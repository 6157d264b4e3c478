#!/usr/bin/env python
"""Bitwise A/B of the two time-parallel renderers through the C-ABI: one sha256 per output, one JSON line each.  Run it
once per build (NVSP_LIB selects the library) and compare the lines; every hash must match.

  kernel (b), speechPlayer_synthesizeLong: every pre-queued scenario of tests/scenarios.py at chunk length 64, and the
      whole-sample pitch-period streams (150 / 225 Hz at 22 050 Hz) at chunk lengths 64 and 1024
  kernel (b), batched: a ragged 40-stream batch (empty queues, a NULL-only queue, a one-request queue, per-stream caps, one
      stream on the serial phase fallback) by the host and the device route, at chunk lengths 64 and 1024: samples,
      outOffsets and serialPhase
  pull path (SPEECHPLAYER_PRECISION_STREAM): one player through every scenario script, purges included"""
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nvspeechplayer_b200 import player, workloads  # noqa: E402
from tests import scenarios  # noqa: E402

SR = 22050


def emit(name, *arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    print(json.dumps({"output": name, "sha256": h.hexdigest(), "n": int(sum(np.size(a) for a in arrays))}), flush=True)


def whole_period_queue():
    fr = np.zeros((2, 47))
    for j, hz in enumerate((150.0, 225.0)):
        fr[j, workloads.P["voicePitch"]] = fr[j, workloads.P["endVoicePitch"]] = hz
        for p in ("voiceAmplitude", "preFormantGain", "outputGain"):
            fr[j, workloads.P[p]] = 1.0
        workloads.set_frame(fr[j], "a")
    return fr, np.array([33075, 33075], np.uint32), np.array([441, 441], np.uint32), np.zeros(2, np.uint8), np.zeros(2, np.int32)


def ragged_batch():
    rng = np.random.default_rng(4711)
    qs = [workloads.random_stream(7000 + k, float(s), SR) for k, s in enumerate(np.exp(rng.uniform(np.log(0.02), np.log(25.0), 35)))]
    empty = (np.zeros((0, 47)), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint8), np.zeros(0, np.int32))
    null_only = (np.zeros((4, 47)), np.array([300, 0, 9, 2000], np.uint32), np.array([60, 0, 40, 7], np.uint32), np.ones(4, np.uint8),
                 np.zeros(4, np.int32))
    fr = workloads.random_stream(7099, 0.05, SR)[0]
    tiny = (fr[:1].copy(), np.array([12], np.uint32), np.array([3], np.uint32), np.zeros(1, np.uint8), np.zeros(1, np.int32))
    for k, q in ((0, empty), (8, null_only), (15, tiny), (21, empty), (30, whole_period_queue())):
        qs.insert(k, q)
    fb = workloads._concat(SR, qs, np.arange(len(qs), dtype=np.uint64) * 104729 + 3)
    caps = fb.timeline_samples().astype(np.uint64)
    for k in (2, 9, 17):
        caps[k] = max(int(caps[k]) // 4, 1)
    caps[26] = 0
    return fb, caps


def to_device(fb):
    import torch
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return workloads.FrameBatch(sample_rate=fb.sample_rate, offsets=t(fb.offsets), frames=t(fb.frames), min_dur=t(fb.min_dur.view(np.int32)),
                                fade_dur=t(fb.fade_dur.view(np.int32)), is_null=t(fb.is_null), user_index=None, stream_ids=fb.stream_ids)


class PullAdapter:
    def __init__(self, sr):
        self.p = player.SpeechPlayer(sr, precision=player.PRECISION_STREAM, noise=player.NOISE_PHILOX, seed=scenarios.SEED,
                                     streamId=scenarios.STREAM)

    def queue_frame(self, fr, m, f, ux, purge):
        self.p.queue_frame(fr, m, f, ux, purge)

    def synthesize(self, n):
        return self.p.synthesize_np(n)

    def last_index(self):
        return self.p.last_index()

    def close(self):
        self.p.close()


def main():
    print(json.dumps({"library": player.LIB_PATH}), flush=True)
    for name, sc in sorted(scenarios.all_scenarios().items()):
        ops = sc["ops"]
        first_s = next(i for i, o in enumerate(ops) if o[0] == "s")
        if all(o[0] == "q" and not o[5] for o in ops[:first_s]) and all(o[0] == "s" for o in ops[first_s:]):
            qs = [o for o in ops if o[0] == "q"]
            fr = np.stack([np.zeros(47) if o[1] is None else np.asarray(o[1], dtype=np.float64) for o in qs])
            got, _, _ = player.synthesize_long(sc["sr"], fr, [o[2] for o in qs], [o[3] for o in qs], [o[1] is None for o in qs],
                                               seed=scenarios.SEED, stream_id=scenarios.STREAM, chunk_ticks=64,
                                               max_samples=sum(o[1] for o in ops if o[0] == "s"))
            emit("long/" + name, got)
        pcm, counts, idx = scenarios.run_script(PullAdapter, sc)
        emit("pull/" + name, pcm, np.array(counts), np.array(idx))
    fr, m, f, _, _ = whole_period_queue()
    for chunk in (64, 1024):
        for k, sl in (("both", slice(0, 2)), ("150", slice(0, 1)), ("225", slice(1, 2))):
            emit("long/whole_period_%s/chunk%d" % (k, chunk), player.synthesize_long(SR, fr[sl], m[sl], f[sl], None, seed=11, stream_id=3,
                                                                                      chunk_ticks=chunk)[0])
    fb, caps = ragged_batch()
    dfb = to_device(fb)
    for chunk in (64, 1024):
        for route, q in (("host", fb), ("device", dfb)):
            pcm, off, serial, _, _ = player.synthesize_long_batch(q, seed=0xB200, chunk_ticks=chunk, max_samples=caps)
            emit("long_batch/%s/chunk%d" % (route, chunk), pcm, off, serial)
            print(json.dumps({"output": "long_batch/%s/chunk%d" % (route, chunk), "serial_streams": np.flatnonzero(serial).tolist()}), flush=True)


if __name__ == "__main__":
    main()
