#!/usr/bin/env python
"""IPA text -> PCM in HBM for N whole utterances through three routes:

  (a) host_long     ipa.frames_for_texts (host producer, every CPU thread) + speechPlayer_synthesizeLongBatch, which uploads
                    the queues (player.synthesize_long_batch on the host FrameBatch)
  (b) device_long   ipa.frames_for_texts_device + speechPlayer_synthesizeLongBatchDevice, which reads the queues in place
                    (player.synthesize_long_batch on the DeviceFrameBatch), both on one non-default torch stream
  (c) device_batch  ipa.frames_for_texts_device + player.Batch FP32 set_frames_device + synthesize_device: one thread per
                    stream (the ring scheduler above NVSP_ROUNDS_MIN_STREAMS streams), every stream to its end

Texts: the 8 lines of sampleIpa.txt (tests/golden/ipa_frames.npz) at speed 0.6 with 150 ms of trailing silence, 22.05 kHz;
stream s queues consecutive lines from line s mod 8 on until it holds at least --seconds of audio.  (a) and (b) render the
same queues with the same noise streams (0..N-1) and must give the same PCM, bit for bit: the script checks it.

Every route is warmed up once, then timed --reps times by the host clock from the list of texts to the PCM in HBM; each
run ends in a device synchronise.  The median is reported.  (b) is also split into its preparation -- the offsets copied
back, the ticks kernel, the ticks copied back: timed alone as a size query (player.long_batch_size) -- and its render (the
call's render_ms: CUDA events around the groups' launch sequences).  The card's name and power limit are read in the same run.

    python tools/long_batch_text_bench.py [--streams 64,512,1024,2048,4096] [--seconds 10] [--reps 5]
                                          [--out profiles/r05_long_batch_text_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nvspeechplayer_b200 import ipa, player  # noqa: E402

SR, SPEED, SILENCE, SEED = 22050, 0.6, 150.0, 0xB200


def card(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60).stdout.strip().split(",")
        info.update(smi_name=q[0].strip(), power_limit_w=float(q[1]), sm_max_mhz=float(q[2]))
    except Exception as e:  # noqa: BLE001 -- the numbers are still reported, the power limit marked as unknown
        info.update(power_limit_w=None, nvidia_smi=repr(e))
    return info


def texts_for(lines, line_s, n, seconds):
    texts, so = [], [0]
    for s in range(n):
        acc, k = 0.0, s % len(lines)
        while acc < seconds:
            texts.append(lines[k])
            acc += line_s[k]
            k = (k + 1) % len(lines)
        so.append(len(texts))
    return texts, np.asarray(so, dtype=np.int64)


def median_ms(fn, reps):
    fn()  # warm-up: module loads, scratch pools, the allocator
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), ts


def run(torch, lines, line_s, n, seconds, reps):
    texts, so = texts_for(lines, line_s, n, seconds)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    kw = dict(speed=SPEED, sample_rate=SR, trailing_silence_ms=SILENCE)
    db = ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)
    total, off = player.long_batch_size(db, cuda_stream=stream)
    law = np.diff(off)
    count = int(law.max())
    audio_s = total / SR
    row = {"streams": n, "texts": len(texts), "frames": int(db.frames.shape[0]), "samples": int(total), "audio_seconds": audio_s,
           "stream_seconds_min": float(law.min()) / SR, "stream_seconds_max": count / SR}
    del db
    out_a = torch.empty(total + 64, dtype=torch.int16, device=dev)
    out_b = torch.empty(total + 64, dtype=torch.int16, device=dev)
    rows_c = torch.empty((n, count), dtype=torch.int16, device=dev)
    torch.cuda.synchronize()

    def host_long():
        fb = ipa.frames_for_texts(texts, threads=0, **kw)
        fb.offsets = fb.offsets[so]
        fb.stream_ids = np.arange(n, dtype=np.uint64)
        player.synthesize_long_batch(fb, seed=SEED, device_out=out_a.data_ptr())  # ends in a device synchronise

    split = {"render_ms": [], "call_ms": []}

    def device_long():
        db = ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)
        t0 = time.perf_counter()
        _, _, _, render_ms, _ = player.synthesize_long_batch(db, seed=SEED, device_out=out_b.data_ptr(), cuda_stream=stream)
        split["call_ms"].append(1e3 * (time.perf_counter() - t0))
        split["render_ms"].append(render_ms)

    batch = player.Batch(SR, n, precision=player.PRECISION_FP32, noise=player.NOISE_PHILOX, seed=SEED)

    def device_batch():
        db = ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)
        batch.set_frames_device(db, cuda_stream=stream)
        batch.synthesize_device(count, rows_c.data_ptr(), count, None, stream.cuda_stream)
        stream.synchronize()

    row["host_long_ms"], row["host_long_runs_ms"] = median_ms(host_long, reps)
    row["device_long_ms"], row["device_long_runs_ms"] = median_ms(device_long, reps)
    row["device_batch_ms"], row["device_batch_runs_ms"] = median_ms(device_batch, reps)
    batch.close()
    row["pcm_a_equals_b"] = bool(torch.equal(out_a[:total], out_b[:total]))

    # (b) split: the preparation alone (a size query on the produced queues) and the render of the calls timed above
    db = ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)
    stream.synchronize()
    row["device_long_prepare_ms"], _ = median_ms(lambda: player.long_batch_size(db, cuda_stream=stream), reps)
    row["device_long_render_ms"] = float(np.median(split["render_ms"][1:]))
    row["device_long_call_ms"] = float(np.median(split["call_ms"][1:]))
    for k in ("host_long", "device_long", "device_batch"):
        row[k + "_audio_s_per_s"] = audio_s / (row[k + "_ms"] / 1e3)
    row["device_long_saves_vs_host_long_ms"] = row["host_long_ms"] - row["device_long_ms"]
    row["device_batch_over_device_long"] = row["device_batch_ms"] / row["device_long_ms"]
    del db, out_a, out_b, rows_c
    torch.cuda.empty_cache()
    return row


def crossover(rows):
    """where the faster of (b) and (c) changes, between two measured batch sizes"""
    win = [(r["streams"], "device_long" if r["device_long_ms"] <= r["device_batch_ms"] else "device_batch") for r in rows]
    for (n0, w0), (n1, w1) in zip(win, win[1:]):
        if w0 != w1:
            return {"between_streams": [n0, n1], "below": w0, "above": w1, "winners": win}
    return {"between_streams": None, "winners": win, "note": "the same route is faster at every measured size"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="64,512,1024,2048,4096")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_long_batch_text_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("long_batch_text_bench: no CUDA device (the measurement has no CPU fallback)")
    info = card(torch)
    print("card: %s, power limit %s W" % (info["name"], info["power_limit_w"]), flush=True)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "ipa_frames.npz"))
    lines = [str(t) for t in gold["texts"][:8]]
    line_s = ipa.frames_for_texts(lines, **dict(speed=SPEED, sample_rate=SR, trailing_silence_ms=SILENCE)).timeline_samples() / SR
    rows = []
    for n in [int(x) for x in a.streams.split(",")]:
        rows.append(run(torch, lines, line_s, n, a.seconds, a.reps))
        print(json.dumps({k: (round(v, 3) if isinstance(v, float) else v) for k, v in rows[-1].items() if not k.endswith("runs_ms")}),
              flush=True)
    res = {"tool": "tools/long_batch_text_bench.py", "card": info, "sample_rate": SR, "speed": SPEED, "trailing_silence_ms": SILENCE,
           "seconds_per_stream": a.seconds, "reps": a.reps, "cpu_threads": os.cpu_count(),
           "timing": "host clock from the texts to the PCM in HBM, ending in a device synchronise; median of reps after one warm-up",
           "rows": rows, "long_vs_batch_crossover": crossover(rows)}
    print(json.dumps(res["long_vs_batch_crossover"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
