"""Batched long-utterance path against today's routes for a batch of whole, pre-queued utterances.

N streams of workloads.random_frames, 10 s each at 22.05 kHz, through
  long_batch   speechPlayer_synthesizeLongBatch (all streams' chunks in one launch sequence), at the default chunk length
               and at every chunk length from 1024 down to 64 (the sweep the default's fill threshold is read from);
  batch_f32    player.Batch FP32 with synthesize_device: one thread per stream (one launch below NVSP_ROUNDS_MIN_STREAMS,
               the ring scheduler above);
  long_solo    N consecutive speechPlayer_synthesizeLong calls (N <= 512).
Every route is warmed up, then timed with CUDA events around `--reps` repetitions, device output (no copy to the host).
Reports audio-seconds per second of each route with the card name and power limit, and writes JSON under profiles/.

    python tools/long_batch_bench.py [--streams 1,8,64,512,4096] [--seconds 10] [--reps 3] [--out profiles/long_batch_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from nvspeechplayer_b200 import player, workloads  # noqa: E402

SR = 22050
SEED = 0xB200


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0])
        info["sm_max_mhz"] = float(q[1])
    except Exception as e:  # the number is still reported, marked as unknown
        info["power_limit_w"] = None
        info["nvidia_smi"] = repr(e)
    return info


def timed(fn, reps):
    fn()  # warm-up: module loads, scratch pools
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="1,8,64,512,4096")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--solo-max", type=int, default=512)
    ap.add_argument("--chunks", default="1024,512,256,128,64")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_batch_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_batch_bench: no CUDA device (the measurement has no CPU fallback)")
    info = card()
    print("card: %s, power limit %s W" % (info["name"], info["power_limit_w"]), flush=True)
    rows = []
    for n in [int(x) for x in a.streams.split(",")]:
        t0 = time.time()
        fb = workloads.random_frames(n, a.seconds, SR, first_stream=1)
        law = fb.timeline_samples()
        samples = int(law.sum())
        audio_s = samples / SR
        d_out = torch.empty(samples + 64, dtype=torch.int16, device="cuda")
        row = {"streams": n, "seconds_per_stream": a.seconds, "samples": samples, "gen_s": round(time.time() - t0, 1)}

        def long_batch(chunk):
            return lambda: player.synthesize_long_batch(fb, seed=SEED, chunk_ticks=chunk, device_out=d_out.data_ptr())
        row["long_batch_default_ms"] = timed(long_batch(0), a.reps)
        for c in [int(x) for x in a.chunks.split(",")]:
            row["long_batch_chunk%d_ms" % c] = timed(long_batch(c), a.reps)
        # kernel (a): every stream whole (count = the longest queue), rows of the longest length
        count = int(law.max())
        d_rows = torch.empty((n, count), dtype=torch.int16, device="cuda")
        b = player.Batch(SR, n, precision=player.PRECISION_FP32, seed=SEED, stream_ids=fb.stream_ids)

        def batch_f32():
            b.set_frames_host(fb)
            b.synthesize_device(count, d_rows.data_ptr(), count)
        row["batch_f32_ms"] = timed(batch_f32, a.reps)
        b.close()
        del d_rows
        if n <= a.solo_max:
            def solo():
                for s in range(n):
                    fr, m, f, nul, _ = fb.stream(s)
                    player.synthesize_long(SR, fr, m, f, nul, seed=SEED, stream_id=int(fb.stream_ids[s]), device_out=d_out.data_ptr())
            row["long_solo_ms"] = timed(solo, max(1, a.reps if n <= 64 else 1))
        for k in list(row):
            if k.endswith("_ms"):
                row[k] = round(row[k], 3)
                row[k[:-3] + "_audio_s_per_s"] = round(audio_s / (row[k] / 1e3), 1)
        row["long_batch_speedup_vs_batch_f32"] = round(row["batch_f32_ms"] / row["long_batch_default_ms"], 2)
        if "long_solo_ms" in row:
            row["long_batch_speedup_vs_long_solo"] = round(row["long_solo_ms"] / row["long_batch_default_ms"], 2)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del d_out
        torch.cuda.empty_cache()
    res = {"tool": "tools/long_batch_bench.py", "card": info, "sample_rate": SR, "reps": a.reps,
           "timing": "CUDA events around reps calls after one warm-up call; device output; includes host-side setup of each call",
           "rows": rows}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
