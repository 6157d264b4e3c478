#!/usr/bin/env python
"""IPA text -> frame queues -> PCM in HBM: the host producer (speechPlayer_ipaFrames, all threads) + batchSetFramesHost
against the device producer (speechPlayer_ipaFramesDevice) + batchSetFramesDevice, with the FP32 ring render of the same
batch for scale.  Prints one JSON object (and writes it to --out).

  (a) sampleIpa.txt's 8 lines x 4096 at speed 0.6, 150 ms of trailing silence, 22.05 kHz, one text per stream
  (b) config-3 shaped: 65 536 streams of >= 10 s, each a run of consecutive lines (stream s starts at line s mod 8),
      rendered for 10 s like bench.py's config 3

Device times are CUDA events on the producer's stream around the Python call (which includes packing the texts on the
host); the device work alone (uploads, kernels, copies) and its split come from one torch.profiler pass of its own.
Audio-seconds are the timeline samples of the produced queues (sum of max(M+1, max(F,1)+2)) over the sample rate."""
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

SR, SPEED, SILENCE = 22050, 0.6, 150.0


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi query failed: %s" % e
    return q


def workloads(lines, reps_a, streams_b, seconds_b):
    a = dict(texts=lines * reps_a, stream_offsets=None, count=None)
    fb = ipa.frames_for_texts(lines, speed=SPEED, sample_rate=SR, trailing_silence_ms=SILENCE)
    line_s = fb.timeline_samples() / SR
    texts, so = [], [0]
    for s in range(streams_b):
        acc, k = 0.0, s % len(lines)
        while acc < seconds_b:
            texts.append(lines[k])
            acc += line_s[k]
            k = (k + 1) % len(lines)
        so.append(len(texts))
    b = dict(texts=texts, stream_offsets=np.asarray(so, dtype=np.int64), count=int(round(seconds_b * SR)))
    return {"a": a, "b": b}


def run(name, w, torch, steps):
    texts, so = w["texts"], w["stream_offsets"]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    kw = dict(speed=SPEED, sample_rate=SR, trailing_silence_ms=SILENCE)
    res = {"texts": len(texts)}

    def produce():
        return ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)

    db = produce()  # warm-up: module load, scratch growth, allocator
    stream.synchronize()
    ns = db.num_streams
    frames = int(db.frames.shape[0])
    timeline = db.timeline_samples.cpu().numpy()
    count = w["count"] or int(timeline.max())
    audio_s = float(np.minimum(timeline, count).sum()) / SR
    res.update(streams=ns, frames=frames, render_samples_per_stream=count, audio_seconds=audio_s,
               frame_rows_bytes=frames * 376)

    # ---- device producer: events around the call on its stream, and host wall time (the call includes its one sync) ----
    ev_ms, call_s, done_s = [], [], []
    for _ in range(steps):
        del db
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        t0 = time.perf_counter()
        db = produce()
        t1 = time.perf_counter()
        b.record(stream)
        stream.synchronize()
        t2 = time.perf_counter()
        ev_ms.append(a.elapsed_time(b))
        call_s.append(t1 - t0)
        done_s.append(t2 - t0)
    # events bracket the whole Python call: packing the str texts into one UTF-8 blob (host) is inside them
    res["device_producer"] = {"call_event_ms_median": float(np.median(ev_ms)), "call_event_ms": ev_ms,
                              "host_wall_call_ms_median": 1e3 * float(np.median(call_s)),
                              "host_wall_to_rows_written_ms_median": 1e3 * float(np.median(done_s)),
                              "audio_seconds_per_second": audio_s / float(np.median(done_s))}

    # ---- the split: one profiled call ----
    from torch.profiler import ProfilerActivity, profile
    del db
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        db = produce()
        stream.synchronize()
    split = {}
    for e in prof.key_averages():
        if "ipa_" in e.key or "Memcpy" in e.key or "Memset" in e.key:
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            split[e.key[:60]] = round(t / 1e3, 3)  # ms
    res["device_producer"]["profiled_split_ms"] = split
    res["device_producer"]["device_work_ms"] = round(sum(v for k, v in split.items() if not k.startswith("cuda")), 3)

    # ---- FP32 ring render of the same batch ----
    out = torch.empty((ns, (count + 7) // 8 * 8), dtype=torch.int16, device=dev)
    batch = player.Batch(SR, ns, precision=player.PRECISION_FP32, noise=player.NOISE_PHILOX, seed=0xB200)
    render_ms = []
    for i in range(steps + 1):
        batch.set_frames_device(db, cuda_stream=stream)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        batch.synthesize_device(count, out.data_ptr(), out.shape[1], None, stream.cuda_stream)
        b.record(stream)
        stream.synchronize()
        if i:
            render_ms.append(a.elapsed_time(b))
    r = float(np.median(render_ms))
    res["fp32_render"] = {"ms_median": r, "ms": render_ms, "audio_seconds_per_second": audio_s / (r * 1e-3)}
    res["device_producer"]["device_work_share_of_render"] = res["device_producer"]["device_work_ms"] / r
    res["device_producer"]["call_share_of_render"] = res["device_producer"]["call_event_ms_median"] / r

    # ---- text -> PCM in HBM, device route ----
    dev_route = []
    for _ in range(steps):
        del db
        stream.synchronize()
        t0 = time.perf_counter()
        db = produce()
        batch.set_frames_device(db, cuda_stream=stream)
        batch.synthesize_device(count, out.data_ptr(), out.shape[1], None, stream.cuda_stream)
        stream.synchronize()
        dev_route.append(time.perf_counter() - t0)
    pcm_dev = out[:, :count].clone()
    batch.close()
    del db

    # ---- host producer (all threads) + batchSetFramesHost, and the host route to PCM in HBM ----
    t0 = time.perf_counter()
    fb = ipa.frames_for_texts(texts, threads=0, **kw)
    t1 = time.perf_counter()
    if so is not None:
        fb.offsets = fb.offsets[so]
        fb.stream_ids = np.arange(ns, dtype=np.uint64)
    hb = player.Batch(SR, ns, precision=player.PRECISION_FP32, noise=player.NOISE_PHILOX, seed=0xB200)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    hb.set_frames_host(fb)
    t3 = time.perf_counter()
    hb.synthesize_device(count, out.data_ptr(), out.shape[1], None, None)
    torch.cuda.synchronize()
    t4 = time.perf_counter()
    host_route = (t1 - t0) + (t4 - t2)
    same = bool(torch.equal(out[:, :count], pcm_dev))
    hb.close()
    res["host_producer"] = {"producer_ms": 1e3 * (t1 - t0), "set_frames_host_ms": 1e3 * (t3 - t2), "threads": os.cpu_count(),
                            "audio_seconds_per_second": audio_s / (t1 - t0 + t3 - t2)}
    res["text_to_pcm_in_hbm"] = {
        "device_route_ms_median": 1e3 * float(np.median(dev_route)), "host_route_ms": 1e3 * host_route,
        "device_route_audio_seconds_per_second": audio_s / float(np.median(dev_route)),
        "host_route_audio_seconds_per_second": audio_s / host_route, "pcm_identical": same}
    del out
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps-a", type=int, default=4096)
    ap.add_argument("--streams-b", type=int, default=65536)
    ap.add_argument("--seconds-b", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--only", choices=["a", "b"], default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("ipa_device_bench: needs a CUDA device")
    gold = np.load(os.path.join(ROOT, "tests", "golden", "ipa_frames.npz"))
    lines = [str(t) for t in gold["texts"][:8]]
    ws = workloads(lines, args.reps_a, args.streams_b, args.seconds_b)
    result = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "sample_rate": SR, "speed": SPEED,
              "trailing_silence_ms": SILENCE, "workloads": {}}
    for name in ("a", "b"):
        if args.only in (None, name):
            result["workloads"][name] = run(name, ws[name], torch, args.steps)
            print(json.dumps({name: result["workloads"][name]}), flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
