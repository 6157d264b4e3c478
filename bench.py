#!/usr/bin/env python
"""bench.py -- the headline benchmark of the B200-native Klatt engine.

Metric (BASELINE.json): audio-seconds synthesized per wall-second, batched streams, and the fraction of the FP32
CUDA-core FMA roofline from counted flops W(phi) = 128 + 270*phi per sample (SURVEY.md section 8d).
Workload: BASELINE config 3 -- synthetic random-frame batch, 65 536 streams x 10 s at 22 050 Hz PER GPU (weak
scaling: rank r renders stream ids [r*65536, (r+1)*65536), no data-path collective, streams are independent).

A "step" is one pass of the hot path over one batch: reset every stream to its initial state, then frame manager
+ generator for streams x seconds x rate ticks.
  value    : inputs (frames, durations) already resident in HBM, output left in HBM (speechPlayer_batch*Device)
  e2e      : same step through the host-buffer C-ABI: frames H2D from pinned memory, int16 D2H into pinned memory
  roofline : counted flops / CUDA-event kernel time, against (a) FP32 FMA peak measured on this GPU by an FFMA
             loop and (b) SMs x 128 x 2 x max clock; plus the output stream's share of the measured HBM peak
  cpu_baseline : the reference C++ (oracle/_ref) on the host cores, one process per core, bounded sample

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--streams S] [--seconds T] [--dump-outputs DIR]
N>1 is launched with torch.distributed.run (one rank per GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: NCCL's version banner (NCCL_DEBUG=VERSION in some images) goes nowhere near it
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

W_HOLD, W_FADE_EXTRA = 128.0, 270.0  # flops per sample: hold tick, extra on a fade tick (SURVEY.md 8d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--streams", type=int, default=65536, help="streams per GPU")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--sample-rate", type=int, default=22050)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--seed", type=lambda s: int(s, 0), default=0xB200)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-slice-seconds", type=float, default=2.0,
                    help="the e2e leg pulls the audio in slices of this length into ONE pinned host buffer (a streaming "
                         "consumer): 65536 x 2 s = 5.8 GB pinned per rank instead of 28.9 GB, so 8 ranks fit the host")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run oracle check of random output rows")
    ap.add_argument("--parity-streams", type=int, default=16)
    ap.add_argument("--cpu-streams-per-core", type=int, default=16)
    ap.add_argument("--workload", default="batch", choices=["batch", "vowel", "midi", "long", "pull"],
                    help="batch: BASELINE config 3 (default, the headline); vowel: config 2, vowel-chart pairs x --voices "
                         "voices at 16 kHz (one fresh player per (voice, pair)); midi: config 5, midi-sing style streams "
                         "(--streams per GPU x 5 s); long: config 4, ONE stream of --long-seconds at --long-rate through "
                         "the time-parallel kernel")
    ap.add_argument("--voices", type=int, default=1024, help="--workload vowel: voices per GPU (1369 pairs each)")
    ap.add_argument("--pull-samples", type=int, default=8192, help="--workload pull: samples per speechPlayer_synthesize call")
    ap.add_argument("--pull-players", type=int, default=148, help="--workload pull: players of the batched-pull leg")
    ap.add_argument("--long-seconds", type=float, default=3600.0)
    ap.add_argument("--long-rate", type=int, default=44100)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy in float32 / "
                         "float64, at most 64 MB in all: a fixed, seeded sample where the output is larger, so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm renders in worker processes and keeps no outputs")
    return args


DUMP_BYTES = 64 * 10**6


def dump_outputs(path, arrays):
    """Write {name: float32 / float64 array} as path/<name>.npy; together they stay within DUMP_BYTES."""
    import numpy as np
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, "--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_BYTES)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def sample_pcm(d_out, count, written, seed, points=1 << 20):
    """What a caller receives -- int16 rows on the device, row i valid up to written[i] -- as float32 / float64 arrays:
    `written` of every row; `points` at a seeded sample of positions over all rows (`points_index` = row * count + sample);
    whole `rows` of a seeded sample of rows (`rows_index`), as many as the rest of DUMP_BYTES holds.  Samples past a row's
    written count are not output and read as 0."""
    import numpy as np
    import torch
    rows_n, stride = d_out.shape
    rng = np.random.default_rng(seed)
    flat = np.sort(rng.choice(rows_n * count, size=min(points, rows_n * count), replace=False))
    r, c = flat // count, flat % count
    pts = d_out.view(-1)[torch.from_numpy(r * stride + c).to(d_out.device)].cpu().numpy().astype(np.float32)
    pts[c >= written[r]] = 0
    left = DUMP_BYTES - rows_n * 8 - flat.size * 12 - (1 << 20)
    sel = np.sort(rng.choice(rows_n, size=max(0, min(rows_n, left // (count * 4 + 8))), replace=False))
    rows = d_out[torch.from_numpy(sel).to(d_out.device), :count].cpu().numpy().astype(np.float32)
    rows[np.arange(count)[None, :] >= written[sel][:, None]] = 0
    return {"written": written.astype(np.float64), "points": pts, "points_index": flat.astype(np.float64),
            "rows": rows, "rows_index": sel.astype(np.float64)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); power.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(dev_index):
    """Pin this rank's threads to the CPUs next to its GPU (NVML's ideal affinity) BEFORE the pinned host buffers are
    allocated: first-touch puts them on that NUMA node, so the eight ranks of a box do not copy 231 GB per step through
    whatever socket the scheduler happened to start them on.  (On the pool this was measured on, every GPU reports the
    same single node and the binding changes nothing: the host side caps the eight concurrent D2H streams at ~88 GB/s in
    aggregate, 8-GPU e2e = 2.0x the 1-GPU figure, while the HBM-resident value scales 8.0x.)"""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(dev_index)
        try:
            bus = "%08x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(dev_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (oracle/_ref when it
    was compiled, else the plain-C port).  Rank 0 alone runs it."""
    if rank != 0:
        return
    from oracle import cpu_bench
    runs = []
    for i in range(args.warmup + args.steps):
        r = cpu_bench.run(streams_per_core=max(args.cpu_streams_per_core // 4, 2), seconds=args.seconds,
                          sample_rate=args.sample_rate, seed=args.seed, first_stream=0)
        if i >= args.warmup:
            runs.append(r)
    value = sum(r["value"] for r in runs) / len(runs)
    ms = 1e3 * sum(r["synth_seconds_slowest_core"] for r in runs) / len(runs)
    last = runs[-1]
    line = {
        "impl": "reference", "metric": "audio-seconds synthesized/sec (batched streams)", "value": value,
        "unit": "audio-seconds/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "config3 random-frame batch, bounded sample: " + last["sample"],
                   "sample_rate": args.sample_rate, "seconds_per_stream": args.seconds},
        "cpu_baseline": {"value": value, "unit": "audio-seconds/s", "cores": last["cores"], "kind": last["kind"],
                         "sample": last["sample"], "ns_per_sample_core": last["ns_per_sample_core"]},
        "e2e": {"value": value, "unit": "audio-seconds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def long_arm(args, rank, world, local_rank):
    """BASELINE config 4: a single long stream (config-3 frame generator at 44.1 kHz) through kernel (b).  The path does
    not shard (one stream): N > 1 runs N independent replicas, one per GPU ("replicas only")."""
    import numpy as np
    import torch
    from nvspeechplayer_b200 import player, workloads
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")  # control plane only (barrier, max over ranks): no NCCL anywhere in this path
    sr, secs = args.long_rate, args.long_seconds
    fr, m, f, nul, ux = workloads.random_stream(4_000_000 + rank, secs, sr, seed=args.seed)
    n = int(round(secs * sr))
    fb = workloads._concat(sr, [(fr, m, f, nul, ux)], [4_000_000 + rank])
    phi = fb.fade_fraction(n)
    flops_per_sample = W_HOLD + W_FADE_EXTRA * phi
    d_out = torch.empty(n + 64, dtype=torch.int16, device=dev)
    lib = player.load_library()
    lib.speechPlayer_debugFp32PeakTflops.restype = __import__("ctypes").c_double
    peak_tf = float(lib.speechPlayer_debugFp32PeakTflops())
    sampler = ClockSampler(local_rank)
    times, launches = [], 0
    for i in range(max(args.warmup, 3) + args.steps):
        if i == max(args.warmup, 3) and rank == 0:
            sampler.start()
        torch.cuda.synchronize()
        got, ms, launches = player.synthesize_long(sr, fr, m, f, nul, seed=args.seed, stream_id=4_000_000 + rank, max_samples=n,
                                                   device_out=d_out.data_ptr())
        assert got == n, (got, n)
        if i >= max(args.warmup, 3):
            times.append(ms)
    clocks = sampler.stop() if rank == 0 else None
    ms = sum(times) / len(times)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sample_pcm(d_out[None, :], n, np.array([got]), args.seed))
    # e2e: host frames in, host int16 out, wall clock around the C-ABI call
    h_out = np.zeros(n, dtype=np.int16)
    t0 = time.perf_counter()
    out, _, _ = player.synthesize_long(sr, fr, m, f, nul, seed=args.seed, stream_id=4_000_000 + rank, max_samples=n, out=h_out)
    e2e_s = time.perf_counter() - t0
    same = bool(np.array_equal(out[:100000], d_out[:100000].cpu().numpy()))
    if world > 1:
        t = torch.tensor([ms, e2e_s], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle
            ref = oracle.RefLib(philox=False) if oracle.have_ref() else None
            cn = int(30.0 * sr)  # bounded sample: the first 30 s of the same stream, one core (a stream is serial on a CPU)
            t0 = time.perf_counter()
            if ref is not None:
                got_cpu = ref.render(sr, fr, m, f, nul, max_samples=cn, seed=1)
            else:
                got_cpu = oracle.PortLib().render(sr, fr, m, f, nul, max_samples=cn, noise=("libc",))
            dt = time.perf_counter() - t0
            cpu = {"value": len(got_cpu) / sr / dt, "unit": "audio-seconds/s", "cores": 1, "kind": "reference" if ref else "port",
                   "sample": "first 30 s of the same stream incl. queueing its frames, one core"}
        par = None
        if not args.no_parity:
            # the WHOLE stream on the oracle with the same Philox noise (one core, ~25 s for an hour at 44.1 kHz), compared over
            # its final 10 s: drift of any scanned quantity over all chunks would show there
            from oracle import oracle
            from tests import parity as parity_mod
            if not oracle.have_port():
                oracle.build(quiet=True)
            t0 = time.perf_counter()
            want = oracle.PortLib().render(sr, fr, m, f, nul, ux, max_samples=n, noise=("philox", args.seed, 4_000_000 + rank))
            t_or = time.perf_counter() - t0
            tail = min(n, 10 * sr)
            got_tail = d_out[n - tail:n].cpu().numpy()
            w1_, ex_, snr_, mx_ = parity_mod.metrics(got_tail, want[n - tail:n])
            w1_all = parity_mod.metrics(d_out[:n].cpu().numpy(), want)[0] if n <= 200_000_000 else None
            lib.speechPlayer_debugLongSerialFallbacks.restype = __import__("ctypes").c_ulonglong
            par = {"samples_checked": int(tail), "of": "the final 10 s of the stream", "within_1lsb": w1_, "snr_db": snr_,
                   "max_abs_diff": mx_, "within_1lsb_whole_stream": w1_all, "oracle_seconds": round(t_or, 1),
                   "oracle": "oracle/klatt_oracle.c (port) with the same Philox noise",
                   "serial_phase_fallbacks": int(lib.speechPlayer_debugLongSerialFallbacks())}
        achieved = n * flops_per_sample / (ms * 1e-3) / 1e12
        line = {"metric": "audio-seconds synthesized/sec (single long stream)", "value": world * secs / (ms * 1e-3),
                "unit": "audio-seconds/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
                "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "config4: single %.0f s stream @ %d Hz, random frames, time-parallel kernel (b)" % (secs, sr),
                           "frames": int(len(m)), "fade_fraction_phi": round(phi, 4), "flops_per_sample_W": round(flops_per_sample, 1),
                           "l2": "no flush needed: the stage signals (5 x %.2f GB) exceed the 126 MB L2" % (n * 4 / 1e9)},
                "roofline": {"bound": "fp32_fma", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                             "traffic": None, "kernel": "klatt_long_* (27 launches)",
                             "note": "algorithmic flops of the SERIAL path; the scan formulation executes about 3x of them"},
                "cpu_baseline": cpu, "parity": par,
                "e2e": {"value": world * secs / e2e_s, "unit": "audio-seconds/s", "h2d_bytes_per_step": int(fr.nbytes + m.nbytes + f.nbytes + nul.nbytes),
                        "d2h_bytes_per_step": int(n * 2), "matches_device_path": same},
                "gpu_launches": int(launches) * args.steps, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def pull_arm(args, rank, world, local_rank):
    """SURVEY 8f rank 3: ONE player driven like the NVDA audio thread drives the reference -- speechPlayer_synthesize pulls
    of --pull-samples (8192) through the five-symbol C-ABI with host buffers -- on the low-latency path
    (SPEECHPLAYER_PRECISION_STREAM: host frame manager + one time-parallel block launch per pull).  A step is one pull;
    the number that matters is its latency.  One stream does not shard: N > 1 runs N replicas ("replicas only")."""
    import numpy as np
    import torch
    from nvspeechplayer_b200 import player, workloads
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    sr, pull = args.sample_rate, args.pull_samples
    warm, steps = max(args.warmup, 3), args.steps
    secs = (warm + steps + 2) * pull / sr
    fr, m, f, nul, ux = workloads.random_stream(5_000_000 + rank, secs, sr, seed=args.seed)
    fb = workloads._concat(sr, [(fr, m, f, nul, ux)], [5_000_000 + rank])
    phi = fb.fade_fraction(int(secs * sr))
    flops_per_sample = W_HOLD + W_FADE_EXTRA * phi
    lib = player.load_library()
    lib.speechPlayer_debugFp32PeakTflops.restype = __import__("ctypes").c_double
    peak_tf = float(lib.speechPlayer_debugFp32PeakTflops())

    def timed_pulls(make):
        p = make()
        p.queue_frames(fr, m, f, ux, nul) if hasattr(p, "queue_frames") else [
            p.queue_frame(None if nul[j] else fr[j], int(m[j]), int(f[j]), int(ux[j])) for j in range(len(m))]
        syn = p.synthesize_np if hasattr(p, "synthesize_np") else p.synthesize
        ts = []
        for i in range(warm + steps):
            t0 = time.perf_counter()
            c = syn(pull)
            dt = time.perf_counter() - t0
            assert len(c) == pull
            if i >= warm:
                ts.append(dt)
        p.close()
        return np.array(ts), c

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    res, last = {}, {}
    for name, prec in (("stream", player.PRECISION_STREAM), ("fp32_serial", player.PRECISION_FP32)):
        res[name], last[name] = timed_pulls(lambda: player.SpeechPlayer(sr, precision=prec, noise=player.NOISE_PHILOX,
                                                                        seed=args.seed, streamId=5_000_000 + rank))
    # many interactive players in one launch (speechPlayer_synthesizeBatch over stream handles: one block per player)
    nb = args.pull_players
    bsecs = (warm + steps + 2) * pull / sr
    bstreams = [workloads.random_stream(6_000_000 + rank * nb + k, bsecs, sr, seed=args.seed) for k in range(nb)]
    bps = [player.SpeechPlayer(sr, precision=player.PRECISION_STREAM, noise=player.NOISE_PHILOX, seed=args.seed,
                               streamId=6_000_000 + rank * nb + k) for k in range(nb)]
    for p_, (fr_, m_, f_, nul_, ux_) in zip(bps, bstreams):
        p_.queue_frames(fr_, m_, f_, ux_, nul_)
    bts = []
    bh, bout, bw = player.batch_handles(bps), np.zeros((nb, pull), dtype=np.int16), np.zeros(nb, dtype=np.uint32)
    for i in range(warm + steps):
        t0 = time.perf_counter()
        bout, bw = player.synthesize_batch(bps, pull, out=bout, written=bw, handles=bh)  # (a caller's loop reuses its buffers)
        dt = time.perf_counter() - t0
        assert (bw == pull).all()
        if i >= warm:
            bts.append(dt)
    for p_ in bps:
        p_.close()
    bts = np.array(bts)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pull": last["stream"].astype(np.float32), "pull_fp32_serial": last["fp32_serial"].astype(np.float32),
                                         "batch": bout.astype(np.float32), "batch_written": bw.astype(np.float64)})
    ts = res["stream"]
    total_s = float(ts.sum())
    if world > 1:
        t = torch.tensor([total_s], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_s = float(t[0])
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle
            if oracle.have_ref():
                ref = oracle.RefLib(philox=False)
                rts, _ = timed_pulls(lambda: ref.player(sr))
                kind = "reference"
            else:
                port = oracle.PortLib()
                rts, _ = timed_pulls(lambda: port.player(sr))
                kind = "port"
            cpu = {"value": pull / sr / float(np.median(rts)), "unit": "audio-seconds/s", "cores": 1, "kind": kind,
                   "sample": "the same %d pulls of %d samples on one player, one core" % (steps, pull),
                   "ms_per_pull_median": float(np.median(rts)) * 1e3, "ms_per_pull_p95": float(np.percentile(rts, 95)) * 1e3}
        value = world * steps * pull / sr / total_s
        achieved = steps * pull * flops_per_sample / float(ts.sum()) / 1e12
        e2e = {"value": value, "unit": "audio-seconds/s", "h2d_bytes_per_step": int(fr.nbytes + m.nbytes + f.nbytes) // steps,
               "d2h_bytes_per_step": pull * 2, "note": "the path is host-to-host by construction: value IS the end-to-end number"}
        line = {"metric": "audio-seconds synthesized/sec (one handle, %d-sample pulls)" % pull, "value": value,
                "unit": "audio-seconds/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": total_s / steps * 1e3,
                "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "pull: one player, random frames @ %d Hz, speechPlayer_synthesize(%d) per step through the "
                                       "five-symbol C-ABI, SPEECHPLAYER_PRECISION_STREAM" % (sr, pull),
                           "fade_fraction_phi": round(phi, 4), "flops_per_sample_W": round(flops_per_sample, 1),
                           "l2": "not applicable: one block, working set in shared memory"},
                "latency_ms": {"median": float(np.median(ts)) * 1e3, "p95": float(np.percentile(ts, 95)) * 1e3, "max": float(ts.max()) * 1e3,
                               "fp32_serial_kernel_median": float(np.median(res["fp32_serial"])) * 1e3},
                "batch_of_players": {"players": nb, "samples_per_call": pull, "calls": steps, "ms_per_call_median": float(np.median(bts)) * 1e3,
                                     "audio_seconds_per_s": nb * pull / sr / float(np.median(bts)),
                                     "note": "speechPlayer_synthesizeBatch over %d stream handles: one launch, one block per player" % nb},
                "roofline": {"bound": "latency", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                             "traffic": None, "kernel": "klatt_pull_kernel (1 block of 512 threads per pull)",
                             "note": "one SM of 148 and a serial FP64 phase recurrence: the bound is dependent-issue latency, "
                                     "not a throughput roof; per-phase cycles: NVSP_PULL_DEBUG=1"},
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": steps, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.workload == "pull":
        pull_arm(args, rank, world, local_rank)
        return
    if args.workload == "long":
        long_arm(args, rank, world, local_rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from nvspeechplayer_b200 import player, sharding, workloads

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # The data plane has no collective at all (streams are independent: each rank renders its own stream ids into its own
        # buffers); the control plane -- the barriers around the timed region and the max over ranks -- runs over gloo on the
        # host, so no NCCL communicator is ever created (BASELINE north star: "no NCCL").
        dist.init_process_group("gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sr, S, secs = args.sample_rate, args.streams, args.seconds
    if args.workload == "vowel":    # config 2: 16 kHz (the NVDA rate), 13 926 ticks per (voice, pair) stream
        sr, secs = 16000, 13926 / 16000.0
        S = args.voices * 1369
    elif args.workload == "midi":   # config 5: 5 s per stream; 2^20 streams over 8 GPUs = 131 072 per GPU
        secs = 5.0 if args.seconds == 10.0 else args.seconds
        S = 131072 if args.streams == 65536 else args.streams
    count = int(round(secs * sr))
    prec = player.PRECISION_FP32 if args.precision == "fp32" else player.PRECISION_FP64

    def make_workload(n, first):
        if args.workload == "vowel":
            return workloads.vowel_chart(max(n // 1369, 1), sr, seed=args.seed, first_stream=first)
        if args.workload == "midi":
            return workloads.midi_sing(n, secs, sr, seed=args.seed, first_stream=first)
        return workloads.random_frames(n, secs, sr, seed=args.seed, first_stream=first)

    workload_name = {"batch": "config3: synthetic random-frame batch", "vowel": "config2: vowel-chart pairs x voices (fresh player per pair)",
                     "midi": "config5: midi-sing style pitch-sweep streams"}[args.workload]

    # ---- CPU baseline first (spawns processes; keep it away from the timed GPU region) ----
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import cpu_bench
        cpu = cpu_bench.run(streams_per_core=args.cpu_streams_per_core, seconds=secs, sample_rate=sr, seed=args.seed)

    cpus_bound = bind_to_gpu_numa_node(local_rank) if world > 1 else None  # after the CPU baseline: its workers inherit affinity

    # ---- workload: this rank's shard of config 3 ----
    t_gen = time.time()
    first_stream, _ = sharding.weak_shard(S, rank)  # weak scaling: rank r renders stream ids [r*S, (r+1)*S), no collective
    fb = make_workload(S, first_stream)
    phi = fb.fade_fraction(count) if S <= 4096 else make_workload(1369 if args.workload == "vowel" else 1024,
                                                                  first_stream).fade_fraction(count)
    t_gen = time.time() - t_gen
    flops_per_sample = W_HOLD + W_FADE_EXTRA * phi
    total_frames = int(fb.offsets[-1])

    lib = player.load_library()
    lib.speechPlayer_debugFp32PeakTflops.restype = __import__("ctypes").c_double
    fp32_peak_measured = float(lib.speechPlayer_debugFp32PeakTflops())
    props = torch.cuda.get_device_properties(dev)

    # ---- HBM-resident inputs ----
    d_off = torch.from_numpy(fb.offsets.astype(np.int64)).to(dev)
    d_frames = torch.from_numpy(fb.frames).to(dev)
    d_min = torch.from_numpy(fb.min_dur.astype(np.int32)).to(dev)   # same bits as uint32
    d_fade = torch.from_numpy(fb.fade_dur.astype(np.int32)).to(dev)
    d_uix = torch.from_numpy(fb.user_index).to(dev)
    d_null = torch.from_numpy(fb.is_null).to(dev)
    stride = (count + 7) // 8 * 8
    d_out = torch.empty((S, stride), dtype=torch.int16, device=dev)
    d_written = torch.zeros(S, dtype=torch.int32, device=dev)

    batch = player.Batch(sr, S, precision=prec, noise=player.NOISE_PHILOX, seed=args.seed, stream_ids=fb.stream_ids)
    stream = torch.cuda.current_stream().cuda_stream
    batch.set_frames_device(d_off.data_ptr(), d_frames.data_ptr(), d_min.data_ptr(), d_fade.data_ptr(),
                            d_uix.data_ptr(), d_null.data_ptr(), stream)

    kev = []  # (before, after) CUDA events around the render kernel alone, on the launching stream
    enqueue_s = []  # host time spent enqueueing one synthesize call (asynchronous launches)

    def step(timed=False):
        # a step = hand the (HBM-resident) queues to fresh players, then plan + render them: SetFrames resets every
        # stream and invalidates the fade plans, so the plan kernel runs inside the timed synthesize call
        batch.set_frames_device(d_off.data_ptr(), d_frames.data_ptr(), d_min.data_ptr(), d_fade.data_ptr(),
                                d_uix.data_ptr(), d_null.data_ptr(), stream)
        if timed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        t_host = time.perf_counter()
        batch.synthesize_device(count, d_out.data_ptr(), stride, d_written.data_ptr(), stream)
        if timed:
            enqueue_s.append(time.perf_counter() - t_host)
            b.record()
            kev.append((a, b))

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    if args.workload == "batch":
        assert int(d_written.min()) == count, "a stream drained early: workload shorter than the render"
    rendered = int(d_written.to(torch.int64).sum())  # midi streams end at their own length: count what was rendered
    launches0, _ = batch.launch_stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        step(timed=True)
        ev[i + 1].record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches1, _ = batch.launch_stats()
    elapsed_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / len(kev)
    t = torch.tensor([elapsed_ms], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    rendered_all = torch.tensor([float(rendered)], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(rendered_all, op=dist.ReduceOp.SUM)
    rendered_all = float(rendered_all.item())                            # samples rendered per step, all ranks
    value = rendered_all / sr * args.steps / (elapsed_ms * 1e-3)          # audio-seconds per wall-second, whole job
    samples_per_s_gpu = rendered * args.steps / (elapsed_ms * 1e-3)       # per GPU
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sample_pcm(d_out, count, d_written.cpu().numpy(), args.seed))

    # ---- e2e: host buffers through the C-ABI (H2D of the frames + D2H of the int16 inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        slice_ticks = min(count, max(int(args.e2e_slice_seconds * sr) // 64 * 64, 64))
        h_out = torch.empty((S, slice_ticks), dtype=torch.int16).pin_memory()
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        h_off, h_frames = pin(fb.offsets.astype(np.int64)), pin(fb.frames)
        h_min, h_fade = pin(fb.min_dur.astype(np.int32)), pin(fb.fade_dur.astype(np.int32))
        h_uix, h_null = pin(fb.user_index), pin(fb.is_null)
        h2d = sum(x.numel() * x.element_size() for x in (h_off, h_frames, h_min, h_fade, h_uix, h_null))
        d2h = S * count * 2 + S * 16
        eb = player.Batch(sr, S, precision=prec, noise=player.NOISE_PHILOX, seed=args.seed, stream_ids=fb.stream_ids)
        L = eb._L

        def e2e_step():
            eb.reset(None)
            rc = L.speechPlayer_batchSetFramesHost(eb._h, h_off.data_ptr(), h_frames.data_ptr(), h_min.data_ptr(),
                                                   h_fade.data_ptr(), h_uix.data_ptr(), h_null.data_ptr(), None)
            assert rc == 0, player.last_error()
            done = 0
            while done < count:  # every slice lands in the same pinned buffer; the first one is kept for the check below
                n_now = min(slice_ticks, count - done)
                dst = h_out if done == 0 else h_scratch
                got = L.speechPlayer_batchSynthesizeHost(eb._h, n_now, dst.data_ptr(), None)
                assert got >= 0 and (args.workload != "batch" or got == S * n_now), (got, player.last_error())
                done += n_now

        h_scratch = torch.empty((S, slice_ticks), dtype=torch.int16).pin_memory() if count > slice_ticks else h_out
        e2e_step()  # warm-up (staging buffers, pinned result buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        # The ceiling the end-to-end number lives under, measured in the same run: every rank copies its device rows into its
        # pinned host buffer at the same time, in the engine's gather shape (2-D, one 2-s slice of every row), with no kernel
        # running.  At N > 1 this is the HOST's concurrent device->pinned bandwidth (tools/d2h_probe.cu, profiles/r02_d2h_probe_*:
        # 55 / 68 / 73 / 92 GB/s for 1 / 2 / 4 / 8 GPUs on this pool's boxes), not a property of the engine.
        reps = 3
        h_out.copy_(d_out[:, :slice_ticks], non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            h_out.copy_(d_out[:, :slice_ticks], non_blocking=True)
        torch.cuda.synchronize()
        dtp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dtp, op=dist.ReduceOp.MAX)
        host_ceiling = world * reps * S * slice_ticks * 2 / float(dtp.item()) / 1e9
        e2e_launches = eb.launch_stats()[0]
        # the device-resident and the host path must agree bit for bit
        same = bool(torch.equal(d_out[:64, :slice_ticks].cpu(), h_out[:64]))
        e2e = {"value": rendered_all / sr * args.e2e_steps / float(dt.item()), "unit": "audio-seconds/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
               "ms_per_step": 1e3 * float(dt.item()) / args.e2e_steps, "matches_device_path": same,
               "slice_seconds": slice_ticks / sr, "rank_cpus_bound_to_gpu_numa_node": cpus_bound,
               "kernel_launches_total": int(e2e_launches),
               "d2h_GBps_achieved": world * d2h * args.e2e_steps / float(dt.item()) / 1e9,
               "host_d2h_GBps_all_ranks_concurrent": host_ceiling,
               "note": "PCIe / host bound: d2h_GBps_achieved is the int16 of all ranks over the e2e wall time (H2D of the queues, planning "
                       "and the first render included); host_d2h_GBps_all_ranks_concurrent is the same copies alone, all ranks at once"}
        eb.close()

    # ---- parity of what was just timed (outside the timed region): random rows of d_out against the oracle, whole length ----
    par = None
    if rank == 0 and not args.no_parity and args.workload == "batch":
        from oracle import oracle
        from tests import parity as parity_mod
        if not oracle.have_port():
            oracle.build(quiet=True)
        port = oracle.PortLib()
        rows = np.random.default_rng(args.seed).choice(S, size=min(args.parity_streams, S), replace=False)
        w1s, snrs, exacts, worst = [], [], [], 0.0
        for s_ in rows:
            got = d_out[int(s_), :count].cpu().numpy()
            fr_, m_, f_, nul_, ux_ = fb.stream(int(s_))
            want = port.render(sr, fr_, m_, f_, nul_, ux_, max_samples=count, noise=("philox", args.seed, int(fb.stream_ids[int(s_)])))
            w1_, ex_, snr_, mx_ = parity_mod.metrics(got, want)
            assert len(want) == count
            w1s.append(w1_); snrs.append(snr_); exacts.append(ex_); worst = max(worst, mx_)
        par = {"streams": int(len(rows)), "samples_per_stream": count, "within_1lsb_min": min(w1s), "snr_db_min": min(snrs),
               "exact_min": min(exacts), "max_abs_diff": worst, "oracle": "oracle/klatt_oracle.c (port, pinned to the compiled reference)",
               "bar": "fp32: <=1 LSB on >= 99.9 % and >= 60 dB; fp64: exact on >= 99.99 %"}

    # which kernel rendered, and the DRAM traffic of one launch of it from the committed ncu capture of this very command
    # (tools/ncu_summary.py --json; per launch = per step, like `achieved`)
    sched = os.environ.get("NVSP_SCHED", "rings")
    if prec != player.PRECISION_FP32:
        kernel_name, cap = "klatt_batch_f64_kernel", None
    elif sched == "rounds":
        kernel_name, cap = "klatt_f32_hold_kernel + klatt_f32_general_pair_kernel (rounds)", None
    elif sched != "block" or S < int(os.environ.get("NVSP_BLOCK_MIN_STREAMS", "16384")):
        kernel_name, cap = "klatt_f32_sched_kernel (ring scheduler: hold and general chunks of all streams in one launch)", "r02_sched_traffic.json"
    else:
        kernel_name = ("klatt_f32_block_kernel (block scheduler: streams owned by one thread block, hold / fade / general cells, "
                       "the whole call in one launch)")
        cap = "r02_block_traffic.json"
    traffic, traffic_src = None, None
    if cap and args.workload == "batch" and S == 65536 and abs(secs - 10.0) < 1e-9:
        try:
            rec = json.load(open(os.path.join(ROOT, "profiles", cap)))["launches"][0]
            traffic, traffic_src = rec["dram_bytes"], "profiles/" + cap + " (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one launch)"
        except Exception:
            pass

    if rank == 0:
        peaks = measured_peaks()
        achieved_tf = rendered * flops_per_sample / (kernel_ms * 1e-3) / 1e12  # dominant kernel alone
        sm_max = (clocks or {}).get("sm_max_mhz") or (peaks or {}).get("sm_max_mhz") or 1965.0
        nominal_tf = props.multi_processor_count * 128 * 2 * sm_max * 1e6 / 1e12
        peak_tf = fp32_peak_measured if fp32_peak_measured > 0 else nominal_tf
        out_bytes_per_s = samples_per_s_gpu * 2.0 + total_frames * (47 * 8 + 13) * args.steps / (elapsed_ms * 1e-3)
        hbm_peak = (peaks or {}).get("hbm_gbs", 6650.0)
        line = {
            "metric": "audio-seconds synthesized/sec (batched streams)", "value": value, "unit": "audio-seconds/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if prec == player.PRECISION_FP32 else "f64", "data": "synthetic",
            "config": {"workload": "%s, %d streams x %.2f s @ %d Hz per GPU (seed 0x%X)" % (workload_name, S, secs, sr, args.seed),
                       "rendered_fraction": rendered / float(S * count),
                       "streams_per_gpu": S, "seconds_per_stream": secs, "sample_rate": sr, "frames_per_gpu": total_frames,
                       "fade_fraction_phi": round(phi, 4), "flops_per_sample_W": round(flops_per_sample, 1),
                       "noise": "philox4x32-10", "precision": args.precision,
                       "l2": "no flush needed: each step writes %.1f GB of int16 (>> 126 MB L2)" % (S * stride * 2 / 1e9),
                       "real_time_factor_per_gpu": samples_per_s_gpu / sr,
                       "host_enqueue_ms_per_step": round(1e3 * sum(enqueue_s) / max(len(enqueue_s), 1), 2)},
            "roofline": {"bound": "fp32_fma", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf,
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel (klatt_f32_sched_kernel:
                         # one launch = one step of config 3), ncu --set full capture summarised in
                         # profiles/r01_v4_ncu_summary.txt; algorithmic bytes of that launch: 36.6 GB (int16 out + queues + plans)
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "FFMA loop measured on this GPU in this run (MEASURED_PEAKS.json has no FP32 entry)"
                                        if fp32_peak_measured > 0 else "SMs x 128 x 2 x max SM clock",
                         "peak_nominal": nominal_tf, "frac_of_nominal": achieved_tf / nominal_tf,
                         "kernel": kernel_name,
                         "flops_per_launch": rendered * flops_per_sample, "kernel_ms": kernel_ms,
                         "kernel_share_of_step": kernel_ms / ms_per_step},
            "roofline_hbm": {"bound": "hbm", "achieved": out_bytes_per_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": out_bytes_per_s / 1e9 / hbm_peak,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                             "algorithmic_bytes_per_sample": 2.0},
            "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "ns_per_sample_core")} if cpu else None),
            "parity": par,
            "e2e": e2e,
            "gpu_launches": int(launches1 - launches0),
            "clocks": clocks,
            "setup": {"workload_generation_s": round(t_gen, 1), "gpu": props.name, "sms": props.multi_processor_count},
        }
        print(json.dumps(line), flush=True)
    batch.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
