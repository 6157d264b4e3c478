"""GPU: the long-utterance path (kernel b: chunks rendered in parallel, phase and resonator state recovered by scans)
against the reference restatement, through the C-ABI.

Bar (BASELINE.json north_star, FP32 variant): <= 1 LSB on >= 99.9 % of samples and >= 60 dB SNR; the sample count
follows the timeline law.  Config 4's recipe (config-1 frames looped, 44.1 kHz) at a length the oracle renders in
seconds; the full hour is exercised by bench.py --workload long."""
import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads
from tests import parity, scenarios
from tests.test_long_stream_numerics_cpu import LONG_MAX_ABS, LONG_SNR_DB

pytestmark = pytest.mark.gpu


def _looped_config1(g, sr, repeats):
    scale = sr / 22050.0
    m = np.tile((g["min_dur"] * scale).astype(np.uint32), repeats)
    f = np.tile((g["fade_dur"] * scale).astype(np.uint32), repeats)
    return np.tile(g["frames"], (repeats, 1)), m, f, np.tile(g["is_null"], repeats)


@pytest.mark.parametrize("sr,repeats,chunk", [(44100, 2, 1024), (22050, 1, 256), (16000, 1, 4096)])
def test_long_config1_looped(port, golden_config1, sr, repeats, chunk):
    fr, m, f, nul = _looped_config1(golden_config1, sr, repeats)
    want = port.render(sr, fr, m, f, nul, noise=("philox", 5, 9))
    got, ms, launches = player.synthesize_long(sr, fr, m, f, nul, seed=5, stream_id=9, chunk_ticks=chunk)
    assert launches >= 20
    assert len(got) == len(want) == workloads._concat(sr, [(fr, m, f, nul, np.zeros(len(m), np.int32))], [9]).timeline_samples()[0]
    w1, exact, snr, mx = parity.assert_f32_parity(got, want, "long config1 @%d" % sr)
    assert snr >= 80.0


@pytest.mark.parametrize("sr,chunk", [(22050, 1024), (44100, 512)])
def test_long_random_frames(port, sr, chunk):
    """all 47 params randomised, 5 % NULL requests, fades from 5 ms to 0.6 M: every stage's scan is exercised"""
    fr, m, f, nul, ux = workloads.random_stream(31337, 6.0, sr)
    want = port.render(sr, fr, m, f, nul, ux, noise=("philox", 0xB200, 31337))
    got, ms, _ = player.synthesize_long(sr, fr, m, f, nul, seed=0xB200, stream_id=31337, chunk_ticks=chunk)
    assert len(got) == len(want)
    parity.assert_f32_parity(got, want, "long random @%d" % sr)


def test_long_matches_batch_kernel_and_chunk_sizes():
    """same stream through kernel (a) (FP32 batch path) and kernel (b) at two chunk sizes: within 1 LSB of each other"""
    sr = 22050
    fr, m, f, nul, ux = workloads.random_stream(77, 3.0, sr)
    fb = workloads._concat(sr, [(fr, m, f, nul, ux)], [77])
    n = int(fb.timeline_samples()[0])
    b = player.Batch(sr, 1, precision=player.PRECISION_FP32, seed=3, stream_ids=fb.stream_ids)
    b.set_frames_host(fb)
    a_out, written = b.synthesize_host(n)
    b.close()
    assert written[0] == n
    outs = [player.synthesize_long(sr, fr, m, f, nul, seed=3, stream_id=77, chunk_ticks=c)[0] for c in (128, 2048)]
    for o in outs:
        assert len(o) == n
        parity.assert_f32_parity(o, a_out[0], "kernel b vs kernel a")
    parity.assert_f32_parity(outs[0], outs[1], "chunk 128 vs 2048")


def test_long_truncated_and_null_only():
    sr = 22050
    fr, m, f, nul, ux = workloads.random_stream(5, 1.0, sr)
    full, _, _ = player.synthesize_long(sr, fr, m, f, nul, seed=1, stream_id=5)
    part, _, _ = player.synthesize_long(sr, fr, m, f, nul, seed=1, stream_id=5, max_samples=10000)
    assert len(part) == 10000
    parity.assert_f32_parity(part, full[:10000], "truncated")
    # a queue of NULL requests only renders silence of the lawful length (reference src/frame.cpp:59-63)
    got, _, _ = player.synthesize_long(sr, np.zeros((2, 47)), [100, 0], [50, 30], is_null=[1, 1], seed=1, stream_id=5)
    assert len(got) == 101 + 32 and not got.any()


def _fallbacks():
    import ctypes
    L = player.load_library()
    L.speechPlayer_debugLongSerialFallbacks.restype = ctypes.c_ulonglong
    return L.speechPlayer_debugLongSerialFallbacks()


def _prequeued(sc):
    """scenario scripts kernel (b) can take: every frame queued before the first pull, no purge"""
    ops = sc["ops"]
    first_s = next(i for i, o in enumerate(ops) if o[0] == "s")
    return all(o[0] == "q" and not o[5] for o in ops[:first_s]) and all(o[0] == "s" for o in ops[first_s:])


@pytest.mark.parametrize("name", sorted(n for n, sc in scenarios.all_scenarios().items() if _prequeued(sc)))
def test_long_scenarios(golden_scenarios, name):
    """The frame-manager / generator scenarios of tests/scenarios.py (timeline law, NULL-frame rewrites, NaN keep, NaN gain,
    clamp, fade longer than hold, glide to zero, source features, random frames at three rates) through kernel (b), against
    the goldens the compiled reference rendered.  `clamp` (gain 1e6: every sample is +-32000, a wrap one tick off flips
    hundreds of them) and `fade_gt_hold` are the two the round-1 fixed-point phase could not pass."""
    sc = scenarios.all_scenarios()[name]
    qs = [o for o in sc["ops"] if o[0] == "q"]
    want = golden_scenarios[name + "/pcm"]
    asked = sum(o[1] for o in sc["ops"] if o[0] == "s")
    fr = np.stack([np.zeros(47) if o[1] is None else np.asarray(o[1], dtype=np.float64) for o in qs])
    m = np.array([o[2] for o in qs], dtype=np.uint32)
    f = np.array([o[3] for o in qs], dtype=np.uint32)
    nul = np.array([o[1] is None for o in qs], dtype=np.uint8)
    got, _, _ = player.synthesize_long(sc["sr"], fr, m, f, nul, seed=scenarios.SEED, stream_id=scenarios.STREAM, chunk_ticks=64,
                                       max_samples=asked)
    assert len(got) == len(want) == sum(golden_scenarios[name + "/counts"])
    parity.assert_f32_parity(got, want, "long " + name)


@pytest.mark.parametrize("chunk", [64, 1024])
def test_long_whole_sample_pitch_periods_wrap_with_the_reference(port, chunk):
    """150 Hz and 225 Hz at 22 050 Hz (147 / 98 samples per period), constant pitch, no vibrato: the sawtooth wrap hangs on
    the last bit of the reference's FP64 phase sum (src/speechWaveGenerator.cpp:55).  Kernel (b) runs that recurrence
    itself (klatt_long_phase.cuh), so it wraps on the reference's tick -- through the verified parallel construction or,
    when a run fails its end-to-start check, through the serial fallback."""
    sr = 22050
    fr = np.zeros((2, 47))
    for j, hz in enumerate((150.0, 225.0)):
        fr[j, workloads.P["voicePitch"]] = fr[j, workloads.P["endVoicePitch"]] = hz
        fr[j, workloads.P["voiceAmplitude"]] = 1.0
        fr[j, workloads.P["preFormantGain"]] = 1.0
        fr[j, workloads.P["outputGain"]] = 1.0
        workloads.set_frame(fr[j], "a")
    m = np.array([33075, 33075], dtype=np.uint32)
    f = np.array([441, 441], dtype=np.uint32)
    want = port.render(sr, fr, m, f, None, None, noise=("philox", 11, 3))
    got, _, _ = player.synthesize_long(sr, fr, m, f, None, seed=11, stream_id=3, chunk_ticks=chunk)
    assert len(got) == len(want)
    w1, exact, snr, mx = parity.assert_f32_parity(got, want, "long whole-sample periods")
    assert snr >= 80.0, snr


def test_long_ten_minutes_at_44k_last_five_seconds(port):
    """26.5 M ticks of random frames at 44.1 kHz (a sixth of BASELINE config 4) compared with the oracle over the LAST five
    seconds: any drift of the timeline, the vibrato phase, the glottal phase or the scanned resonator states over 25 000
    chunks would show there.  The parallel phase must have verified (no serial fallback on a generic stream)."""
    sr, secs = 44100, 600.0
    fr, m, f, nul, ux = workloads.random_stream(424242, secs, sr)
    n = int(secs * sr)
    before = _fallbacks()
    got, ms, launches = player.synthesize_long(sr, fr, m, f, nul, seed=0xB200, stream_id=424242, max_samples=n)
    assert len(got) == n
    assert _fallbacks() == before, "the speculative phase failed its check on a generic stream"
    want = port.render(sr, fr, m, f, nul, ux, max_samples=n, noise=("philox", 0xB200, 424242))
    assert len(want) == n
    tail = 5 * sr
    w1, exact, snr, mx = parity.assert_f32_parity(got[-tail:], want[-tail:], "last 5 s of 10 min")
    print("10 min @44.1k in %.1f ms: last 5 s <=1LSB %.5f, SNR %.1f dB; whole stream <=1LSB %.5f" %
          (ms, w1, snr, parity.metrics(got, want)[0]))
    # the whole stream to the long-stream bar (an FP32 vibrato depth left 60.8 dB, max|d| 1350 here)
    parity.assert_whole_stream(got, want, "kernel b 10 min whole stream", LONG_MAX_ABS, LONG_SNR_DB, m, f)


def test_long_serial_fallback_is_the_same_audio(port, monkeypatch):
    """NVSP_LONG_PHASE=serial forces the fallback (the plain recurrence on one thread).  Same phase values by construction;
    the samples agree to the last bit except where the runs of the two modes start on different ticks and the 64-tick
    warm-up of the noise colouring filter (0.75^64 = 1e-8) rounds differently."""
    import subprocess, sys, os, tempfile
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from nvspeechplayer_b200 import player, workloads; "
            "fr, m, f, nul, ux = workloads.random_stream(9, 1.5, 22050); "
            "np.save(sys.argv[1], player.synthesize_long(22050, fr, m, f, nul, seed=4, stream_id=9, chunk_ticks=256)[0])"
            % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    outs = []
    for mode in ("", "serial"):
        with tempfile.TemporaryDirectory() as d:
            env = dict(os.environ, NVSP_LONG_PHASE=mode)
            subprocess.run([sys.executable, "-c", code, os.path.join(d, "o.npy")], check=True, env=env, timeout=300)
            outs.append(np.load(os.path.join(d, "o.npy")))
    assert len(outs[0]) == len(outs[1])
    w1, exact, snr, mx = parity.metrics(outs[0], outs[1])
    assert mx <= 1 and exact >= 0.99 and snr >= 85.0, (exact, snr, mx)
