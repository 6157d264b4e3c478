"""GPU: speechPlayer_synthesizeLongBatch -- many pre-queued streams through the long-utterance path (kernel b) in one launch
sequence.  Every row is checked against what speechPlayer_synthesizeLong renders for that stream alone (same seed, stream
id, chunk length), against the reference restatement and the committed goldens, and against kernel (a).

A row may differ from its solo render only where a resonator chunk's start state, composed in double by a scan whose
association depends on where the stream sits among the scan's blocks, rounds differently in its last bit; the phase and
excitation are bit for bit the same.  The bar against the solo render is therefore max|d| <= 1 on >= 99.99 % identical
samples, and the number of differing samples is printed (zero is what is expected)."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads
from tests import parity, scenarios
from tests.test_gpu_long import _fallbacks, _prequeued
from tests.test_long_stream_numerics_cpu import LONG_MAX_ABS, LONG_SNR_DB

pytestmark = pytest.mark.gpu

SR = 22050
SEED = 0xB200


def _empty():
    return (np.zeros((0, 47)), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint8), np.zeros(0, np.int32))


def _single(m, f):
    """one real request of random frames with min duration m and fade f (m + 1 ticks when m + 1 >= f + 2)"""
    fr, _, _, _, _ = workloads.random_stream(4242, 0.05, SR)
    return (fr[:1].copy(), np.array([m], np.uint32), np.array([f], np.uint32), np.zeros(1, np.uint8), np.zeros(1, np.int32))


def _ragged_batch():
    """~40 streams: random lengths from 0.05 s to 20 s, an empty queue, a NULL-only queue, a stream shorter than one chunk,
    one of exactly 4096 ticks (a whole number of chunks at 64 and at 1024), and per-stream caps on some of them"""
    rng = np.random.default_rng(2026)
    secs = np.exp(rng.uniform(np.log(0.05), np.log(20.0), 34))
    qs = [workloads.random_stream(1000 + k, float(s), SR) for k, s in enumerate(secs)]
    null_only = (np.zeros((3, 47)), np.array([100, 0, 500], np.uint32), np.array([50, 30, 10], np.uint32), np.ones(3, np.uint8),
                 np.zeros(3, np.int32))
    qs[3:3] = [_empty()]
    qs[10:10] = [null_only]
    qs[17:17] = [_single(40, 5)]      # 41 ticks
    qs[23:23] = [_single(4095, 100)]  # 4096 ticks
    qs.append(_empty())
    ids = np.arange(len(qs), dtype=np.uint64) * 7919 + 5
    fb = workloads._concat(SR, qs, ids)
    law = fb.timeline_samples()
    caps = law.astype(np.uint64).copy()
    for k in (1, 5, 12, 30):
        caps[k] = max(int(law[k]) // 3, 1)
    caps[20] = 0
    return fb, caps


def _solo(fb, s, chunk, cap=None, seed=SEED):
    fr, m, f, nul, _ = fb.stream(s)
    if len(m) == 0:
        return np.zeros(0, np.int16), 0
    before = _fallbacks()
    got, _, _ = player.synthesize_long(fb.sample_rate, fr, m, f, nul, seed=seed, stream_id=int(fb.stream_ids[s]), chunk_ticks=chunk,
                                       max_samples=None if cap is None else int(cap))
    return got, _fallbacks() - before


def _assert_rows_equal_solo(rows, fb, chunk, caps, what):
    differing = total = 0
    for s, row in enumerate(rows):
        want, _ = _solo(fb, s, chunk, None if caps is None else caps[s])
        assert len(row) == len(want), (what, s, len(row), len(want))
        if len(row) == 0:
            continue
        d = np.abs(row.astype(np.int32) - want.astype(np.int32))
        differing += int((d != 0).sum())
        total += len(row)
        assert d.max() <= 1, (what, s, int(d.max()))
    print("%s: %d of %d samples differ from the solo renders" % (what, differing, total))
    assert differing <= 1e-4 * total, (what, differing, total)


@pytest.fixture(scope="module")
def ragged():
    return _ragged_batch()


@pytest.mark.parametrize("chunk", [64, 1024])
def test_rows_equal_the_solo_calls(ragged, chunk):
    fb, caps = ragged
    pcm, off, serial, ms, launches = player.synthesize_long_batch(fb, seed=SEED, chunk_ticks=chunk, max_samples=caps)
    law = np.minimum(fb.timeline_samples(), caps.astype(np.int64))
    assert (np.diff(off) == law).all() and len(pcm) == law.sum()
    assert launches >= 45
    rows = player.split_rows(pcm, off)
    assert len(rows[3]) == 0 and len(rows[20]) == 0
    assert not rows[10].any()  # NULL-only: silence of the lawful length
    assert len(rows[17]) == 41 and len(rows[23]) == 4096
    _assert_rows_equal_solo(rows, fb, chunk, caps, "ragged batch, chunk %d" % chunk)


def test_one_stream_is_bitwise_synthesize_long():
    fr, m, f, nul, ux = workloads.random_stream(31337, 6.0, SR)
    fb = workloads._concat(SR, [(fr, m, f, nul, ux)], np.array([31337], np.uint64))
    for chunk in (256, 1024):
        pcm, off, serial, _, launches = player.synthesize_long_batch(fb, seed=7, chunk_ticks=chunk)
        want, _, want_launches = player.synthesize_long(SR, fr, m, f, nul, seed=7, stream_id=31337, chunk_ticks=chunk)
        assert off[-1] == len(want) and np.array_equal(pcm, want)
        assert launches == want_launches and not serial.any()


@pytest.mark.parametrize("sr", sorted({sc["sr"] for sc in scenarios.all_scenarios().values() if _prequeued(sc)}))
def test_scenarios_in_one_batch(golden_scenarios, sr):
    """the pre-queued scenarios of tests/scenarios.py at one sample rate, as the streams of one batch, capped at the samples
    the script asks for, against the goldens the compiled reference rendered"""
    names = sorted(n for n, sc in scenarios.all_scenarios().items() if _prequeued(sc) and sc["sr"] == sr)
    qs, caps = [], []
    for name in names:
        sc = scenarios.all_scenarios()[name]
        q = [o for o in sc["ops"] if o[0] == "q"]
        fr = np.stack([np.zeros(47) if o[1] is None else np.asarray(o[1], dtype=np.float64) for o in q])
        m = np.array([o[2] for o in q], dtype=np.uint32)
        f = np.array([o[3] for o in q], dtype=np.uint32)
        nul = np.array([o[1] is None for o in q], dtype=np.uint8)
        qs.append((fr, m, f, nul, np.zeros(len(m), np.int32)))
        caps.append(sum(o[1] for o in sc["ops"] if o[0] == "s"))
    fb = workloads._concat(sr, qs, np.full(len(qs), scenarios.STREAM, dtype=np.uint64))
    pcm, off, _, _, _ = player.synthesize_long_batch(fb, seed=scenarios.SEED, chunk_ticks=64, max_samples=np.array(caps, np.uint64))
    for name, row in zip(names, player.split_rows(pcm, off)):
        want = golden_scenarios[name + "/pcm"]
        assert len(row) == len(want) == sum(golden_scenarios[name + "/counts"]), name
        parity.assert_f32_parity(row, want, "long batch " + name)


def _whole_sample_period_streams():
    """the queue of test_long_whole_sample_pitch_periods_wrap_with_the_reference (150 Hz then 225 Hz), and each pitch alone"""
    fr = np.zeros((2, 47))
    for j, hz in enumerate((150.0, 225.0)):
        fr[j, workloads.P["voicePitch"]] = fr[j, workloads.P["endVoicePitch"]] = hz
        fr[j, workloads.P["voiceAmplitude"]] = 1.0
        fr[j, workloads.P["preFormantGain"]] = 1.0
        fr[j, workloads.P["outputGain"]] = 1.0
        workloads.set_frame(fr[j], "a")
    m = np.array([33075, 33075], dtype=np.uint32)
    f = np.array([441, 441], dtype=np.uint32)
    z = np.zeros(2, np.uint8), np.zeros(2, np.int32)
    return [(fr, m, f, *z), (fr[:1], m[:1], f[:1], z[0][:1], z[1][:1]), (fr[1:], m[1:], f[1:], z[0][1:], z[1][1:])]


@pytest.mark.parametrize("chunk", [64, 1024])
def test_per_stream_serial_fallback(port, chunk):
    """streams whose constant whole-sample pitch periods may fail the speculative phase's check, among random streams: the
    serial fallback is taken for exactly the streams whose solo call takes it, and the others keep their verified phase"""
    special = _whole_sample_period_streams()
    qs = [workloads.random_stream(50 + k, 1.5, SR) for k in range(6)]
    for k, q in zip((1, 3, 6), special):
        qs.insert(k, q)
    ids = np.arange(len(qs), dtype=np.uint64) + 300
    fb = workloads._concat(SR, qs, ids)
    solo = [_solo(fb, s, chunk, seed=11) for s in range(fb.num_streams)]
    want_flags = np.array([fell for _, fell in solo], np.uint8)
    before = _fallbacks()
    pcm, off, serial, _, _ = player.synthesize_long_batch(fb, seed=11, chunk_ticks=chunk)
    assert _fallbacks() - before == int(want_flags.sum())
    assert np.array_equal(serial, want_flags), (serial, want_flags)
    print("chunk %d: %d of %d streams took the serial fallback" % (chunk, int(want_flags.sum()), fb.num_streams))
    for s, row in enumerate(player.split_rows(pcm, off)):
        fr, m, f, nul, ux = fb.stream(s)
        want = port.render(SR, fr, m, f, nul, ux, noise=("philox", 11, int(ids[s])))
        assert len(row) == len(want)
        parity.assert_f32_parity(row, want, "long batch fallback stream %d" % s)
        d = np.abs(row.astype(np.int32) - solo[s][0].astype(np.int32))
        assert len(row) == len(solo[s][0]) and d.max() <= 1


def test_three_minute_streams_whole_stream(port):
    """three 3-minute streams at 44.1 kHz among short fillers, to the long-stream bar over the whole stream (the reference
    renders of tests/test_gpu_long_streams.py)"""
    sr, seed = 44100, 0xB200
    long_ids = (31337, 8675309, 271828)
    qs, ids, secs = [], [], []
    for k, sid in enumerate(long_ids):
        qs.append(workloads.random_stream(sid, 180.0, sr)); ids.append(sid); secs.append(180.0)
        qs.append(workloads.random_stream(900 + k, 0.4, sr)); ids.append(900 + k); secs.append(0.4)
    fb = workloads._concat(sr, qs, np.array(ids, dtype=np.uint64))
    caps = np.array([int(s * sr) for s in secs], np.uint64)
    pcm, off, serial, ms, _ = player.synthesize_long_batch(fb, seed=seed, max_samples=caps)
    assert not serial.any()
    for s, row in enumerate(player.split_rows(pcm, off)):
        q = fb.stream(s)
        want = port.render(sr, *q, max_samples=int(caps[s]), noise=("philox", seed, ids[s]))
        assert len(row) == len(want) == caps[s]
        parity.assert_whole_stream(row, want, "long batch %d %g s" % (ids[s], secs[s]), LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


def test_agrees_with_kernel_a():
    """rows within the FP32 bar of player.Batch FP32 (kernel a) at the same seed and stream ids"""
    fb = workloads.random_frames(24, 2.0, SR, first_stream=4000)
    pcm, off, _, _, _ = player.synthesize_long_batch(fb, seed=3)
    law = fb.timeline_samples()
    b = player.Batch(SR, fb.num_streams, precision=player.PRECISION_FP32, seed=3, stream_ids=fb.stream_ids)
    try:
        b.set_frames_host(fb)
        a_out, written = b.synthesize_host(int(law.max()))
    finally:
        b.close()
    for s, row in enumerate(player.split_rows(pcm, off)):
        assert len(row) == law[s] == written[s]
        parity.assert_f32_parity(row, a_out[s, :law[s]], "long batch vs kernel a, stream %d" % s)


def test_device_output_equals_host_output(ragged):
    import torch
    fb, caps = ragged
    pcm, off, _, _, _ = player.synthesize_long_batch(fb, seed=SEED, chunk_ticks=512, max_samples=caps)
    d = torch.full((len(pcm) + 8,), -7, dtype=torch.int16, device="cuda")
    got, off_d, _, _, _ = player.synthesize_long_batch(fb, seed=SEED, chunk_ticks=512, max_samples=caps, device_out=d.data_ptr())
    torch.cuda.synchronize()
    h = d.cpu().numpy()
    assert got == len(pcm) and np.array_equal(off, off_d)
    assert np.array_equal(h[:got], pcm) and (h[got:] == -7).all()


def test_small_group_budget_forces_groups(ragged):
    """NVSP_LONG_BATCH_TICKS small enough for at least three groups (read once per process: a subprocess)"""
    fb, caps = ragged
    law = np.minimum(fb.timeline_samples(), caps.astype(np.int64))
    budget = int(law.sum()) // 4
    assert (law > budget).sum() <= 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from nvspeechplayer_b200 import player; "
            "from tests.test_gpu_long_batch import _ragged_batch; fb, caps = _ragged_batch(); "
            "pcm, off, serial, ms, launches = player.synthesize_long_batch(fb, seed=%d, chunk_ticks=1024, max_samples=caps); "
            "np.savez(sys.argv[1], pcm=pcm, off=off, launches=launches)" % (root, SEED))
    with tempfile.TemporaryDirectory() as d:
        env = dict(os.environ, NVSP_LONG_BATCH_TICKS=str(budget))
        subprocess.run([sys.executable, "-c", code, os.path.join(d, "o.npz")], check=True, env=env, timeout=600)
        z = np.load(os.path.join(d, "o.npz"))
        pcm, off, launches = z["pcm"], z["off"], int(z["launches"])
    _, want_off = player.long_batch_size(fb, max_samples=caps)
    assert np.array_equal(off, want_off)
    assert launches >= 3 * 47, launches  # plan + timeline + 45 per group
    _assert_rows_equal_solo(player.split_rows(pcm, off), fb, 1024, caps, "three or more groups")
