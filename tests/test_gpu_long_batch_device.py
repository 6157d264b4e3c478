"""GPU: speechPlayer_synthesizeLongBatchDevice -- the batched long-utterance path reading queues that already live in device
memory.  It groups, chunks and scans exactly as the host entry does, so every check here is BITWISE against
speechPlayer_synthesizeLongBatch on the same queues: samples, output offsets and serial-fallback flags, and a kernel count
that is the host route's plus the one ticks kernel."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from nvspeechplayer_b200 import ipa, player, workloads
from tests.test_gpu_long import _fallbacks
from tests.test_gpu_long_batch import _whole_sample_period_streams

pytestmark = pytest.mark.gpu

SR = 22050
SEED = 0xB200
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _queue(k, secs):
    return workloads.random_stream(7000 + k, secs, SR)


def _ragged_batch():
    """40 streams: lengths from 0.02 s to 25 s, three empty queues, a NULL-only queue, one request shorter than a tile, and
    per-stream caps on some of them (one cap of 0)"""
    rng = np.random.default_rng(4711)
    secs = np.exp(rng.uniform(np.log(0.02), np.log(25.0), 35))
    qs = [_queue(k, float(s)) for k, s in enumerate(secs)]
    empty = (np.zeros((0, 47)), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint8), np.zeros(0, np.int32))
    null_only = (np.zeros((4, 47)), np.array([300, 0, 9, 2000], np.uint32), np.array([60, 0, 40, 7], np.uint32), np.ones(4, np.uint8),
                 np.zeros(4, np.int32))
    fr, _, _, _, _ = _queue(99, 0.05)
    tiny = (fr[:1].copy(), np.array([12], np.uint32), np.array([3], np.uint32), np.zeros(1, np.uint8), np.zeros(1, np.int32))
    qs.insert(0, empty)
    qs.insert(8, null_only)
    qs.insert(15, tiny)
    qs.insert(21, empty)
    qs.append(empty)
    ids = np.arange(len(qs), dtype=np.uint64) * 104729 + 3
    fb = workloads._concat(SR, qs, ids)
    law = fb.timeline_samples()
    caps = law.astype(np.uint64).copy()
    for k in (2, 9, 17, 30):
        caps[k] = max(int(law[k]) // 4, 1)
    caps[26] = 0
    return fb, caps


def _to_device(fb, with_is_null=True):
    """fb's queues as CUDA tensors in the layout of speechPlayer_batchSetFramesDevice"""
    import torch
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return workloads.FrameBatch(sample_rate=fb.sample_rate, offsets=t(fb.offsets), frames=t(fb.frames), min_dur=t(fb.min_dur.view(np.int32)),
                                fade_dur=t(fb.fade_dur.view(np.int32)), is_null=t(fb.is_null) if with_is_null else None, user_index=None,
                                stream_ids=fb.stream_ids)


def _without_is_null(fb):
    return workloads.FrameBatch(fb.sample_rate, fb.offsets, fb.frames, fb.min_dur, fb.fade_dur, None, fb.user_index, fb.stream_ids)


def _assert_same(dev, host, what):
    pcm_d, off_d, ser_d, _, launches_d = dev
    pcm_h, off_h, ser_h, _, launches_h = host
    np.testing.assert_array_equal(off_d, off_h, err_msg=what + ": out_offsets")
    np.testing.assert_array_equal(ser_d, ser_h, err_msg=what + ": serial_phase")
    assert len(pcm_d) == len(pcm_h), what
    np.testing.assert_array_equal(pcm_d, pcm_h, err_msg=what + ": samples")
    assert launches_d == launches_h + 1, (what, launches_d, launches_h)


@pytest.fixture(scope="module")
def ragged():
    fb, caps = _ragged_batch()
    return fb, caps, _to_device(fb)


@pytest.mark.parametrize("chunk", [64, 1024, 0])
def test_device_queues_render_the_host_route_bitwise(ragged, chunk):
    fb, caps, dfb = ragged
    host = player.synthesize_long_batch(fb, seed=SEED, chunk_ticks=chunk, max_samples=caps)
    dev = player.synthesize_long_batch(dfb, seed=SEED, chunk_ticks=chunk, max_samples=caps)
    _assert_same(dev, host, "chunk %d" % chunk)
    rows = player.split_rows(dev[0], dev[1])
    assert len(rows[0]) == len(rows[21]) == len(rows[26]) == 0
    assert len(rows[15]) == 13 and not rows[8].any()
    assert np.abs(dev[0]).max() > 1000


@pytest.mark.parametrize("with_is_null,device_out", [(False, False), (False, True), (True, True)])
def test_without_is_null_and_into_device_memory(ragged, with_is_null, device_out):
    """dIsNull = NULL (every request real, on both routes), and the samples written to device memory"""
    import torch
    fb, caps, dfb = ragged
    hfb = fb if with_is_null else _without_is_null(fb)
    host = player.synthesize_long_batch(hfb, seed=SEED, max_samples=caps)
    d = dfb if with_is_null else _to_device(fb, with_is_null=False)
    if not device_out:
        _assert_same(player.synthesize_long_batch(d, seed=SEED, max_samples=caps), host, "no isNull")
        return
    buf = torch.full((len(host[0]) + 16,), -7, dtype=torch.int16, device="cuda")
    got, off, serial, ms, launches = player.synthesize_long_batch(d, seed=SEED, max_samples=caps, device_out=buf.data_ptr())
    h = buf.cpu().numpy()
    assert got == len(host[0]) and (h[got:] == -7).all()
    _assert_same((h[:got], off, serial, ms, launches), host, "device output, isNull %s" % with_is_null)


def test_size_query_equals_the_host_arrays(ragged):
    fb, caps, dfb = ragged
    for mx in (None, caps, 5000):
        total_d, off_d = player.long_batch_size(dfb, max_samples=mx)
        total_h, off_h = player.long_batch_size(fb, max_samples=mx)
        assert total_d == total_h
        np.testing.assert_array_equal(off_d, off_h)


def test_ticks_kernel_at_ten_million_requests_and_a_million_streams():
    """the ticks kernel against the host law: one stream of 10^7 requests with durations over the whole u32 range, and
    2^20 + 5 small streams (more streams than the kernel's grid: a block takes several)"""
    import torch
    rng = np.random.default_rng(17)
    for lens in ([10 ** 7, 3, 0], rng.integers(0, 4, (1 << 20) + 5)):
        lens = np.asarray(lens, np.int64)
        total = int(lens.sum())
        m = rng.integers(0, 1 << 32, total, dtype=np.uint64).astype(np.uint32)
        f = rng.integers(0, 1 << 32, total, dtype=np.uint64).astype(np.uint32)
        small = rng.random(total) < 0.5  # ordinary durations for half of them, the 0 / 1 fade edge included
        m[small] = rng.integers(0, 3000, int(small.sum()))
        f[small] = rng.integers(0, 3, int(small.sum()))
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        occ = np.maximum(m.astype(np.uint64) + 1, np.maximum(f.astype(np.uint64), 1) + 2)
        c = np.concatenate([[0], np.cumsum(occ, dtype=np.uint64)]).astype(np.uint64)
        law = c[offsets[1:]] - c[offsets[:-1]]
        dfb = workloads.FrameBatch(SR, torch.from_numpy(offsets).cuda(), torch.empty((total, 47), dtype=torch.float64, device="cuda"),
                                   torch.from_numpy(m.view(np.int32)).cuda(), torch.from_numpy(f.view(np.int32)).cuda(), None, None, None)
        got, off = player.long_batch_size(dfb)
        np.testing.assert_array_equal(np.diff(off).astype(np.uint64), law)
        del dfb
        torch.cuda.empty_cache()


@pytest.mark.parametrize("chunk", [64, 1024])
def test_serial_fallback_flags_match_the_host_route(chunk):
    """constant whole-sample pitch periods (150 Hz and 225 Hz at 22 050 Hz: 147 and 98 ticks, each alone and one after the
    other) among random streams: at least one stream takes the per-stream serial fallback, and the device route sends
    exactly the streams there that the host route sends"""
    special = _whole_sample_period_streams()
    qs = [_queue(200 + k, 1.5) for k in range(5)]
    for k, q in zip((0, 2, 5), special):
        qs.insert(k, q)
    fb = workloads._concat(SR, qs, np.arange(len(qs), dtype=np.uint64) + 900)
    before = _fallbacks()
    host = player.synthesize_long_batch(fb, seed=11, chunk_ticks=chunk)
    mid = _fallbacks()
    dev = player.synthesize_long_batch(_to_device(fb), seed=11, chunk_ticks=chunk)
    after = _fallbacks()
    print("chunk %d: serial fallback flags %s" % (chunk, host[2].tolist()))
    assert host[2].any()
    assert after - mid == mid - before == int(host[2].sum())
    _assert_same(dev, host, "serial fallback, chunk %d" % chunk)


def test_queue_arrays_are_only_read(ragged):
    import torch
    fb, caps, dfb = ragged
    fields = ("offsets", "frames", "min_dur", "fade_dur", "is_null")
    before = [getattr(dfb, k).view(torch.uint8).clone() for k in fields]
    buf = torch.empty(int(player.long_batch_size(fb)[0]) + 8, dtype=torch.int16, device="cuda")
    player.synthesize_long_batch(dfb, seed=SEED, chunk_ticks=256, device_out=buf.data_ptr())
    player.synthesize_long_batch(dfb, seed=SEED, max_samples=caps)
    for k, b in zip(fields, before):
        assert torch.equal(getattr(dfb, k).view(torch.uint8), b), k


def test_queues_written_on_a_side_stream_need_no_synchronisation(ragged):
    """the queues are written on a non-default torch stream behind ~0.1 s of pending work, and the render is issued on that
    stream right away: it must see the written queues, not the zeros that were there before"""
    import torch
    fb, caps, src = ragged
    dst = workloads.FrameBatch(SR, *[torch.zeros_like(getattr(src, k)) for k in ("offsets", "frames", "min_dur", "fade_dur", "is_null")],
                               None, fb.stream_ids)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        for k in ("offsets", "frames", "min_dur", "fade_dur", "is_null"):
            getattr(dst, k).copy_(getattr(src, k))
        buf = torch.full((int(player.long_batch_size(fb, max_samples=caps)[0]) + 8,), -7, dtype=torch.int16, device="cuda")
    got, off, serial, ms, launches = player.synthesize_long_batch(dst, seed=SEED, max_samples=caps, device_out=buf.data_ptr(),
                                                                  cuda_stream=side)
    side.synchronize()
    host = player.synthesize_long_batch(fb, seed=SEED, max_samples=caps)
    _assert_same((buf.cpu().numpy()[:got], off, serial, ms, launches), host, "side stream")


@pytest.mark.parametrize("side_stream", [False, True])
def test_text_to_pcm(side_stream):
    """frames_for_texts_device(..., stream_offsets) -> the device long batch, against frames_for_texts (its per-text queues
    joined by the same stream_offsets) -> the host long batch.  With side_stream the producer and the render run on a
    non-default torch stream with no synchronisation in between."""
    import torch
    gold = np.load(os.path.join(GOLDEN, "ipa_frames.npz"))
    lines = [str(t) for t in gold["texts"][:8]]
    texts = [lines[(i * 5) % 8] for i in range(120)]
    so = np.concatenate([[0], np.cumsum(np.tile([1, 6, 3, 2, 0, 4, 5, 3], 5))])  # 40 streams, an empty one among them
    assert so[-1] == len(texts)
    kw = dict(speed=0.8, sample_rate=SR, trailing_silence_ms=150.0)
    stream = torch.cuda.Stream() if side_stream else None
    db = ipa.frames_for_texts_device(texts, stream_offsets=so, cuda_stream=stream, **kw)
    dev = player.synthesize_long_batch(db, seed=SEED, cuda_stream=stream)
    fb = ipa.frames_for_texts(texts, **kw)
    fb.offsets = fb.offsets[so]
    fb.stream_ids = np.arange(len(so) - 1, dtype=np.uint64)
    host = player.synthesize_long_batch(fb, seed=SEED)
    _assert_same(dev, host, "text to PCM")
    assert (np.diff(host[1]) == 0).any() and np.abs(host[0]).max() > 1000


def test_small_group_budget_forces_groups(ragged):
    """NVSP_LONG_BATCH_TICKS small enough for at least three groups (read once per process: a subprocess running both routes)"""
    fb, caps, _ = ragged
    law = np.minimum(fb.timeline_samples(), caps.astype(np.int64))
    budget = int(law.sum()) // 4
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from nvspeechplayer_b200 import player; "
            "from tests.test_gpu_long_batch_device import _ragged_batch, _to_device; fb, caps = _ragged_batch(); "
            "h = player.synthesize_long_batch(fb, seed=%d, chunk_ticks=1024, max_samples=caps); "
            "d = player.synthesize_long_batch(_to_device(fb), seed=%d, chunk_ticks=1024, max_samples=caps); "
            "np.savez(sys.argv[1], **{k + w: v for w, r in (('h', h), ('d', d)) for k, v in zip(('pcm', 'off', 'ser', 'ms', 'n'), r)})"
            % (root, SEED, SEED))
    with tempfile.TemporaryDirectory() as tmp:
        env = dict(os.environ, NVSP_LONG_BATCH_TICKS=str(budget))
        subprocess.run([sys.executable, "-c", code, os.path.join(tmp, "o.npz")], check=True, env=env, timeout=600)
        z = dict(np.load(os.path.join(tmp, "o.npz")))
    host = tuple(z[k + "h"] for k in ("pcm", "off", "ser", "ms", "n"))
    dev = tuple(z[k + "d"] for k in ("pcm", "off", "ser", "ms", "n"))
    assert int(host[4]) >= 3 * 47, int(host[4])  # plan + timeline + 45 per group
    _assert_same(dev, host, "three or more groups")


def test_pointers_that_are_not_device_memory_are_refused(ragged):
    import torch
    fb, caps, dfb = ragged
    L = player.load_library()
    n = fb.num_streams
    out_offsets = np.zeros(n + 1, np.int64)
    args = [dfb.offsets.data_ptr(), dfb.frames.data_ptr(), dfb.min_dur.data_ptr(), dfb.fade_dur.data_ptr(), dfb.is_null.data_ptr()]
    for k, host_ptr in enumerate([fb.offsets.ctypes.data, fb.frames.ctypes.data, fb.min_dur.ctypes.data]):
        bad = list(args)
        bad[k] = host_ptr
        got = L.speechPlayer_synthesizeLongBatchDevice(SR, n, *bad, SEED, None, 0, None, None, out_offsets.ctypes.data, 0, None, None, None,
                                                       None)
        assert got == -1 and "not device memory" in player.last_error(), (k, player.last_error())
    # offsets that break the host entry's rules, with the host entry's message, before any kernel reads the queues
    for offs, msg in (([1] + [int(fb.offsets[-1])] * n, "offsets[0]"), ([0, 5, 3] + [int(fb.offsets[-1])] * (n - 2), "non-decreasing")):
        d = torch.tensor(offs, dtype=torch.int64, device="cuda")
        got = L.speechPlayer_synthesizeLongBatchDevice(SR, n, d.data_ptr(), *args[1:], SEED, None, 0, None, None, out_offsets.ctypes.data, 0,
                                                       None, None, None, None)
        assert got == -1 and msg in player.last_error(), player.last_error()
