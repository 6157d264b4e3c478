"""GPU: minutes-long streams through every FP32 render path, compared with the reference over the WHOLE stream.

The glottal phase integrates any constant pitch error for as long as a stream lives, and a wrap that lands on the
neighbouring tick is a full-scale burst; renders of a few seconds cannot see it (tests/test_long_stream_numerics_cpu.py has
the mechanism on the host build of the same arithmetic).  Kernel b's 10-minute stream is in tests/test_gpu_long.py."""
import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads
from tests import parity
from tests.test_long_stream_numerics_cpu import LONG_MAX_ABS, LONG_SNR_DB, SEED, directed_stream

pytestmark = pytest.mark.gpu

SR = 44100
# one batch: the 10-minute stream of the CPU test and three more of 3 minutes (one thread renders each whole stream)
BATCH = ((424242, 600.0), (31337, 180.0), (8675309, 180.0), (271828, 180.0))


def _render_batch(fb, count, precision, chunk=30 * SR):
    b = player.Batch(SR, fb.num_streams, precision=precision, seed=SEED, stream_ids=fb.stream_ids)
    try:
        b.set_frames_host(fb)
        parts, left = [], count
        while left > 0:
            o, _ = b.synthesize_host(min(chunk, left))
            parts.append(o)
            left -= o.shape[1]
        return np.concatenate(parts, axis=1)
    finally:
        b.close()


@pytest.fixture(scope="module")
def batch_streams(port):
    streams = [workloads.random_stream(sid, secs, SR) for sid, secs in BATCH]
    fb = workloads._concat(SR, streams, np.array([sid for sid, _ in BATCH], dtype=np.uint64))
    wants = [port.render(SR, *q, max_samples=int(secs * SR), noise=("philox", SEED, sid))
             for q, (sid, secs) in zip(streams, BATCH)]
    return streams, fb, wants


@pytest.mark.parametrize("mode", ["rings", "block", "single_launch"])
def test_batch_f32_long_streams_whole_stream(monkeypatch, batch_streams, mode):
    """player.Batch FP32 under the ring scheduler, the block scheduler and the one-thread-per-stream single launch (the
    environment of test_f32_rounds_equal_single_launch_bitwise, so that four streams take each path)."""
    monkeypatch.setenv("NVSP_ROUNDS_MIN_STREAMS", "100000000" if mode == "single_launch" else "1")
    monkeypatch.setenv("NVSP_SCHED", {"rings": "rings", "block": "block"}.get(mode, "rounds"))
    monkeypatch.setenv("NVSP_BLOCK_MIN_STREAMS", "1")
    streams, fb, wants = batch_streams
    got = _render_batch(fb, int(max(s for _, s in BATCH) * SR), player.PRECISION_FP32)
    for k, ((sid, secs), q, want) in enumerate(zip(BATCH, streams, wants)):
        g = got[k, :len(want)]
        parity.assert_whole_stream(g, want, "batch f32 %s %d %g s" % (mode, sid, secs), LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


def test_batch_f64_control_three_minutes(port):
    """The FP64 engine on a 3-minute stream holds the FP64 bar over the whole stream: the reference arithmetic has no drift."""
    sid, secs = 31337, 180.0
    q = workloads.random_stream(sid, secs, SR)
    n = int(secs * SR)
    fb = workloads._concat(SR, [q], np.array([sid], dtype=np.uint64))
    got = _render_batch(fb, n, player.PRECISION_FP64)[0, :n]
    want = port.render(SR, *q, max_samples=n, noise=("philox", SEED, sid))
    w1, exact, snr, mx = parity.assert_whole_stream(got, want, "batch f64 %d %g s" % (sid, secs), 1, 0.0, q[1], q[2])
    assert exact >= 0.9999, exact


def _pull(sr, q, n, seed, stream, pull=8192):
    fr, m, f, nul, ux = q
    p = player.SpeechPlayer(sr, precision=player.PRECISION_STREAM, noise=player.NOISE_PHILOX, seed=seed, streamId=stream)
    try:
        p.queue_frames(fr, m, f, ux, nul)
        out, left = [], n
        while left > 0:
            c = p.synthesize_np(min(pull, left))
            assert c.size == min(pull, left)
            out.append(c)
            left -= c.size
        return np.concatenate(out)
    finally:
        p.close()


def test_pull_ten_minutes_whole_stream(batch_streams):
    """The low-latency pull path the way NVDA drives it: one player, 8192 samples per pull, for 10 minutes."""
    streams, _, wants = batch_streams
    q, want = streams[0], wants[0]
    got = _pull(SR, q, len(want), SEED, BATCH[0][0])
    parity.assert_whole_stream(got, want, "pull 424242 600 s", LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


def test_directed_vibrato_depth_stream_all_paths(port):
    """The CPU test's directed stream (a depth error adds up every vibrato cycle) through the batch and the pull kernels."""
    sr, secs = 22050, 30.0
    q = directed_stream(sr, secs)
    n = int(secs * sr)
    want = port.render(sr, *q, max_samples=n, noise=("philox", SEED, 1))
    b = player.Batch(sr, 1, precision=player.PRECISION_FP32, seed=SEED, stream_ids=np.array([1], dtype=np.uint64))
    try:
        b.set_frames_host(workloads._concat(sr, [q], np.array([1], dtype=np.uint64)))
        got, _ = b.synthesize_host(n)
    finally:
        b.close()
    parity.assert_whole_stream(got[0, :n], want, "directed, batch f32", 1, 90.0, q[1], q[2])
    parity.assert_whole_stream(_pull(sr, q, n, SEED, 1), want, "directed, pull", 1, 90.0, q[1], q[2])
