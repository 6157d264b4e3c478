"""GPU: the host layer's objects give back the device memory they take.  Players of all three precisions, FP64 and FP32
batches (one of them on the ring scheduler), and a one-device multi-GPU batch are created, used once and destroyed, 20
times over; afterwards free device memory is where it was after one warm-up cycle (which creates the process-lifetime
scratch: the batched-pull items)."""
import ctypes

import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads

pytestmark = pytest.mark.gpu

SR = 22050


def _free_device_bytes():
    """cuMemGetInfo on the context the library made current on this thread."""
    cu = ctypes.CDLL("libcuda.so.1")
    free, total = ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert cu.cuMemGetInfo_v2(ctypes.byref(free), ctypes.byref(total)) == 0
    return free.value


def _cycle(fb, stream):
    fr, m, f, nul, ux = stream
    for prec in (player.PRECISION_FP64, player.PRECISION_FP32, player.PRECISION_STREAM):
        p = player.SpeechPlayer(SR, precision=prec, noise=player.NOISE_PHILOX, seed=3, streamId=1)
        p.queue_frames(fr, m, f, ux, nul)
        assert p.synthesize_np(1024).size > 0
        p.close()
    pair = [player.SpeechPlayer(SR, precision=player.PRECISION_STREAM, noise=player.NOISE_PHILOX, seed=3, streamId=s)
            for s in range(2)]
    for p in pair:
        p.queue_frames(fr, m, f, ux, nul)
    _, written = player.synthesize_batch(pair, 1024)
    assert (written > 0).all()
    for p in pair:
        p.close()
    # 2048 samples per call: more than the ring scheduler's 384-tick general chunk, so with NVSP_ROUNDS_MIN_STREAMS=1 the
    # FP32 batch renders through it
    for prec in (player.PRECISION_FP64, player.PRECISION_FP32):
        b = player.Batch(SR, fb.num_streams, precision=prec, seed=5, stream_ids=fb.stream_ids)
        b.set_frames_host(fb)
        _, written = b.synthesize_host(2048)
        assert (written > 0).all()
        b.close()
    mb = player.MultiBatch(SR, fb.num_streams, [0], seed=5, stream_ids=fb.stream_ids)
    mb.set_frames_host(fb)
    _, written = mb.synthesize_host(2048)
    assert (written > 0).all()
    mb.close()


def test_create_destroy_cycles_return_device_memory(monkeypatch):
    monkeypatch.setenv("NVSP_ROUNDS_MIN_STREAMS", "1")
    fb = workloads.random_frames(64, 0.3, SR, seed=17)
    stream = workloads.random_stream(7, 0.3, SR)
    _cycle(fb, stream)
    base = _free_device_bytes()
    for _ in range(20):
        _cycle(fb, stream)
    after = _free_device_bytes()
    assert base - after <= 32 << 20, (base - after) / 2**20
