"""CPU: speechPlayer_synthesizeLongBatchDevice's argument checks happen before any device work, and without a device the call
reports that there is no CPU fallback."""
import ctypes

import numpy as np
import pytest

from nvspeechplayer_b200 import player


def _call(sr=22050, n=2, d_offsets=0x1000, out_offsets=True):
    """the device entry with stand-in device addresses: every case here is refused before one is dereferenced"""
    L = player.load_library()
    oo = np.zeros(max(n, 0) + 1, np.int64) if out_offsets else None
    fake = ctypes.c_void_p(0x2000)
    got = L.speechPlayer_synthesizeLongBatchDevice(sr, n, None if d_offsets is None else ctypes.c_void_p(d_offsets), fake, fake, fake, None,
                                                   0, None, 0, None, None, None if oo is None else oo.ctypes.data, 0, None, None, None,
                                                   None)
    return got, player.last_error()


@pytest.mark.parametrize("kw,msg", [
    (dict(d_offsets=None), "null offsets"),
    (dict(n=0), "numStreams"),
    (dict(out_offsets=False), "null outOffsets"),
    (dict(sr=0), "sampleRate"),
])
def test_argument_errors_need_no_device(kw, msg):
    got, err = _call(**kw)
    assert got == -1
    assert msg in err, err


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    offsets = np.array([0, 0], np.int64)
    out_offsets = np.zeros(2, np.int64)
    got = player.load_library().speechPlayer_synthesizeLongBatchDevice(22050, 1, offsets.ctypes.data, None, None, None, None, 0, None, 0,
                                                                       None, None, out_offsets.ctypes.data, 0, None, None, None, None)
    assert got == -1
    assert "no usable CUDA device" in player.last_error() and "no CPU fallback" in player.last_error()
