"""Noise draws for the replay tests: Philox4x32-10 in numpy, restated from nvspeechplayer_b200/csrc/philox.cuh.

Draw d of the Philox stream keyed (seed, stream) is word d & 3 of block d >> 2, shifted right by one (the reference's
rand() range).  The FP64 kernel draws word >> 1 and the FP32 paths use word >> 9, while a replayed draw reaches FP64 as is
and the FP32 paths as draw << 1.  So replaying these draws renders, on every path, exactly what Philox noise keyed
(seed, stream) renders.
"""
import numpy as np

from nvspeechplayer_b200.workloads import P

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters (c0..c3, uint32 arrays) under key (k0, k1) -> uint32 [n, 4]."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _LO for c in (c0, c1, c2, c3))
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & _LO,
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & _LO)
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def philox_draws(seed, stream, n):
    """The first n draws (int32, 0..2^31-1) of the Philox noise keyed (seed, stream); both keys are 64-bit."""
    blocks = np.arange((n + 3) // 4, dtype=np.uint64)
    w = philox4x32_10(blocks & _LO, blocks >> np.uint64(32), np.full_like(blocks, stream & 0xFFFFFFFF),
                      np.full_like(blocks, stream >> 32), seed & 0xFFFFFFFF, seed >> 32)
    return (w.reshape(-1)[:n] >> 1).astype(np.int32)


def noisy(frames, aspiration=0.3, frication=0.4, turbulence=0.2):
    """Frames with aspiration, frication (through the parallel bypass) and voice turbulence added, so that every noise draw
    reaches the output."""
    fr = np.array(frames, dtype=np.float64).reshape(-1, 47)
    fr[:, P["aspirationAmplitude"]] = aspiration
    fr[:, P["fricationAmplitude"]] = frication
    fr[:, P["parallelBypass"]] = np.maximum(fr[:, P["parallelBypass"]], 0.5)
    fr[:, P["voiceTurbulenceAmplitude"]] = turbulence
    return fr
