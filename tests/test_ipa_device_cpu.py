"""CPU: speechPlayer_ipaFramesDevice's argument checks (no device needed), no CPU fallback without a device, and the pitch
factors the host precomputes (ipa_core.h ipaPercents) covering every percent the rules produce over a random corpus."""
import ctypes

import numpy as np
import pytest

from nvspeechplayer_b200 import ipa, player
from tests import ipa_corpus


def _call(table, text, toff, n, sample_rate=22050, d_min=None):
    L = ipa._lib()
    return L.speechPlayer_ipaFramesDevice(table, text, None if toff is None else toff.ctypes.data, n, None, None, None, None,
                                          sample_rate, -1.0, None, None, d_min, None, None, None, None, None, 0, None)


def test_argument_errors_need_no_device():
    t = ipa.table()
    toff = np.array([0, 3], dtype=np.int64)
    cases = [
        (dict(table=None, text=b"abc", toff=toff, n=1), b"null table"),
        (dict(table=t, text=None, toff=toff, n=1), b"null text"),
        (dict(table=t, text=b"abc", toff=None, n=1), b"null text"),
        (dict(table=t, text=b"abcdef", toff=np.array([0, 4, 2], dtype=np.int64), n=2), b"decrease"),
        (dict(table=t, text=b"abc", toff=toff, n=1, sample_rate=0, d_min=ctypes.c_void_p(0x1000)), b"sampleRate"),
    ]
    for kw, msg in cases:
        assert _call(**kw) == -1, kw
        assert msg in player.load_library().speechPlayer_lastError(), (kw, player.last_error())


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    toff = np.array([0, 5], dtype=np.int64)
    assert _call(ipa.table(), "hælou".encode()[:5], toff, 1) == -1
    assert b"CUDA" in player.load_library().speechPlayer_lastError()
    with pytest.raises(player.EngineError):
        ipa.frames_for_texts_device(["hælou"])


def test_random_corpus_has_no_pitch_factor_miss():
    """The host producer uses the same factor look-up as the device: a percent without a factor would make it return -1."""
    texts, sp, bp, inf, cl = ipa_corpus.corpus(100000, seed=99)
    # many distinct inflections (one factor row each) and long heads with many stressed syllables, every clause type
    texts += [("ˈbɑ " * k + "ˌtɑ ˈpæ").encode() for k in range(1, 40)] * 4
    extra = len(texts) - len(sp)
    sp = np.concatenate([sp, np.ones(extra)])
    bp = np.concatenate([bp, np.full(extra, 100.0)])
    inf = np.concatenate([inf, np.linspace(0.0, 2.0, extra)])
    cl += b"".join([b".", b",", b"?", b"!"][i % 4] for i in range(extra))
    out = ipa_corpus.host_frames(texts, sp, bp, inf, cl, sample_rate=22050, trailing_silence_ms=150.0)
    assert out["offsets"][-1] == len(out["is_null"]) > 10 ** 6
    voiced = out["is_null"] == 0
    assert np.isfinite(out["frames"][voiced][:, [0, 46]]).all()
