"""GPU: the device IPA producer (speechPlayer_ipaFramesDevice) is bit for bit the host producer (speechPlayer_ipaFrames),
which the CPU suite checks against fixtures made by the reference's own ipa.py.  Covers the fixtures themselves, a random
corpus of 10^5 texts at three sample rates, the rules' edge cases, partitions, the capacity contract, and text -> PCM on
the device against the host route."""
import os

import numpy as np
import pytest

from nvspeechplayer_b200 import ipa, player
from tests import ipa_corpus

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KEYS = ("frames", "min_dur", "fade_dur", "is_null", "duration_ms", "fade_ms")


def _np(db):
    """A DeviceFrameBatch as host arrays with the host producer's dtypes (floats compared through their int64 view)."""
    return dict(offsets=db.text_offsets.cpu().numpy(), frames=db.frames.cpu().numpy(), min_dur=db.min_dur.cpu().numpy().view(np.uint32),
                fade_dur=db.fade_dur.cpu().numpy().view(np.uint32), is_null=db.is_null.cpu().numpy(),
                duration_ms=db.duration_ms.cpu().numpy(), fade_ms=db.fade_ms.cpu().numpy(),
                timeline=db.timeline_samples.cpu().numpy().view(np.uint64))


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64) if a.dtype == np.float64 else a


def _assert_same(dev, host, what=""):
    np.testing.assert_array_equal(dev["offsets"], host["offsets"], err_msg=what + " offsets")
    for k in KEYS:
        assert dev[k].shape == host[k].shape, (what, k)
        np.testing.assert_array_equal(_bits(dev[k]), _bits(host[k]), err_msg="%s %s" % (what, k))


def _timeline(out):
    m = out["min_dur"].astype(np.int64)
    f = np.maximum(out["fade_dur"].astype(np.int64), 1)
    c = np.concatenate([[0], np.cumsum(np.maximum(m + 1, f + 2))])
    return (c[out["offsets"][1:]] - c[out["offsets"][:-1]]).astype(np.uint64)


def _both(texts, sp=None, bp=None, inf=None, cl=None, sample_rate=22050, trailing_silence_ms=-1.0):
    kw = dict(sample_rate=sample_rate, trailing_silence_ms=trailing_silence_ms)
    dev = _np(ipa.frames_for_texts_device(texts, speed=sp, basePitch=bp, inflection=inf, clauseType=cl, with_ms=True, **kw))
    host = ipa_corpus.host_frames(texts, sp, bp, inf, cl, **kw)
    return dev, host


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLDEN, "ipa_frames.npz"))


def test_golden_fixtures_bit_for_bit(gold):
    texts = [str(t) for t in gold["texts"]]
    clause = [str(c) or "." for c in gold["clause"]]
    db = ipa.frames_for_texts_device(texts, speed=gold["speed"], basePitch=gold["base_pitch"], inflection=gold["inflection"],
                                     clauseType=clause, sample_rate=16000, with_ms=True)
    d = _np(db)
    np.testing.assert_array_equal(d["offsets"], gold["offsets"])
    np.testing.assert_array_equal(_bits(d["frames"]), _bits(gold["frames"]))
    np.testing.assert_array_equal(_bits(d["duration_ms"]), _bits(gold["duration_ms"]))
    np.testing.assert_array_equal(_bits(d["fade_ms"]), _bits(gold["fade_ms"]))
    np.testing.assert_array_equal(d["is_null"], gold["is_null"])


def test_config1_queue_as_one_stream(gold, golden_config1):
    g = golden_config1
    lines = [str(t) for t in gold["texts"][:8]]
    db = ipa.frames_for_texts_device(lines, speed=0.6, sample_rate=int(g["sample_rate"]), trailing_silence_ms=150.0, stream_offsets=[0, 8])
    assert db.num_streams == 1
    assert db.offsets.cpu().tolist() == [0, len(g["is_null"])]
    np.testing.assert_array_equal(db.is_null.cpu().numpy(), g["is_null"])
    np.testing.assert_array_equal(db.min_dur.cpu().numpy().view(np.uint32), g["min_dur"])
    np.testing.assert_array_equal(db.fade_dur.cpu().numpy().view(np.uint32), g["fade_dur"])
    np.testing.assert_array_equal(_bits(db.frames.cpu().numpy()), _bits(g["frames"]))
    m = g["min_dur"].astype(np.int64)
    f = np.maximum(g["fade_dur"].astype(np.int64), 1)
    assert int(db.timeline_samples.cpu()[0]) == int(np.maximum(m + 1, f + 2).sum())


@pytest.mark.parametrize("sample_rate", [16000, 22050, 44100])
@pytest.mark.parametrize("trailing", [-1.0, 150.0])
def test_random_corpus_bitwise(sample_rate, trailing):
    texts, sp, bp, inf, cl = ipa_corpus.corpus(100000, seed=sample_rate + int(trailing))
    dev, host = _both(texts, sp, bp, inf, cl, sample_rate, trailing)
    assert len(host["is_null"]) > 10 ** 6
    _assert_same(dev, host, "corpus %d %g" % (sample_rate, trailing))
    np.testing.assert_array_equal(dev["timeline"], _timeline(host))


PITFALLS = [
    # _copyAdjacent: h beside h, h first / last / before a pre-stop gap, post-stop aspiration beside a copy-adjacent phoneme
    "hh", "hhh", "h", "hɑ", "ɑh", "hæh", "ɑht", "hkɑ", "ɑhp", "pha", "thɑ", "phhɑ", "kɦɑ", "ɑ h t", "ˈhɑ ˈhh",
    "tɑ phɑ", "sph", "ph", "hʔ", "ʔh",
    # tie bars and length marks at the end of a text, and pairs the table has or lacks
    "d͡ʒ", "t͡ʃɑ", "d͡", "ɑ͡", "͡", "͡ɑ", "ɑ͡ɪ", "t͡", "t͡s", "ɑː", "ː", "ɑːː", "iː", "ɑ͡ː", "t͡ʃː", "d͡ʒːɑ",
    # stress marks alone, at the end, doubled
    "ˈ", "ˌ", "ɑˈ", "ˈˌɑ", "ˈ ˈɑ",
    # long heads: many stressed syllables cycle the head steps
    " ".join(["ˈbɑ"] * 30), " ".join(["ˈpɑtə", "ˌkɑ", "ˈmɪn"] * 12), "ˈtɑ" * 25 + "ɑ",
]


@pytest.mark.parametrize("clause", [".", ",", "?", "!", "\0", "x"])
def test_rule_edge_cases(clause):
    texts = [s.encode() for s in PITFALLS]
    # UTF-8 edge cases: embedded NUL, empty, no phoneme at all, malformed and truncated sequences
    texts += [b"h\x00\xc3\xa6lou", b"\x00abc", b"", b"   ", b"xq1", b"\xff\xfe", b"\xc3", b"ba\xc3", b"ba\xe2\x80", b"\xc3ba",
              b"\xc0\x80b", b"t\xcd", b"t\xcd\xa1", b"b\xcb\x90", "ɑ".encode() + b"\xcb", "ˈ".encode()[:1] + b"ba"]
    n = len(texts)
    rng = np.random.default_rng(5)
    sp, bp, inf = rng.uniform(0.5, 2, n), rng.uniform(80, 200, n), rng.uniform(0, 1, n)
    dev, host = _both(texts, sp, bp, inf, clause.encode() * n, 22050, 150.0)
    _assert_same(dev, host, "clause %r" % clause)
    assert dev["offsets"][texts.index(b"") + 1] - dev["offsets"][texts.index(b"")] == 1  # the trailing silence only
    np.testing.assert_array_equal(dev["timeline"], _timeline(host))


def test_large_inputs():
    """One text of >= 10^5 code points beside short ones; there is no fixed per-thread list size."""
    rng = np.random.default_rng(11)
    ks = ipa_corpus.keys()
    long_text = b"".join(ipa_corpus.random_text(rng, ks, 60) for _ in range(5000))
    assert len(long_text.decode("utf8", "replace")) >= 10 ** 5
    texts = [b"h\xc3\xa6lou", long_text, ("ˈbɑ " * 40000).encode(), b"ba"]
    dev, host = _both(texts, np.array([1.0, 0.7, 1.3, 2.0]), None, np.array([0.5, 0.9, 0.1, 0.3]), b".?!,", 22050, 150.0)
    _assert_same(dev, host, "large")
    assert dev["offsets"][2] - dev["offsets"][1] > 10 ** 5


def test_partition_independence():
    texts, sp, bp, inf, cl = ipa_corpus.corpus(20000, seed=3)
    kw = dict(sample_rate=22050, trailing_silence_ms=150.0, with_ms=True)
    whole = _np(ipa.frames_for_texts_device(texts, speed=sp, basePitch=bp, inflection=inf, clauseType=cl, **kw))
    cuts = [0] + sorted(np.random.default_rng(4).choice(np.arange(1, 20000), 9, replace=False).tolist()) + [20000]
    parts = [_np(ipa.frames_for_texts_device(texts[a:b], speed=sp[a:b], basePitch=bp[a:b], inflection=inf[a:b], clauseType=cl[a:b], **kw))
             for a, b in zip(cuts[:-1], cuts[1:])]
    for k in KEYS + ("timeline",):
        np.testing.assert_array_equal(_bits(np.concatenate([p[k] for p in parts])), _bits(whole[k]), err_msg=k)
    offs = np.concatenate([[0]] + [p["offsets"][1:] + base for p, base in
                                   zip(parts, np.cumsum([0] + [p["offsets"][-1] for p in parts])[:-1])])
    np.testing.assert_array_equal(offs, whole["offsets"])


def test_capacity_contract():
    import torch
    L = ipa._lib()
    texts, sp, bp, inf, cl = ipa_corpus.corpus(300, seed=8)
    blob = b"".join(texts)
    toff = np.concatenate([[0], np.cumsum([len(t) for t in texts])]).astype(np.int64)
    n = len(texts)
    host = ipa_corpus.host_frames(texts, sp, bp, inf, cl, 22050, 150.0)
    total = int(host["offsets"][-1])
    dev = torch.device("cuda", 0)
    offs = torch.full((n + 1,), -7, dtype=torch.int64, device=dev)
    arrays = dict(frames=torch.full((total, 47), -3.0, dtype=torch.float64, device=dev), m=torch.full((total,), -5, dtype=torch.int32, device=dev),
                  f=torch.full((total,), -5, dtype=torch.int32, device=dev), nul=torch.full((total,), 9, dtype=torch.uint8, device=dev),
                  dms=torch.full((total,), -1.0, dtype=torch.float64, device=dev), fms=torch.full((total,), -1.0, dtype=torch.float64, device=dev),
                  tl=torch.full((n,), -9, dtype=torch.int64, device=dev))
    before = {k: v.clone() for k, v in arrays.items()}
    a = arrays
    args = lambda cap: (ipa.table(), blob, toff.ctypes.data, n, sp.ctypes.data, bp.ctypes.data, inf.ctypes.data, cl, 22050, 150.0, offs.data_ptr(),
                        a["frames"].data_ptr(), a["m"].data_ptr(), a["f"].data_ptr(), a["nul"].data_ptr(), a["dms"].data_ptr(),
                        a["fms"].data_ptr(), a["tl"].data_ptr(), cap, None)
    assert L.speechPlayer_ipaFramesDevice(*args(total - 1)) == total
    torch.cuda.synchronize()
    np.testing.assert_array_equal(offs.cpu().numpy(), host["offsets"])
    for k in arrays:
        assert torch.equal(arrays[k], before[k]), k
    assert L.speechPlayer_ipaFramesDevice(*args(total)) == total
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_bits(a["frames"].cpu().numpy()), _bits(host["frames"]))
    np.testing.assert_array_equal(a["nul"].cpu().numpy(), host["is_null"])
    tl = a["tl"].cpu().numpy().view(np.uint64)
    lib = player.load_library()
    for i in range(n):
        s, e = int(host["offsets"][i]), int(host["offsets"][i + 1])
        want = lib.speechPlayer_timelineSamples(host["min_dur"][s:].ctypes.data, host["fade_dur"][s:].ctypes.data, e - s)
        assert tl[i] == want, i
    # no outputs at all: a size query
    assert L.speechPlayer_ipaFramesDevice(ipa.table(), blob, toff.ctypes.data, n, None, None, None, None, 22050, 150.0, None, None, None,
                                          None, None, None, None, None, 0, None) == \
        int(ipa_corpus.host_frames(texts, sample_rate=22050, trailing_silence_ms=150.0)["offsets"][-1])


@pytest.mark.parametrize("precision", [player.PRECISION_FP32, player.PRECISION_FP64])
@pytest.mark.parametrize("voices", [False, True])
def test_text_to_pcm_on_the_device(gold, precision, voices):
    """ipaFramesDevice -> batchSetFramesDevice -> (batchApplyVoices) -> batchSynthesizeDevice on a non-default stream with no
    synchronisation in between, against frames_for_texts -> batchSetFramesHost."""
    import torch
    lines = [str(t) for t in gold["texts"][:8]]
    texts = [lines[i % 8] for i in range(96)]
    so = np.arange(0, 97, 3)  # 32 streams of three lines each
    sr, ns = 22050, 32
    va = np.full((2, 47), np.nan)
    va[1, 3] = 1200.0
    vm = np.ones((2, 47))
    vm[0, 5] = 1.1
    stream = torch.cuda.Stream()
    db = ipa.frames_for_texts_device(texts, speed=0.8, sample_rate=sr, trailing_silence_ms=150.0, stream_offsets=so, cuda_stream=stream)
    count = int(db.timeline_samples.max())
    with torch.cuda.stream(stream):
        out_dev = torch.zeros((ns, count), dtype=torch.int16, device="cuda")
    b = player.Batch(sr, ns, precision=precision, noise=player.NOISE_PHILOX, seed=0xB200)
    b.set_frames_device(db, cuda_stream=stream)
    if voices:
        b.apply_voices(va, vm, cuda_stream=stream.cuda_stream)
    b.synthesize_device(count, out_dev.data_ptr(), count, None, stream.cuda_stream)
    stream.synchronize()
    fb = ipa.frames_for_texts(texts, speed=0.8, sample_rate=sr, trailing_silence_ms=150.0)
    fb.offsets = fb.offsets[so]
    fb.stream_ids = np.arange(ns, dtype=np.uint64)
    np.testing.assert_array_equal(db.timeline_samples.cpu().numpy(), fb.timeline_samples())
    h = player.Batch(sr, ns, precision=precision, noise=player.NOISE_PHILOX, seed=0xB200)
    h.set_frames_host(fb)
    if voices:
        h.apply_voices(va, vm)
    want, _ = h.synthesize_host(count)
    np.testing.assert_array_equal(out_dev.cpu().numpy(), want)
    assert np.abs(want).max() > 1000
    b.close()
    h.close()
