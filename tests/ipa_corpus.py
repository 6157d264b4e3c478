"""Seeded random IPA corpus for the producer tests: texts as UTF-8 bytes that mix the phoneme table's keys, stress marks, tie
bars, length marks, blanks, characters that are not phonemes and invalid or truncated UTF-8, with per-text speed, pitch,
inflection and clause type (including 0 and characters that are not clause types)."""
import ctypes

import numpy as np

from nvspeechplayer_b200 import ipa, player, workloads

STRESS = ["ˈ", "ˌ"]
TIE, LONG = "͡", "ː"
OTHER = ["x", "q", "1", ",", ".", "é", "ɑ̃", "—", "\U0001f600"]
BAD = [b"\xff", b"\xc3", b"\xe2\x80", b"\xc0\x80", b"\x80", b"\xf0\x9f\x98", b"\xed\xa0\x80"]
CLAUSES = [b".", b",", b"?", b"!", b"\x00", b"x", b";"]


def keys():
    return [str(n) for n in workloads.phoneme_table()["names"]]


def random_text(rng, ks, max_len=40):
    """One text as bytes."""
    parts = []
    for _ in range(int(rng.integers(0, max_len + 1))):
        r = rng.random()
        if r < 0.55:
            k = ks[int(rng.integers(len(ks)))]
            if len(k) > 1 and rng.random() < 0.5:  # a key's first code point alone, then maybe a tie / length mark
                k = k[0]
            parts.append(k.encode())
        elif r < 0.65:
            parts.append(STRESS[int(rng.integers(2))].encode())
        elif r < 0.72:
            parts.append(TIE.encode())
        elif r < 0.79:
            parts.append(LONG.encode())
        elif r < 0.90:
            parts.append(b" ")
        elif r < 0.96:
            parts.append(OTHER[int(rng.integers(len(OTHER)))].encode())
        else:
            parts.append(BAD[int(rng.integers(len(BAD)))])
    return b"".join(parts)


def corpus(n, seed=1234, max_len=40):
    """n texts (bytes) and per-text speed, basePitch, inflection (float64) and clause type (bytes of length n)."""
    rng = np.random.default_rng(seed)
    ks = keys()
    texts = [random_text(rng, ks, max_len) for _ in range(n)]
    speed = rng.uniform(0.3, 2.5, n)
    base_pitch = rng.uniform(60.0, 300.0, n)
    inflection = np.round(rng.uniform(0.0, 1.0, n), 2)
    clause = b"".join(CLAUSES[i] for i in rng.integers(0, len(CLAUSES), n))
    return texts, speed, base_pitch, inflection, clause


def host_frames(texts, speed=None, base_pitch=None, inflection=None, clause=None, sample_rate=22050, trailing_silence_ms=-1.0,
                threads=0, lib=None, table=None):
    """speechPlayer_ipaFrames over byte texts (each ends at its first NUL, as a C string does): a dict of every output array."""
    L = lib or ipa._lib()
    t = table or ipa.table()
    n = len(texts)
    arr = (ctypes.c_char_p * max(n, 1))(*texts)
    ptr = lambda a: None if a is None else np.ascontiguousarray(a).ctypes.data
    keep = [None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (speed, base_pitch, inflection)]
    ct = None if clause is None else np.frombuffer(clause, dtype=np.uint8).copy()
    cap = max(2 * sum(len(s) for s in texts) + n, 1)
    out = dict(offsets=np.zeros(n + 1, np.int64), frames=np.empty((cap, 47)), min_dur=np.empty(cap, np.uint32),
               fade_dur=np.empty(cap, np.uint32), is_null=np.empty(cap, np.uint8), duration_ms=np.empty(cap), fade_ms=np.empty(cap))
    total = L.speechPlayer_ipaFrames(t, arr, n, ptr(keep[0]), ptr(keep[1]), ptr(keep[2]), ptr(ct), sample_rate, float(trailing_silence_ms),
                                     out["offsets"].ctypes.data, out["frames"].ctypes.data, out["min_dur"].ctypes.data,
                                     out["fade_dur"].ctypes.data, out["is_null"].ctypes.data, out["duration_ms"].ctypes.data,
                                     out["fade_ms"].ctypes.data, cap, threads)
    if total < 0:
        raise player.EngineError(player.last_error())
    assert total <= cap
    for k in ("frames", "min_dur", "fade_dur", "is_null", "duration_ms", "fade_ms"):
        out[k] = out[k][:total]
    return out
