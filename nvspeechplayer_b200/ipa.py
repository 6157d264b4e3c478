"""IPA text -> Klatt frame queues through the native bulk producer (include/speechPlayer_ipa.h).

Mirrors the caller-facing names of the reference's ipa.py (generateFramesAndTiming, reference ipa.py:336-353) so that a
script written against it runs unchanged, and adds the bulk form the batch engine wants: many utterances in one native
call, straight into the flat arrays of speechPlayer_batchSetFramesHost (no per-frame ctypes call, no Frame objects;
SURVEY.md section 8f rank 1).  The phoneme table is the numeric content of the reference's data.py
(nvspeechplayer_b200/data/phoneme_table.npz, written by tests/golden/make_golden.py)."""
import ctypes
from dataclasses import dataclass

import numpy as np

from . import player, workloads

_FLAG_BITS = {"_isNasal": 1, "_isStop": 2, "_isLiquid": 4, "_isVowel": 8, "_isVoiced": 16, "_isAfricate": 32,
              "_copyAdjacent": 64, "_isSemivowel": 128}
_table = None


def _lib():
    L = player.load_library()
    if not getattr(L, "_ipa_ready", False):
        vp = ctypes.c_void_p
        L.speechPlayer_ipaTableCreate.restype = vp
        L.speechPlayer_ipaTableCreate.argtypes = [vp, vp, vp, vp, ctypes.c_uint]
        L.speechPlayer_ipaTableDestroy.restype = None
        L.speechPlayer_ipaTableDestroy.argtypes = [vp]
        L.speechPlayer_ipaFrames.restype = ctypes.c_longlong
        L.speechPlayer_ipaFrames.argtypes = [vp, vp, ctypes.c_uint, vp, vp, vp, vp, ctypes.c_int, ctypes.c_double, vp, vp, vp, vp,
                                             vp, vp, vp, ctypes.c_ulonglong, ctypes.c_uint]
        L.speechPlayer_ipaFramesDevice.restype = ctypes.c_longlong
        L.speechPlayer_ipaFramesDevice.argtypes = [vp, vp, vp, ctypes.c_uint, vp, vp, vp, vp, ctypes.c_int, ctypes.c_double, vp, vp, vp,
                                                   vp, vp, vp, vp, vp, ctypes.c_ulonglong, vp]
        L._ipa_ready = True
    return L


def table():
    """The native phoneme table handle (created once from the shipped .npz)."""
    global _table
    if _table is None:
        t = workloads.phoneme_table()
        n = len(t["names"])
        keys = np.zeros((n, 3), dtype=np.uint32)
        for i, name in enumerate(t["names"]):
            cps = [ord(c) for c in name]
            keys[i, :len(cps)] = cps
        flags = np.zeros(n, dtype=np.uint32)
        for fname, bit in _FLAG_BITS.items():
            flags |= (np.asarray(t["flags"][fname]) != 0).astype(np.uint32) * np.uint32(bit)
        values = np.ascontiguousarray(t["table"], dtype=np.float64)
        present = np.ascontiguousarray(t["present"], dtype=np.uint8)
        h = _lib().speechPlayer_ipaTableCreate(keys.ctypes.data, values.ctypes.data, present.ctypes.data, flags.ctypes.data, n)
        if not h:
            raise player.EngineError(player.last_error())
        _table = h
    return _table


def _per_text(x, n, dtype=np.float64):
    if x is None:
        return None
    a = np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=dtype), (n,)))
    return a


def frames_for_texts(texts, speed=1, basePitch=100, inflection=0.5, clauseType=None, sample_rate=22050,
                     trailing_silence_ms=-1.0, stream_ids=None, threads=0, with_ms=False):
    """Many IPA clauses -> one workloads.FrameBatch (durations in samples at sample_rate), one stream per clause.
    speed / basePitch / inflection / clauseType: scalars or per-text sequences.  trailing_silence_ms >= 0 appends the
    NULL frame reference test_speakIpa.py:26 queues after each line."""
    L, t = _lib(), table()
    n = len(texts)
    enc = [s.encode("utf8") for s in texts]
    arr = (ctypes.c_char_p * max(n, 1))(*enc)
    sp, bp, inf = _per_text(speed, n), _per_text(basePitch, n), _per_text(inflection, n)
    ct = None
    if clauseType is not None:
        cl = [clauseType] * n if isinstance(clauseType, str) or clauseType is None else list(clauseType)
        ct = np.frombuffer(b"".join((c or ".").encode("ascii")[:1] for c in cl), dtype=np.uint8).copy()
    ptr = lambda a: None if a is None else a.ctypes.data
    offsets = np.zeros(n + 1, dtype=np.int64)
    # one native pass: a character yields at most three entries (aspiration, gap, phoneme), plus the trailing silence
    cap = max(3 * sum(len(s) for s in texts) + n, 1)
    frames = np.empty((cap, 47))
    m = np.empty(cap, dtype=np.uint32)
    f = np.empty(cap, dtype=np.uint32)
    nul = np.empty(cap, dtype=np.uint8)
    dms = np.empty(cap) if with_ms else None
    fms = np.empty(cap) if with_ms else None
    total = L.speechPlayer_ipaFrames(t, arr, n, ptr(sp), ptr(bp), ptr(inf), ptr(ct), sample_rate, float(trailing_silence_ms),
                                     offsets.ctypes.data, frames.ctypes.data, m.ctypes.data, f.ctypes.data, nul.ctypes.data,
                                     ptr(dms), ptr(fms), cap, threads)
    if total < 0 or total > cap:
        raise player.EngineError(player.last_error() or "frame capacity estimate too small")
    k = int(total)
    ids = np.arange(n, dtype=np.uint64) if stream_ids is None else np.asarray(stream_ids, dtype=np.uint64)
    fb = workloads.FrameBatch(sample_rate=sample_rate, offsets=offsets, frames=frames[:k], min_dur=m[:k], fade_dur=f[:k],
                              is_null=nul[:k], user_index=np.full(k, -1, dtype=np.int32), stream_ids=ids)
    return (fb, dms[:k], fms[:k]) if with_ms else fb


@dataclass
class DeviceFrameBatch:
    """The device counterpart of workloads.FrameBatch that frames_for_texts_device returns: torch tensors on one CUDA device.
    min_dur / fade_dur hold uint32 bits in int32 tensors, timeline_samples uint64 bits in an int64 tensor."""
    sample_rate: int
    offsets: object           # int64 [numStreams+1] into the flat arrays
    frames: object            # float64 [total, 47]
    min_dur: object           # int32 (uint32) [total], samples
    fade_dur: object          # int32 (uint32) [total], samples
    is_null: object           # uint8 [total]
    timeline_samples: object  # int64 (uint64) [numStreams]: samples each stream yields, sum of max(M+1, max(F,1)+2)
    text_offsets: object      # int64 [numTexts+1]: the frames of each text
    duration_ms: object = None  # float64 [total] (with_ms=True)
    fade_ms: object = None

    @property
    def num_streams(self):
        return self.offsets.numel() - 1


def _clause_bytes(clauseType, n):
    if clauseType is None:
        return None
    if isinstance(clauseType, (bytes, bytearray)) and len(clauseType) == n and n != 1:
        return np.frombuffer(bytes(clauseType), dtype=np.uint8).copy()
    cl = [clauseType] * n if isinstance(clauseType, (str, bytes)) else list(clauseType)
    enc = [(c if isinstance(c, bytes) else (c or ".").encode("ascii"))[:1] or b"." for c in cl]
    return np.frombuffer(b"".join(enc), dtype=np.uint8).copy()


def frames_for_texts_device(texts, speed=1, basePitch=100, inflection=0.5, clauseType=None, sample_rate=22050,
                            trailing_silence_ms=-1.0, stream_offsets=None, device=None, cuda_stream=None, with_ms=False):
    """frames_for_texts on the GPU (speechPlayer_ipaFramesDevice): the same frames, bit for bit, written in device memory;
    only the UTF-8 bytes and the per-text parameters are uploaded.  texts: str or bytes (a text ends at its first NUL).
    stream_offsets: text indices [numStreams+1]; stream s queues texts [stream_offsets[s], stream_offsets[s+1]) one after
    another (default: one stream per text).  device: CUDA device index (default: the current one); cuda_stream: a
    torch.cuda.Stream or raw handle (default: the device's current torch stream).  The rows are still being written on
    that stream when this returns, so work queued on it (Batch.set_frames_device) needs no synchronisation.
    Returns a DeviceFrameBatch."""
    import torch
    if not torch.cuda.is_available():
        raise player.EngineError("frames_for_texts_device: no usable CUDA device (there is no CPU fallback)")
    L, t = _lib(), table()
    n = len(texts)
    enc = [s if isinstance(s, (bytes, bytearray)) else s.encode("utf8") for s in texts]
    blob = b"".join(enc)
    toff = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, enc), dtype=np.int64, count=n), out=toff[1:])
    sp, bp, inf = _per_text(speed, n), _per_text(basePitch, n), _per_text(inflection, n)
    ct = _clause_bytes(clauseType, n)
    ptr = lambda a: None if a is None else a.ctypes.data
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev) if cuda_stream is None else cuda_stream
        handle = st.cuda_stream if hasattr(st, "cuda_stream") else st
        # one call: a code point yields at most two entries (a phoneme and either its post-stop aspiration or its
        # pre-stop gap; frames_for_texts allows three), plus the trailing silence
        chars = sum(len(s) for s in texts)
        cap = max(2 * chars + n, 1)
        i64 = dict(dtype=torch.int64, device=dev)
        text_offsets = torch.empty(n + 1, **i64)
        frames = torch.empty((cap, 47), dtype=torch.float64, device=dev)
        m = torch.empty(cap, dtype=torch.int32, device=dev)
        f = torch.empty(cap, dtype=torch.int32, device=dev)
        nul = torch.empty(cap, dtype=torch.uint8, device=dev)
        tl = torch.empty(max(n, 1), **i64)
        dms = torch.empty(cap, dtype=torch.float64, device=dev) if with_ms else None
        fms = torch.empty(cap, dtype=torch.float64, device=dev) if with_ms else None
        dp = lambda x: None if x is None else x.data_ptr()
        total = L.speechPlayer_ipaFramesDevice(t, blob, toff.ctypes.data, n, ptr(sp), ptr(bp), ptr(inf), ptr(ct), sample_rate,
                                               float(trailing_silence_ms), dp(text_offsets), dp(frames), dp(m), dp(f), dp(nul),
                                               dp(dms), dp(fms), dp(tl), cap, handle)
        if total < 0 or total > cap:
            raise player.EngineError(player.last_error() or "frame capacity estimate too small")
        k = int(total)
        tl = tl[:n]
        if stream_offsets is None:
            offsets, timeline = text_offsets, tl
        else:
            with torch.cuda.stream(st if isinstance(st, torch.cuda.Stream) else torch.cuda.ExternalStream(handle, device=dev)):
                so = torch.as_tensor(np.asarray(stream_offsets, dtype=np.int64)).to(dev)
                offsets = text_offsets[so]  # a stream's frames are its texts' frames, back to back
                cs = torch.cat([torch.zeros(1, **i64), torch.cumsum(tl, 0)])
                timeline = cs[so[1:]] - cs[so[:-1]]
    return DeviceFrameBatch(sample_rate=sample_rate, offsets=offsets, frames=frames[:k], min_dur=m[:k], fade_dur=f[:k], is_null=nul[:k],
                            timeline_samples=timeline, text_offsets=text_offsets, duration_ms=None if dms is None else dms[:k],
                            fade_ms=None if fms is None else fms[:k])


def generateFramesAndTiming(ipaText, speed=1, basePitch=100, inflection=0.5, clauseType=None):
    """Same generator as reference ipa.py:336-353: yields (Frame or None, durationMs, fadeMs)."""
    fb, dms, fms = frames_for_texts([ipaText], speed, basePitch, inflection, clauseType, with_ms=True)
    for j in range(len(dms)):
        if fb.is_null[j]:
            yield None, float(dms[j]), float(fms[j])
        else:
            fr = player.Frame()
            for name, v in zip(player.PARAM_NAMES, fb.frames[j]):
                setattr(fr, name, float(v))
            yield fr, float(dms[j]), float(fms[j])
