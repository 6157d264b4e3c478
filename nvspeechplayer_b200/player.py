"""ctypes binding of libspeechPlayer.so -- the host-side mirror of the reference's Python interface.

``Frame`` and ``SpeechPlayer`` keep the names, argument meaning (durations in MILLISECONDS, converted with
``int(ms*(sampleRate/1000.0))``), return conventions (``synthesize`` -> ctypes short array with ``.length`` or
``None``) and error behaviour of the reference wrapper (reference speechPlayer.py:20-68), so code written against
it -- including the reference's own ipa.py frame pipeline -- runs unchanged.  ``Batch`` exposes the batched /
device-resident entry points of include/speechPlayer_batch.h.

The library is CUDA-only.  Loading fails loudly if it has not been built (``python -c "import
__graft_entry__ as g; g.build()"``); creating a player fails loudly without a CUDA device.
"""
import ctypes
import os

import numpy as np

from .workloads import NUM_PARAMS, PARAM_NAMES

PRECISION_FP64, PRECISION_FP32, PRECISION_STREAM = 0, 1, 2
NOISE_PHILOX, NOISE_GLIBC, NOISE_REPLAY = 0, 1, 2

_HERE = os.path.dirname(os.path.abspath(__file__))
# NVSP_LIB: an A/B build of the same library (tools/_variants/, csrc/Makefile LIB=...); never anything but this engine
LIB_PATH = os.environ.get("NVSP_LIB") or os.path.join(_HERE, "libspeechPlayer.so")
dllPath = os.path.join(_HERE, "speechPlayer.dll")  # the name the reference wrapper loads (speechPlayer.py:42)

speechPlayer_frameParam_t = ctypes.c_double


class Frame(ctypes.Structure):
    """speechPlayer_frame_t: 47 doubles in ABI order (reference src/frame.h:20-47)."""
    _fields_ = [(name, speechPlayer_frameParam_t) for name in PARAM_NAMES]


assert ctypes.sizeof(Frame) == 8 * NUM_PARAMS

_lib = None


def load_library():
    """Load libspeechPlayer.so and declare every prototype of include/speechPlayer.h and speechPlayer_batch.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(LIB_PATH + " is missing: the CUDA engine has not been built (run __graft_entry__.build()); "
                          "there is no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    vp, u32, i32, u64 = ctypes.c_void_p, ctypes.c_uint, ctypes.c_int, ctypes.c_uint64
    L.speechPlayer_initialize.restype = vp
    L.speechPlayer_initialize.argtypes = [i32]
    L.speechPlayer_initializeEx.restype = vp
    L.speechPlayer_initializeEx.argtypes = [i32, i32, i32, u64, u64]
    L.speechPlayer_queueFrame.restype = None
    L.speechPlayer_queueFrame.argtypes = [vp, vp, u32, u32, i32, ctypes.c_bool]
    L.speechPlayer_queueFrames.restype = i32
    L.speechPlayer_queueFrames.argtypes = [vp, vp, vp, vp, vp, vp, u32]
    L.speechPlayer_synthesize.restype = i32
    L.speechPlayer_synthesize.argtypes = [vp, u32, vp]
    L.speechPlayer_synthesizeBatch.restype = ctypes.c_longlong
    L.speechPlayer_synthesizeBatch.argtypes = [vp, u32, u32, vp, vp]
    L.speechPlayer_getLastIndex.restype = i32
    L.speechPlayer_getLastIndex.argtypes = [vp]
    L.speechPlayer_terminate.restype = None
    L.speechPlayer_terminate.argtypes = [vp]
    L.speechPlayer_setNoiseReplay.restype = i32
    L.speechPlayer_setNoiseReplay.argtypes = [vp, vp, ctypes.c_size_t]
    L.speechPlayer_seedNoise.restype = None
    L.speechPlayer_seedNoise.argtypes = [u32]
    L.speechPlayer_lastError.restype = ctypes.c_char_p
    L.speechPlayer_version.restype = ctypes.c_char_p
    L.speechPlayer_timelineSamples.restype = ctypes.c_ulonglong
    L.speechPlayer_timelineSamples.argtypes = [vp, vp, u32]
    L.speechPlayer_batchCreate.restype = vp
    L.speechPlayer_batchCreate.argtypes = [i32, u32, i32, i32, u64, vp]
    L.speechPlayer_batchDestroy.restype = None
    L.speechPlayer_batchDestroy.argtypes = [vp]
    L.speechPlayer_batchReset.restype = i32
    L.speechPlayer_batchReset.argtypes = [vp, vp]
    L.speechPlayer_batchSetFramesHost.restype = i32
    L.speechPlayer_batchSetFramesHost.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.speechPlayer_batchSetFramesDevice.restype = i32
    L.speechPlayer_batchSetFramesDevice.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.speechPlayer_batchApplyVoices.restype = i32
    L.speechPlayer_batchApplyVoices.argtypes = [vp, vp, vp, vp, u32, vp]
    L.speechPlayer_batchSetNoiseReplayDevice.restype = i32
    L.speechPlayer_batchSetNoiseReplayDevice.argtypes = [vp, vp, ctypes.c_size_t]
    L.speechPlayer_batchSynthesizeDevice.restype = i32
    L.speechPlayer_batchSynthesizeDevice.argtypes = [vp, u32, vp, ctypes.c_size_t, vp, vp]
    L.speechPlayer_batchSynthesizeHost.restype = ctypes.c_longlong
    L.speechPlayer_batchSynthesizeHost.argtypes = [vp, u32, vp, vp]
    L.speechPlayer_batchToFloat32Device.restype = i32
    L.speechPlayer_batchToFloat32Device.argtypes = [vp, ctypes.c_size_t, u32, u32, vp, ctypes.c_size_t, vp]
    L.speechPlayer_batchConcatenateDevice.restype = i32
    L.speechPlayer_batchConcatenateDevice.argtypes = [vp, ctypes.c_size_t, u32, u32, vp, vp, vp, vp]
    L.speechPlayer_batchGetLastIndices.restype = i32
    L.speechPlayer_batchGetLastIndices.argtypes = [vp, vp]
    L.speechPlayer_batchGetLaunchStats.restype = i32
    L.speechPlayer_batchGetLaunchStats.argtypes = [vp, vp, vp]
    L.speechPlayer_multiBatchCreate.restype = vp
    L.speechPlayer_multiBatchCreate.argtypes = [i32, u32, i32, i32, u64, vp, vp, u32]
    L.speechPlayer_multiBatchDestroy.restype = None
    L.speechPlayer_multiBatchDestroy.argtypes = [vp]
    L.speechPlayer_multiBatchSetFramesHost.restype = i32
    L.speechPlayer_multiBatchSetFramesHost.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.speechPlayer_multiBatchSynthesizeHost.restype = ctypes.c_longlong
    L.speechPlayer_multiBatchSynthesizeHost.argtypes = [vp, u32, vp, vp]
    L.speechPlayer_multiBatchGetShards.restype = i32
    L.speechPlayer_multiBatchGetShards.argtypes = [vp, vp]
    L.speechPlayer_multiBatchGetLastIndices.restype = i32
    L.speechPlayer_multiBatchGetLastIndices.argtypes = [vp, vp]
    L.speechPlayer_synthesizeLong.restype = ctypes.c_longlong
    L.speechPlayer_synthesizeLong.argtypes = [i32, vp, vp, vp, vp, u32, u64, u64, u32, vp, ctypes.c_ulonglong, i32, vp, vp]
    L.speechPlayer_synthesizeLongBatch.restype = ctypes.c_longlong
    L.speechPlayer_synthesizeLongBatch.argtypes = [i32, u32, vp, vp, vp, vp, vp, u64, vp, u32, vp, vp, vp, i32, vp, vp, vp]
    _lib = L
    return L


def last_error():
    return load_library().speechPlayer_lastError().decode()


class EngineError(RuntimeError):
    pass


def _check(rc, what):
    if rc is None or rc < 0:
        raise EngineError("%s failed: %s" % (what, last_error()))
    return rc


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class SpeechPlayer(object):
    """One reference player.  ``precision`` / ``noise`` default to the library's environment-driven defaults
    (FP64 parity arithmetic, process-global glibc-compatible noise: what a Linux build of the reference does)."""

    def __init__(self, sampleRate, precision=None, noise=None, seed=0xB200, streamId=0):
        self.sampleRate = sampleRate
        self._dll = load_library()
        if precision is None and noise is None:
            self._speechHandle = self._dll.speechPlayer_initialize(sampleRate)
        else:
            self._speechHandle = self._dll.speechPlayer_initializeEx(
                sampleRate, PRECISION_FP64 if precision is None else precision,
                NOISE_GLIBC if noise is None else noise, seed, streamId)
        if not self._speechHandle:
            raise EngineError("speechPlayer_initialize failed: " + last_error())

    # ---- the reference interface (speechPlayer.py:51-65) ----
    def queueFrame(self, frame, minFrameDuration, fadeDuration, userIndex=-1, purgeQueue=False):
        frame = ctypes.byref(frame) if frame else None
        self._dll.speechPlayer_queueFrame(self._speechHandle, frame, int(minFrameDuration * (self.sampleRate / 1000.0)),
                                          int(fadeDuration * (self.sampleRate / 1000.0)), userIndex, purgeQueue)

    def synthesize(self, numSamples):
        buf = (ctypes.c_short * numSamples)()
        res = self._dll.speechPlayer_synthesize(self._speechHandle, numSamples, buf)
        if res > 0:
            buf.length = min(res, len(buf))
            return buf
        if res < 0:
            raise EngineError("speechPlayer_synthesize failed: " + last_error())
        return None

    def getLastIndex(self):
        return self._dll.speechPlayer_getLastIndex(self._speechHandle)

    # ---- sample-unit / numpy conveniences used by the tests and the bench ----
    def queue_frame(self, frame, min_dur, fade_dur, user_index=-1, purge=False):
        """Durations in SAMPLES; frame is None or 47 doubles."""
        if frame is None:
            ptr = None
        else:
            buf = np.ascontiguousarray(frame, dtype=np.float64)
            assert buf.size == NUM_PARAMS
            ptr = buf.ctypes.data_as(ctypes.c_void_p)
        self._dll.speechPlayer_queueFrame(self._speechHandle, ptr, int(min_dur), int(fade_dur), int(user_index), bool(purge))

    def queue_frames(self, frames, min_dur, fade_dur, user_index=None, is_null=None):
        frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, NUM_PARAMS)
        m = np.ascontiguousarray(min_dur, dtype=np.uint32)
        f = np.ascontiguousarray(fade_dur, dtype=np.uint32)
        ux = None if user_index is None else np.ascontiguousarray(user_index, dtype=np.int32)
        nul = None if is_null is None else np.ascontiguousarray(is_null, dtype=np.uint8)
        _check(self._dll.speechPlayer_queueFrames(self._speechHandle, _ptr(frames), _ptr(m), _ptr(f), _ptr(ux), _ptr(nul),
                                                  len(m)), "speechPlayer_queueFrames")

    def synthesize_np(self, n):
        buf = np.zeros(n, dtype=np.int16)
        got = _check(self._dll.speechPlayer_synthesize(self._speechHandle, n, _ptr(buf)), "speechPlayer_synthesize")
        return buf[:got]

    def set_noise_replay(self, draws):
        d = np.ascontiguousarray(draws, dtype=np.int32)
        _check(self._dll.speechPlayer_setNoiseReplay(self._speechHandle, _ptr(d), d.size), "speechPlayer_setNoiseReplay")

    # aliases so test scripts can drive oracle players and engine players alike
    def last_index(self):
        return self.getLastIndex()

    def close(self):
        if getattr(self, "_speechHandle", None):
            self._dll.speechPlayer_terminate(self._speechHandle)
            self._speechHandle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def synthesize_batch(players, num_samples, out=None, written=None, handles=None):
    """speechPlayer_synthesizeBatch over a list of SpeechPlayer objects -> (int16 [n, num_samples], written[n]).
    A caller in a loop passes the arrays of its previous call back in (out, written, and handles = batch_handles(players))
    so that a call costs the library call alone, not fresh pages for the result."""
    L = load_library()
    n = len(players)
    if handles is None:
        handles = batch_handles(players)
    if out is None:
        out = np.zeros((n, num_samples), dtype=np.int16)
    if written is None:
        written = np.zeros(n, dtype=np.uint32)
    assert out.shape == (n, num_samples) and out.dtype == np.int16 and out.flags.c_contiguous
    _check(L.speechPlayer_synthesizeBatch(handles, n, num_samples, _ptr(out), _ptr(written)), "speechPlayer_synthesizeBatch")
    return out, written


def batch_handles(players):
    """The handle array speechPlayer_synthesizeBatch takes, for reuse across calls."""
    return (ctypes.c_void_p * len(players))(*[p._speechHandle for p in players])


def synthesize_long(sample_rate, frames, min_dur, fade_dur, is_null=None, seed=0xB200, stream_id=0, chunk_ticks=0,
                    max_samples=None, out=None, device_out=None):
    """speechPlayer_synthesizeLong: one pre-queued stream rendered with parallelism in time (kernel b).
    Returns (int16 samples, render_ms, kernel_launches); with device_out (a raw device address) the samples stay in
    HBM and the first element is the sample count."""
    L = load_library()
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, NUM_PARAMS)
    m = np.ascontiguousarray(min_dur, dtype=np.uint32)
    f = np.ascontiguousarray(fade_dur, dtype=np.uint32)
    nul = None if is_null is None else np.ascontiguousarray(is_null, dtype=np.uint8)
    if max_samples is None:
        mm, ff = m.astype(np.int64), np.maximum(f.astype(np.int64), 1)
        max_samples = int(np.maximum(mm + 1, ff + 2).sum())
    ms, launches = ctypes.c_double(0), ctypes.c_ulonglong(0)
    if device_out is not None:
        got = L.speechPlayer_synthesizeLong(sample_rate, _ptr(frames), _ptr(m), _ptr(f), _ptr(nul), len(m), seed, stream_id,
                                            chunk_ticks, device_out, max_samples, 1, ctypes.byref(ms), ctypes.byref(launches))
        _check(got, "speechPlayer_synthesizeLong")
        return got, ms.value, launches.value
    if out is None:
        out = np.zeros(max_samples, dtype=np.int16)
    got = L.speechPlayer_synthesizeLong(sample_rate, _ptr(frames), _ptr(m), _ptr(f), _ptr(nul), len(m), seed, stream_id,
                                        chunk_ticks, _ptr(out), max_samples, 0, ctypes.byref(ms), ctypes.byref(launches))
    _check(got, "speechPlayer_synthesizeLong")
    return out[:got], ms.value, launches.value


def synthesize_long_batch(fb, seed=0xB200, chunk_ticks=0, max_samples=None, device_out=None):
    """speechPlayer_synthesizeLongBatch: every stream of ``fb`` (a workloads.FrameBatch of whole, pre-queued queues) rendered
    with parallelism in time, all streams' chunks in one launch sequence.  Row s is what ``synthesize_long`` renders for
    stream s with noise stream ``fb.stream_ids[s]``.  ``max_samples``: None, one cap for all streams, or one per stream.
    Returns (packed int16 samples, out_offsets int64 [N+1], serial_phase uint8 [N], render_ms, kernel_launches); stream s is
    ``samples[out_offsets[s]:out_offsets[s+1]]`` (``split_rows``).  With ``device_out`` (a raw device address of at least
    ``long_batch_size(...)`` int16) the samples stay in HBM and the first element is the total sample count."""
    L = load_library()
    n = fb.num_streams
    offsets = np.ascontiguousarray(fb.offsets, dtype=np.int64)
    frames = np.ascontiguousarray(fb.frames, dtype=np.float64).reshape(-1, NUM_PARAMS)
    m = np.ascontiguousarray(fb.min_dur, dtype=np.uint32)
    f = np.ascontiguousarray(fb.fade_dur, dtype=np.uint32)
    nul = np.ascontiguousarray(fb.is_null, dtype=np.uint8)
    ids = np.ascontiguousarray(fb.stream_ids, dtype=np.uint64)
    caps = None if max_samples is None else np.ascontiguousarray(np.broadcast_to(np.asarray(max_samples, dtype=np.uint64), (n,)))
    out_offsets = np.zeros(n + 1, dtype=np.int64)
    serial = np.zeros(n, dtype=np.uint8)
    ms, launches = ctypes.c_double(0), ctypes.c_ulonglong(0)

    def call(out_ptr, on_device):
        return L.speechPlayer_synthesizeLongBatch(fb.sample_rate, n, _ptr(offsets), _ptr(frames), _ptr(m), _ptr(f), _ptr(nul), seed,
                                                  _ptr(ids), chunk_ticks, _ptr(caps), out_ptr, _ptr(out_offsets), on_device,
                                                  _ptr(serial), ctypes.byref(ms), ctypes.byref(launches))
    if device_out is not None:
        got = _check(call(device_out, 1), "speechPlayer_synthesizeLongBatch")
        return got, out_offsets, serial, ms.value, launches.value
    total = _check(call(None, 0), "speechPlayer_synthesizeLongBatch")
    out = np.zeros(max(total, 1), dtype=np.int16)
    got = _check(call(_ptr(out), 0), "speechPlayer_synthesizeLongBatch")
    return out[:got], out_offsets, serial, ms.value, launches.value


def long_batch_size(fb, max_samples=None):
    """(total samples, out_offsets) of synthesize_long_batch for ``fb``: a size query, no device needed."""
    L = load_library()
    n = fb.num_streams
    offsets = np.ascontiguousarray(fb.offsets, dtype=np.int64)
    m = np.ascontiguousarray(fb.min_dur, dtype=np.uint32)
    f = np.ascontiguousarray(fb.fade_dur, dtype=np.uint32)
    caps = None if max_samples is None else np.ascontiguousarray(np.broadcast_to(np.asarray(max_samples, dtype=np.uint64), (n,)))
    out_offsets = np.zeros(n + 1, dtype=np.int64)
    got = L.speechPlayer_synthesizeLongBatch(fb.sample_rate, n, _ptr(offsets), None, _ptr(m), _ptr(f), None, 0, None, 0, _ptr(caps),
                                             None, _ptr(out_offsets), 0, None, None, None)
    return _check(got, "speechPlayer_synthesizeLongBatch"), out_offsets


def split_rows(samples, out_offsets):
    """The packed output of synthesize_long_batch as one array (a view) per stream."""
    return [samples[int(out_offsets[s]):int(out_offsets[s + 1])] for s in range(len(out_offsets) - 1)]


class Batch(object):
    """N independent streams rendered by one launch (include/speechPlayer_batch.h)."""

    def __init__(self, sample_rate, num_streams, precision=PRECISION_FP32, noise=NOISE_PHILOX, seed=0xB200, stream_ids=None):
        self._L = load_library()
        self.sample_rate, self.num_streams, self.precision, self.noise = sample_rate, num_streams, precision, noise
        ids = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint64)
        assert ids is None or ids.size == num_streams
        self._h = self._L.speechPlayer_batchCreate(sample_rate, num_streams, precision, noise, seed, _ptr(ids))
        if not self._h:
            raise EngineError("speechPlayer_batchCreate failed: " + last_error())
        self._keep = None

    def reset(self, cuda_stream=None):
        _check(self._L.speechPlayer_batchReset(self._h, cuda_stream), "speechPlayer_batchReset")

    def set_frames_host(self, fb, cuda_stream=None):
        """fb: workloads.FrameBatch (host numpy arrays)."""
        assert fb.num_streams == self.num_streams
        off = np.ascontiguousarray(fb.offsets, dtype=np.int64)
        _check(self._L.speechPlayer_batchSetFramesHost(self._h, _ptr(off), _ptr(fb.frames), _ptr(fb.min_dur), _ptr(fb.fade_dur),
                                                       _ptr(fb.user_index), _ptr(fb.is_null), cuda_stream),
               "speechPlayer_batchSetFramesHost")

    def set_frames_device(self, d_offsets, d_frames, d_min, d_fade, d_user_index=None, d_is_null=None, cuda_stream=None):
        """Arguments are raw device addresses (ints), e.g. tensor.data_ptr()."""
        _check(self._L.speechPlayer_batchSetFramesDevice(self._h, d_offsets, d_frames, d_min, d_fade, d_user_index, d_is_null,
                                                         cuda_stream), "speechPlayer_batchSetFramesDevice")

    def apply_voices(self, voice_abs, voice_mul, voice_of_stream=None, cuda_stream=None):
        """Rewrite the queued frames with per-stream voices on the device (reference applyVoiceToFrame,
        nvdaAddon/synthDrivers/nvSpeechPlayer/__init__.py:117-125): value = abs if not NaN else frame; frame = value * mul.
        voice_abs / voice_mul: [numVoices][47] doubles; voice_of_stream: [numStreams] or None (stream s -> voice s % numVoices)."""
        va = np.ascontiguousarray(voice_abs, dtype=np.float64)
        vm = np.ascontiguousarray(voice_mul, dtype=np.float64)
        assert va.shape == vm.shape and va.ndim == 2 and va.shape[1] == 47
        vs = None if voice_of_stream is None else np.ascontiguousarray(voice_of_stream, dtype=np.uint32)
        assert vs is None or vs.shape == (self.num_streams,)
        _check(self._L.speechPlayer_batchApplyVoices(self._h, _ptr(va), _ptr(vm), None if vs is None else _ptr(vs), va.shape[0],
                                                     cuda_stream), "speechPlayer_batchApplyVoices")

    def set_noise_replay_device(self, d_draws, draws_per_stream):
        _check(self._L.speechPlayer_batchSetNoiseReplayDevice(self._h, d_draws, draws_per_stream),
               "speechPlayer_batchSetNoiseReplayDevice")

    def synthesize_device(self, num_samples, d_out, row_stride, d_written=None, cuda_stream=None):
        _check(self._L.speechPlayer_batchSynthesizeDevice(self._h, num_samples, d_out, row_stride, d_written, cuda_stream),
               "speechPlayer_batchSynthesizeDevice")

    def synthesize_host(self, num_samples, out=None):
        if out is None:
            out = np.zeros((self.num_streams, num_samples), dtype=np.int16)
        assert out.shape == (self.num_streams, num_samples) and out.dtype == np.int16 and out.flags.c_contiguous
        written = np.zeros(self.num_streams, dtype=np.uint32)
        _check(self._L.speechPlayer_batchSynthesizeHost(self._h, num_samples, _ptr(out), _ptr(written)),
               "speechPlayer_batchSynthesizeHost")
        return out, written

    def last_indices(self):
        out = np.zeros(self.num_streams, dtype=np.int32)
        _check(self._L.speechPlayer_batchGetLastIndices(self._h, _ptr(out)), "speechPlayer_batchGetLastIndices")
        return out

    def launch_stats(self):
        a, b = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        _check(self._L.speechPlayer_batchGetLaunchStats(self._h, ctypes.byref(a), ctypes.byref(b)), "launch stats")
        return a.value, b.value

    def close(self):
        if getattr(self, "_h", None):
            self._L.speechPlayer_batchDestroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiBatch(object):
    """N streams over several GPUs of one box, in-library (include/speechPlayer_batch.h speechPlayer_multiBatch*): contiguous
    stream ranges balanced by ticks, one host thread per device, no collective, one host buffer."""

    def __init__(self, sample_rate, num_streams, devices, precision=PRECISION_FP32, noise=NOISE_PHILOX, seed=0xB200, stream_ids=None):
        self._L = load_library()
        self.sample_rate, self.num_streams, self.devices = sample_rate, num_streams, list(devices)
        ids = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint64)
        dv = np.ascontiguousarray(self.devices, dtype=np.int32)
        self._h = self._L.speechPlayer_multiBatchCreate(sample_rate, num_streams, precision, noise, seed, _ptr(ids), _ptr(dv), len(dv))
        if not self._h:
            raise EngineError("speechPlayer_multiBatchCreate failed: " + last_error())

    def set_frames_host(self, fb):
        off = np.ascontiguousarray(fb.offsets, dtype=np.int64)
        _check(self._L.speechPlayer_multiBatchSetFramesHost(self._h, _ptr(off), _ptr(fb.frames), _ptr(fb.min_dur), _ptr(fb.fade_dur),
                                                            _ptr(fb.user_index), _ptr(fb.is_null)), "speechPlayer_multiBatchSetFramesHost")

    def synthesize_host(self, num_samples, out=None):
        if out is None:
            out = np.zeros((self.num_streams, num_samples), dtype=np.int16)
        written = np.zeros(self.num_streams, dtype=np.uint32)
        _check(self._L.speechPlayer_multiBatchSynthesizeHost(self._h, num_samples, _ptr(out), _ptr(written)),
               "speechPlayer_multiBatchSynthesizeHost")
        return out, written

    def shards(self):
        first = np.zeros(len(self.devices) + 1, dtype=np.uint32)
        _check(self._L.speechPlayer_multiBatchGetShards(self._h, _ptr(first)), "speechPlayer_multiBatchGetShards")
        return first

    def last_indices(self):
        out = np.zeros(self.num_streams, dtype=np.int32)
        _check(self._L.speechPlayer_multiBatchGetLastIndices(self._h, _ptr(out)), "speechPlayer_multiBatchGetLastIndices")
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._L.speechPlayer_multiBatchDestroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ----------------------------------------------------------------------------------------------
# Output sinks (SURVEY.md section 8f rank 4): what the reference's demo players do with the int16 buffers
# ----------------------------------------------------------------------------------------------
def to_float32_device(d_pcm, row_stride, num_streams, num_samples, d_out, out_stride, cuda_stream=None):
    """speechPlayer_batchToFloat32Device: int16 rows in HBM -> float32 rows in HBM (value / 32767.0, reference lavPlayer.py:17).
    Arguments are raw device addresses."""
    _check(load_library().speechPlayer_batchToFloat32Device(d_pcm, row_stride, num_streams, num_samples, d_out, out_stride, cuda_stream),
           "speechPlayer_batchToFloat32Device")


def concatenate_device(d_pcm, row_stride, num_streams, num_samples, d_written, d_offsets, d_packed, cuda_stream=None):
    """speechPlayer_batchConcatenateDevice: the ragged rows packed back to back in stream order, offsets = exclusive scan."""
    _check(load_library().speechPlayer_batchConcatenateDevice(d_pcm, row_stride, num_streams, num_samples, d_written, d_offsets,
                                                              d_packed, cuda_stream), "speechPlayer_batchConcatenateDevice")


def to_float32(pcm):
    """int16 -> float32 in [-1, 1] exactly as reference lavPlayer.py:17 feeds its audio graph (value / 32767.0)."""
    return (np.asarray(pcm, dtype=np.int16).astype(np.float64) / 32767.0).astype(np.float32)


def write_wav(path, pcm, sample_rate):
    """Mono 16-bit PCM WAV of one stream (1-D int16) or the concatenation of the rows of a batch (2-D, with a matching
    `written` handled by the caller slicing rows first)."""
    import wave
    data = np.ascontiguousarray(np.asarray(pcm, dtype=np.int16).reshape(-1))
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(int(sample_rate))
        w.writeframes(data.astype("<i2").tobytes())


def nvda_voice_tables(voices):
    """[(abs[47], mul[47])] tables for Batch.apply_voices from NVDA-style voice dicts ({'cb1_mul': 1.3, 'cf4': 3770, ...},
    reference nvdaAddon/synthDrivers/nvSpeechPlayer/__init__.py:86-115)."""
    names = [f[0] for f in Frame._fields_]
    va = np.full((len(voices), 47), np.nan)
    vm = np.ones((len(voices), 47))
    for i, v in enumerate(voices):
        for k, x in v.items():
            if k.endswith("_mul"):
                vm[i, names.index(k[:-4])] = x
            else:
                va[i, names.index(k)] = x
    return va, vm
