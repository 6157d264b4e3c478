"""TEST INFRASTRUCTURE ONLY (oracle/): ctypes harness around the two CPU oracles.

* ``RefLib``  -- the UNMODIFIED reference C++ compiled by ``oracle/Makefile`` into
  ``oracle/_ref/libspeechPlayer_ref{,_philox}.so`` (the five exports of
  ``src/speechPlayer.h:25-31``).  ``_philox`` has the reference's ``rand()`` bound to
  the per-stream Philox of ``oracle/philox.h``; the plain one uses glibc ``rand()``.
* ``PortLib`` -- the plain-C restatement ``oracle/klatt_oracle.c``.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs import this module.  The product never does.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
REF_SO = os.path.join(REF_DIR, "libspeechPlayer_ref.so")
REF_PHILOX_SO = os.path.join(REF_DIR, "libspeechPlayer_ref_philox.so")
PORT_SO = os.path.join(HERE, "libklatt_oracle.so")
# A checkout of the original NVSpeechPlayer to compile the reference from; the repository does not contain one, and what
# needs the reference itself (rather than the committed goldens rendered by it) skips without it.
REFERENCE = os.environ.get("NVSP_REFERENCE_DIR", "")
NUM_PARAMS = 47

NOISE_LIBC, NOISE_PHILOX, NOISE_REPLAY = 0, 1, 2


def build(reference=REFERENCE, quiet=True):
    """Compile the port always, and the reference .so files when the reference tree is present."""
    out = subprocess.DEVNULL if quiet else None
    subprocess.check_call(["make", "-C", HERE, "port"], stdout=out)
    if reference and os.path.isdir(os.path.join(reference, "src")):
        subprocess.check_call(["make", "-C", HERE, "ref", "REF=" + reference], stdout=out)
    return have_ref()


def have_ref():
    return os.path.exists(REF_SO) and os.path.exists(REF_PHILOX_SO)


def have_port():
    return os.path.exists(PORT_SO)


_libc = None


def libc():
    global _libc
    if _libc is None:
        _libc = ctypes.CDLL("libc.so.6")
        _libc.srand.argtypes = [ctypes.c_uint]
        _libc.rand.restype = ctypes.c_int
    return _libc


def libc_rand_sequence(seed, n):
    """n successive glibc rand() values after srand(seed) (RAND_MAX = 2^31-1)."""
    lc = libc()
    lc.srand(seed)
    out = np.empty(n, dtype=np.int32)
    r = lc.rand
    for i in range(n):
        out[i] = r()
    return out


class RefLib:
    """The compiled reference, driven through explicit prototypes (the reference's own wrapper leaves restype unset)."""

    def __init__(self, philox=False):
        path = REF_PHILOX_SO if philox else REF_SO
        if not os.path.exists(path):
            raise FileNotFoundError(path + " missing: run `make -C oracle ref REF=<NVSpeechPlayer checkout>`")
        self.philox = philox
        L = self.lib = ctypes.CDLL(path)
        L.speechPlayer_initialize.restype = ctypes.c_void_p
        L.speechPlayer_initialize.argtypes = [ctypes.c_int]
        L.speechPlayer_queueFrame.restype = None
        L.speechPlayer_queueFrame.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint,
                                              ctypes.c_int, ctypes.c_bool]
        L.speechPlayer_synthesize.restype = ctypes.c_int
        L.speechPlayer_synthesize.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p]
        L.speechPlayer_getLastIndex.restype = ctypes.c_int
        L.speechPlayer_getLastIndex.argtypes = [ctypes.c_void_p]
        L.speechPlayer_terminate.restype = None
        L.speechPlayer_terminate.argtypes = [ctypes.c_void_p]
        if philox:
            L.oracle_noise_seed.restype = None
            L.oracle_noise_seed.argtypes = [ctypes.c_uint64, ctypes.c_uint64]
            L.oracle_noise_ndraws.restype = ctypes.c_uint64

    def seed(self, seed, stream=0):
        """Philox build: key the next stream.  Plain build: srand(seed) (process-global, one stream at a time)."""
        if self.philox:
            self.lib.oracle_noise_seed(seed, stream)
        else:
            libc().srand(seed)

    def player(self, sample_rate):
        return RefPlayer(self, sample_rate)

    def render(self, sample_rate, frames, min_dur, fade_dur, is_null=None, user_index=None, max_samples=None,
               seed=1, stream=0):
        """Queue every frame up front, then synthesize until the queue drains. Returns int16 array."""
        frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, NUM_PARAMS)
        n = len(min_dur)
        if max_samples is None:
            max_samples = timeline_samples(min_dur, fade_dur) + 16
        self.seed(seed, stream)
        p = self.player(sample_rate)
        for j in range(n):
            null = bool(is_null[j]) if is_null is not None else False
            p.queue_frame(None if null else frames[j], int(min_dur[j]), int(fade_dur[j]),
                          -1 if user_index is None else int(user_index[j]))
        out = p.synthesize(max_samples)
        p.close()
        return out


class RefPlayer:
    def __init__(self, lib, sample_rate):
        self._L = lib.lib
        self.h = self._L.speechPlayer_initialize(sample_rate)

    def queue_frame(self, frame, min_dur, fade_dur, user_index=-1, purge=False):
        """Durations in SAMPLES (the C side's unit, src/speechPlayer.h:28)."""
        if frame is None:
            ptr = None
        else:
            buf = np.ascontiguousarray(frame, dtype=np.float64)
            assert buf.size == NUM_PARAMS
            ptr = buf.ctypes.data_as(ctypes.c_void_p)
        self._L.speechPlayer_queueFrame(self.h, ptr, min_dur, fade_dur, user_index, purge)

    def synthesize(self, n):
        buf = np.zeros(n, dtype=np.int16)
        got = self._L.speechPlayer_synthesize(self.h, n, buf.ctypes.data_as(ctypes.c_void_p))
        return buf[:max(got, 0)]

    def last_index(self):
        return self._L.speechPlayer_getLastIndex(self.h)

    def close(self):
        if self.h:
            self._L.speechPlayer_terminate(self.h)
            self.h = None


class PortLib:
    def __init__(self):
        if not os.path.exists(PORT_SO):
            raise FileNotFoundError(PORT_SO + " missing: run `make -C oracle port`")
        L = self.lib = ctypes.CDLL(PORT_SO)
        vp, u64, u32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint
        L.klatt_oracle_create.restype = vp
        L.klatt_oracle_create.argtypes = [ctypes.c_int]
        L.klatt_oracle_destroy.argtypes = [vp]
        L.klatt_oracle_noise_libc.argtypes = [vp]
        L.klatt_oracle_noise_philox.argtypes = [vp, u64, u64]
        L.klatt_oracle_noise_replay.argtypes = [vp, vp, ctypes.c_size_t]
        L.klatt_oracle_queue_frame.argtypes = [vp, vp, u32, u32, ctypes.c_int, ctypes.c_int]
        L.klatt_oracle_synthesize.restype = ctypes.c_int
        L.klatt_oracle_synthesize.argtypes = [vp, u32, vp]
        L.klatt_oracle_get_last_index.restype = ctypes.c_int
        L.klatt_oracle_get_last_index.argtypes = [vp]
        for name in ("klatt_oracle_ticks", "klatt_oracle_fade_ticks", "klatt_oracle_draws"):
            getattr(L, name).restype = u64
            getattr(L, name).argtypes = [vp]
        L.klatt_oracle_render.restype = ctypes.c_int
        L.klatt_oracle_render.argtypes = [ctypes.c_int, vp, vp, vp, vp, vp, u32, ctypes.c_int, u64, u64, vp,
                                          ctypes.c_size_t, u32, vp, vp]

    def player(self, sample_rate):
        return PortPlayer(self, sample_rate)

    def render(self, sample_rate, frames, min_dur, fade_dur, is_null=None, user_index=None, max_samples=None,
               noise=("philox", 0, 0), return_phi=False):
        """noise: ("libc",) | ("philox", seed, stream) | ("replay", int32 array)."""
        frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, NUM_PARAMS)
        n = len(min_dur)
        min_dur = np.ascontiguousarray(min_dur, dtype=np.uint32)
        fade_dur = np.ascontiguousarray(fade_dur, dtype=np.uint32)
        nul = None if is_null is None else np.ascontiguousarray(is_null, dtype=np.uint8)
        uix = None if user_index is None else np.ascontiguousarray(user_index, dtype=np.int32)
        if max_samples is None:
            max_samples = timeline_samples(min_dur, fade_dur) + 16
        out = np.zeros(max_samples, dtype=np.int16)
        mode, seed, stream, draws = NOISE_LIBC, 0, 0, None
        if noise[0] == "philox":
            mode, seed, stream = NOISE_PHILOX, noise[1], noise[2]
        elif noise[0] == "replay":
            mode, draws = NOISE_REPLAY, np.ascontiguousarray(noise[1], dtype=np.int32)
        fade_ticks = ctypes.c_uint64(0)
        ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
        got = self.lib.klatt_oracle_render(sample_rate, ptr(frames), ptr(min_dur), ptr(fade_dur), ptr(uix), ptr(nul),
                                           n, mode, seed, stream, ptr(draws), 0 if draws is None else draws.size,
                                           max_samples, ptr(out), ctypes.byref(fade_ticks))
        res = out[:max(got, 0)]
        if return_phi:
            return res, (fade_ticks.value / max(got, 1))
        return res


class PortPlayer:
    def __init__(self, lib, sample_rate):
        self._L = lib.lib
        self.h = self._L.klatt_oracle_create(sample_rate)
        self._keep = None

    def noise_libc(self):
        self._L.klatt_oracle_noise_libc(self.h)

    def noise_philox(self, seed, stream):
        self._L.klatt_oracle_noise_philox(self.h, seed, stream)

    def noise_replay(self, draws):
        self._keep = np.ascontiguousarray(draws, dtype=np.int32)
        self._L.klatt_oracle_noise_replay(self.h, self._keep.ctypes.data_as(ctypes.c_void_p), self._keep.size)

    def queue_frame(self, frame, min_dur, fade_dur, user_index=-1, purge=False):
        if frame is None:
            ptr = None
        else:
            buf = np.ascontiguousarray(frame, dtype=np.float64)
            assert buf.size == NUM_PARAMS
            ptr = buf.ctypes.data_as(ctypes.c_void_p)
        self._L.klatt_oracle_queue_frame(self.h, ptr, min_dur, fade_dur, user_index, int(purge))

    def synthesize(self, n):
        buf = np.zeros(n, dtype=np.int16)
        got = self._L.klatt_oracle_synthesize(self.h, n, buf.ctypes.data_as(ctypes.c_void_p))
        return buf[:max(got, 0)]

    def last_index(self):
        return self._L.klatt_oracle_get_last_index(self.h)

    def phi(self):
        t = self._L.klatt_oracle_ticks(self.h)
        return self._L.klatt_oracle_fade_ticks(self.h) / max(t, 1)

    def close(self):
        if self.h:
            self._L.klatt_oracle_destroy(self.h)
            self.h = None


def timeline_samples(min_dur, fade_dur):
    """Samples a fully pre-queued stream yields: sum_j max(M_j+1, max(F_j,1)+2)  (SURVEY.md 3.3.1 law)."""
    m = np.asarray(min_dur, dtype=np.int64)
    f = np.maximum(np.asarray(fade_dur, dtype=np.int64), 1)
    return int(np.maximum(m + 1, f + 2).sum())
