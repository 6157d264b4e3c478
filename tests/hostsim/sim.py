"""TEST INFRASTRUCTURE ONLY: ctypes access to the host build of the FP32 kernel arithmetic + parity metrics."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libhostsim.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-C", HERE], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(SO)
        vp = ctypes.c_void_p
        L.hostsim_render_f32.restype = ctypes.c_int
        L.hostsim_render_f32.argtypes = [ctypes.c_int, vp, vp, vp, vp, vp, ctypes.c_uint, ctypes.c_uint64, ctypes.c_uint64,
                                         ctypes.c_uint, vp, ctypes.c_uint, vp, ctypes.c_int, ctypes.c_uint, ctypes.c_uint, vp, vp,
                                         ctypes.c_uint64]
        L.hostsim_render_f32_cells.restype = ctypes.c_int
        L.hostsim_render_f32_cells.argtypes = [ctypes.c_int, vp, vp, vp, vp, vp, ctypes.c_uint, ctypes.c_uint64, ctypes.c_uint64,
                                               ctypes.c_uint, vp, ctypes.c_uint, ctypes.c_uint, vp, vp, ctypes.c_uint, vp, ctypes.c_uint64]
        _lib = L
    return _lib


def _replay_args(replay):
    if replay is None:
        return None, 0
    d = np.ascontiguousarray(replay, dtype=np.int32)
    return d.ctypes.data_as(ctypes.c_void_p), d.size


def render_f32_cells(sr, frames, min_dur, fade_dur, is_null=None, user_index=None, max_samples=None, seed=0, stream=0,
                     hold_ticks=128, fade_ticks=64, fade_max=0, replay=None):
    """The block scheduler's execution model on one stream: compact state, hold / fade / general cells.  Returns
    (pcm, last_index, [hold ticks, fade ticks, general ticks]).  replay: int32 draws instead of Philox noise (seed, stream)."""
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 47)
    m = np.ascontiguousarray(min_dur, dtype=np.uint32)
    f = np.ascontiguousarray(fade_dur, dtype=np.uint32)
    nul = None if is_null is None else np.ascontiguousarray(is_null, dtype=np.uint8)
    ux = None if user_index is None else np.ascontiguousarray(user_index, dtype=np.int32)
    if max_samples is None:
        mm = m.astype(np.int64)
        ff = np.maximum(f.astype(np.int64), 1)
        max_samples = int(np.maximum(mm + 1, ff + 2).sum()) + 16
    out = np.zeros(max_samples, dtype=np.int16)
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    li = ctypes.c_int32(0)
    used = (ctypes.c_uint32 * 3)()
    n = lib().hostsim_render_f32_cells(sr, ptr(frames), ptr(m), ptr(f), ptr(ux), ptr(nul), len(m), seed, stream, max_samples,
                                       ptr(out), hold_ticks, fade_ticks, used, ctypes.byref(li), fade_max, *_replay_args(replay))
    return out[:n], li.value, list(used)


def render_f32(sr, frames, min_dur, fade_dur, is_null=None, user_index=None, max_samples=None, seed=0, stream=0, chunk=0,
               planned=False, hold_ticks=0, gen_ticks=0, return_hold=False, replay=None):
    """planned=False: inline plans, one general pass per `chunk` ticks.  planned=True: precomputed plans and rounds of
    hold_ticks pure-hold / gen_ticks general chunks, as the batch engine schedules them.  replay: int32 draws instead of
    Philox noise (seed, stream)."""
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 47)
    m = np.ascontiguousarray(min_dur, dtype=np.uint32)
    f = np.ascontiguousarray(fade_dur, dtype=np.uint32)
    nul = None if is_null is None else np.ascontiguousarray(is_null, dtype=np.uint8)
    ux = None if user_index is None else np.ascontiguousarray(user_index, dtype=np.int32)
    if max_samples is None:
        mm = m.astype(np.int64)
        ff = np.maximum(f.astype(np.int64), 1)
        max_samples = int(np.maximum(mm + 1, ff + 2).sum()) + 16
    out = np.zeros(max_samples, dtype=np.int16)
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    li = ctypes.c_int32(0)
    hold = ctypes.c_uint32(0)
    n = lib().hostsim_render_f32(sr, ptr(frames), ptr(m), ptr(f), ptr(ux), ptr(nul), len(m), seed, stream, max_samples,
                                 ptr(out), chunk, ctypes.byref(li), int(bool(planned)), hold_ticks, gen_ticks,
                                 ctypes.byref(hold), *_replay_args(replay))
    if return_hold:
        return out[:n], li.value, hold.value
    return out[:n], li.value


def parity(got, want):
    """(fraction within 1 LSB, fraction exact, SNR dB, max |diff|)"""
    n = min(len(got), len(want))
    g = got[:n].astype(np.float64)
    w = want[:n].astype(np.float64)
    d = g - w
    sig = float((w * w).sum())
    err = float((d * d).sum())
    snr = float("inf") if err == 0 else 10 * np.log10(max(sig, 1e-30) / err)
    return float((np.abs(d) <= 1).mean()), float((d == 0).mean()), snr, float(np.abs(d).max())


class PullPlayer:
    """The low-latency pull path on the host: the product's request-level frame manager (pull_manager.h) driving a
    thread-by-thread emulation of klatt_pull_kernel.  Same surface as the players `scenarios.run_script` drives."""

    def __init__(self, sr, seed=0, stream=0, max_ticks=0, max_segs=0, phase_mode=1):
        L = lib()
        vp = ctypes.c_void_p
        L.hostsim_pull_create.restype = vp
        L.hostsim_pull_create.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64]
        L.hostsim_pull_destroy.argtypes = [vp]
        L.hostsim_pull_queue.argtypes = [vp, vp, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_int]
        L.hostsim_pull_last_index.restype = ctypes.c_int
        L.hostsim_pull_last_index.argtypes = [vp]
        L.hostsim_pull_synthesize.restype = ctypes.c_int
        L.hostsim_pull_synthesize.argtypes = [vp, ctypes.c_uint, vp, ctypes.c_uint, ctypes.c_uint]
        self.L = L
        L.hostsim_pull_phase_mode.argtypes = [vp, ctypes.c_int]
        self.h = L.hostsim_pull_create(sr, seed, stream)
        L.hostsim_pull_phase_mode(self.h, int(phase_mode))
        self.max_ticks, self.max_segs = max_ticks, max_segs

    def queue_frame(self, frame, min_dur, fade_dur, user_index=-1, purge=False):
        if frame is None:
            self.L.hostsim_pull_queue(self.h, None, int(min_dur), int(fade_dur), int(user_index), int(bool(purge)))
        else:
            fr = np.ascontiguousarray(frame, dtype=np.float64)
            assert fr.size == 47
            self.L.hostsim_pull_queue(self.h, fr.ctypes.data_as(ctypes.c_void_p), int(min_dur), int(fade_dur),
                                      int(user_index), int(bool(purge)))

    def synthesize(self, n):
        out = np.zeros(max(int(n), 1), dtype=np.int16)
        got = self.L.hostsim_pull_synthesize(self.h, int(n), out.ctypes.data_as(ctypes.c_void_p), self.max_ticks,
                                             self.max_segs)
        return out[:got]

    def last_index(self):
        return self.L.hostsim_pull_last_index(self.h)

    def close(self):
        if self.h:
            self.L.hostsim_pull_destroy(self.h)
            self.h = None


def pull_runs_stats():
    """(launches rendered with the run decomposition of the phase, special ticks in them) since the library was loaded"""
    a, b = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    lib().hostsim_pull_runs_stats(ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def phase(inc, pos0, mode):
    """The glottal-phase recurrence over an increment sequence (<= 8192 ticks): mode 0 the plain FP64 loop, mode 1 the run
    decomposition.  Returns (phase after every tick, carried phase, special ticks visited | -1 = handed back to the loop)."""
    L = lib()
    L.hostsim_phase.restype = ctypes.c_int
    L.hostsim_phase.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    inc = np.ascontiguousarray(inc, dtype=np.float64)
    out = np.empty_like(inc)
    carry = ctypes.c_double(0)
    visited = L.hostsim_phase(inc.ctypes.data, len(inc), float(pos0), int(mode), out.ctypes.data, ctypes.byref(carry))
    return out, carry.value, visited


def sin_turns(t):
    """sinTurns (the FP32 vibrato sine of every FP32 path) of float32 phases in turns, |t| <= 0.5"""
    L = lib()
    L.hostsim_sin_turns.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p]
    t = np.ascontiguousarray(t, dtype=np.float32)
    out = np.empty_like(t)
    L.hostsim_sin_turns(t.ctypes.data, len(t), out.ctypes.data)
    return out


def vibrato_depth(vibrato_pitch_offset):
    """what the FP32 paths multiply the vibrato sine by for a frame's vibratoPitchOffset"""
    L = lib()
    L.hostsim_vibrato_depth.restype = ctypes.c_double
    L.hostsim_vibrato_depth.argtypes = [ctypes.c_double]
    return L.hostsim_vibrato_depth(float(vibrato_pitch_offset))
