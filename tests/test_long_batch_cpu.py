"""CPU: speechPlayer_synthesizeLongBatch without a device -- the size query (out = NULL) follows the timeline law per
stream, caps and empty queues included, and every malformed argument is refused before any device is touched."""
import ctypes

import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads


def _lib():
    return player.load_library()


def _ragged():
    sr = 22050
    streams = [workloads.random_stream(11, 0.3, sr), workloads.random_stream(12, 1.0, sr)]
    empty = (np.zeros((0, 47)), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint8), np.zeros(0, np.int32))
    null_only = (np.zeros((2, 47)), np.array([100, 0], np.uint32), np.array([50, 30], np.uint32), np.ones(2, np.uint8),
                 np.zeros(2, np.int32))
    qs = [streams[0], empty, null_only, streams[1], empty]
    return workloads._concat(sr, qs, np.array([11, 0, 1, 12, 2], dtype=np.uint64))


def test_size_query_is_the_timeline_law():
    fb = _ragged()
    law = fb.timeline_samples()
    assert law[1] == 0 and law[4] == 0 and law[2] == 101 + 32
    total, off = player.long_batch_size(fb)
    assert total == law.sum()
    assert (np.diff(off) == law).all() and off[0] == 0


def test_size_query_with_caps():
    fb = _ragged()
    law = fb.timeline_samples()
    caps = np.array([1000, 5, 0, 10 ** 12, 7], dtype=np.uint64)
    total, off = player.long_batch_size(fb, max_samples=caps)
    want = np.minimum(law, caps.astype(np.int64))
    assert total == want.sum()
    assert (np.diff(off) == want).all()
    # one cap for every stream
    total, off = player.long_batch_size(fb, max_samples=40)
    assert (np.diff(off) == np.minimum(law, 40)).all()


def test_size_query_needs_no_device_and_touches_no_output_arguments():
    """out = NULL: serialPhase, renderMs and kernelLaunches are zeroed, nothing else happens"""
    fb = _ragged()
    L = _lib()
    n = fb.num_streams
    off = np.zeros(n + 1, np.int64)
    serial = np.full(n, 7, np.uint8)
    ms, launches = ctypes.c_double(5.0), ctypes.c_ulonglong(9)
    got = L.speechPlayer_synthesizeLongBatch(fb.sample_rate, n, fb.offsets.ctypes.data, fb.frames.ctypes.data, fb.min_dur.ctypes.data,
                                             fb.fade_dur.ctypes.data, fb.is_null.ctypes.data, 1, None, 0, None, None,
                                             off.ctypes.data, 0, serial.ctypes.data, ctypes.byref(ms), ctypes.byref(launches))
    assert got == fb.timeline_samples().sum() == off[-1]
    assert not serial.any() and ms.value == 0 and launches.value == 0


def _call(sr=22050, n=2, offsets=(0, 1, 2), m=(10, 10), f=(5, 5), out_offsets=True):
    L = _lib()
    offs = None if offsets is None else np.asarray(offsets, np.int64)
    mm = None if m is None else np.asarray(m, np.uint32)
    ff = None if f is None else np.asarray(f, np.uint32)
    oo = np.zeros(max(n, 0) + 1, np.int64) if out_offsets else None
    p = lambda a: None if a is None else a.ctypes.data
    got = L.speechPlayer_synthesizeLongBatch(sr, n, p(offs), None, p(mm), p(ff), None, 0, None, 0, None, None, p(oo), 0, None, None, None)
    return got, player.last_error()


@pytest.mark.parametrize("kw,msg", [
    (dict(sr=0), "sampleRate"),
    (dict(sr=-22050), "sampleRate"),
    (dict(n=0, offsets=(0,)), "numStreams"),
    (dict(offsets=None), "offsets"),
    (dict(out_offsets=False), "outOffsets"),
    (dict(offsets=(1, 1, 2)), "offsets[0]"),
    (dict(offsets=(0, 2, 1)), "non-decreasing"),
    (dict(m=None), "durations"),
    (dict(f=None), "durations"),
])
def test_malformed_arguments_are_refused(kw, msg):
    got, err = _call(**kw)
    assert got == -1
    assert msg in err, err


def test_empty_requests_need_no_durations():
    """a batch of empty queues renders nothing and needs no duration arrays"""
    got, err = _call(n=3, offsets=(0, 0, 0, 0), m=None, f=None)
    assert got == 0, err
