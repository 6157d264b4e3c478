"""CPU: minutes-long streams through the FP32 arithmetic (klatt_f32_core.cuh and klatt_pull_core.cuh compiled for the host
by tests/hostsim, test infrastructure only) against the reference restatement, held to a bar over the WHOLE stream.

The glottal phase is FP64 and exact per tick, but it is never reset: it integrates any constant pitch error for as long as a
player lives, and after minutes a sawtooth wrap lands on the neighbouring tick -- a full-scale impulse that rings through the
resonators for 10^2..10^3 samples.  The vibrato depth used to be such an error (rounded to FP32: up to 2^-24 relative for a
whole request), and so is the gain of the FP32 vibrato sine; short renders cannot see either.  The GPU kernels run the same streams in tests/test_gpu_long_streams.py."""
import numpy as np
import pytest

from nvspeechplayer_b200 import workloads
from tests import parity
from tests.hostsim import sim

P = workloads.P
SEED = 0xB200

# measured on the host build: 91.8 dB, max|d| 2 (57 samples at 2 LSB) over the 10-minute stream; FP32 depth: 60.8 dB, 1350
LONG_SNR_DB = 88.0
LONG_MAX_ABS = 2


def long_stream(sid, seconds, sr):
    fr, m, f, nul, ux = workloads.random_stream(sid, seconds, sr)
    return (fr, m, f, nul, ux), int(seconds * sr)


def pull_render(sr, q, n, seed, stream, pull=8192):
    """the NVDA pattern: one player for the whole session, every request queued, pulled `pull` samples at a time"""
    fr, m, f, nul, ux = q
    p = sim.PullPlayer(sr, seed=seed, stream=stream)
    try:
        for j in range(len(m)):
            p.queue_frame(None if nul[j] else fr[j], int(m[j]), int(f[j]), int(ux[j]))
        out, left = [], n
        while left > 0:
            c = p.synthesize(min(pull, left))
            assert len(c) > 0
            out.append(c)
            left -= len(c)
        return np.concatenate(out)
    finally:
        p.close()


def directed_stream(sr, seconds, speed=0.5, period_hi=55, period_lo=350):
    """A stream built to expose a constant error of the vibrato depth within seconds of audio.  Each request lasts half a
    cycle of a slow vibrato at full depth, high pitch while the vibrato raises the pitch and low while it lowers it, so a
    depth error moves the glottal phase the same way every cycle instead of averaging out.  Every depth sits 0.49 ulp below
    a float32 value (its FP32 rounding errs by the same sign in every request), and the pitches have whole-sample periods."""
    half = int(round(sr / (2 * speed)))
    n = int(np.ceil(seconds * sr / half)) + 1
    fr0 = workloads.random_stream(77, 1.0, sr)[0]
    fr = fr0[np.arange(n) % len(fr0)].copy()
    d32 = np.linspace(0.7, 0.99, n).astype(np.float32)
    fr[:, P["vibratoPitchOffset"]] = d32.astype(np.float64) - 0.49 * np.spacing(d32).astype(np.float64)
    fr[:, P["vibratoSpeed"]] = speed
    pitch = np.where(np.arange(n) % 2 == 0, sr / period_hi, sr / period_lo)
    fr[:, P["voicePitch"]] = pitch
    fr[:, P["endVoicePitch"]] = pitch
    for k in ("voiceAmplitude", "preFormantGain", "outputGain"):
        fr[:, P[k]] = 1.0
    m = np.full(n, half - 1, np.uint32)  # occupancy M + 1 = half a vibrato cycle
    f = np.full(n, int(0.005 * sr), np.uint32)
    return fr, m, f, np.zeros(n, np.uint8), np.arange(n, dtype=np.int32)


def test_batch_arithmetic_ten_minutes_at_44k(port):
    """The batch kernels' arithmetic on stream 424242: 10 minutes at 44.1 kHz in one render."""
    sr = 44100
    q, n = long_stream(424242, 600.0, sr)
    want = port.render(sr, *q, max_samples=n, noise=("philox", SEED, 424242))
    got, _ = sim.render_f32(sr, *q, max_samples=n, seed=SEED, stream=424242)
    parity.assert_whole_stream(got, want, "batch f32 10 min @44100", LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


def test_pull_renderer_ten_minutes_at_44k(port):
    """The same stream through the low-latency pull path (host frame manager + the pull kernel's passes), 8192 samples per
    pull.  Measured: 92.7 dB, max|d| 1."""
    sr = 44100
    q, n = long_stream(424242, 600.0, sr)
    want = port.render(sr, *q, max_samples=n, noise=("philox", SEED, 424242))
    got = pull_render(sr, q, n, SEED, 424242)
    parity.assert_whole_stream(got, want, "pull f32 10 min @44100", LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


@pytest.mark.parametrize("sr,sid,seconds", [(16000, 31337, 240.0), (22050, 8675309, 240.0)])
def test_batch_arithmetic_four_minutes(port, sr, sid, seconds):
    q, n = long_stream(sid, seconds, sr)
    want = port.render(sr, *q, max_samples=n, noise=("philox", SEED, sid))
    got, _ = sim.render_f32(sr, *q, max_samples=n, seed=SEED, stream=sid)
    parity.assert_whole_stream(got, want, "batch f32 %g s @%d" % (seconds, sr), LONG_MAX_ABS, LONG_SNR_DB, q[1], q[2])


def test_directed_vibrato_depth_stream(port):
    """30 s built so that a vibrato depth off by a constant fraction of an FP32 ulp moves wraps within seconds (an FP32 depth
    failed after 12.4 s: 48.5 dB, max|d| 1032).  Measured: 95.8 dB, max|d| 1, on the batch and the pull arithmetic."""
    sr, secs = 22050, 30.0
    q = directed_stream(sr, secs)
    n = int(secs * sr)
    want = port.render(sr, *q, max_samples=n, noise=("philox", 3, 1))
    got, _ = sim.render_f32(sr, *q, max_samples=n, seed=3, stream=1)
    parity.assert_whole_stream(got, want, "directed vibrato depth, batch", 1, 92.0, q[1], q[2])
    got = pull_render(sr, q, n, 3, 1)
    parity.assert_whole_stream(got, want, "directed vibrato depth, pull", 1, 92.0, q[1], q[2])


def test_vibrato_sine_has_the_reference_gain():
    """sinTurns times the depth the FP32 paths use has the amplitude of the reference's sin(2 pi t) * 0.06 * offset: a gain
    error of the vibrato's fundamental is a constant pitch error like a wrong depth.  (The FP32 coefficients of sinTurns make
    its fundamental 3.86e-8 too large; the depth divides that out.)"""
    t = (np.arange(-2 ** 22, 2 ** 22) / 2.0 ** 23).astype(np.float32)
    s = np.sin(2 * np.pi * t.astype(np.float64))
    q = sim.sin_turns(t).astype(np.float64)
    gain = float((q * s).sum() / (s * s).sum())
    assert abs(gain - 1) < 1e-7                                 # the sine itself: measured 3.86e-8
    assert abs(gain * sim.vibrato_depth(1.0) / 0.06 - 1) < 1e-10  # with the depth: measured 3e-13
    for v in (0.0, 0.3, 1.0, 0.123456789):
        assert sim.vibrato_depth(v) == pytest.approx(0.06 * v / gain, rel=1e-10, abs=0)
