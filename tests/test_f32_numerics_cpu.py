"""CPU: the FP32 production ARITHMETIC (klatt_f32_core.cuh compiled for the host by tests/hostsim, test
infrastructure only) against the reference restatement.  This pins the numerics of the formulation (delta-form
resonators, pole recurrences, FP64 phase) in the CPU-only container; the CUDA kernel itself is checked by
tests/test_gpu_parity_f32.py on the B200."""
import numpy as np
import pytest

from nvspeechplayer_b200 import workloads
from tests import parity, scenarios
from tests.hostsim import sim
from tests.noise import noisy, philox_draws


def test_config1_f32_arithmetic(port, golden_config1):
    g = golden_config1
    got, _ = sim.render_f32(int(g["sample_rate"]), g["frames"], g["min_dur"], g["fade_dur"], g["is_null"],
                            seed=int(g["philox_seed"]), stream=int(g["philox_stream"]))
    w1, exact, snr, mx = parity.assert_f32_parity(got, g["pcm_philox"], "config1")
    assert w1 >= 0.9999 and snr >= 90.0   # measured: 100 % / 96.5 dB


@pytest.mark.parametrize("sr,within,snr", [(16000, 0.9999, 85.0), (22050, 0.9999, 85.0), (44100, 0.9999, 85.0)])
def test_random_frames_f32_arithmetic(port, sr, within, snr):
    fr, m, f, nul, ux = workloads.random_stream(4242, 3.0, sr)
    n = int(3.0 * sr)
    want = port.render(sr, fr, m, f, nul, ux, max_samples=n, noise=("philox", 9, 4242))
    got, li = sim.render_f32(sr, fr, m, f, nul, ux, max_samples=n, seed=9, stream=4242)
    parity.assert_f32_parity(got, want, "random@%d" % sr, within=within, snr_db=snr)


def test_chunked_equals_one_shot_bitwise():
    """State save/restore between launches is exact: any chunking renders the same int16."""
    sr = 22050
    fr, m, f, nul, ux = workloads.random_stream(7, 1.0, sr)
    n = int(1.0 * sr)
    one, _ = sim.render_f32(sr, fr, m, f, nul, ux, max_samples=n, seed=1, stream=7)
    for chunk in (1, 7, 777, 8192):
        part, _ = sim.render_f32(sr, fr, m, f, nul, ux, max_samples=n, seed=1, stream=7, chunk=chunk)
        np.testing.assert_array_equal(part, one)


def test_counts_and_user_index_follow_the_timeline_law():
    sr = 22050
    fr, m, f, nul, ux = workloads.random_stream(11, 0.5, sr)
    got, li = sim.render_f32(sr, fr, m, f, nul, ux, seed=1, stream=11)
    assert len(got) == workloads._concat(sr, [(fr, m, f, nul, ux)], [11]).timeline_samples()[0]
    assert li == ux[-1]


def test_long_fades_do_not_drift(port):
    """config 2 recipe: 400 ms fades (6400 ticks at 16 kHz) -- the per-tick pole recurrence alone drifts to ~70 dB
    here; with the 64-tick re-basing it stays within 1 LSB everywhere."""
    fb = workloads.vowel_chart(1, pairs=6)
    for s in range(fb.num_streams):
        fr, m, f, nul, ux = fb.stream(s)
        want = port.render(16000, fr, m, f, nul, ux, noise=("philox", 8, s))
        got, _ = sim.render_f32(16000, fr, m, f, nul, ux, seed=8, stream=s)
        w1, exact, snr, mx = parity.assert_f32_parity(got, want, "vowel pair %d" % s)
        assert mx <= 1 and snr >= 80.0


@pytest.mark.parametrize("hold,fade", [(128, 64), (64, 64), (256, 64)])
def test_cells_equal_one_shot_bitwise(golden_config1, hold, fade):
    """The block scheduler's execution model (klatt_f32_block.cu): the stream in the compact StreamStateLite, every 64-sample
    cell handed to the hold loop, the straight-line fade loop (renderFadeF32T) or the general loop.  Same bits as the
    one-shot general render, on random frames, on config 1 and on the vowel chart's 400 ms fades; and most ticks must
    actually run in the two fast loops."""
    sr = 22050
    for sid, secs in ((7, 2.0), (4242, 3.0)):
        fr, m, f, nul, ux = workloads.random_stream(sid, secs, sr)
        n = int(secs * sr)
        one, li = sim.render_f32(sr, fr, m, f, nul, ux, max_samples=n, seed=1, stream=sid)
        got, li2, used = sim.render_f32_cells(sr, fr, m, f, nul, ux, max_samples=n, seed=1, stream=sid, hold_ticks=hold, fade_ticks=fade)
        np.testing.assert_array_equal(got, one)
        assert li2 == li and sum(used) == n
        assert used[0] > 0.3 * n and used[1] > 0.1 * n, used
    g = golden_config1
    one, _ = sim.render_f32(int(g["sample_rate"]), g["frames"], g["min_dur"], g["fade_dur"], g["is_null"], seed=5, stream=9)
    got, _, used = sim.render_f32_cells(int(g["sample_rate"]), g["frames"], g["min_dur"], g["fade_dur"], g["is_null"], seed=5, stream=9,
                                        hold_ticks=hold, fade_ticks=fade)
    np.testing.assert_array_equal(got, one)
    fb = workloads.vowel_chart(1, pairs=3)
    for s in range(fb.num_streams):
        fr, m, f, nul, ux = fb.stream(s)
        one, _ = sim.render_f32(16000, fr, m, f, nul, ux, seed=8, stream=s)
        got, _, used = sim.render_f32_cells(16000, fr, m, f, nul, ux, seed=8, stream=s, hold_ticks=hold, fade_ticks=fade)
        np.testing.assert_array_equal(got, one)
        assert used[1] > 0.4 * len(one), used   # 60 % of these ticks are fade ticks
    _replay_cells_equal_one_shot(hold, fade, 0)


def _replay_cells_equal_one_shot(hold, fade, fade_max):
    """A replay stream under the cells model renders its caller's draws: the fade loop draws Philox noise only, so interior
    fades must go to the general loop.  The draws are the Philox words of another key (>> 1): a fade cell that drew the
    stream's own key would change the bits, and the one-shot render under that other key is the answer."""
    fb = workloads.vowel_chart(1, pairs=2)
    for s in range(fb.num_streams):
        fr, m, f, nul, ux = fb.stream(s)
        fr = noisy(fr)   # the vowels are voiced only: give the noise a way into the output
        one, _ = sim.render_f32(16000, fr, m, f, nul, ux, seed=0x51, stream=(1 << 40) + s)
        draws = philox_draws(0x51, (1 << 40) + s, 2 * len(one))
        rep, _ = sim.render_f32(16000, fr, m, f, nul, ux, seed=8, stream=s, replay=draws)
        np.testing.assert_array_equal(rep, one)
        got, _, used = sim.render_f32_cells(16000, fr, m, f, nul, ux, seed=8, stream=s, hold_ticks=hold, fade_ticks=fade,
                                            fade_max=fade_max, replay=draws)
        np.testing.assert_array_equal(got, one)
        assert used[1] == 0, used


@pytest.mark.parametrize("hold,fade,fade_max", [(256, 128, 0), (256, 128, 512), (256, 64, 4096), (256, 192, 320)])
def test_long_fade_chunks_equal_one_shot_bitwise(hold, fade, fade_max):
    """The ring scheduler's fade class (klatt_f32_sched.cu): a fade chunk is several 64-tick cells of renderFadeF32T in one
    call (the coarse re-base at the head of every cell), stretched to the interior fade ticks the stream has left.  Same
    bits as the one-shot general render."""
    sr = 22050
    for sid, secs in ((11, 2.0), (977, 2.5)):
        fr, m, f, nul, ux = workloads.random_stream(sid, secs, sr)
        n = int(secs * sr)
        one, li = sim.render_f32(sr, fr, m, f, nul, ux, max_samples=n, seed=3, stream=sid)
        got, li2, used = sim.render_f32_cells(sr, fr, m, f, nul, ux, max_samples=n, seed=3, stream=sid, hold_ticks=hold, fade_ticks=fade,
                                              fade_max=fade_max)
        np.testing.assert_array_equal(got, one)
        assert li2 == li and sum(used) == n
        assert used[1] > 0.05 * n, used
    fb = workloads.vowel_chart(1, pairs=2)
    for s in range(fb.num_streams):
        fr, m, f, nul, ux = fb.stream(s)
        one, _ = sim.render_f32(16000, fr, m, f, nul, ux, seed=8, stream=s)
        got, _, used = sim.render_f32_cells(16000, fr, m, f, nul, ux, seed=8, stream=s, hold_ticks=hold, fade_ticks=fade, fade_max=fade_max)
        np.testing.assert_array_equal(got, one)
        assert used[1] > 0.4 * len(one), used
    _replay_cells_equal_one_shot(hold, fade, fade_max)
