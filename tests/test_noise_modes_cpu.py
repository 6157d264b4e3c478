"""CPU: the noise sources without a device -- the numpy Philox the replay tests build their draws with is the oracle's
and the engine's, and speechPlayer_multiBatchCreate refuses the precisions and noise modes a multi-batch cannot render
before it looks for a device."""
import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads
from tests.noise import philox4x32_10, philox_draws


def test_philox_known_answers():
    """Random123's published vectors for Philox4x32-10"""
    z = np.zeros(1, np.uint64)
    assert philox4x32_10(z, z, z, z, 0, 0)[0].tolist() == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    f = np.full(1, 0xFFFFFFFF, np.uint64)
    assert philox4x32_10(f, f, f, f, 0xFFFFFFFF, 0xFFFFFFFF)[0].tolist() == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    c = [np.full(1, v, np.uint64) for v in (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344)]
    assert philox4x32_10(*c, 0xA4093822, 0x299F31D0)[0].tolist() == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


@pytest.mark.parametrize("seed,stream", [(99, 33), (0xB200, (1 << 32) + 7), ((1 << 40) + 3, 5), ((1 << 63) + 1, (1 << 63) + (1 << 32))])
def test_replayed_philox_draws_are_philox_noise(port, seed, stream):
    """The oracle renders replayed draws of key (seed, stream) bit for bit as its own Philox noise of that key: the premise of
    every exact replay check in test_gpu_noise_modes.py, for keys with high words too"""
    sr = 22050
    fr, m, f, nul, ux = workloads.random_stream(41, 0.4, sr)
    want = port.render(sr, fr, m, f, nul, ux, noise=("philox", seed, stream))
    got = port.render(sr, fr, m, f, nul, ux, noise=("replay", philox_draws(seed, stream, 2 * len(want) + 8)))
    np.testing.assert_array_equal(got, want)
    other = port.render(sr, fr, m, f, nul, ux, noise=("philox", seed, stream ^ (1 << 32)))
    assert (other != want).any()


@pytest.mark.parametrize("precision,noise,msg", [
    (player.PRECISION_STREAM, player.NOISE_PHILOX, "SPEECHPLAYER_PRECISION_STREAM is a per-handle mode"),
    (7, player.NOISE_PHILOX, "unknown precision"),
    (player.PRECISION_FP32, player.NOISE_GLIBC, "noise mode must be PHILOX"),
    (player.PRECISION_FP64, player.NOISE_REPLAY, "noise mode must be PHILOX"),
    (player.PRECISION_FP32, player.NOISE_REPLAY, "noise mode must be PHILOX"),
])
def test_multi_batch_create_refuses_what_it_cannot_render(precision, noise, msg):
    """refused at create, before the device query (so also here, without a device), with batchCreate's words"""
    with pytest.raises(player.EngineError, match=msg):
        player.MultiBatch(22050, 4, [0], precision=precision, noise=noise)
