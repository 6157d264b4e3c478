"""GPU: the three noise sources on every render path that takes them.

* REPLAY of Philox draws is Philox noise.  Replaying the draws of key (s2, id2) (tests/noise.py) must render bit for bit
  what Philox noise keyed (s2, id2) renders: on FP64, FP32 and STREAM players, and on FP64 / FP32 batches under every
  FP32 scheduler.  The replaying handle's own key is a different one, so a loop that drew its own Philox noise instead of
  the caller's draws changes the bits.
* REPLAY of arbitrary draws (uniform, runs of 0 and 2^31-1, a sequence shorter than the render) against the oracle's
  replay, on requests where each of the two draws of a sample reaches the output on its own.
* GLIBC against the oracle's own libc rand(): one player per precision, interleaved players, and speechPlayer_synthesizeBatch
  against the same calls made one after another (rows, and where the process-global generator is left).
* Philox keys with bits above 2^32 in the seed and the stream id, on the players, Batch and the long-utterance paths.
"""
import numpy as np
import pytest

from nvspeechplayer_b200 import player, workloads
from oracle import oracle
from tests import parity, scenarios
from tests.noise import noisy, philox_draws

pytestmark = pytest.mark.gpu

P = workloads.P
PRECISIONS = {"fp64": player.PRECISION_FP64, "fp32": player.PRECISION_FP32, "stream": player.PRECISION_STREAM}
KEY = ((1 << 44) + 0x5EED, (1 << 36) + 99)  # the key the replayed draws come from
OWN = (0xB200, 7)                             # the replaying handles' own Philox key
HI_SEED, HI_ID = (1 << 40) + 0xB200, (1 << 35) + 17


def _assert_bar(prec, got, want, what):
    if prec == player.PRECISION_FP64:
        assert len(got) == len(want), what
        np.testing.assert_array_equal(got, want, err_msg=what)
    else:
        parity.assert_f32_parity(got, want, what)


class _Engine:
    def __init__(self, sr, precision, noise, key=OWN, draws=None):
        self.p = player.SpeechPlayer(sr, precision=precision, noise=noise, seed=key[0], streamId=key[1])
        if draws is not None:
            self.p.set_noise_replay(draws)

    def queue_frame(self, fr, m, f, ux=-1, purge=False):
        self.p.queue_frame(fr, m, f, ux, purge)

    def synthesize(self, n):
        return self.p.synthesize_np(n)

    def last_index(self):
        return self.p.last_index()

    def close(self):
        self.p.close()


class _Oracle:
    def __init__(self, port, sr, noise):
        self.p = port.player(sr)
        if noise[0] == "libc":
            self.p.noise_libc()
        elif noise[0] == "philox":
            self.p.noise_philox(noise[1], noise[2])
        else:
            self.p.noise_replay(noise[1])

    def queue_frame(self, fr, m, f, ux=-1, purge=False):
        self.p.queue_frame(fr, m, f, ux, purge)

    def synthesize(self, n):
        return self.p.synthesize(n)

    def last_index(self):
        return self.p.last_index()

    def close(self):
        self.p.close()


def _noisy_script(sc):
    """the scenario with noise in every real frame"""
    ops = [("q", None if op[1] is None else noisy(op[1])[0]) + tuple(op[2:]) if op[0] == "q" else op for op in sc["ops"]]
    return dict(sr=sc["sr"], ops=ops)


def _pulled(sc):
    return sum(op[1] for op in sc["ops"] if op[0] == "s")


def _long_pull():
    fr, m, f, nul, ux = workloads.random_stream(4711, 1.2, 22050)
    ops = [("q", None if nul[j] else fr[j], int(m[j]), int(f[j]), int(ux[j]), False) for j in range(len(m))]
    return dict(sr=22050, ops=ops + [("s", 20000), ("s", 9000)])


PLAYER_SCENARIOS = ("purge_mid_fade", "purge_mid_hold", "purge_twice", "purge_idle_then_speak", "drain_resume", "chunk_777",
                    "null_first", "source_features", "random_16000", "random_22050", "random_44100")


@pytest.mark.parametrize("prec", sorted(PRECISIONS))
def test_player_replay_of_philox_draws_is_philox_noise(prec):
    scs = scenarios.all_scenarios()
    cases = [(name, _noisy_script(scs[name])) for name in PLAYER_SCENARIOS]
    if prec == "stream":
        cases.append(("pull of 20000 samples", _long_pull()))   # more than one launch of 8192 ticks
    pr = PRECISIONS[prec]
    for name, sc in cases:
        draws = philox_draws(*KEY, 2 * _pulled(sc))
        want, wc, wi = scenarios.run_script(lambda sr: _Engine(sr, pr, player.NOISE_PHILOX, key=KEY), sc)
        got, gc, gi = scenarios.run_script(lambda sr: _Engine(sr, pr, player.NOISE_REPLAY, draws=draws), sc)
        assert (gc, gi) == (wc, wi), name
        np.testing.assert_array_equal(got, want, err_msg=name)
        if name == "source_features":   # the noise reaches these samples: the handle's own key renders other bits
            own, _, _ = scenarios.run_script(lambda sr: _Engine(sr, pr, player.NOISE_PHILOX), sc)
            assert (own != want).any()


# the FP32 schedulers, forced as test_gpu_parity_f32.py::test_f32_rounds_equal_single_launch_bitwise forces them
_SCHED_COMMON = dict(NVSP_GROUPS="3", NVSP_SCHED_FADE_TICKS="0", NVSP_SCHED_FADE_MAX="320", NVSP_BLOCK_MIN_STREAMS="1",
                     NVSP_BLOCK_BLOCKS="3", NVSP_SCHED_BLOCKS="3", NVSP_SCHED_HOLD_TICKS="256", NVSP_SCHED_GEN_TICKS="128")
SCHEDULERS = {
    "single": dict(NVSP_ROUNDS_MIN_STREAMS="100000000", NVSP_SCHED="rounds"),
    "rounds": dict(NVSP_ROUNDS_MIN_STREAMS="1", NVSP_SCHED="rounds"),
    "rings": dict(NVSP_ROUNDS_MIN_STREAMS="1", NVSP_SCHED="rings"),
    "rings_fade": dict(NVSP_ROUNDS_MIN_STREAMS="1", NVSP_SCHED="rings", NVSP_SCHED_FADE_TICKS="128"),
    "block": dict(NVSP_ROUNDS_MIN_STREAMS="1", NVSP_SCHED="block"),
}
# kernels per synthesize call beyond the one-launch kernel's: import, seed, workers, export | import, workers, export
EXTRA_LAUNCHES = {"rings": 3, "rings_fade": 3, "block": 2}


def _batch_streams():
    """16 kHz: vowel-chart streams (400 ms fades, so the fade cells run) and random-frame streams, noise in every frame"""
    vc = workloads.vowel_chart(1, pairs=40)
    streams = [vc.stream(s) for s in range(vc.num_streams)] + [workloads.random_stream(600 + s, 1.0, 16000) for s in range(24)]
    streams = [(noisy(fr),) + tuple(rest) for fr, *rest in streams]
    return workloads._concat(16000, streams, np.arange(len(streams), dtype=np.uint64) + 300)


def _render_batch(b, fb, calls):
    """the calls, then batchReset + the first call again, then a second SetFrames + all of it in one call"""
    l0 = b.launch_stats()[0]
    parts, written = [], []
    for c in calls:
        o, w = b.synthesize_host(c)
        parts.append(o)
        written.append(w)
    launches = b.launch_stats()[0] - l0
    b.reset()
    again, _ = b.synthesize_host(calls[0])
    b.set_frames_host(fb)
    whole, _ = b.synthesize_host(sum(calls))
    return np.concatenate(parts, axis=1), np.sum(written, axis=0), b.last_indices(), launches, again, whole


@pytest.mark.parametrize("prec,sched", [("fp64", "single")] + [("fp32", s) for s in SCHEDULERS])
def test_batch_replay_of_philox_draws_is_philox_noise(monkeypatch, prec, sched):
    import torch
    for k, v in dict(_SCHED_COMMON, **SCHEDULERS[sched]).items():
        monkeypatch.setenv(k, v)
    fb = _batch_streams()
    n, count = fb.num_streams, 16000
    calls = (9000, 777, count - 9777)   # calls that end inside chunks
    ids2 = fb.stream_ids + np.uint64((1 << 33) + 5)
    draws = np.stack([philox_draws(KEY[0], int(i), 2 * count) for i in ids2])
    d_draws = torch.from_numpy(draws).cuda()
    pr = PRECISIONS[prec]
    ref = player.Batch(16000, n, precision=pr, noise=player.NOISE_PHILOX, seed=KEY[0], stream_ids=ids2)
    ref.set_frames_host(fb)
    want = _render_batch(ref, fb, calls)
    ref.close()
    rep = player.Batch(16000, n, precision=pr, noise=player.NOISE_REPLAY, seed=OWN[0], stream_ids=fb.stream_ids)
    rep.set_frames_host(fb)
    rep.set_noise_replay_device(d_draws.data_ptr(), draws.shape[1])
    got = _render_batch(rep, fb, calls)
    rep.close()
    torch.cuda.synchronize()
    assert want[0].any() and (want[1] > 0).all()
    for k, what in enumerate(("samples", "written", "last indices")):
        np.testing.assert_array_equal(got[k], want[k], err_msg="%s %s: %s" % (prec, sched, what))
    assert got[3] == want[3]
    # batchReset and a second SetFrames restart every stream at draw 0
    np.testing.assert_array_equal(got[4], want[0][:, :calls[0]], err_msg="after batchReset")
    np.testing.assert_array_equal(got[5], want[0], err_msg="after a second SetFrames")
    if sched in EXTRA_LAUNCHES:
        for k, v in SCHEDULERS["single"].items():
            monkeypatch.setenv(k, v)
        one = player.Batch(16000, n, precision=pr, noise=player.NOISE_PHILOX, seed=KEY[0], stream_ids=ids2)
        one.set_frames_host(fb)
        single = _render_batch(one, fb, calls)
        one.close()
        assert want[3] == single[3] + EXTRA_LAUNCHES[sched] * len(calls), "the %s scheduler did not run" % sched
        np.testing.assert_array_equal(single[0], want[0])


# ---- replayed draws that are not Philox-shaped, against the oracle ----
def _noise_queue():
    """a voiced request with turbulence, an aspiration-only and a frication-only request (each draw of a sample reaches the
    output on its own), silence, and a mixed request"""
    base = scenarios._vowel(130, 110)
    turb = base.copy()
    turb[P["voiceTurbulenceAmplitude"]], turb[P["glottalOpenQuotient"]] = 0.5, 0.4
    asp = scenarios._vowel(120)
    asp[P["voiceAmplitude"]], asp[P["aspirationAmplitude"]] = 0.0, 1.0
    fric = scenarios._vowel(120)
    fric[P["voiceAmplitude"]], fric[P["fricationAmplitude"]], fric[P["parallelBypass"]] = 0.0, 1.0, 1.0
    mix = noisy(scenarios._vowel(150, 180))[0]
    q = [(turb, 3000, 200), (asp, 2500, 300), (fric, 2500, 300), (None, 400, 200), (mix, 3000, 400)]
    return q, sum(max(m + 1, max(f, 1) + 2) for _, m, f in q)


def _arbitrary_draws(n, seed):
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 2 ** 31 - 1, n, endpoint=True, dtype=np.int64)
    d[n // 5:n // 5 + 3001] = 0
    d[n // 2:n // 2 + 2999] = 2 ** 31 - 1
    return d.astype(np.int32)


def _play(p, queue, pulls=4096):
    for j, (fr, m, f) in enumerate(queue):
        p.queue_frame(fr, m, f, j)
    out = []
    while True:
        o = p.synthesize(pulls)
        if len(o) == 0:
            break
        out.append(np.asarray(o, dtype=np.int16))
    p.close()
    return np.concatenate(out)


@pytest.mark.parametrize("prec", sorted(PRECISIONS))
def test_player_replay_against_oracle(port, prec):
    pr = PRECISIONS[prec]
    queue, total = _noise_queue()
    full = _arbitrary_draws(2 * total, 12)
    short = full[:2 * 7000 + 1]   # ends after the aspiration draw of sample 7000: the rest are 0
    for what, draws in (("arbitrary draws", full), ("short replay", short)):
        want = _play(_Oracle(port, 22050, ("replay", draws)), queue)
        got = _play(_Engine(22050, pr, player.NOISE_REPLAY, draws=draws), queue)
        _assert_bar(pr, got, want, "%s %s" % (prec, what))
        if what == "arbitrary draws":   # the bar is tight enough to see a swapped or shifted draw
            for wrong in (full.reshape(-1, 2)[:, ::-1].ravel(), np.roll(full, 1)):
                w1, _, snr, _ = parity.metrics(_play(_Oracle(port, 22050, ("replay", wrong)), queue), want)
                assert w1 < parity.F32_WITHIN_1LSB and snr < parity.F32_SNR_DB
    # a sequence set after the handle has rendered is indexed from the handle's first sample
    other = _arbitrary_draws(2 * total, 13)
    p = _Engine(22050, pr, player.NOISE_REPLAY, draws=full)
    for j, (fr, m, f) in enumerate(queue):
        p.queue_frame(fr, m, f, j)
    first = p.synthesize(5000)
    p.p.set_noise_replay(other)
    rest = [p.synthesize(4096) for _ in range(total // 4096 + 2)]
    p.close()
    got = np.concatenate([first] + rest)
    spliced = np.concatenate([full[:2 * 5000], other[2 * 5000:]])
    _assert_bar(pr, got, _play(_Oracle(port, 22050, ("replay", spliced)), queue), "%s replay set mid-stream" % prec)


@pytest.mark.parametrize("prec", ["fp64", "fp32"])
def test_batch_replay_against_oracle(port, prec):
    import torch
    queue, total = _noise_queue()
    fr = np.stack([np.zeros(47) if q[0] is None else q[0] for q in queue])
    one = (fr, np.array([q[1] for q in queue], np.uint32), np.array([q[2] for q in queue], np.uint32),
           np.array([q[0] is None for q in queue], np.uint8), np.arange(len(queue), dtype=np.int32))
    n = 4
    fb = workloads._concat(22050, [one] * n, np.arange(n, dtype=np.uint64))
    dps = 2 * total
    draws = np.stack([_arbitrary_draws(dps, 20 + s) for s in range(n)])
    draws[3, 2 * 6000:] = 0   # what a shorter sequence gives
    d_draws = torch.from_numpy(draws).cuda()
    b = player.Batch(22050, n, precision=PRECISIONS[prec], noise=player.NOISE_REPLAY, seed=OWN[0])
    b.set_frames_host(fb)
    b.set_noise_replay_device(d_draws.data_ptr(), dps)
    out, written = b.synthesize_host(total)
    b.close()
    for s in range(n):
        want = port.render(22050, *one[:4], one[4], noise=("replay", draws[s] if s < 3 else draws[s][:2 * 6000]))
        assert written[s] == len(want)
        _assert_bar(PRECISIONS[prec], out[s][:written[s]], want, "%s batch stream %d" % (prec, s))


# ---- glibc: the engine's process-global generator against the oracle's libc rand() ----
def _seed(s):
    """seed both generators: other tests consume them, the result must not depend on test order"""
    player.load_library().speechPlayer_seedNoise(s)
    oracle.libc().srand(s)


@pytest.mark.parametrize("prec", sorted(PRECISIONS))
def test_glibc_single_player_against_libc(port, prec):
    pr = PRECISIONS[prec]
    queue, _ = _noise_queue()
    res = {}
    for s in (0, 1, 0xB200):
        _seed(s)
        res[s] = got = _play(_Engine(22050, pr, player.NOISE_GLIBC), queue)
        _seed(s)
        want = _play(_Oracle(port, 22050, ("libc",)), queue)
        _assert_bar(pr, got, want, "%s glibc seed %d" % (prec, s))
    np.testing.assert_array_equal(res[0], res[1])   # seed 0 is seed 1, as in glibc
    assert (res[1] != res[0xB200]).any()


def _interleaved(make):
    """three glibc players driven in one order: calls of different sizes, a drain, a purge, a player created mid-way"""
    q, _ = _noise_queue()
    out = {0: [], 1: [], 2: []}
    p0, p1 = make(), make()
    for j, (fr, m, f) in enumerate(q):
        p0.queue_frame(fr, m, f, j)
    for j, (fr, m, f) in enumerate(q[::-1]):
        p1.queue_frame(fr, m, f, j)
    out[0].append(p0.synthesize(1000))
    out[1].append(p1.synthesize(700))
    out[0].append(p0.synthesize(30000))          # drains
    p1.queue_frame(q[2][0], 2000, 300, 9, True)  # purge
    p2 = make()
    for j, (fr, m, f) in enumerate(q[1:3]):
        p2.queue_frame(fr, m, f, j)
    out[2].append(p2.synthesize(2500))
    out[1].append(p1.synthesize(5000))
    out[0].append(p0.synthesize(500))            # idle: no sample, no draw
    p0.queue_frame(q[1][0], 1500, 200, 20)
    out[0].append(p0.synthesize(3000))
    out[2].append(p2.synthesize(20000))
    out[1].append(p1.synthesize(20000))
    for p in (p0, p1, p2):
        p.close()
    return [np.concatenate([np.asarray(o, np.int16) for o in out[k]]) for k in range(3)]


def test_glibc_interleaved_players_against_libc(port):
    _seed(77)
    got = _interleaved(lambda: _Engine(22050, player.PRECISION_FP64, player.NOISE_GLIBC))
    _seed(77)
    want = _interleaved(lambda: _Oracle(port, 22050, ("libc",)))
    for k in range(3):
        np.testing.assert_array_equal(got[k], want[k], err_msg="player %d" % k)


def _handle_queues(prec):
    """per handle: idle (nothing queued), one that drains mid-call, a long one; STREAM adds one of 60 short requests"""
    q, _ = _noise_queue()
    short = [q[1]]
    long = q + q
    queues = [[], short, long]
    if prec == "stream":
        queues.append([(q[k % 3][0], 90 + k, 40) for k in range(60)])
    return queues


def _make(sr, pr, queue):
    p = _Engine(sr, pr, player.NOISE_GLIBC)
    for j, (fr, m, f) in enumerate(queue):
        p.queue_frame(fr, m, f, j)
    return p


def _after(make):
    """one more FP64 glibc player: shows where the generator was left"""
    p = make()
    q, _ = _noise_queue()
    return _play(p, q[::-1])


@pytest.mark.parametrize("prec", sorted(PRECISIONS))
def test_glibc_synthesize_batch_is_sequential_calls(port, prec):
    pr = PRECISIONS[prec]
    queues = _handle_queues(prec)
    count = 20000 if prec == "stream" else 6000   # STREAM: more than one launch of 8192 ticks per call
    calls = 2
    _seed(5)
    ps = [_make(22050, pr, q) for q in queues]
    batch = [player.synthesize_batch([p.p for p in ps], count) for _ in range(calls)]
    for p in ps:
        p.close()
    d_batch = _after(lambda: _Engine(22050, player.PRECISION_FP64, player.NOISE_GLIBC))
    _seed(5)
    ps = [_make(22050, pr, q) for q in queues]
    seq = []
    for _ in range(calls):
        rows, written = np.zeros((len(ps), count), np.int16), np.zeros(len(ps), np.uint32)
        for i, p in enumerate(ps):
            o = p.synthesize(count)
            rows[i, :len(o)], written[i] = o, len(o)
        seq.append((rows, written))
    for p in ps:
        p.close()
    d_seq = _after(lambda: _Engine(22050, player.PRECISION_FP64, player.NOISE_GLIBC))
    assert seq[0][1][0] == 0 and 0 < seq[0][1][1] < count and seq[0][1][2] == count
    for c in range(calls):
        np.testing.assert_array_equal(batch[c][1], seq[c][1], err_msg="written, call %d" % c)
        np.testing.assert_array_equal(batch[c][0], seq[c][0], err_msg="rows, call %d" % c)
    np.testing.assert_array_equal(d_batch, d_seq)
    # and the sequential calls draw what the reference's rand() hands out
    _seed(5)
    ops = [_make_oracle(port, q) for q in queues]
    for _ in range(calls):
        for o in ops:
            o.synthesize(count)
    for o in ops:
        o.close()
    np.testing.assert_array_equal(d_batch, _after(lambda: _Oracle(port, 22050, ("libc",))))


def _make_oracle(port, queue):
    p = _Oracle(port, 22050, ("libc",))
    for j, (fr, m, f) in enumerate(queue):
        p.queue_frame(fr, m, f, j)
    return p


# ---- Philox keys with bits above 2^32 ----
def _hi_stream():
    fr, m, f, nul, ux = workloads.random_stream(808, 0.5, 22050)
    return noisy(fr), m, f, nul, ux


@pytest.mark.parametrize("prec", sorted(PRECISIONS))
def test_philox_high_key_words_players(port, prec):
    pr = PRECISIONS[prec]
    fr, m, f, nul, ux = _hi_stream()
    q = [(None if nul[j] else fr[j], int(m[j]), int(f[j])) for j in range(len(m))]
    want = port.render(22050, fr, m, f, nul, np.arange(len(m), dtype=np.int32), noise=("philox", HI_SEED, HI_ID))
    got = _play(_Engine(22050, pr, player.NOISE_PHILOX, key=(HI_SEED, HI_ID)), q)
    _assert_bar(pr, got, want, "%s high key words" % prec)
    other = _play(_Engine(22050, pr, player.NOISE_PHILOX, key=(HI_SEED, HI_ID + (1 << 32))), q)
    assert len(other) == len(got) and (other != got).any()


@pytest.mark.parametrize("prec", ["fp64", "fp32"])
def test_philox_high_key_words_batch(port, prec):
    st = _hi_stream()
    ids = np.array([HI_ID, HI_ID + (1 << 32), (1 << 63) + 1], dtype=np.uint64)
    fb = workloads._concat(22050, [st] * len(ids), ids)
    count = int(fb.timeline_samples()[0])
    b = player.Batch(22050, len(ids), precision=PRECISIONS[prec], noise=player.NOISE_PHILOX, seed=HI_SEED, stream_ids=ids)
    b.set_frames_host(fb)
    out, written = b.synthesize_host(count)
    b.close()
    for s in range(len(ids)):
        want = port.render(22050, *st[:4], st[4], max_samples=count, noise=("philox", HI_SEED, int(ids[s])))
        _assert_bar(PRECISIONS[prec], out[s], want, "%s batch stream id %#x" % (prec, ids[s]))
    assert (out[0] != out[1]).any()


def test_philox_high_key_words_long_paths(port):
    fr, m, f, nul, ux = _hi_stream()
    ids = [HI_ID, HI_ID + (1 << 32)]
    want = [port.render(22050, fr, m, f, nul, ux, noise=("philox", HI_SEED, i))[:oracle.timeline_samples(m, f)] for i in ids]
    assert (want[0] != want[1]).any()
    for k, i in enumerate(ids):
        got, _, _ = player.synthesize_long(22050, fr, m, f, nul, seed=HI_SEED, stream_id=i, chunk_ticks=256)
        parity.assert_f32_parity(got, want[k], "synthesize_long id %#x" % i)
    fb = workloads._concat(22050, [(fr, m, f, nul, ux)] * 2, np.array(ids, dtype=np.uint64))
    samples, offs, _, _, _ = player.synthesize_long_batch(fb, seed=HI_SEED, chunk_ticks=256)
    rows = player.split_rows(samples, offs)
    for k, i in enumerate(ids):
        parity.assert_f32_parity(rows[k], want[k], "synthesize_long_batch id %#x" % i)
    assert (rows[0] != rows[1]).any()
