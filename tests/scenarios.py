"""Small frame-manager / generator scenarios shared by the golden generator and the parity tests.

Each scenario is a script of C-ABI calls on ONE player:
    ("q", frame47 | None, minDurSamples, fadeDurSamples, userIndex, purge)   -> speechPlayer_queueFrame
    ("s", n)                                                               -> speechPlayer_synthesize(n)
`run_script` drives any object with queue_frame/synthesize/last_index/close and returns
(concatenated pcm, [count returned by each "s"], [getLastIndex after each "s"]).

The behaviours covered are the ones SURVEY.md section 4 lists as probe-verified on the
compiled reference (timeline law, drain/resume, purge snapshot, clamp/NaN, chunk invariance,
userIndex) plus the NULL-frame rewrites of reference src/frame.cpp:59-67.
"""
import numpy as np

from nvspeechplayer_b200.workloads import NUM_PARAMS, P, PARAM_NAMES, RANDOM_RANGES, random_stream  # noqa: F401

SEED, STREAM = 0xB200, 7  # Philox noise key used for every scenario
# random-frame streams (sample rate, stream id) of 1.5 s with Philox key (RANDOM_SEED, stream id): what the live port-vs-reference
# test renders, and what `tests/golden/make_golden.py random_streams` records from the reference
RANDOM_STREAMS, RANDOM_SECONDS, RANDOM_SEED = ((16000, 31), (22050, 32), (44100, 33)), 1.5, 99


def _rand_frame(rng):
    lo = np.array([RANDOM_RANGES[n][0] for n in PARAM_NAMES])
    hi = np.array([RANDOM_RANGES[n][1] for n in PARAM_NAMES])
    return lo + (hi - lo) * rng.random(NUM_PARAMS)


def _vowel(pitch=120.0, end=None, gain=1.0):
    """A plain 'a'-like voiced frame with hand-set formants (no table needed)."""
    f = np.zeros(NUM_PARAMS)
    f[P["voicePitch"]] = pitch
    f[P["endVoicePitch"]] = pitch if end is None else end
    f[P["voiceAmplitude"]] = 1.0
    f[P["glottalOpenQuotient"]] = 0.1
    for k, (cf, cb) in enumerate([(700, 130), (1220, 70), (2600, 160), (3300, 250), (3750, 200), (4900, 1000)]):
        f[P["cf1"] + k] = cf
        f[P["cb1"] + k] = cb
        f[P["pf1"] + k] = cf
        f[P["pb1"] + k] = cb
    f[P["cfN0"]], f[P["cbN0"]], f[P["cfNP"]], f[P["cbNP"]] = 450, 100, 270, 100
    f[P["preFormantGain"]] = 1.0
    f[P["outputGain"]] = gain
    return f


def all_scenarios():
    sc = {}
    rng = np.random.default_rng(20261017)

    # --- timeline law max(M+1, F+2): one frame each, pulled in one big call -------------------
    for m, f in [(10, 4), (10, 1), (4, 10), (1, 1), (10, 9), (10, 10), (10, 0), (2000, 300)]:
        sc["law_M%d_F%d" % (m, f)] = dict(sr=22050, ops=[("q", _rand_frame(rng), m, f, 5, False), ("s", 4096)])
    sc["law_two_frames"] = dict(sr=22050, ops=[("q", _rand_frame(rng), 300, 100, 1, False),
                                               ("q", _rand_frame(rng), 50, 200, 2, False), ("s", 4096)])
    # NULL frame with M=0 is legal (frame.cpp:63 overwrites the inc)
    sc["law_null_M0"] = dict(sr=22050, ops=[("q", _vowel(), 400, 50, -1, False), ("q", None, 0, 30, -1, False),
                                            ("s", 4096)])
    # --- chunk-size invariance: same queue drained with different pull sizes ------------------
    frames = [(_rand_frame(rng), int(rng.integers(200, 1500)), int(rng.integers(1, 900))) for _ in range(6)]
    for chunk in (1, 7, 777, 8192):
        ops = [("q", fr, m, f, j, False) for j, (fr, m, f) in enumerate(frames)]
        total = sum(max(m + 1, max(f, 1) + 2) for _, m, f in frames)
        ops += [("s", chunk)] * (total // chunk + 2)
        sc["chunk_%d" % chunk] = dict(sr=22050, ops=ops)
    # --- drain, idle, resume (frame.cpp:73-75) -----------------------------------------------
    sc["drain_resume"] = dict(sr=16000, ops=[
        ("q", _vowel(100, 140), 800, 160, 11, False), ("s", 600), ("s", 600), ("s", 600), ("s", 64),
        ("q", None, 320, 160, 12, False), ("s", 1000), ("s", 10),
        ("q", _vowel(200, 90), 500, 100, 13, False), ("q", None, 100, 100, -1, False), ("s", 2000)])
    # --- purge (frame.cpp:103-112) -------------------------------------------------------------
    a, b = _vowel(110, 130), _vowel(180, 90, gain=1.5)
    b[P["cf1"]], b[P["cf2"]] = 300, 2300
    sc["purge_mid_fade"] = dict(sr=22050, ops=[
        ("q", a, 2205, 110, 1, False), ("q", b, 2205, 4000, 2, False), ("s", 3000),
        ("q", None, 441, 4410, 3, True), ("s", 8192)])
    sc["purge_mid_hold"] = dict(sr=22050, ops=[
        ("q", a, 5000, 200, 1, False), ("q", b, 3000, 500, 2, False), ("s", 1500),
        ("q", b, 1000, 300, 9, True), ("q", None, 100, 200, 10, False), ("s", 8192)])
    sc["purge_idle_then_speak"] = dict(sr=16000, ops=[
        ("q", None, 0, 320, -1, True), ("q", a, 4800, 800, 4, False), ("q", b, 8000, 6400, 5, False),
        ("q", None, 800, 800, 6, False), ("s", 20000)])
    sc["purge_twice"] = dict(sr=22050, ops=[
        ("q", a, 3000, 1000, 1, False), ("s", 500), ("q", b, 800, 400, 2, True), ("q", a, 700, 300, 3, True),
        ("s", 4000)])
    # --- clamp / NaN semantics of the Win32 min/max macros (speechWaveGenerator.cpp:208) -------
    g = _vowel(150)
    g[P["outputGain"]] = np.nan
    sc["nan_gain"] = dict(sr=22050, ops=[("q", g, 400, 50, -1, False), ("s", 1024)])
    g = _vowel(150)
    g[P["outputGain"]] = 1e6
    sc["clamp"] = dict(sr=22050, ops=[("q", g, 400, 50, -1, False), ("s", 1024)])
    # NaN in a target param keeps the old value for that fade (utils.h:21)
    k1, k2 = _vowel(120), _vowel(160)
    k2[P["cf2"]] = np.nan
    k2[P["pa3"]] = np.nan
    sc["nan_keep"] = dict(sr=22050, ops=[("q", k1, 600, 100, -1, False), ("q", k2, 600, 300, -1, False), ("s", 900)])
    # --- NULL first / NULL after NULL -----------------------------------------------------------
    sc["null_first"] = dict(sr=22050, ops=[("q", None, 100, 50, 1, False), ("q", None, 10, 10, 2, False),
                                           ("q", _vowel(), 300, 60, 3, False), ("q", None, 50, 50, 4, False),
                                           ("q", None, 50, 20, 5, False), ("s", 2048)])
    # --- fade longer than hold, fade of 0 (clamped to 1 by speechPlayer.cpp:36) ----------------
    sc["fade_gt_hold"] = dict(sr=22050, ops=[("q", _rand_frame(rng), 20, 500, -1, False),
                                             ("q", _rand_frame(rng), 30, 0, -1, False),
                                             ("q", _rand_frame(rng), 1, 700, -1, False), ("s", 4096)])
    # --- source features: vibrato, turbulence, open quotient, aspiration, frication ------------
    v = _vowel(140, 210)
    v[P["vibratoPitchOffset"]], v[P["vibratoSpeed"]] = 0.3, 5.5
    v[P["voiceTurbulenceAmplitude"]], v[P["glottalOpenQuotient"]] = 0.4, 0.35
    v[P["aspirationAmplitude"]], v[P["fricationAmplitude"]] = 0.6, 0.8
    for k in range(6):
        v[P["pa1"] + k] = 0.3 + 0.1 * k
    v[P["parallelBypass"]], v[P["caNP"]] = 0.4, 0.7
    sc["source_features"] = dict(sr=22050, ops=[("q", v, 6000, 400, -1, False), ("q", None, 200, 200, -1, False),
                                                ("s", 8192)])
    # pitch gliding to zero (test_sayHannah.py leaves endVoicePitch at 0)
    h = _vowel(160, 0.0)
    sc["glide_to_zero"] = dict(sr=22050, ops=[("q", h, 3000, 200, -1, False), ("s", 4096)])
    # --- longer random streams at the three sample rates ----------------------------------------
    for sr in (16000, 22050, 44100):
        fr, m, f, nul, ux = random_stream(1000 + sr, 0.6, sr)
        ops = [("q", None if nul[j] else fr[j], int(m[j]), int(f[j]), int(ux[j]), False) for j in range(len(m))]
        ops += [("s", int(0.6 * sr))]
        sc["random_%d" % sr] = dict(sr=sr, ops=ops)
    return sc


def run_script(make_player, scenario):
    p = make_player(scenario["sr"])
    pcm, counts, idx = [], [], []
    for op in scenario["ops"]:
        if op[0] == "q":
            _, fr, m, f, ux, purge = op
            p.queue_frame(fr, m, f, ux, purge)
        else:
            out = p.synthesize(op[1])
            pcm.append(np.asarray(out, dtype=np.int16))
            counts.append(len(out))
            idx.append(p.last_index())
    p.close()
    return (np.concatenate(pcm) if pcm else np.zeros(0, np.int16)), counts, idx
