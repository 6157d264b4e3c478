"""Regenerate the committed golden fixtures from the REFERENCE ITSELF.

Run where an NVSpeechPlayer checkout is at hand (NVSP_REFERENCE_DIR names it; oracle/_ref is built
from it); the tests only read the .npz files.

  config1.npz    BASELINE config 1: sampleIpa.txt through the reference's UNCHANGED
                 ipa.py + speechPlayer.py (recipe test_speakIpa.py:20-27, 22 050 Hz,
                 speed=0.6) driving the compiled reference.  Stores the exact
                 queueFrame call sequence (in samples) and the int16 render under
                 (a) glibc rand() from the default seed and (b) the Philox noise contract.
  scenarios.npz  the small state-machine scenarios of tests/scenarios.py rendered by
                 the compiled reference (Philox noise), incl. purge / drain-resume /
                 NaN gain / chunked pulls.
  phonemes       nvspeechplayer_b200/data/phoneme_table.npz: the numeric content of the
                 reference's data.py (49 phonemes x 47 params + flags) used by the
                 vowel-chart and midi-sing workload generators.
  random_streams.npz  the random-frame streams of scenarios.RANDOM_STREAMS rendered by the
                 compiled reference (Philox noise); `make_golden.py random_streams` writes
                 only this file and needs only the compiled reference.
"""
import ctypes
import hashlib
import importlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402
from tests import scenarios  # noqa: E402

REF = oracle.REFERENCE
HERE = os.path.dirname(os.path.abspath(__file__))
SEED, STREAM = 0xB200, 0


def reference_package(so_path):
    """A throw-away package dir that lets the UNCHANGED reference python files import each other
    (ipa.py:18 uses a relative import) and find the library under the literal name speechPlayer.dll
    (speechPlayer.py:42)."""
    d = tempfile.mkdtemp(prefix="nvsp_refpkg_")
    pkg = os.path.join(d, "nvsp_ref")
    os.mkdir(pkg)
    open(os.path.join(pkg, "__init__.py"), "w").close()
    for name in ("speechPlayer.py", "ipa.py", "data.py"):
        os.symlink(os.path.join(REF, name), os.path.join(pkg, name))
    os.symlink(so_path, os.path.join(pkg, "speechPlayer.dll"))
    sys.path.insert(0, d)
    return importlib.import_module("nvsp_ref.ipa"), importlib.import_module("nvsp_ref.speechPlayer")


def config1():
    ipa, sp = reference_package(oracle.REF_SO)
    sr = 22050
    calls = []  # (frame47 or None, minDurSamples, fadeDurSamples)
    player = sp.SpeechPlayer(sr)
    oracle.libc().srand(1)  # glibc's default seed, made explicit

    def queue(frame, dur_ms, fade_ms):
        player.queueFrame(frame, dur_ms, fade_ms)
        m = int(dur_ms * (sr / 1000.0))  # speechPlayer.py:53
        f = int(fade_ms * (sr / 1000.0))
        vals = None if frame is None else np.array([getattr(frame, n) for n, _ in sp.Frame._fields_])
        calls.append((vals, m, f))

    import codecs
    text = codecs.open(os.path.join(REF, "sampleIpa.txt"), "r", "utf8").read()
    for line in text.splitlines():
        for args in ipa.generateFramesAndTiming(line.strip(), speed=0.6):
            queue(*args)
        queue(None, 150, 0)
    chunks = []
    while True:
        buf = player.synthesize(8192)
        if buf is None:
            break
        chunks.append(np.frombuffer(buf, dtype=np.int16, count=buf.length).copy())
    pcm_libc = np.concatenate(chunks)
    n = len(calls)
    frames = np.zeros((n, 47))
    is_null = np.zeros(n, dtype=np.uint8)
    for j, (vals, _, _) in enumerate(calls):
        if vals is None:
            is_null[j] = 1
        else:
            frames[j] = vals
    min_dur = np.array([c[1] for c in calls], dtype=np.uint32)
    fade_dur = np.array([c[2] for c in calls], dtype=np.uint32)
    ref_px = oracle.RefLib(philox=True)
    pcm_philox = ref_px.render(sr, frames, min_dur, fade_dur, is_null, seed=SEED, stream=STREAM)
    sha = hashlib.sha256(pcm_libc.tobytes()).hexdigest()
    print("config1: %d frames (%d NULL), %d samples, sha256(libc)=%s" % (n, is_null.sum(), pcm_libc.size, sha))
    np.savez_compressed(os.path.join(HERE, "config1.npz"), sample_rate=sr, frames=frames, min_dur=min_dur,
                        fade_dur=fade_dur, is_null=is_null, pcm_libc=pcm_libc, pcm_philox=pcm_philox,
                        sha256_libc=sha, philox_seed=SEED, philox_stream=STREAM)
    return ipa


def phoneme_table(ipa):
    names = sorted(ipa.data.keys())
    fields = scenarios.PARAM_NAMES
    table = np.zeros((len(names), 47))
    present = np.zeros((len(names), 47), dtype=np.uint8)
    flags = {}
    for i, k in enumerate(names):
        for pk, pv in ipa.data[k].items():
            if pk in fields:
                table[i, fields.index(pk)] = pv
                present[i, fields.index(pk)] = 1
            elif pk.startswith("_"):
                flags.setdefault(pk, np.zeros(len(names), dtype=np.uint8))[i] = 1 if pv else 0
    out = os.path.join(ROOT, "nvspeechplayer_b200", "data")
    os.makedirs(out, exist_ok=True)
    np.savez_compressed(os.path.join(out, "phoneme_table.npz"), names=np.array(names), table=table, present=present,
                        **{"flag" + k: v for k, v in flags.items()})
    print("phoneme table: %d phonemes, %d voiced" % (len(names), int(flags["_isVoiced"].sum())))


def scenario_goldens():
    ref_px = oracle.RefLib(philox=True)
    out = {}
    for name, sc in scenarios.all_scenarios().items():
        pcm, counts, idx = scenarios.run_script(lambda sr: _RefAdapter(ref_px, sr), sc)
        out[name + "/pcm"] = pcm
        out[name + "/counts"] = np.array(counts, dtype=np.int64)
        out[name + "/last_index"] = np.array(idx, dtype=np.int64)
        print("scenario %-28s %7d samples" % (name, pcm.size))
    np.savez_compressed(os.path.join(HERE, "scenarios.npz"), **out)


def random_stream_goldens():
    """scenarios.RANDOM_STREAMS through the compiled reference with Philox noise, every frame queued up front."""
    ref_px = oracle.RefLib(philox=True)
    out = {}
    for sr, sid in scenarios.RANDOM_STREAMS:
        fr, m, f, nul, ux = scenarios.random_stream(sid, scenarios.RANDOM_SECONDS, sr)
        out["%d_%d" % (sr, sid)] = ref_px.render(sr, fr, m, f, nul, ux, seed=scenarios.RANDOM_SEED, stream=sid)
        print("random stream %d @ %d Hz: %d samples" % (sid, sr, out["%d_%d" % (sr, sid)].size))
    np.savez_compressed(os.path.join(HERE, "random_streams.npz"), **out)


class _RefAdapter:
    def __init__(self, lib, sr):
        lib.seed(scenarios.SEED, scenarios.STREAM)
        self.p = lib.player(sr)

    def queue_frame(self, frame, m, f, user_index, purge):
        self.p.queue_frame(frame, m, f, user_index, purge)

    def synthesize(self, n):
        return self.p.synthesize(n)

    def last_index(self):
        return self.p.last_index()

    def close(self):
        self.p.close()


if __name__ == "__main__":
    assert oracle.build(REF, quiet=True), "reference .so not built"
    if sys.argv[1:] != ["random_streams"]:  # the one step that needs only the compiled reference, not its Python files
        ipa_mod = config1()
        phoneme_table(ipa_mod)
        scenario_goldens()
    random_stream_goldens()
