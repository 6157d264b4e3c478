"""The zero-change route (BASELINE north star: "the speechPlayer.py ctypes wrapper and the ipa.py frame pipeline drive it
unchanged"): the engine behind an UNTYPED ctypes binding, exactly as reference speechPlayer.py:42-65 uses its DLL."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = oracle.REFERENCE


@pytest.mark.gpu
def test_untyped_wrapper_renders_config1_like_the_reference(tmp_path, golden_config1):
    """Fresh process (the library's default noise is the process-global glibc rand() replica from the default seed, like a
    fresh process of the reference), FP64 parity arithmetic: the reference's own PCM, sample for sample."""
    out = str(tmp_path / "pcm.npy")
    env = {k: v for k, v in os.environ.items() if not k.startswith("NVSP_")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "untyped_wrapper_driver.py"), out], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    pcm, want = np.load(out), golden_config1["pcm_libc"]
    assert len(pcm) == len(want) == 288454
    d = np.abs(pcm.astype(np.int64) - want.astype(np.int64))
    exact = float((d == 0).mean())
    print("untyped wrapper, config 1: exact %.6f, max |d| %d" % (exact, d.max()))
    assert exact >= 0.9999 and d.max() <= 1


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))),
                    reason="needs the reference's own Python files: an NVSpeechPlayer checkout in NVSP_REFERENCE_DIR")
def test_reference_python_files_load_and_queue_against_the_engine_library(tmp_path):
    """The reference's real speechPlayer.py / ipa.py / data.py, unmodified, in a throw-away package next to the engine's
    speechPlayer.dll: import, construct, run sampleIpa.txt through ipa.generateFramesAndTiming and queue every frame.
    Without a CUDA device speechPlayer_initialize returns NULL and every later call is a no-op on a bad handle (the
    reference has no error channel either), so this runs on the CPU box; with a device it renders."""
    code = r'''
import codecs, importlib, os, sys
pkg = os.path.join(sys.argv[1], "nvsp_ref")
os.mkdir(pkg)
open(os.path.join(pkg, "__init__.py"), "w").close()
for name in ("speechPlayer.py", "ipa.py", "data.py"):
    os.symlink(os.path.join(sys.argv[2], name), os.path.join(pkg, name))
os.symlink(os.path.join(sys.argv[3], "nvspeechplayer_b200", "speechPlayer.dll"), os.path.join(pkg, "speechPlayer.dll"))
sys.path.insert(0, sys.argv[1])
ipa = importlib.import_module("nvsp_ref.ipa")
sp = importlib.import_module("nvsp_ref.speechPlayer")
player = sp.SpeechPlayer(22050)
n = 0
for line in codecs.open(os.path.join(sys.argv[2], "sampleIpa.txt"), "r", "utf8").read().splitlines():
    for args in ipa.generateFramesAndTiming(line.strip(), speed=0.6):
        player.queueFrame(*args)
        n += 1
    player.queueFrame(None, 150, 0)
    n += 1
total = 0
while True:
    buf = player.synthesize(8192)
    if buf is None:
        break
    total += buf.length
print("queued", n, "rendered", total, "handle", player._speechHandle)
'''
    r = subprocess.run([sys.executable, "-c", code, str(tmp_path), REF, ROOT], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    words = r.stdout.split()
    assert words[0] == "queued" and int(words[1]) == 193, r.stdout
    if int(words[5]) != 0:  # a device was there: the whole utterance came out
        assert int(words[3]) == 288454, r.stdout
