#!/usr/bin/env python
"""Frame-producer throughput: the native bulk producer (include/speechPlayer_ipa.h) against the reference's ipa.py
(the reference leg runs when NVSP_REFERENCE_DIR names an NVSpeechPlayer checkout, imported through tests/golden/make_golden.py).
Workload: the eight lines of sampleIpa.txt, speed 0.6, repeated; audio-seconds = sum of max(M+1, F+2) ticks / 22 050."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nvspeechplayer_b200 import ipa  # noqa: E402

gold = np.load(os.path.join(ROOT, "tests", "golden", "ipa_frames.npz"))
lines = [str(t) for t in gold["texts"][:8]]
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
texts = lines * reps
for threads in (1, 0):
    t0 = time.perf_counter()
    fb = ipa.frames_for_texts(texts, speed=0.6, sample_rate=22050, trailing_silence_ms=150.0, threads=threads)
    dt = time.perf_counter() - t0
    audio = float(fb.timeline_samples().sum()) / 22050.0
    print("native producer, %s: %d clauses, %d frames in %.3f s = %.0f clauses/s, %.3g audio-seconds/s"
          % ("1 thread" if threads == 1 else "%d threads" % os.cpu_count(), len(texts), int(fb.offsets[-1]), dt, len(texts) / dt, audio / dt))
if os.environ.get("NVSP_REFERENCE_DIR"):
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden import oracle, reference_package
    ref_ipa, sp = reference_package(oracle.REF_SO)
    n = max(reps // 50, 4)
    t0 = time.perf_counter()
    frames = 0
    for _ in range(n):
        for l in lines:
            for fr, d, f in ref_ipa.generateFramesAndTiming(l, speed=0.6):
                frames += 1
    dt = time.perf_counter() - t0
    audio_ref = audio / reps * n
    print("reference ipa.py, 1 core (frame objects built, no queueFrame call): %d clauses, %d frames in %.3f s = %.0f clauses/s, %.3g audio-seconds/s"
          % (8 * n, frames, dt, 8 * n / dt, audio_ref / dt))
