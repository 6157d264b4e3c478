"""Regenerate tests/golden/ipa_frames.npz from the REFERENCE's own ipa.py (needs an NVSpeechPlayer checkout named by
NVSP_REFERENCE_DIR, and oracle/_ref built from it).  For every (text, speed, basePitch, inflection, clauseType) case it stores what
ipa.generateFramesAndTiming yields -- the 47 frame values (zeros + isNull for silence), durationMs, fadeMs -- so that the
native bulk producer (include/speechPlayer_ipa.h) can be checked value for value where the reference is absent.

Cases: the eight lines of sampleIpa.txt with the recipe of test_speakIpa.py (speed 0.6) and with other speeds, pitches,
inflections and the four clause types; plus constructed strings that walk the rules: stress marks (primary / secondary),
tie bars (with and without a table entry for the pair), length marks, stops / affricates (pre-stop gaps, post-stop
aspiration), h between vowels and at the edges (_copyAdjacent), unknown characters, repeated blanks, the empty string."""
import codecs
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import REF, oracle, reference_package  # noqa: E402


def cases():
    lines = [l.strip() for l in codecs.open(os.path.join(REF, "sampleIpa.txt"), "r", "utf8").read().splitlines()]
    out = [(l, 0.6, 100, 0.5, None) for l in lines]
    out += [(l, 1.0, 120, 0.35, c) for l, c in zip(lines, [".", ",", "?", "!", ".", ",", "?", "!"])]
    out += [(lines[1], 1.7, 80, 1.0, "?"), (lines[2], 0.45, 210, 0.0, "!"), (lines[5], 2.5, 95, 0.75, ",")]
    made = [
        "",
        " ",
        "a",
        "ˈa",
        "hə",
        "əh",
        "aha",
        "ˈpɑ tɑ kɑ",
        "ˈtɑ ˌtɑ tɑ ˈtɑ tɑ",
        "spɪt stɪk skɪp",
        "t͡ʃɑt͡ʃ d͡ʒʌd͡ʒ",
        "a͡ɪ o͡ʊ e͡ɪ",
        "iː uː ɑː ɔː",
        "ˈsiːŋɪŋ ˌlɔːŋ ˈsɔŋz",
        "mɑlənə nɑməl",
        "lɑ wɑ jɑ ɹɑ",
        "ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ˈɑ ɑ",
        "ɑ ɑ ɑ ˈɑ ɑ ɑ ˈɑ ɑ ɑ ɑ ˈɑ ɑ",
        "x7q#  ˈkæt!  dɔɡ",
        "ˌɪntəˈnæʃənəl ˌɒpəˈɹeɪʃən",
        "ðə kwɪk bɹaʊn fɒks d͡ʒʌmps oʊvə ðə leɪzi dɒɡ",
        "ˈbʌtə ˈlɪtəl ˈbɒtəl",
        "θɪŋk ðɪs ʃʊd ʒɑ",
    ]
    for k, t in enumerate(made):
        out.append((t, [1.0, 0.6, 1.3][k % 3], [100, 140, 75][k % 3], [0.5, 0.25, 0.9][k % 3], [None, ".", ",", "?", "!"][k % 5]))
    return out


def main():
    ipa, sp = reference_package(oracle.REF_SO)
    names = [f[0] for f in sp.Frame._fields_]
    cs = cases()
    frames, dms, fms, nul, offsets = [], [], [], [], [0]
    for text, speed, pitch, infl, clause in cs:
        for fr, d, f in ipa.generateFramesAndTiming(text, speed=speed, basePitch=pitch, inflection=infl, clauseType=clause):
            frames.append(np.zeros(47) if fr is None else np.array([getattr(fr, n) for n in names]))
            nul.append(1 if fr is None else 0)
            dms.append(d)
            fms.append(f)
        offsets.append(len(dms))
    np.savez_compressed(os.path.join(HERE, "ipa_frames.npz"), texts=np.array([c[0] for c in cs]),
                        speed=np.array([c[1] for c in cs], dtype=np.float64), base_pitch=np.array([c[2] for c in cs], dtype=np.float64),
                        inflection=np.array([c[3] for c in cs], dtype=np.float64), clause=np.array([c[4] or "" for c in cs]),
                        offsets=np.array(offsets, dtype=np.int64), frames=np.array(frames).reshape(-1, 47), duration_ms=np.array(dms),
                        fade_ms=np.array(fms), is_null=np.array(nul, dtype=np.uint8))
    print("ipa golden: %d cases, %d frames (%d silence)" % (len(cs), len(dms), int(np.sum(nul))))


if __name__ == "__main__":
    main()
