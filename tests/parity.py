"""Shared parity metrics and bars (BASELINE.json north_star).

FP64 kernel : int16 bit-exact on >= 99.99 % of samples, <= 1 LSB on the rest.
FP32 kernel : <= 1 LSB on >= 99.9 % of samples and >= 60 dB SNR against the reference.
"""
import numpy as np

F32_WITHIN_1LSB = 0.999
F32_SNR_DB = 60.0


def metrics(got, want):
    """(fraction within 1 LSB, fraction exact, SNR dB, max |diff|) over the common prefix."""
    n = min(len(got), len(want))
    g = np.asarray(got[:n], dtype=np.float64)
    w = np.asarray(want[:n], dtype=np.float64)
    d = g - w
    sig, err = float((w * w).sum()), float((d * d).sum())
    snr = float("inf") if err == 0 else 10 * np.log10(max(sig, 1e-30) / err)
    if n == 0:
        return 1.0, 1.0, float("inf"), 0.0
    return float((np.abs(d) <= 1).mean()), float((d == 0).mean()), snr, float(np.abs(d).max())


def assert_f32_parity(got, want, what="", within=F32_WITHIN_1LSB, snr_db=F32_SNR_DB, short_ok=2):
    """The FP32 bar.  Two allowances, both for SHORT or SILENT renders only, and the margins are printed so the log shows
    how far inside the bar every case sits (pytest -s / -rA):
      * fewer than `short_ok` samples off by more than 1 LSB pass whatever the percentage (a 12-sample scenario cannot meet
        a 99.9 % bar with one 2-LSB sample);
      * the SNR bar is waived when the reference is silent (peak < 50) or -- for renders of at most 10 000 samples -- when
        no sample is off by more than 1 LSB."""
    assert len(got) == len(want), "%s: %d vs %d samples" % (what, len(got), len(want))
    w1, exact, snr, mx = metrics(got, want)
    bad = int(round((1 - w1) * len(want)))
    print("parity %-44s n=%8d  <=1LSB %.6f  exact %.6f  SNR %6.1f dB  max|d| %g" % (what, len(want), w1, exact, snr, mx))
    assert w1 >= within or bad <= short_ok, "%s: only %.5f within 1 LSB (max %g, snr %.1f dB)" % (what, w1, mx, snr)
    quiet = float(np.abs(np.asarray(want, dtype=np.float64)).max()) < 50 if len(want) else True
    short_and_tight = len(want) <= 10000 and mx <= 1
    assert snr >= snr_db or quiet or short_and_tight, "%s: SNR %.1f dB (max %g)" % (what, snr, mx)
    return w1, exact, snr, mx


def clusters(got, want, gap=2000):
    """Runs of samples off by more than 1 LSB, split where two of them are more than `gap` samples apart:
    [(first index, length, peak |d|)]."""
    n = min(len(got), len(want))
    d = np.abs(np.asarray(got[:n], dtype=np.int64) - np.asarray(want[:n], dtype=np.int64))
    bad = np.nonzero(d > 1)[0]
    if len(bad) == 0:
        return []
    runs = np.split(bad, np.nonzero(np.diff(bad) > gap)[0] + 1)
    return [(int(r[0]), int(r[-1] - r[0] + 1), int(d[r[0]:r[-1] + 1].max())) for r in runs]


def where_in_queue(index, min_dur, fade_dur):
    """(request, tick in that request, "pop" / "fade" / "hold") of output sample `index` of a queue rendered from a fresh
    player: request j occupies max(M+1, F+2) ticks (F = max(fadeDuration, 1)); its tick 0 pops it, ticks 1..F-1 fade."""
    m = np.asarray(min_dur, dtype=np.int64)
    f = np.maximum(np.asarray(fade_dur, dtype=np.int64), 1)
    start = np.concatenate([[0], np.cumsum(np.maximum(m + 1, f + 2))])
    j = int(np.searchsorted(start, index, side="right") - 1)
    c = int(index - start[j])
    return j, c, "pop" if c == 0 else ("fade" if c < f[min(j, len(f) - 1)] else "hold")


def assert_whole_stream(got, want, what, max_abs, snr_db, min_dur=None, fade_dur=None):
    """Maximum |difference| and SNR over the WHOLE stream (a long render must not hide a burst in its average).  On failure
    the message lists every cluster of samples off by more than 1 LSB (first index, length, peak), and, given the queue
    (min_dur, fade_dur), the request, tick and phase each cluster starts in."""
    assert len(got) == len(want), "%s: %d vs %d samples" % (what, len(got), len(want))
    w1, exact, snr, mx = metrics(got, want)
    print("parity %-44s n=%8d  <=1LSB %.6f  exact %.6f  SNR %6.1f dB  max|d| %g  (whole stream)" % (what, len(want), w1, exact, snr, mx))
    if mx <= max_abs and snr >= snr_db:
        return w1, exact, snr, mx
    lines = []
    for first, length, peak in clusters(got, want):
        line = "  at sample %d: %d samples, peak %d" % (first, length, peak)
        if min_dur is not None and fade_dur is not None:
            line += "  request %d tick %d (%s)" % where_in_queue(first, min_dur, fade_dur)
        lines.append(line)
    raise AssertionError("%s: SNR %.1f dB (bar %.1f), max|d| %g (bar %g), %d clusters of |d| > 1:\n%s"
                         % (what, snr, snr_db, mx, max_abs, len(lines), "\n".join(lines)))
