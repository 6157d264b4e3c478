// The rules of the reference's ipa.py (file:line at each step), stated once for the host producer (ipa_frames.cpp, g++)
// and the device producer (ipa_device.cu, nvcc).  No std:: containers: a text is a UTF-8 byte range read through a
// four-code-point window, and a phoneme list is an array of compact records (Rec, 40 bytes) that name table rows instead
// of carrying the 47 values.  The values are resolved only when a frame row is written (ipaCell): the phoneme's own row,
// then the row of its _copyAdjacent source for the parameters it lacks, then the two pitches.
//
// Why one source row is enough: _copyAdjacent (ipa.py:123-135) copies from the next phoneme unless it is silence, and the
// next phoneme has not been visited yet, so it contributes its table values.  When it copies from the previous phoneme,
// that one's values "after its own copy" are its table values plus what it took from its own next phoneme -- which is the
// phoneme being corrected -- so the parameters the corrected phoneme lacks come from the previous phoneme's table row.
//
// pow() is not called here: pitchPath's factors 2 ** (((pct - 50) / 50) * inflection) are computed by the host with
// std::pow (glibc, what ipa.py's ** uses) for every percent a clause type can produce (ipaPercents), and looked up by
// the exact value of the percent.  CUDA's pow differs from glibc's in the last bits.
//
// All arithmetic is in double in the reference's order of operations; the device unit builds with -fmad=false and the
// host with no contraction, so both give the same bits.
#pragma once
#include <stdint.h>

#include "../../include/speechPlayer_ipa.h"

#if defined(__CUDACC__)
#define NVSP_HD __host__ __device__
#else
#define NVSP_HD
#endif

namespace ipa {

constexpr int kParams = 47;
constexpr int kVoicePitch = 0, kPreFormantGain = 44, kOutputGain = 45, kEndVoicePitch = 46;  // src/frame.h:20-47
constexpr int kMaxPercents = 64;  // distinct pitch percents of one clause type (at most 46 with the reference's tables)
constexpr int kClauseTypes = 4;
constexpr uint32_t kNone = 0xFFFFFFFFu;  // no code point (before the first / after the last)

// decorations of a list entry (the reference's '_' keys) and which pitches pitchPath set
enum : uint16_t {
	kSilence = 1, kPreStopGap = 2, kPostStopAspiration = 4, kSyllableStart = 8, kWordStart = 16, kTiedTo = 32,
	kTiedFrom = 64, kLengthened = 128, kHasVoicePitch = 256, kHasEndVoicePitch = 512
};

struct Rec {
	double duration, fade, voicePitch, endVoicePitch;  // milliseconds; pitches valid where kHas*Pitch is set
	int16_t entry;     // table row, -1 for silence
	int16_t copyFrom;  // table row that fills the parameters `entry` lacks (_copyAdjacent), -1 for none
	uint16_t deco;
	uint8_t flags;     // SPEECHPLAYER_IPA_* of the table row
	int8_t stress;     // 0, 1 primary, 2 secondary
};
static_assert(sizeof(Rec) == 40, "a list entry is 40 bytes");

// The phoneme table as sorted arrays: keys are up to three code points, 21 bits each (first in the low bits).
struct TableView {
	const uint64_t *keys;
	const uint8_t *flags;
	const uint64_t *present;  // bit p: the row holds parameter p
	const double *values;     // [n][kParams]; read only by ipaCell
	int n, h;                 // h: the row of "h" (post-stop aspiration, ipa.py:104)
	NVSP_HD int find(uint64_t key) const {
		int lo = 0, hi = n;
		while (lo < hi) {
			const int mid = (lo + hi) >> 1;
			if (keys[mid] < key) lo = mid + 1;
			else hi = mid;
		}
		return (lo < n && keys[lo] == key) ? lo : -1;
	}
};

NVSP_HD inline uint64_t packKey(uint32_t a, uint32_t b = kNone, uint32_t c = kNone) {
	uint64_t k = a & 0x1FFFFFu;
	if (b != kNone) k |= (uint64_t)(b & 0x1FFFFFu) << 21;
	if (c != kNone) k |= (uint64_t)(c & 0x1FFFFFu) << 42;
	return k;
}

// UTF-8 over [p, end), ending early at a NUL byte; malformed or truncated sequences give U+FFFD
struct Utf8 {
	const unsigned char *p, *end;
	NVSP_HD bool next(uint32_t &c) {
		if (p >= end || *p == 0) return false;
		c = *p;
		const int extra = c < 0x80 ? 0 : (c >> 5) == 0x6 ? 1 : (c >> 4) == 0xE ? 2 : (c >> 3) == 0x1E ? 3 : -1;
		++p;
		if (extra < 0) { c = 0xFFFD; return true; }
		if (extra) c &= (0x3Fu >> extra);
		for (int k = 0; k < extra; ++k) {
			if (p >= end || (*p & 0xC0) != 0x80) { c = 0xFFFD; break; }
			c = (c << 6) | (*p & 0x3Fu);
			++p;
		}
		return true;
	}
};

// code points i-1 .. i+2 of a text (kNone outside it): all the look-around the rules use
struct Window {
	Utf8 src;
	uint32_t w[4];
	NVSP_HD explicit Window(Utf8 s) : src(s) {
		w[0] = kNone;
		for (int k = 1; k < 4; ++k) w[k] = pull();
	}
	NVSP_HD uint32_t pull() {
		uint32_t c;
		return src.next(c) ? c : kNone;
	}
	NVSP_HD void advance() {
		w[0] = w[1]; w[1] = w[2]; w[2] = w[3];
		w[3] = pull();
	}
};

// ipa.py:213-275
struct Intonation {
	double preHeadStart, preHeadEnd;
	int headExtendFrom, numSteps;
	double headStart, headEnd;
	double headSteps[9];
	double headStressEndDelta, headUnstressedRunStartDelta, headUnstressedRunEndDelta;
	double nucleus0Start, nucleus0End, nucleusStart, nucleusEnd, tailStart, tailEnd;
};
#define NVSP_IPA_INTONATION                                                                                                  \
	{{46, 57, 4, 9, 80, 50, {100, 75, 50, 25, 0, 63, 38, 13, 0}, -16, -8, -5, 64, 8, 70, 18, 24, 8},  /* '.' */          \
	 {46, 57, 4, 9, 80, 60, {100, 75, 50, 25, 0, 63, 38, 13, 0}, -16, -8, -5, 34, 52, 78, 34, 34, 52}, /* ',' */          \
	 {45, 56, 3, 8, 75, 43, {100, 75, 50, 20, 60, 35, 11, 0}, -16, -7, 0, 34, 68, 86, 21, 34, 68},     /* '?' */          \
	 {46, 57, 3, 8, 90, 50, {100, 75, 50, 16, 82, 50, 32, 16}, -16, -9, 0, 92, 4, 92, 80, 76, 4}}      /* '!' */
static const Intonation kIntonationHost[kClauseTypes] = NVSP_IPA_INTONATION;
#if defined(__CUDACC__)
__constant__ Intonation kIntonationDev[kClauseTypes] = NVSP_IPA_INTONATION;
#endif
NVSP_HD inline const Intonation &intonation(int clause) {
#if defined(__CUDA_ARCH__)
	return kIntonationDev[clause];
#else
	return kIntonationHost[clause];
#endif
}
// clause type character -> index into the intonation tables; 0 and unknown characters mean '.'
NVSP_HD inline int clauseIndex(char c) { return c == ',' ? 1 : c == '?' ? 2 : c == '!' ? 3 : 0; }

// the percents of the head (ipa.py:313-330), shared by the rules and by ipaPercents
NVSP_HD inline double headStepPercent(const Intonation &in, int step) {
	const int ns = in.numSteps;  // chain(steps, cycle(steps[extendFrom:]))
	const double v = step < ns ? in.headSteps[step] : in.headSteps[in.headExtendFrom + (step - ns) % (ns - in.headExtendFrom)];
	return in.headEnd + (((in.headStart - in.headEnd) / 100.0) * v);
}
NVSP_HD inline double stressEndPercent(const Intonation &in, double startP) { return startP + in.headStressEndDelta; }
NVSP_HD inline double runStartPercent(const Intonation &in, double stressEnd) { return stressEnd + in.headUnstressedRunStartDelta; }
NVSP_HD inline double runEndPercent(const Intonation &in, double stressEnd) { return stressEnd + in.headUnstressedRunEndDelta; }

// Every percent pitchPath can be given for one clause type, sorted and distinct, padded to kMaxPercents with +inf (the
// look-up's sentinel).  Host only in practice; it runs once per call.
inline int ipaPercents(const Intonation &in, double *out) {
	double v[kMaxPercents];
	int n = 0;
	const double fixed[8] = {in.preHeadStart, in.preHeadEnd, in.nucleus0Start, in.nucleus0End, in.nucleusStart, in.nucleusEnd,
	                         in.tailStart, in.tailEnd};
	for (double f : fixed) v[n++] = f;
	v[n++] = runStartPercent(in, 0.0);  // an unstressed run before any stressed step closed: stressEndPitch is still 0
	v[n++] = runEndPercent(in, 0.0);
	for (int s = 0; s < in.numSteps; ++s) {  // the cycle only revisits these steps
		const double startP = headStepPercent(in, s), endP = stressEndPercent(in, startP);
		v[n++] = startP;
		v[n++] = endP;
		v[n++] = runStartPercent(in, endP);
		v[n++] = runEndPercent(in, endP);
	}
	for (int i = 1; i < n; ++i)
		for (int j = i; j > 0 && v[j] < v[j - 1]; --j) { const double t = v[j]; v[j] = v[j - 1]; v[j - 1] = t; }
	int m = 0;
	for (int i = 0; i < n; ++i)
		if (m == 0 || v[i] != out[m - 1]) out[m++] = v[i];
	for (int i = m; i < kMaxPercents; ++i) out[i] = __builtin_inf();
	return m;
}

// pitchPath's factors of one (clause type, inflection): pct is the clause type's ipaPercents row, factor[k] belongs to pct[k]
struct Factors {
	const double *pct, *factor;
	NVSP_HD bool get(double percent, double &f) const {
		int lo = 0, hi = kMaxPercents;
		while (lo < hi) {
			const int mid = (lo + hi) >> 1;
			if (pct[mid] < percent) lo = mid + 1;
			else hi = mid;
		}
		if (lo == kMaxPercents || pct[lo] != percent) return false;
		f = factor[lo];
		return true;
	}
};

NVSP_HD inline Rec fromTable(const TableView &tab, int e) {
	Rec r;
	r.duration = r.fade = r.voicePitch = r.endVoicePitch = 0;
	r.entry = (int16_t)e;
	r.copyFrom = -1;
	r.deco = e < 0 ? kSilence : 0;
	r.flags = e < 0 ? 0 : tab.flags[e];
	r.stress = 0;
	return r;
}

// list sinks: the builder runs once counting entries and once writing them
struct CountSink {
	int64_t n = 0;
	NVSP_HD int64_t push(const Rec &) { return n++; }
	NVSP_HD void markSyllableStart(int64_t) {}
	NVSP_HD void setStress(int64_t, int) {}
};
struct WriteSink {
	Rec *r;
	int64_t n = 0;
	NVSP_HD int64_t push(const Rec &x) { r[n] = x; return n++; }
	NVSP_HD void markSyllableStart(int64_t i) { r[i].deco |= kSyllableStart; }
	NVSP_HD void setStress(int64_t i, int s) { r[i].stress = (int8_t)s; }
};

// ipa.py:39-121: characters -> phoneme list (the helper's per-character look-up and the list builder's syllable /
// aspiration / gap rules fused).  The rules read only the table flags of the previous entry, so the sink need not be
// readable.
template <class Sink>
NVSP_HD void buildList(const TableView &tab, Utf8 text, Sink &list) {
	const uint32_t kPrimary = 0x02C8, kSecondary = 0x02CC, kLong = 0x02D0, kTie = 0x0361;
	int pendingStress = 0;
	bool newWord = true;
	int64_t last = -1, syllableStartIdx = -1;
	uint8_t lastFlags = 0;
	for (Window t(text); t.w[1] != kNone; t.advance()) {
		const uint32_t ch = t.w[1];
		if (ch == kPrimary) { pendingStress = 1; continue; }
		if (ch == kSecondary) { pendingStress = 2; continue; }
		const bool lengthened = t.w[2] == kLong;
		const bool tiedTo = t.w[2] == kTie;
		const bool tiedFrom = t.w[0] == kTie;
		int e = -1, skip = 0;
		if (tiedTo) {  // ipa.py:60-62: the tied pair as one phoneme if the table has it (min(3, n - i) code points)
			e = tab.find(packKey(ch, t.w[2], t.w[3]));
			skip = e >= 0 ? 2 : 1;
		} else if (lengthened) {  // :63-65
			e = tab.find(packKey(ch, t.w[2]));
			skip = 1;
		}
		if (e < 0) e = tab.find(packKey(ch));
		if (e < 0) {  // :68-70: not a phoneme; a blank starts a new word (:93-94)
			if (ch == 0x20) newWord = true;
			for (; skip; --skip) t.advance();
			continue;
		}
		Rec ph = fromTable(tab, e);
		const int stress = pendingStress;  // :72-74 and the pop at :97
		pendingStress = 0;
		if (tiedFrom) ph.deco |= kTiedFrom;  // :75-78
		else if (tiedTo) ph.deco |= kTiedTo;
		if (lengthened) ph.deco |= kLengthened;
		// ---- list builder, ipa.py:96-120 ----
		bool selfSyllableStart = false;
		if (last >= 0 && !(lastFlags & SPEECHPLAYER_IPA_VOWEL) && (ph.flags & SPEECHPLAYER_IPA_VOWEL)) {
			list.markSyllableStart(last);  // a consonant before a vowel opens the syllable
			syllableStartIdx = last;
		} else if (stress == 1 && last >= 0 && (lastFlags & SPEECHPLAYER_IPA_VOWEL)) {
			ph.deco |= kSyllableStart;
			selfSyllableStart = true;
		}
		if (last >= 0 && (lastFlags & SPEECHPLAYER_IPA_STOP) && !(lastFlags & SPEECHPLAYER_IPA_VOICED) &&
		    (ph.flags & SPEECHPLAYER_IPA_VOICED) && !(ph.flags & SPEECHPLAYER_IPA_STOP) && !(ph.flags & SPEECHPLAYER_IPA_AFRICATE)) {
			Rec asp = fromTable(tab, tab.h);  // :104-108 post-stop aspiration
			asp.deco |= kPostStopAspiration;
			last = list.push(asp);
			lastFlags = asp.flags;
		}
		if (newWord) {  // :109-113
			newWord = false;
			ph.deco |= kWordStart | kSyllableStart;
			selfSyllableStart = true;
		}
		const bool stopLike = (ph.flags & (SPEECHPLAYER_IPA_STOP | SPEECHPLAYER_IPA_AFRICATE)) != 0;
		if (!stress && stopLike) {  // :116-118 (the elif of the stress test)
			Rec gap = fromTable(tab, -1);
			gap.deco |= kPreStopGap;
			list.push(gap);
		}
		const int64_t self = list.push(ph);
		if (selfSyllableStart) syllableStartIdx = self;
		if (stress && syllableStartIdx >= 0) list.setStress(syllableStartIdx, stress);  // :114-115
		last = self;
		lastFlags = ph.flags;
		for (; skip; --skip) t.advance();
	}
}

// ipa.py:123-135 (see the top of this file for why one source row suffices)
NVSP_HD inline void copyAdjacent(Rec *list, int64_t n) {
	for (int64_t i = 0; i < n; ++i) {
		if (!(list[i].flags & SPEECHPLAYER_IPA_COPY_ADJACENT)) continue;
		const Rec *next = i + 1 < n ? &list[i + 1] : nullptr;
		const Rec *prev = i > 0 ? &list[i - 1] : nullptr;
		const Rec *adj = (next && !(next->deco & kSilence)) ? next : prev;
		if (adj) list[i].copyFrom = adj->entry;  // -1 (silence) holds nothing to copy
	}
}

// ipa.py:137-189
NVSP_HD inline void assignTimes(Rec *list, int64_t n, double baseSpeed) {
	int syllableStress = 0;
	double speed = baseSpeed;
	for (int64_t i = 0; i < n; ++i) {
		Rec &ph = list[i];
		const Rec *next = i + 1 < n ? &list[i + 1] : nullptr;
		const Rec *last = i > 0 ? &list[i - 1] : nullptr;
		if (ph.deco & kSyllableStart) {
			syllableStress = ph.stress;
			if (syllableStress) speed = syllableStress == 1 ? baseSpeed / 1.4 : baseSpeed / 1.1;
			else speed = baseSpeed;
		}
		double dur = 60.0 / speed, fade = 10.0 / speed;
		if (ph.deco & kPreStopGap) {
			dur = 41.0 / speed;
		} else if (ph.deco & kPostStopAspiration) {
			dur = 20.0 / speed;
		} else if (ph.flags & SPEECHPLAYER_IPA_STOP) {
			const double d = 6.0 / speed;
			dur = (6.0 < d) ? 6.0 : d;  // std::min(6.0 / speed, 6.0)
			fade = 0.001;
		} else if (ph.flags & SPEECHPLAYER_IPA_AFRICATE) {
			dur = 24.0 / speed;
			fade = 0.001;
		} else if (!(ph.flags & SPEECHPLAYER_IPA_VOICED)) {
			dur = 45.0 / speed;
		} else if (ph.flags & SPEECHPLAYER_IPA_VOWEL) {
			if (last && (last->flags & (SPEECHPLAYER_IPA_LIQUID | SPEECHPLAYER_IPA_SEMIVOWEL))) fade = 25.0 / speed;
			if (ph.deco & kTiedTo) {
				dur = 40.0 / speed;
			} else if (ph.deco & kTiedFrom) {
				dur = 20.0 / speed;
				fade = 20.0 / speed;
			} else if (!syllableStress && !(ph.deco & kSyllableStart) && next && !(next->deco & kWordStart) &&
			           (next->flags & (SPEECHPLAYER_IPA_LIQUID | SPEECHPLAYER_IPA_NASAL))) {
				dur = (next->flags & SPEECHPLAYER_IPA_LIQUID) ? 30.0 / speed : 40.0 / speed;
			}
		} else {  // voiced consonant
			dur = 30.0 / speed;
			if (ph.flags & (SPEECHPLAYER_IPA_LIQUID | SPEECHPLAYER_IPA_SEMIVOWEL)) fade = 20.0 / speed;
		}
		if (ph.deco & kLengthened) dur *= 1.05;
		ph.duration = dur;
		ph.fade = fade;
	}
}

// ipa.py:191-211; false when a percent has no factor
NVSP_HD inline bool pitchPath(Rec *list, int64_t start, int64_t end, double basePitch, const Factors &fx, double startPercent,
                              double endPercent) {
	double fs, fe;
	if (!fx.get(startPercent, fs) || !fx.get(endPercent, fe)) return false;
	const double startPitch = basePitch * fs;
	const double endPitch = basePitch * fe;
	double voiced = 0;
	for (int64_t i = start; i < end; ++i)
		if (list[i].flags & SPEECHPLAYER_IPA_VOICED) voiced += list[i].duration;
	double cur = 0;
	const double delta = endPitch - startPitch;
	double pitch = startPitch;
	for (int64_t i = start; i < end; ++i) {
		Rec &ph = list[i];
		ph.voicePitch = pitch;
		if (ph.flags & SPEECHPLAYER_IPA_VOICED) {
			cur += ph.duration;
			const double ratio = cur / voiced;
			pitch = startPitch + (delta * ratio);
		}
		ph.endVoicePitch = pitch;
		ph.deco |= kHasVoicePitch | kHasEndVoicePitch;
	}
	return true;
}

// ipa.py:277-334: pre-head, head (stressed steps and unstressed runs), nucleus, tail.  False on a factor miss.
NVSP_HD inline bool assignPitches(Rec *list, int64_t n, double basePitch, int clause, const Factors &fx) {
	const Intonation &in = intonation(clause);
	bool ok = true;
	auto isStart = [&](int64_t i) { return (list[i].deco & kSyllableStart) != 0; };
	int64_t preHeadEnd = n;
	for (int64_t i = 0; i < n; ++i)
		if (isStart(i) && list[i].stress == 1) { preHeadEnd = i; break; }
	if (preHeadEnd > 0) ok &= pitchPath(list, 0, preHeadEnd, basePitch, fx, in.preHeadStart, in.preHeadEnd);
	int64_t nucleusStart = n, nucleusEnd = n, tailStart = n;
	const int64_t tailEnd = n;
	for (int64_t i = nucleusEnd - 1; i >= preHeadEnd; --i) {
		if (!isStart(i)) continue;
		if (list[i].stress == 1) { nucleusStart = i; break; }
		nucleusEnd = tailStart = i;
	}
	const bool hasTail = tailEnd - tailStart > 0;
	if (hasTail) ok &= pitchPath(list, tailStart, tailEnd, basePitch, fx, in.tailStart, in.tailEnd);
	if (nucleusEnd - nucleusStart > 0) {
		if (hasTail) ok &= pitchPath(list, nucleusStart, nucleusEnd, basePitch, fx, in.nucleusStart, in.nucleusEnd);
		else ok &= pitchPath(list, nucleusStart, nucleusEnd, basePitch, fx, in.nucleus0Start, in.nucleus0End);
	}
	if (preHeadEnd < nucleusStart) {
		int64_t stressRunStart = -1, unstressedRunStart = -1;
		double stressEndPitch = 0;
		int step = 0;
		for (int64_t i = preHeadEnd; i <= nucleusStart && i < n; ++i) {
			if (!isStart(i)) continue;
			if (stressRunStart >= 0) {
				const double startP = headStepPercent(in, step++);
				stressEndPitch = stressEndPercent(in, startP);
				ok &= pitchPath(list, stressRunStart, i, basePitch, fx, startP, stressEndPitch);
				stressRunStart = -1;
			}
			if (list[i].stress == 1) {
				if (unstressedRunStart >= 0) {
					ok &= pitchPath(list, unstressedRunStart, i, basePitch, fx, runStartPercent(in, stressEndPitch),
					                runEndPercent(in, stressEndPitch));
					unstressedRunStart = -1;
				}
				stressRunStart = i;
			} else if (unstressedRunStart < 0) {
				unstressedRunStart = i;
			}
		}
	}
	return ok;
}

// entries of one text: the phoneme list plus the trailing silence
NVSP_HD inline int64_t ipaCount(const TableView &tab, Utf8 text, double trailingSilenceMs) {
	CountSink c;
	buildList(tab, text, c);
	return c.n + (trailingSilenceMs >= 0 ? 1 : 0);
}

// ipa.py:336-353 + the trailing silence of reference test_speakIpa.py:26: writes ipaCount entries to out.  False on a
// factor miss.
NVSP_HD inline bool ipaRecords(const TableView &tab, Utf8 text, double speed, double basePitch, int clause, const Factors &fx,
                               double trailingSilenceMs, Rec *out, int64_t *written) {
	WriteSink w{out};
	buildList(tab, text, w);
	bool ok = true;
	if (w.n) {
		copyAdjacent(out, w.n);
		assignTimes(out, w.n, speed);
		ok = assignPitches(out, w.n, basePitch, clause, fx);
	}
	if (trailingSilenceMs >= 0) {
		Rec s = fromTable(tab, -1);
		s.duration = trailingSilenceMs;
		w.push(s);
	}
	*written = w.n;
	return ok;
}

// parameter p of the frame row of entry r (ipa.py:349-351): silence rows are zero; otherwise preFormantGain 1 and
// outputGain 2 under the phoneme's own values, the copied values and the pitches
NVSP_HD inline double ipaCell(const TableView &tab, const Rec &r, int p) {
	if (r.deco & kSilence) return 0.0;
	if (p == kVoicePitch && (r.deco & kHasVoicePitch)) return r.voicePitch;
	if (p == kEndVoicePitch && (r.deco & kHasEndVoicePitch)) return r.endVoicePitch;
	if (tab.present[r.entry] >> p & 1) return tab.values[(size_t)r.entry * kParams + p];
	if (r.copyFrom >= 0 && (tab.present[r.copyFrom] >> p & 1)) return tab.values[(size_t)r.copyFrom * kParams + p];
	return p == kPreFormantGain ? 1.0 : p == kOutputGain ? 2.0 : 0.0;
}

// reference speechPlayer.py:51-53: int(ms * (sampleRate / 1000.0))
NVSP_HD inline unsigned int msToSamples(double ms, double perMs) { return (unsigned int)(long long)(ms * perMs); }

}  // namespace ipa
