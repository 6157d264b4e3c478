// klatt_pull: the low-latency path of the per-handle API (SURVEY 8f rank 3): ONE pull of one player
// (speechPlayer_synthesize(handle, n, buf), the call the NVDA audio thread makes, reference
// nvdaAddon/synthDrivers/nvSpeechPlayer/__init__.py:56-82) rendered by ONE thread block, parallel in time, with the
// state of the stream carried in and out.  It is klatt_long.cu's scheme (affine maps of the two-pole sections over a
// chunk, composed by a scan) brought down to chunks of <= 16 ticks held in shared memory, and the tick both render is
// klatt_tick_core.cuh's:
//
//   host   the frame manager runs at REQUEST granularity in FP64, exactly as reference src/frame.cpp:41-115 (pop,
//          NULL-frame rewrites, swap, hold glide, drain, purge): pull_manager.h.  For a pull it emits the runs of ticks
//          (PullSeg) the pull consists of, each with the fade plan of its request (planFade, klatt_f32_core.cuh) and the
//          values in force on the pop tick.  Everything a tick needs is then a closed form of (segment, sampleCounter).
//   device 512 threads, thread i renders ticks [i*L, (i+1)*L) of the pull, L = ceil(n / 512).  Source (vibrato, the two
//          coloured noises; the glottal phase recurrence is the one serial step, see "source" below), parallel bank,
//          rN0+rNP, r6 ... r1: per stage, pass 1 runs the chunk from zero state and accumulates its affine map, a block scan
//          (warp shuffles, seeded with the carried-in state) gives every chunk its true start state, pass 2 renders the
//          chunk in place in shared memory.  The last stage fuses mix, gain, clamp and the int16 store.
//
// The per-thread passes below are written against plain pointers (KLATT_HD) so that tests/hostsim can run the very
// same arithmetic "thread by thread" on the host; only the block scans differ (shuffles on the device, a plain loop in
// the test build).  The arithmetic of a tick is the FP32 formulation of klatt_f32_core.cuh; parity with the reference is
// by the FP32 bar (<= 1 LSB on >= 99.9 %, >= 60 dB), not bit for bit (the scan re-associates).
#pragma once
#include "klatt_common.h"
#include "klatt_f32_core.cuh"
#include "klatt_tick_core.cuh"

namespace klatt {

constexpr int kPullThreads = 512;
constexpr uint32_t kPullMaxTicks = 8192;  // per launch: <= 16 ticks per thread, two float signals = 64 KB of shared memory
constexpr uint32_t kPullMaxSegs = 32;     // requests one launch may touch (a longer pull is cut into several launches)

// One run of consecutive ticks of one request inside a pull.
struct alignas(16) PullSeg {
	FadePlanF32 plan;                       // fade old -> new of the request (src/frame.cpp:49-52), pitch excluded
	double fb[kNumResonators][4];           // f0, f1, b0, b1 of each section (NaN targets resolved): exact pole on re-basing
	double pitchStale, pitchOld, pitchNew;  // cur.voicePitch on the pop tick; end points of the fade (frame.cpp:61,71)
	double pitchInc;                        // hold glide (frame.cpp:77,98)
	uint64_t vibPosAtPop;                   // vibrato phase before the pop tick, 2^-64 cycles
	int64_t vibIncStale;                    // vibrato increment on the pop tick
	double depthStale;                      // vibrato depth 0.06 * vibratoPitchOffset on the pop tick
	float dirStale[kNumDirect];             // direct params on the pop tick (curFrame is not touched there, frame.cpp:55-72)
	float zStaleRe[kNumResonators], zStaleIm[kNumResonators];
	uint32_t n0InvStale;
	uint32_t F;          // numFadeSamples, >= 1 (reference src/speechPlayer.cpp:36)
	uint32_t c0;         // sampleCounter on the run's first tick (0 = the pop tick)
	uint32_t tickStart;  // first tick of the run, counted from the start of the pull
	uint32_t count;
	uint32_t pad[1];
};
static_assert(sizeof(PullSeg) % 16 == 0, "segments are copied as 16-byte words");

// What a player carries from one pull to the next (device memory).
struct PullState {
	float y[kNumResonators];  // delta-form memories as in GenStateF32: last output; rN0: last INPUT
	float d[kNumResonators];  //                                          last output difference; rN0: last input difference
	float aspLast, fricLast;  // coloured-noise memories, units of 2^-23
	double pitchPos;          // glottal phase in cycles, FP64 and accumulated exactly like the reference's (:55)
	uint64_t generated;       // samples generated so far == noise draws consumed / 2
};

struct PullPhaseRec;
struct PullCtx {
	const PullSeg *segs;
	uint32_t nSeg, n, L;  // n ticks in this pull, L ticks per thread
	int sampleRate;
	float *sigA, *sigB;   // [L][kPullThreads]: tick t of the pull lives at (t % L) * kPullThreads + t / L
	double *inc;          // same layout: glottal phase increment of every tick, overwritten with the phase after the tick
	// phaseMode 1 ("runs", the default): scratch of the run decomposition of the phase recurrence (see pullRuns*)
	int phaseMode;
	int64_t *runI;        // [L][kPullThreads], 8 bytes per tick: may share the storage of sigA + sigB (both dead until pass 2)
	uint16_t *runMeta;    // [n], by tick: may share the storage of the int16 output (dead until the last stage)
	struct PullPhaseRec *rec;  // [kPullMaxSpecial]
	PullState *state;
	long long *dbg;       // optional (NVSP_PULL_DEBUG): SM cycle counter at the phase boundaries of the launch
	int noiseMode;
	uint64_t seed, streamId;
	const int32_t *draws;  // kNoiseGlibc / kNoiseReplay: rand() values, draw 2g = aspiration, 2g+1 = frication
	uint64_t drawBase, drawLen;
	int16_t *pcm;
};

// one player's pull inside a batched launch (klatt_pull_batch_kernel)
struct PullBatchItem {
	PullCtx ctx;
	const PullSeg *segSrc;
	int16_t *pcmOut;
};

// the pull path's names for the records of klatt_tick_core.cuh (the host model in tests/hostsim uses them)
typedef Affine PullAffine;
typedef PoleWalk PullPole;
template <int STAGE> using PullStageTraits = StageTraits<STAGE>;
constexpr int kPullParallel = kStageParallel, kPullNasal = kStageNasal, kPullCascade = kStageCascade, kPullLast = kStageLast;

struct PullStart {
	float y, d;
};

// the request laws of klatt_tick_core.cuh on tick (seg, c), with the values on the pop tick the segment carries
KLATT_HD uint64_t pullVibBefore(const PullSeg &s, uint32_t c) {
	return vibBeforeLaw(c, s.F, s.vibIncStale, s.plan.vibInc0, s.plan.vibIncStep, s.plan.vibIncFinal);
}
KLATT_HD float pullDirAt(const PullSeg &s, int slot, uint32_t c) {
	return dirLaw(c, s.F, s.dirStale[slot], s.plan.dir0[slot], s.plan.dirStep[slot], s.plan.dirFinal[slot]);
}

// where a tick sits: segment, sampleCounter value on that tick, ticks of the segment still to come (this one included)
struct PullCursor {
	uint32_t s, c, left;
	KLATT_HD void seek(const PullCtx &X, uint32_t t) {
		uint32_t lo = 0, hi = X.nSeg;  // last segment with tickStart <= t
		while (hi - lo > 1) {
			uint32_t mid = (lo + hi) >> 1;
			if (X.segs[mid].tickStart <= t) lo = mid; else hi = mid;
		}
		s = lo;
		c = X.segs[s].c0 + (t - X.segs[s].tickStart);
		left = X.segs[s].count - (t - X.segs[s].tickStart);
	}
	KLATT_HD void next(const PullCtx &X) {
		++c;
		if (--left == 0 && s + 1 < X.nSeg) {
			++s;
			c = X.segs[s].c0;
			left = X.segs[s].count;
		}
	}
};

// zeta of section r on fade tick k from the closed form of the pole (PoleWalk's `exact`).  The arguments are formed in
// double, the exponential and the sine / cosine in FP32 with the cancellation-free expressions of oneMinusExp(): zeta is kept
// in FP32 anyway, and 512 threads x 14 sections x (expm1 + sincos) in double was the largest fixed cost of a launch.
KLATT_HD void pullPoleExact(const PullSeg &S, uint32_t k, int r, double srInv, float &zr, float &zi) {
	const double PI = 3.14159265358979323846;
	const double ratio = (double)((float)k / (float)S.F);
	const double f0 = S.fb[r][0], f1 = S.fb[r][1], b0 = S.fb[r][2], b1 = S.fb[r][3];
	const float x = (float)(-PI * (b0 + ((b1 - b0) * ratio)) * srInv);     // log of the pole radius
	const float hth = (float)(PI * (f0 + ((f1 - f0) * ratio)) * srInv);    // half the pole angle
	const float em1 = expm1f(x);
	const float rad = 1.0f + em1;
	float sh, ch;
	sincosf(hth, &sh, &ch);
	zr = fmaf((2.0f * rad) * sh, sh, -em1);
	zi = -rad * ((2.0f * sh) * ch);
}

// PoleWalk of section r along the pull: the pop tick of a segment sets what was in force before it
KLATT_HD void pullPoleSeek(PoleWalk &w, const PullSeg &S, uint32_t c, int r, double srInv) {
	w.seek(S.plan, c, S.F, r, S.zStaleRe[r], S.zStaleIm[r], [&](uint32_t k, float &zr, float &zi) { pullPoleExact(S, k, r, srInv, zr, zi); });
}
KLATT_HD void pullPoleTick(PoleWalk &w, const PullSeg &S, uint32_t c, int r, double srInv) {
	if (c == 0) w = PoleWalk{S.zStaleRe[r], S.zStaleIm[r], 0.0f, 0.0f};
	else w.tick(S.plan, c, S.F, r, [&](uint32_t k, float &zr, float &zi) { pullPoleExact(S, k, r, srInv, zr, zi); });
}

KLATT_HD uint32_t pullIdx(const PullCtx &X, uint32_t t) { return (t % X.L) * (uint32_t)kPullThreads + t / X.L; }

// the two noise words of generated sample g (word position: the 23 bits used are w >> 9)
KLATT_HD void pullNoiseWords(const PullCtx &X, uint64_t g, Philox4 &blk, uint64_t &blkIndex, uint32_t &wA, uint32_t &wF) {
	if (X.noiseMode == kNoisePhilox) {
		const uint64_t b = g >> 1;
		if (b != blkIndex) { blk = noiseBlock(X.seed, X.streamId, b); blkIndex = b; }
		wA = (g & 1) ? blk.w[2] : blk.w[0];
		wF = (g & 1) ? blk.w[3] : blk.w[1];
	} else {  // rand() values (31 bits): shift into word position
		const uint64_t d0 = 2 * g - X.drawBase;
		wA = (d0 < X.drawLen) ? ((uint32_t)X.draws[d0] << 1) : 0u;
		wF = (d0 + 1 < X.drawLen) ? ((uint32_t)X.draws[d0 + 1] << 1) : 0u;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// source (reference src/speechWaveGenerator.cpp:32-88, :204-206)
//
// The glottal phase is the one quantity of the path that is NOT rendered in parallel: the reference accumulates it as
// fmod(pos + f/sr, 1) in double (src/speechWaveGenerator.cpp:55), and a pitch whose period is a whole number of samples
// (150 Hz at 22 050 Hz) makes the wrap instant a matter of the last bit of that running sum -- a wrap one sample apart
// from the reference's is a full-scale error once per period (klatt_f32_core.cuh OscChain has the same concern).  No
// associative reformulation reproduces a sequence of roundings, so: every thread prepares the per-tick increments of
// its chunk in parallel (vibrato sine, pitch, the correctly rounded division -- the expensive part), and ONE thread then
// runs the bare recurrence pos = frac(pos + inc[t]) over the pull, two dependent FP64 additions per tick.
// ---------------------------------------------------------------------------------------------------------------
struct PullSourceSums {
	float zAsp, zFric;   // colouring filters at the end of the chunk when started from zero
	float decay;         // 0.75 ^ (ticks in the chunk)
	uint64_t phaseFixed; // what the chunk adds to the phase in 2^-64 cycles (exact, associative: the APPROXIMATE phase
	                     // the run decomposition classifies ticks with)
};

struct PullOsc {  // vibrato + pitch along the pull
	PullCursor cur;
	uint64_t vibPos;
	double glide;                     // voicePitch on tick (glideSeg, glideC), the last one pitch() rendered
	uint32_t glideSeg, glideC;
	KLATT_HD void seek(const PullCtx &X, uint32_t t) {
		cur.seek(X, t);
		const PullSeg &S = X.segs[cur.s];
		vibPos = S.vibPosAtPop + pullVibBefore(S, cur.c);
		glide = 0.0; glideSeg = 0xffffffffu; glideC = 0;
	}
	// cur.voicePitch on the current tick (pitchTick)
	KLATT_HD double pitch(const PullSeg &S) {
		const double p = pitchTick(glide, glideSeg == cur.s && glideC + 1u == cur.c, cur.c, S.F, S.pitchStale, S.pitchOld, S.pitchNew,
		                           S.pitchInc);
		glideSeg = cur.s; glideC = cur.c;
		return p;
	}
	// what this tick adds to the glottal phase, in cycles
	KLATT_HD double phaseInc(const PullCtx &X, double srD, double srInv) {
		const PullSeg &S = X.segs[cur.s];
		const uint32_t c = cur.c;
		return glottalInc(vibPos, vibIncLaw(c, S.F, S.vibIncStale, S.plan.vibInc0, S.plan.vibIncStep, S.plan.vibIncFinal), pitch(S),
		                  depthLaw(c, S.F, S.depthStale, S.plan.depth0, S.plan.depthStep, S.plan.depthFinal), srD, srInv);
	}
	KLATT_HD void next(const PullCtx &X) {
		const uint32_t was = cur.s;
		cur.next(X);
		if (cur.s != was) vibPos = X.segs[cur.s].vibPosAtPop + pullVibBefore(X.segs[cur.s], cur.c);
	}
};

KLATT_HD void pullChunkRange(const PullCtx &X, uint32_t ch, uint32_t &t0, uint32_t &t1) {
	const uint64_t a = (uint64_t)ch * X.L;
	t0 = a < X.n ? (uint32_t)a : X.n;
	t1 = (a + X.L < X.n) ? (uint32_t)(a + X.L) : X.n;
}

// pass 1: the phase increment of every tick of the chunk -> X.inc, and what the chunk adds to the two noise filters
KLATT_HD void pullSourcePass1(const PullCtx &X, uint32_t ch, PullSourceSums &out) {
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	out.zAsp = 0.0f; out.zFric = 0.0f; out.decay = 1.0f; out.phaseFixed = 0;
	if (t0 >= t1) return;
	const double srD = (double)X.sampleRate, srInv = 1.0 / srD;
	const uint64_t g0 = X.state->generated;
	PullOsc w;
	w.seek(X, t0);
	Philox4 blk;
	blk.w[0] = blk.w[1] = blk.w[2] = blk.w[3] = 0;
	uint64_t blkIndex = ~0ull;
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		uint32_t wA, wF;
		pullNoiseWords(X, g0 + t, blk, blkIndex, wA, wF);
		out.zAsp = colourNoise(out.zAsp, wA);
		out.zFric = colourNoise(out.zFric, wF);
		out.decay *= 0.75f;
		const double pinc = w.phaseInc(X, srD, srInv);
		X.inc[at] = pinc;
		if (X.phaseMode) out.phaseFixed += (uint64_t)cyclesToFixed(pinc);
		w.next(X);
	}
}

// the recurrence itself (one thread): X.inc[t] <- glottal phase after tick t (src/speechWaveGenerator.cpp:55, :74).
// A wrap happens once per pitch period, so the ticks are taken in groups of up to 8: the running sums of a group are
// formed as if there were no wrap (one dependent FP64 addition per tick, nothing else on the chain), and only if one of
// them left (-1, 1) is the group redone tick by tick with the reference's fmod.  Same roundings either way.
KLATT_HD int32_t pullHiWord(double x) {
#ifdef __CUDA_ARCH__
	return __double2hiint(x);
#else
	int64_t b;
	memcpy(&b, &x, 8);
	return (int32_t)(b >> 32);
#endif
}
template <int LL>
KLATT_HD void pullPhaseSerialL(const PullCtx &X) {
	constexpr int G = LL < 8 ? LL : 8;
	constexpr uint32_t GP = LL / G;  // groups per chunk
	double pos = X.state->pitchPos;
	const uint32_t fullChunks = X.n / LL;
	const uint32_t groups = fullChunks * GP;
	// X.inc is overwritten in place with the phase after each tick (as a double: the conversion to the FP32 sawtooth value
	// is left to the parallel pass that consumes it -- a conversion and a dependent store per tick in THIS loop cost more
	// than the additions).  The increments of the next group are fetched while the current one is summed.
	double a[G], nx[G];
#pragma unroll
	for (int k = 0; k < G; ++k) nx[k] = 0.0;
	if (groups) {
#pragma unroll
		for (int k = 0; k < G; ++k) nx[k] = X.inc[(uint32_t)k * kPullThreads];
	}
	for (uint32_t gi = 0; gi < groups; ++gi) {
		const uint32_t base = (gi % GP) * (uint32_t)(G * kPullThreads) + gi / GP;  // the group's first tick
#pragma unroll
		for (int k = 0; k < G; ++k) a[k] = nx[k];
		if (gi + 1 < groups) {
			const uint32_t nb = ((gi + 1) % GP) * (uint32_t)(G * kPullThreads) + (gi + 1) / GP;
#pragma unroll
			for (int k = 0; k < G; ++k) nx[k] = X.inc[nb + (uint32_t)k * kPullThreads];
		}
		double sum[G];
		sum[0] = pos + a[0];
#pragma unroll
		for (int k = 1; k < G; ++k) sum[k] = sum[k - 1] + a[k];
		int32_t top = 0;
#pragma unroll
		for (int k = 0; k < G; ++k) {
			const int32_t h = pullHiWord(sum[k]) & 0x7fffffff;
			top = h > top ? h : top;
		}
		if (top < 0x3ff00000) {  // every |sum| < 1: no wrap in this group
#pragma unroll
			for (int k = 0; k < G; ++k) X.inc[base + (uint32_t)k * kPullThreads] = sum[k];
			pos = sum[G - 1];
		} else {
#pragma unroll
			for (int k = 0; k < G; ++k) {
				pos = fracRef(a[k] + pos);
				X.inc[base + (uint32_t)k * kPullThreads] = pos;
			}
		}
	}
	const uint32_t tail = X.n - fullChunks * LL;  // the last, shorter chunk
	for (uint32_t i = 0; i < tail; ++i) {
		pos = fracRef(X.inc[i * kPullThreads + fullChunks] + pos);
		X.inc[i * kPullThreads + fullChunks] = pos;
	}
	X.state->pitchPos = pos;
}
KLATT_HD void pullPhaseSerial(const PullCtx &X) {  // X.L is one of the lengths launchKlattPull chooses from
	switch (X.L) {
		case 1: pullPhaseSerialL<1>(X); break;
		case 2: pullPhaseSerialL<2>(X); break;
		case 4: pullPhaseSerialL<4>(X); break;
		case 8: pullPhaseSerialL<8>(X); break;
		default: pullPhaseSerialL<16>(X); break;
	}
}
KLATT_HD uint32_t pullTicksPerThread(uint32_t n) {
	uint32_t L = 1;
	while (L * (uint32_t)kPullThreads < n) L <<= 1;
	return L;
}

// ---------------------------------------------------------------------------------------------------------------
// Run decomposition of the phase recurrence (phaseMode 1, the default; NVSP_PULL_PHASE=serial selects the loop above).
// While the phase stays inside one binade [2^k, 2^(k+1)) every value it takes is a multiple of that binade's ulp
// u = 2^(k-52), so RN(pos + inc) = pos + RN_u(inc) unless inc/u lies exactly half-way: the rounded increments are
// integers on a fixed grid and the recurrence is an integer prefix sum -- associative, scannable, and bit for bit what
// the FP64 additions would have produced.  Only the SPECIAL ticks need the real FP64 addition, in order: wraps, binade
// crossings, ties, non-positive or huge increments, and ticks whose approximate phase (the exact 2^-64 fixed-point
// prefix sum, off by < 1e-12) is within 2^-30 of a binade boundary.  They are 1-20 % of the ticks
// (tools/phase_runs_study.py, which also checks the decomposition bit for bit against the serial loop).
//   classify   per tick, from the approximate phase: normal (k, I = RN_u(inc)/u) or special; per chunk: sum of I behind
//              its last special tick, number of special ticks                       -> segmented block scan
//   offsets    per normal tick: off = (sum of I since the last special tick) * u, exact in double; per special tick a
//              record (off of the tick before, its increment), in order
//   serial     ONE thread, over the special ticks only: pos = fmod((pos + offPrev) + inc, 1)
//   finish     every tick: phase = (phase after the last special tick before it) + off
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t kPullMaxSpecial = 2048;  // more special ticks than this in one launch: the plain serial loop takes over
struct PullPhaseRec {
	double offPrev;  // phase offset of the tick before this special tick from the previous special tick (0 if that is special too)
	double v;        // increment of this tick; replaced by the phase after it
};
struct PullRunSum {   // summary of a chunk, and the element type of the segmented scan
	int64_t sum;       // sum of I behind the last special tick (of everything if there is none)
	uint32_t flag;     // a special tick inside
	uint32_t specials;
};
KLATT_HD PullRunSum pullRunCombine(const PullRunSum &first, const PullRunSum &second) {
	PullRunSum r;
	r.specials = first.specials + second.specials;
	r.flag = first.flag | second.flag;
	r.sum = second.flag ? second.sum : first.sum + second.sum;
	return r;
}
KLATT_HD double pullPow2(int e) {  // 2^e, -1022 <= e <= 1023
	const uint64_t b = (uint64_t)(e + 1023) << 52;
#ifdef __CUDA_ARCH__
	return __longlong_as_double((long long)b);
#else
	double d;
	memcpy(&d, &b, 8);
	return d;
#endif
}
KLATT_HD int pullBinade(double x) { return (int)((pullHiWord(x) >> 20) & 0x7ff) - 1023; }  // x in [2^k, 2^(k+1)), x > 0 normal
KLATT_HD double pullFixedToCycles(uint64_t a) { return (double)(a >> 11) * 1.1102230246251565e-16; }  // top 53 bits * 2^-53

// normal tick?  aPrev: approximate phase before the tick, x: its increment.  I: increment in ulps of binade k.
KLATT_HD bool pullClassify(double aPrev, double x, int64_t &I, int &k) {
	const double margin = 9.313225746154785e-10;  // 2^-30
	if (!(x >= 0.0 && x < 0.5) || !(aPrev >= 9.094947017729282e-13 /* 2^-40 */)) return false;
	const double s = aPrev + x;
	if (!(s < 1.0 - margin)) return false;
	k = pullBinade(s);
	const double lo = pullPow2(k);
	if (pullBinade(aPrev) != k || aPrev < lo * (1.0 + margin) || s > (2.0 * lo) * (1.0 - margin)) return false;
	const double r = x * pullPow2(52 - k);  // x / u, exact
	const double fl = floor(r);
	const double fr = r - fl;               // exact
	if (fr == 0.5) return false;            // tie: round-half-even looks at the parity of pos / u
	I = (int64_t)fl + (fr > 0.5 ? 1 : 0);
	return true;
}

KLATT_HD void pullRunsClassify(const PullCtx &X, uint32_t ch, uint64_t startFixed, PullRunSum &out) {
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	out.sum = 0; out.flag = 0; out.specials = 0;
	uint64_t A = startFixed;
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		const double x = X.inc[at];
		const double aPrev = pullFixedToCycles(A);
		A += (uint64_t)cyclesToFixed(x);
		int64_t I = 0;
		int k = 0;
		// a phase that may turn negative, or an increment the fixed-point approximation cannot hold (|pitch| >= sr/2):
		// leave the whole pull to the serial loop
		if (!(x >= 0.0 && x < 0.5)) out.specials += kPullMaxSpecial + 1;
		if (pullClassify(aPrev, x, I, k)) {
			X.runI[at] = I;
			X.runMeta[t] = (uint16_t)(0x8000 | (k + 64));
			out.sum += I;
		} else {
			X.runI[at] = 0;
			X.runMeta[t] = 0;
			out.sum = 0;
			out.flag = 1;
			out.specials += 1;
		}
	}
}

// before: the exclusive segmented prefix of the chunk (sum of I since the last special tick, special ticks so far)
KLATT_HD void pullRunsOffsets(const PullCtx &X, uint32_t ch, const PullRunSum &before) {
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	if (t0 >= t1) return;
	int64_t O = before.sum;
	uint32_t j = before.specials;
	double lastOff = 0.0;  // offset of the tick before, 0 when that tick is special (or belongs to the previous pull)
	if (t0 > 0) {
		const uint16_t m = X.runMeta[t0 - 1];
		if (m & 0x8000) lastOff = (double)O * pullPow2((int)(m & 0x7fff) - 64 - 52);
	}
	double *off = reinterpret_cast<double *>(X.runI);
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		const uint16_t m = X.runMeta[t];
		if (m & 0x8000) {
			O += X.runI[at];
			lastOff = (double)O * pullPow2((int)(m & 0x7fff) - 64 - 52);  // exact: |O| < 2^53, a power of two
			off[at] = lastOff;
		} else {
			if (j < kPullMaxSpecial) {
				X.rec[j].offPrev = lastOff;
				X.rec[j].v = X.inc[at];
			}
			++j;
			O = 0;
			lastOff = 0.0;
		}
	}
}

// the carried phase as the start of the approximate (fixed-point) phase; negative (only after negative pitches): no runs
KLATT_HD bool pullRunsStart(double pos0, uint64_t &fixed) {
	if (!(pos0 >= 0.0 && pos0 < 1.0)) { fixed = 0; return false; }
	fixed = (uint64_t)(pos0 * 18446744073709551616.0);
	return true;
}

// one thread: the FP64 recurrence over the special ticks only; returns the phase after the last of them
KLATT_HD double pullRunsSerial(const PullCtx &X, uint32_t specials, double pos0) {
	double pos = pos0;
	for (uint32_t j = 0; j < specials; ++j) {
		const double s = (pos + X.rec[j].offPrev) + X.rec[j].v;  // the first addition is exact (same grid, same binade)
		pos = ((pullHiWord(s) & 0x7fffffff) < 0x3ff00000) ? s : fracRef(s);
		X.rec[j].v = pos;
	}
	return pos;
}

// X.inc[t] <- phase after tick t; the pull's last chunk leaves the carry
KLATT_HD void pullRunsFinish(const PullCtx &X, uint32_t ch, uint32_t specialsBefore, double pos0) {
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	if (t0 >= t1) return;
	uint32_t j = specialsBefore;
	double base = j ? X.rec[j - 1].v : pos0;
	const double *off = reinterpret_cast<const double *>(X.runI);
	double p = base;
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		if (X.runMeta[t] & 0x8000) {
			p = base + off[at];  // exact
		} else {
			base = X.rec[j++].v;
			p = base;
		}
		X.inc[at] = p;
	}
	if (t1 == X.n) X.state->pitchPos = p;
}

// pass 2: the two excitation signals of every tick: cascade input -> sigA (:204, :148), parallel input -> sigB (:206, :171)
KLATT_HD void pullSourcePass2(const PullCtx &X, uint32_t ch, float aspStart, float fricStart) {
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	if (t0 >= t1) return;
	const uint64_t g0 = X.state->generated;
	PullCursor cur;
	cur.seek(X, t0);
	float aspLast = aspStart, fricLast = fricStart;
	Philox4 blk;
	blk.w[0] = blk.w[1] = blk.w[2] = blk.w[3] = 0;
	uint64_t blkIndex = ~0ull;
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		uint32_t wA, wF;
		pullNoiseWords(X, g0 + t, blk, blkIndex, wA, wF);
		const PullSeg &S = X.segs[cur.s];
		const uint32_t c = cur.c;
		excitation((float)X.inc[at], wA, wF, pullDirAt(S, dVoiceTurbulenceAmplitude, c), pullDirAt(S, dGlottalOpenQuotient, c),
		           pullDirAt(S, dVoiceAmplitude, c), pullDirAt(S, dAspirationAmplitude, c), pullDirAt(S, dFricationAmplitude, c),
		           pullDirAt(S, dPreFormantGain, c), aspLast, fricLast, X.sigA[at], X.sigB[at]);
		cur.next(X);
	}
	if (t1 == X.n) {  // the pull's last chunk leaves the carry
		X.state->aspLast = aspLast;
		X.state->fricLast = fricLast;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// resonator stages (klatt_tick_core.cuh StageTick): the parallel stage reads and rewrites sigB, the others sigA
// ---------------------------------------------------------------------------------------------------------------
// input of the FIR section before tick t of the pull (t may reach 2 ticks into the previous pull)
KLATT_HD float pullFirInput(const PullCtx &X, int64_t t) {
	if (t >= 0) return X.sigA[pullIdx(X, (uint32_t)t)];
	const float in1 = X.state->y[kResN0];
	return t == -1 ? in1 : in1 - X.state->d[kResN0];
}

// One chunk of one stage.  PASS 1: from zero state, accumulate the affine map.  PASS 2: from the scanned start state,
// overwrite the stage's input signal with its output (or, for the last stage, store the int16 samples).
// fir[2]: the two inputs before the chunk, read in pass 1 (before any thread overwrites sigA) and handed to pass 2.
// poles[NR + 1]: zeta of the sections at the start of the chunk (and of rN0 in the last slot), found in pass 1 -- inside
// a fade that is an exponential and a sine / cosine per section -- and handed to pass 2.
template <int STAGE, int PASS>
KLATT_HD void pullStage(const PullCtx &X, uint32_t ch, int res, Affine *maps, const PullStart *start, float *fir,
                        PoleWalk *poles) {
	constexpr int NR = StageTraits<STAGE>::NR;
	uint32_t t0, t1;
	pullChunkRange(X, ch, t0, t1);
	if (PASS == 1) {
#pragma unroll
		for (int k = 0; k < NR; ++k) maps[k] = Affine{1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.0f};
	}
	if (t0 >= t1) return;
	const double srInv = 1.0 / (double)X.sampleRate;
	float *sig = STAGE == kStageParallel ? X.sigB : X.sigA;
	PullCursor cur;
	cur.seek(X, t0);
	PoleWalk pw[NR], pw0;  // pw0: the FIR anti-resonator of the nasal stage
	if (PASS == 1) {
		const PullSeg &S = X.segs[cur.s];
#pragma unroll
		for (int k = 0; k < NR; ++k) pullPoleSeek(pw[k], S, cur.c, STAGE == kStageParallel ? kResParallel + k : res, srInv);
		if (STAGE == kStageNasal) pullPoleSeek(pw0, S, cur.c, kResN0, srInv);
		else pw0 = PoleWalk{0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
		for (int k = 0; k < NR; ++k) poles[k] = pw[k];
		poles[NR] = pw0;
	} else {
#pragma unroll
		for (int k = 0; k < NR; ++k) pw[k] = poles[k];
		pw0 = poles[NR];
	}
	StageTick<STAGE, PASS> st;
	st.start();
	if (PASS == 2) {
#pragma unroll
		for (int k = 0; k < NR; ++k) { st.y[k] = start[k].y; st.d[k] = start[k].d; }
	}
	if (STAGE == kStageNasal) {
		if (PASS == 1) {
			fir[0] = pullFirInput(X, (int64_t)t0 - 1);
			fir[1] = pullFirInput(X, (int64_t)t0 - 2);
		}
		st.in1 = fir[0]; st.in2 = fir[1];
	}
	// What a tick reads besides its input and the section memories: coefficients and mixing gains, functions of
	// (segment, counter).  Behind the landing tick of a request they are constants, so a chunk that lies inside one hold
	// (most chunks do: a fade is a third of the ticks and 512 consecutive ticks share a warp) evaluates them once.
	StageCoefs<STAGE> co;
	co.extra = co.a0 = co.rho0 = co.rcp0 = 0.0f;
	co.inv = false;
	auto loadCoefs = [&](const PullSeg &S, uint32_t c) {
		if (STAGE == kStageNasal) {
			pullPoleTick(pw0, S, c, kResN0, srInv);
			pw0.coef(co.a0, co.rho0);
			co.inv = n0InvLaw(c, S.F, S.n0InvStale, S.plan.n0InvFade, S.plan.n0InvFinal);
			co.rcp0 = co.inv ? fastRcp(co.a0) : 0.0f;
			co.extra = pullDirAt(S, dCaNP, c);
		}
#pragma unroll
		for (int k = 0; k < NR; ++k) {
			pullPoleTick(pw[k], S, c, STAGE == kStageParallel ? kResParallel + k : res, srInv);
			pw[k].coef(co.a[k], co.rho[k]);
			co.mix[k] = STAGE == kStageParallel ? pullDirAt(S, dPa1 + k, c) : 0.0f;
		}
		if (STAGE == kStageParallel) co.extra = pullDirAt(S, dParallelBypass, c);
		if (STAGE == kStageLast) co.extra = pullDirAt(S, dOutputGain, c);
	};
	const bool hold = cur.c > X.segs[cur.s].F && cur.left >= t1 - t0;
	uint32_t at = ch;
	for (uint32_t t = t0; t < t1; ++t, at += kPullThreads) {
		if (!hold || t == t0) loadCoefs(X.segs[cur.s], cur.c);
		const float o = st(sig[at], STAGE == kStageLast && PASS == 2 ? X.sigB[at] : 0.0f, co);
		if (PASS == 2) {
			if (STAGE == kStageLast) X.pcm[t] = (int16_t)(int)o;
			else sig[at] = o;
		}
		if (!hold) cur.next(X);
	}
	if (PASS == 1) {
#pragma unroll
		for (int k = 0; k < NR; ++k) maps[k] = st.map(k);
	} else if (t1 == X.n) {  // the pull's last chunk leaves the carry
#pragma unroll
		for (int k = 0; k < NR; ++k) {
			const int r = STAGE == kStageParallel ? kResParallel + k : res;
			X.state->y[r] = st.y[k];
			X.state->d[r] = st.d[k];
		}
		if (STAGE == kStageNasal) {
			X.state->y[kResN0] = st.in1;
			X.state->d[kResN0] = st.in1 - st.in2;
		}
	}
}

// Composition of affine maps for the block scans.  FP32 with explicit fmaf (the same bits on the device and in the
// host model below): a pull composes at most 512 maps in a tree of depth 9 + 4, so the scan adds a few 1e-7 relative to
// the start states -- the size of one tick's own rounding.  (klatt_long.cu composes up to 1e5 maps and does it in
// double.)  -DKLATT_PULL_SCAN_DOUBLE switches the scalar for A/B studies.
#ifdef KLATT_PULL_SCAN_DOUBLE
typedef double PullScalar;
KLATT_HD PullScalar pullFma(PullScalar a, PullScalar b, PullScalar c) { return fma(a, b, c); }
#else
typedef float PullScalar;
KLATT_HD PullScalar pullFma(PullScalar a, PullScalar b, PullScalar c) { return fmaf(a, b, c); }
#endif
struct PullAffineD {
	PullScalar p00, p01, p10, p11, zy, zd;
};
KLATT_HD PullAffineD pullIdentity() { return PullAffineD{1, 0, 0, 1, 0, 0}; }
KLATT_HD PullAffineD pullToD(const Affine &m) { return PullAffineD{m.p00, m.p01, m.p10, m.p11, m.zy, m.zd}; }
KLATT_HD PullAffineD pullSeed(float y, float d) { return PullAffineD{1, 0, 0, 1, y, d}; }
// `second` after `first`
KLATT_HD PullAffineD pullCompose(const PullAffineD &second, const PullAffineD &first) {
	PullAffineD r;
	r.p00 = pullFma(second.p00, first.p00, second.p01 * first.p10);
	r.p01 = pullFma(second.p00, first.p01, second.p01 * first.p11);
	r.p10 = pullFma(second.p10, first.p00, second.p11 * first.p10);
	r.p11 = pullFma(second.p10, first.p01, second.p11 * first.p11);
	r.zy = pullFma(second.p00, first.zy, pullFma(second.p01, first.zd, second.zy));
	r.zd = pullFma(second.p10, first.zy, pullFma(second.p11, first.zd, second.zd));
	return r;
}

#ifndef __CUDACC__
// Host model of klatt_pull.cu blockExclusive(): the same compositions in the same order (Kogge-Stone inside each warp of
// 32 chunks, Kogge-Stone over the 16 warp totals, then previous lane -> earlier warps -> seed), so tests/hostsim sees the
// start states the device computes.  own[kPullThreads] -> pre[kPullThreads].
inline void pullBlockExclusiveModel(const PullAffineD *own, const PullAffineD &seed, PullAffineD *pre) {
	constexpr int W = kPullThreads / 32;
	PullAffineD inc[kPullThreads], tot[W];
	for (int w = 0; w < W; ++w) {
		PullAffineD cur[32], nxt[32];
		for (int l = 0; l < 32; ++l) cur[l] = own[w * 32 + l];
		for (int delta = 1; delta < 32; delta <<= 1) {
			for (int l = 0; l < 32; ++l) nxt[l] = l >= delta ? pullCompose(cur[l], cur[l - delta]) : cur[l];
			for (int l = 0; l < 32; ++l) cur[l] = nxt[l];
		}
		for (int l = 0; l < 32; ++l) inc[w * 32 + l] = cur[l];
		tot[w] = cur[31];
	}
	{
		PullAffineD nxt[W];
		for (int delta = 1; delta < W; delta <<= 1) {
			for (int l = 0; l < W; ++l) nxt[l] = l >= delta ? pullCompose(tot[l], tot[l - delta]) : tot[l];
			for (int l = 0; l < W; ++l) tot[l] = nxt[l];
		}
	}
	for (int t = 0; t < kPullThreads; ++t) {
		const int w = t >> 5, l = t & 31;
		PullAffineD p = l == 0 ? pullIdentity() : inc[t - 1];
		if (w > 0) p = pullCompose(p, tot[w - 1]);
		pre[t] = pullCompose(p, seed);
	}
}
#endif

}  // namespace klatt
