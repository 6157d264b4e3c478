// klatt_long: the long-utterance path.  Pre-queued streams are cut into chunks of L ticks and every chunk is rendered by
// its own thread, all chunks of all streams of a launch at once (LongTable: one stream for speechPlayer_synthesizeLong,
// many for speechPlayer_synthesizeLongBatch).  A chunk kernel maps its chunk to (stream, chunk of the stream) and works in
// that stream's own ticks; every scan restarts at a stream's first chunk.  What a chunk needs from its past is recovered
// in closed form or by a scan instead of by running the past:
//
//   frame manager   the occupancy law max(M+1, F+2) (reference src/frame.cpp:41-80) gives every request its first
//                   tick by a prefix sum; a chunk finds its request by bisection and its position in the fade / hold
//                   from the tick index.  Interpolated parameters are a function of that position (src/frame.cpp:49-52),
//                   the hold-phase pitch glide is an arithmetic progression (src/frame.cpp:77).
//   vibrato phase   64-bit fixed point and piecewise-linear increments: an exact arithmetic series per request.
//   glottal phase   the reference's own FP64 recurrence pos = fmod(pos + quot, 1) (src/speechWaveGenerator.cpp:55,74), bit
//                   for bit and parallel in time (klatt_long_phase.cuh): an exact 2^-64 fixed-point prefix sum of the
//                   increments locates an anchor per chunk, every chunk runs the plain recurrence speculatively from its
//                   anchor (two runs, one grid step apart), the chain of roundings is translation-equivariant on the 2^-53
//                   grid so a scan of small integer maps turns the guesses into the true start values, and the source pass
//                   re-runs the plain recurrence from those and CHECKS that every run ends on the next one's start (a miss,
//                   or a stretch of zero / negative pitch without anchors, takes the serial fallback).  The hold glide of
//                   the pitch is the reference's repeated addition (src/frame.cpp:77), seeked in closed form (glideExact).
//   noise           Philox is random access; the 0.75-pole colouring filter (src/speechWaveGenerator.cpp:40) forgets its
//                   past within 64 ticks (0.75^64 = 1e-8), so a chunk warms it up on the 64 ticks before its first one.
//   resonators      each two-pole section is LINEAR in its state for a given input: over a chunk,
//                   state_end = P * state_start + z with P the product of the per-tick 2x2 update matrices and z the
//                   end state reached from zero.  Pass 1 of a stage computes (P, z) per chunk, a parallel scan with
//                   warp shuffles composes these affine maps along the stream (klatt_long_scan_kernel) into the true
//                   start state of every chunk, pass 2 re-runs the chunk from that state and writes the stage's output
//                   signal for the next stage.  rN0 stores INPUTS (src/speechWaveGenerator.cpp:133): it is FIR and needs
//                   no scan.  Stages run in the reference's order: parallel bank (6 sections in one stage), then
//                   rN0+rNP, r6 ... r1; the last stage fuses the mix, gain, clamp and int16 store (:207-208).
//
// The arithmetic of a tick is the FP32 formulation of klatt_f32_core.cuh (delta-form sections, pole recurrences
// during fades, FP64 pitch and phase); inside a fade the pole is re-based on its closed form every 64 ticks.  Parity
// with the serial kernels is by tolerance (re-association), not bit for bit: the bar is the FP32 bar (<= 1 LSB on
// >= 99.9 %, >= 60 dB SNR against the reference).
#include <cuda_runtime.h>
#include "klatt_common.h"
#include "klatt_f32_core.cuh"
#include "klatt_long_phase.cuh"
#include "launch.h"

namespace klatt {

namespace {

// Every chunk kernel is instantiated twice from the same code: MULTI = false for a one-stream launch (the stream's fields
// are kernel parameters, as the per-tick walks want them: reading them from a table in global memory made config 4 24 % slower) and
// MULTI = true for a table of streams.
// the stream that owns chunk ch: the last s with chunkBase[s] <= ch (empty streams own no chunk)
template <bool MULTI>
__device__ __forceinline__ uint32_t streamOfChunk(const LongTable &T, uint32_t ch) {
	if (!MULTI) return 0;
	uint32_t lo = 0, hi = T.numStreams;
	while (hi - lo > 1) {
		const uint32_t mid = (lo + hi) >> 1;
		if (T.chunkBase[mid] <= ch) lo = mid; else hi = mid;
	}
	return lo;
}
template <bool MULTI>
__device__ __forceinline__ const LongStream &streamAt(const LongTable &T, uint32_t s) { return MULTI ? T.streams[s] : T.one; }
// first chunk of stream s, and one past its last
template <bool MULTI>
__device__ __forceinline__ uint32_t chunkBegin(const LongTable &T, uint32_t s) { return MULTI ? T.chunkBase[s] : 0u; }
template <bool MULTI>
__device__ __forceinline__ uint32_t chunkEnd(const LongTable &T, uint32_t s, uint32_t numChunks) { return MULTI ? T.chunkBase[s + 1] : numChunks; }

constexpr int kWarmTicks = 64;

__device__ __forceinline__ bool reqIsNull(const LongStream &L, uint32_t j) { return L.isNull && L.isNull[j] != 0; }

// old / new value of frame parameter p for the fade of request j (plannedFrames() of klatt_f32_core.cuh, one slot)
__device__ void fadeEnds(const LongStream &L, uint32_t j, int p, double &o, double &n) {
	const bool curNull = reqIsNull(L, j);
	const bool prevNull = (j == 0) || reqIsNull(L, j - 1);
	const int32_t pr = L.prevReal[j];
	double PR = pr >= 0 ? L.frames[(size_t)pr * kNumParams + p] : 0.0;
	if (p == kPreFormantGain && prevNull) PR = 0.0;
	if (curNull) {
		o = PR;
		n = (p == kPreFormantGain) ? 0.0 : o;
	} else {
		n = L.frames[(size_t)j * kNumParams + p];
		o = prevNull ? ((p == kPreFormantGain) ? 0.0 : n) : PR;
	}
}

// where a tick sits: request j, sampleCounter value c on that tick (0 on the pop tick), fade length F
struct Cursor {
	uint32_t j, c, F;
	uint64_t left;  // ticks of this request still to come, this one included
	__device__ void load(const LongStream &L) {
		if (j < L.nReq) {
			uint32_t fd = L.fadeDur[j];
			F = fd > 1u ? fd : 1u;
		} else {
			F = 1;
		}
	}
	__device__ void seek(const LongStream &L, uint64_t t) {
		uint32_t lo = 0, hi = L.nReq;  // last j with start[j] <= t
		while (hi - lo > 1) {
			uint32_t mid = (lo + hi) >> 1;
			if (L.start[mid] <= t) lo = mid; else hi = mid;
		}
		j = lo;
		c = (uint32_t)(t - L.start[j]);
		left = L.start[j + 1] - t;
		load(L);
	}
	// n <= left ticks at once (the caller stays inside the request; reaching its end moves on like next())
	__device__ void advance(const LongStream &L, uint32_t n) {
		if (n == 0) return;
		c += n - 1;
		left -= n - 1;
		next(L);
	}
	__device__ void next(const LongStream &L) {
		++c;
		if (--left == 0) {
			++j;
			c = 0;
			if (j < L.nReq) left = L.start[j + 1] - L.start[j];
			load(L);
		}
	}
};

// one directly used parameter along the stream (reference src/frame.cpp:49-52 + the stale pop tick)
struct DirWalk {
	float prevFinal, d0, ds, dF;
	__device__ void load(const LongStream &L, uint32_t j, int slot) {
		prevFinal = j > 0 ? L.plans[j - 1].dirFinal[slot] : 0.0f;
		const FadePlanF32 &p = L.plans[j];
		d0 = p.dir0[slot]; ds = p.dirStep[slot]; dF = p.dirFinal[slot];
	}
	__device__ __forceinline__ float at(uint32_t c, uint32_t F) const {
		return c == 0 ? prevFinal : (c < F ? fmaf((float)c, ds, d0) : dF);
	}
};

// the vibrato depth 0.06 * vibratoPitchOffset along the stream, in double like the serial kernels' (klatt_common.h FadePlanF32)
struct DepthWalk {
	double prevFinal, d0, ds, dF;
	__device__ void load(const LongStream &L, uint32_t j) {
		prevFinal = j > 0 ? L.plans[j - 1].depthFinal : 0.0;
		const FadePlanF32 &p = L.plans[j];
		d0 = p.depth0; ds = p.depthStep; dF = p.depthFinal;
	}
	__device__ __forceinline__ double at(uint32_t c, uint32_t F) const {
		return c == 0 ? prevFinal : (c < F ? fma((double)(float)c, ds, d0) : dF);
	}
};

// zeta = 1 - pole of one section along the stream
struct PoleWalk {
	float zr, zi, wr, wi;
	__device__ void exact(const LongStream &L, uint32_t j, uint32_t k, uint32_t F, int r) {
		double f0, f1, b0, b1;
		fadeEnds(L, j, resFreqParam(r), f0, f1);
		fadeEnds(L, j, resBwParam(r), b0, b1);
		if (f1 != f1) f1 = f0;
		if (b1 != b1) b1 = b0;
		const double ratio = (double)k / (double)F;
		poleTerms(f0 + ((f1 - f0) * ratio), b0 + ((b1 - b0) * ratio), 1.0 / (double)L.sampleRate, zr, zi);
	}
	// state as it is AFTER the tick before (j, c)
	__device__ void seek(const LongStream &L, uint32_t j, uint32_t c, uint32_t F, int r) {
		wr = wi = 0.0f;
		if (c <= 1) {
			if (j > 0) { zr = L.plans[j - 1].zFre[r]; zi = L.plans[j - 1].zFim[r]; }
			else { zr = zi = 0.0f; }
		} else if (c <= F) {  // ticks 1 .. c-1 of the fade are behind us
			if (c - 1 < F) { exact(L, j, c - 1, F, r); wr = L.plans[j].wre[r]; wi = L.plans[j].wim[r]; }
		} else {
			zr = L.plans[j].zFre[r]; zi = L.plans[j].zFim[r];
		}
	}
	// the update of tick (j, c): afterwards (zr, zi) is what the tick renders with
	__device__ __forceinline__ void tick(const LongStream &L, uint32_t j, uint32_t c, uint32_t F, int r) {
		if (c == 0 || c > F) return;  // pop tick: stale; after the landing: constant
		if (c == F) {
			zr = L.plans[j].zFre[r]; zi = L.plans[j].zFim[r]; wr = wi = 0.0f;
			return;
		}
		if (c == 1) {
			const FadePlanF32 &p = L.plans[j];
			zr = p.z0re[r]; zi = p.z0im[r]; wr = p.wre[r]; wi = p.wim[r];
		}
		if ((c & (uint32_t)(kCoarseTicks - 1)) == 0) {
			exact(L, j, c, F, r);  // drift control: back onto the closed form
			return;
		}
		float tr = fmaf(-zr, wr, wr);
		tr = fmaf(zi, wi, tr);
		float ti = fmaf(-zr, wi, wi);
		ti = fmaf(-zi, wr, ti);
		zr += tr;
		zi += ti;
	}
	// a plain interior fade tick (1 < c < F, not a multiple of kCoarseTicks): the last six operations of tick()
	__device__ __forceinline__ void step() {
		float tr = fmaf(-zr, wr, wr);
		tr = fmaf(zi, wi, tr);
		float ti = fmaf(-zr, wi, wi);
		ti = fmaf(-zi, wr, ti);
		zr += tr;
		zi += ti;
	}
	__device__ __forceinline__ void coef(float &a, float &rho) const {
		a = fmaf(zr, zr, zi * zi);
		rho = fmaf(2.0f, zr, -a);
	}
};

__device__ __forceinline__ bool n0InvAt(const LongStream &L, uint32_t j, uint32_t c, uint32_t F) {
	if (c == 0) return j > 0 ? L.plans[j - 1].n0InvFinal != 0 : false;
	return (c < F ? L.plans[j].n0InvFade : L.plans[j].n0InvFinal) != 0;
}

// cur.voicePitch on tick (j, c)
__device__ __forceinline__ double pitchAt(const LongStream &L, uint32_t j, uint32_t c, uint32_t F) {
	if (c == 0) return L.pitchPop[j];
	const double o = L.pitchOld[j], n = L.pitchNew[j];
	if (c < F) return (n != n) ? o : o + ((n - o) * ((double)c / (double)F));
	const double landing = (n != n) ? o : o + ((n - o) * 1.0);
	if (c <= F + 1) return landing;
	return landing + (double)(c - F - 1) * L.pitchInc[j];
}

// vibrato: per-tick increment on tick (j, c), and the phase after the ticks before (j, c)
struct VibWalk {
	int64_t vPrev, v0, vs, vF;
	__device__ void load(const LongStream &L, uint32_t j) {
		vPrev = j > 0 ? L.plans[j - 1].vibIncFinal : 0;
		v0 = L.plans[j].vibInc0; vs = L.plans[j].vibIncStep; vF = L.plans[j].vibIncFinal;
	}
	__device__ __forceinline__ int64_t inc(uint32_t c, uint32_t F) const {
		return c == 0 ? vPrev : (c < F ? v0 + (int64_t)c * vs : vF);
	}
	// sum of inc(c') for c' in [0, c)
	__device__ uint64_t before(uint32_t c, uint32_t F) const {
		if (c == 0) return 0;
		uint64_t s = (uint64_t)vPrev;
		const uint64_t kmax = (c - 1 < F - 1) ? c - 1 : F - 1;  // fade ticks 1 .. kmax are behind us
		s += kmax * (uint64_t)v0 + (uint64_t)vs * (kmax * (kmax + 1) / 2);
		if (c > F) s += (uint64_t)(c - F) * (uint64_t)vF;
		return s;
	}
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// timeline: the queue is walked once, a request per step (the per-tick work is all in the other kernels).  The walk is a
// serial chain (start ticks, the pitch each request inherits, the vibrato phase), but what it READS is not: one block loads
// a tile of requests into shared memory with coalesced accesses, thread 0 runs the chain over the tile out of shared memory,
// and the block writes the tile's results back (round 1 walked global memory directly: 39 ms for the 40 072 requests of
// config 4, 45 % of the whole call, all of it load latency).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kTimelineTile = 256;

// inclusive scan of one uint64 per thread over the block (Hillis-Steele in shared memory: 256 values, 8 steps)
__device__ __forceinline__ uint64_t tileScanAdd(uint64_t v, uint64_t *buf) {
	const int tid = threadIdx.x;
	buf[tid] = v;
	__syncthreads();
	for (int d = 1; d < kTimelineTile; d <<= 1) {
		const uint64_t up = tid >= d ? buf[tid - d] : 0;
		__syncthreads();
		buf[tid] += up;
		__syncthreads();
	}
	return buf[tid];
}

// one block per stream: block s walks streams[s]
template <bool MULTI>
__global__ void __launch_bounds__(kTimelineTile)
klatt_long_timeline_kernel(LongTable T) {
	const LongStream &L = streamAt<MULTI>(T, blockIdx.x);
	__shared__ uint64_t scanBuf[kTimelineTile];
	__shared__ uint8_t sNull[kTimelineTile];
	__shared__ double sP0[kTimelineTile], sPNew[kTimelineTile], sInc[kTimelineTile];  // the frame's voicePitch, new.voicePitch after :71 (real requests), voicePitchInc
	__shared__ uint64_t sHold[kTimelineTile];                          // hold ticks F+2 .. occ-1 of the request
	__shared__ double gLanding[kTimelineTile], gEnd[kTimelineTile];    // the speculative glides
	__shared__ double oPop[kTimelineTile], oOld[kTimelineTile], oNew[kTimelineTile], oInc[kTimelineTile];
	// Everything that is a prefix sum (start ticks, vibrato phase, last real request) is scanned by the whole block.  What is
	// left is the pitch a request inherits: a serial chain through the hold glide of its predecessor -- n repeated FP64
	// additions, exact in closed form (glideExact) but ~1 us each on one thread -- which is speculated and verified in parallel
	// (below).  (Round 1 walked global memory on one thread: 39 ms for the 40 072 requests of config 4, 45 % of the whole
	// call.)
	uint64_t tBase = 0, vibBase = 0;      // carried across tiles (every thread keeps the same copy)
	int64_t vPrevCarry = 0;
	int32_t prevRealCarry = -1;
	double carryEnd = 0.0;       // exact end pitch of the last real request of the earlier tiles (0: none yet, frame.cpp:86)
	bool carryPrevNull = true;   // the request before this tile was a NULL request (or there is none: frame.cpp:87)
	const int tid = threadIdx.x;
	for (uint32_t base = 0; base < L.nReq; base += kTimelineTile) {
		const uint32_t j = base + tid;
		const uint32_t n = L.nReq - base < (uint32_t)kTimelineTile ? L.nReq - base : (uint32_t)kTimelineTile;
		const bool in = j < L.nReq;
		uint64_t occ = 0, vibOwn = 0;
		int64_t vF = 0, v0 = 0, vs = 0;
		uint64_t F = 1;
		bool null = true;
		if (in) {
			const uint64_t M = L.minDur[j];
			const uint32_t fd = L.fadeDur[j];
			F = fd > 1u ? fd : 1u;
			null = reqIsNull(L, j);
			occ = (M + 1 > F + 2) ? M + 1 : F + 2;
			const FadePlanF32 &p = L.plans[j];
			v0 = p.vibInc0; vs = p.vibIncStep; vF = p.vibIncFinal;
			vibOwn = (F - 1) * (uint64_t)v0 + (uint64_t)vs * ((F - 1) * F / 2) + (occ - F) * (uint64_t)vF;  // (+ the predecessor's final increment once)
			double inc = 0.0, pNew = 0.0, pStart = 0.0;
			if (!null) {
				const double p0 = L.frames[(size_t)j * kNumParams + kVoicePitch], p1 = L.frames[(size_t)j * kNumParams + kEndVoicePitch];
				inc = (p1 - p0) / (double)M;       // src/frame.cpp:98
				pNew = p0 + inc * (double)F;      // :71
				pStart = p0;
			}
			sNull[tid] = null ? 1 : 0; sInc[tid] = inc; sPNew[tid] = pNew; sP0[tid] = pStart; sHold[tid] = occ - F - 2;
		}
		// start tick = exclusive sum of the occupancies
		const uint64_t tIncl = tileScanAdd(occ, scanBuf);
		const uint64_t start = tBase + tIncl - occ;
		const uint64_t tTile = scanBuf[kTimelineTile - 1];
		__syncthreads();
		// vibrato phase before the pop tick = exclusive sum of (own sum + the predecessor's final increment)
		scanBuf[tid] = in ? (uint64_t)vF : 0;
		__syncthreads();
		const int64_t vPrev = tid == 0 ? vPrevCarry : (int64_t)scanBuf[tid - 1];
		const int64_t vLast = (int64_t)scanBuf[n - 1];
		__syncthreads();
		const uint64_t vibMine = in ? vibOwn + (uint64_t)vPrev : 0;
		const uint64_t vIncl = tileScanAdd(vibMine, scanBuf);
		const uint64_t vibStart = vibBase + vIncl - vibMine;
		const uint64_t vibTile = scanBuf[kTimelineTile - 1];
		__syncthreads();
		// last real request before j: running maximum of (real ? index + 1 : 0)
		scanBuf[tid] = (in && !null) ? (uint64_t)j + 1 : 0;
		__syncthreads();
		for (int d = 1; d < kTimelineTile; d <<= 1) {
			const uint64_t up = tid >= d ? scanBuf[tid - d] : 0;
			__syncthreads();
			if (up > scanBuf[tid]) scanBuf[tid] = up;
			__syncthreads();
		}
		const uint64_t before = tid == 0 ? 0 : scanBuf[tid - 1];
		const int32_t prevReal = before ? (int32_t)before - 1 : prevRealCarry;
		const uint64_t lastReal = scanBuf[kTimelineTile - 1];
		__syncthreads();
		if (in) { L.start[j] = start; L.vibPosStart[j] = vibStart; L.prevReal[j] = prevReal; }
		tBase += tTile; vibBase += vibTile; vPrevCarry = vLast;
		if (lastReal) prevRealCarry = (int32_t)lastReal - 1;

		// ---- the pitch every request inherits.  A NULL request hands its pitch on unchanged (src/frame.cpp:59-63: new = old,
		// inc = 0), so a request inherits the END pitch of the last REAL request before it (prevReal, scanned above):
		//   1. every real request guesses that value in closed form (landing ~ new pitch, glide = n * inc: good to a few ulps),
		//      forms its landing from the guess and runs its exact glide -- all requests at once;
		//   2. every request recomputes its landing from the EXACT end its predecessor just produced; if all landings of the
		//      tile are confirmed bit for bit, every end is exact by induction from the tile's carried-in value;
		//   3. otherwise (rare) thread 0 walks the tile serially.
		const bool prevNull = in && (j == 0 || (tid == 0 ? carryPrevNull : sNull[tid - 1] != 0));
		const bool realPrevInTile = in && before != 0 && (int64_t)before - 1 >= (int64_t)base;
		const uint32_t rLocal = realPrevInTile ? (uint32_t)(before - 1 - base) : 0u;
		double myInc = 0.0, myPNew = 0.0, myP0 = 0.0;
		uint64_t myHold = 0;
		if (in) { myInc = sInc[tid]; myPNew = sPNew[tid]; myP0 = sP0[tid]; myHold = sHold[tid]; }
		if (in && !null) {
			const double curGuess = realPrevInTile ? sPNew[rLocal] + (double)sHold[rLocal] * sInc[rLocal] : carryEnd;
			const double pOld = prevNull ? myP0 : curGuess;   // :64-67 copies the frame BEFORE :71 moves new.voicePitch
			const double landing = (myPNew != myPNew) ? pOld : pOld + ((myPNew - pOld) * 1.0);
			gLanding[tid] = landing;
			gEnd[tid] = glideExact(landing, myInc, myHold);  // hold ticks F+2 .. occ-1: one addition each (src/frame.cpp:77)
		}
		// 2. fixed-point iteration: every request recomputes its landing from the end its predecessor currently shows; the
		// ones whose landing moved redo their glide.  A pass without a change means every landing is consistent with an exact
		// predecessor, by induction from the tile's carried-in value.  (The landing is insensitive to the last bits of the
		// inherited pitch almost always, so corrections do not travel: two or three passes.)
		double curTrue = 0.0, pOldTrue = 0.0, pNewTrue = 0.0;
		int allOk = 0;
		for (int pass = 0; pass < 12 && !allOk; ++pass) {
			__syncthreads();
			bool changed = false;
			double newEnd = 0.0;
			if (in) {
				curTrue = realPrevInTile ? gEnd[rLocal] : carryEnd;
				if (null) { pOldTrue = curTrue; pNewTrue = curTrue; }
				else {
					pOldTrue = prevNull ? myP0 : curTrue;
					pNewTrue = myPNew;
					const double landing = (pNewTrue != pNewTrue) ? pOldTrue : pOldTrue + ((pNewTrue - pOldTrue) * 1.0);
					changed = __double_as_longlong(landing) != __double_as_longlong(gLanding[tid]);
					if (changed) { gLanding[tid] = landing; newEnd = glideExact(landing, myInc, myHold); }
				}
			}
			allOk = !__syncthreads_or(changed ? 1 : 0);
			if (changed) gEnd[tid] = newEnd;
		}
		__syncthreads();
		if (allOk) {
			if (in) { oPop[tid] = curTrue; oOld[tid] = pOldTrue; oNew[tid] = pNewTrue; oInc[tid] = myInc; }
			if (lastReal && (int64_t)lastReal - 1 >= (int64_t)base) carryEnd = gEnd[(uint32_t)(lastReal - 1 - base)];
		} else {
			if (tid == 0) {  // the true chain, serially
				double pitchCur = carryEnd;
				bool oldIsNull = carryPrevNull;
				for (uint32_t k = 0; k < n; ++k) {
					const bool nul = sNull[k] != 0;
					oPop[k] = pitchCur;
					double pOld = pitchCur, pNew = nul ? pitchCur : sPNew[k];
					if (!nul && (oldIsNull || base + k == 0)) pOld = sP0[k];
					oOld[k] = pOld; oNew[k] = pNew; oInc[k] = sInc[k];
					const double landing = (pNew != pNew) ? pOld : pOld + ((pNew - pOld) * 1.0);
					pitchCur = glideExact(landing, sInc[k], sHold[k]);
					oldIsNull = nul;
				}
				gEnd[0] = pitchCur;  // hand the tile's last value to everybody
			}
			__syncthreads();
			carryEnd = gEnd[0];
		}
		carryPrevNull = sNull[n - 1] != 0;
		__syncthreads();
		if (in) { L.pitchPop[j] = oPop[tid]; L.pitchOld[j] = oOld[tid]; L.pitchNew[j] = oNew[tid]; L.pitchInc[j] = oInc[tid]; }
		__syncthreads();
	}
	if (tid == 0) L.start[L.nReq] = tBase < L.cap ? tBase : L.cap;
}

// ---------------------------------------------------------------------------------------------------------------
// source: vibrato, glottal phase, aspiration / frication noise (reference src/speechWaveGenerator.cpp:72-86, :205-206)
// ---------------------------------------------------------------------------------------------------------------
struct SourceWalk {
	Cursor cur;
	VibWalk vw;
	DepthWalk depth;
	DirWalk vta, goq, va, aa, fa, pfg;
	uint64_t vibPos;
	uint32_t loaded;
	double pPop, pOld, pNew, pInc;  // pitch of the request in force: stale pop-tick value, fade end points, hold glide
	double pitchHold;               // cur.voicePitch while holding, accumulated like the reference does (src/frame.cpp:77)
	__device__ void loadReq(const LongStream &L, bool full) {
		vw.load(L, cur.j);
		depth.load(L, cur.j);
		if (full) {
			vta.load(L, cur.j, dVoiceTurbulenceAmplitude); goq.load(L, cur.j, dGlottalOpenQuotient);
			va.load(L, cur.j, dVoiceAmplitude); aa.load(L, cur.j, dAspirationAmplitude);
			fa.load(L, cur.j, dFricationAmplitude); pfg.load(L, cur.j, dPreFormantGain);
		}
		pPop = L.pitchPop[cur.j]; pOld = L.pitchOld[cur.j]; pNew = L.pitchNew[cur.j]; pInc = L.pitchInc[cur.j];
		loaded = cur.j;
	}
	__device__ __forceinline__ double landing() const { return (pNew != pNew) ? pOld : pOld + ((pNew - pOld) * 1.0); }
	__device__ void seek(const LongStream &L, uint64_t t, bool full) {
		cur.seek(L, t);
		pitchHold = 0.0;
		if (cur.j >= L.nReq) { loaded = cur.j; return; }
		loadReq(L, full);
		vibPos = L.vibPosStart[cur.j] + vw.before(cur.c, cur.F);
		// in the middle of a hold: the value the previous tick used, (c-1) - F - 1 additions after the landing
		if (cur.c >= cur.F + 2) pitchHold = glideExact(landing(), pInc, (uint64_t)(cur.c - cur.F - 2));
	}
	// The increment of the glottal phase on this tick, the double the serial kernel adds (klatt_f32_core.cuh OscChain:
	// vibrato sine in FP32, its depth, pitch * (1 + vibrato) and the correctly rounded division by the sample rate in FP64; reference
	// src/speechWaveGenerator.cpp:73-74).  In a fade the serial kernels sum the depth's steps where this evaluates the depth in
	// closed form: the two differ by a few FP64 ulps.  cur.voicePitch: stale on the pop tick, old+(new-old)*ratio in the fade
	// (src/frame.cpp:49-52), the landing value on the landing and swap ticks, then += inc per tick (:77).
	__device__ __forceinline__ double quotOfTick(double srD, double srInv) {
		const uint32_t c = cur.c, F = cur.F;
		vibPos += (uint64_t)vw.inc(c, F);
		float vph = (float)(int32_t)(uint32_t)(vibPos >> 32) * 2.3283064365386963e-10f;
		const double vib1 = fma((double)sinTurns(vph), depth.at(c, F), 1.0);
		double pitch;
		if (c == 0) pitch = pPop;
		else if (c < F) pitch = (pNew != pNew) ? pOld : pOld + ((pNew - pOld) * ((double)c / (double)F));
		else if (c <= F + 1) { pitch = landing(); pitchHold = pitch; }
		else { pitchHold += pInc; pitch = pitchHold; }
		const double m = pitch * vib1;
		return divideBySampleRate(m, srD, srInv);
	}
	__device__ __forceinline__ void next(const LongStream &L, bool full) {
		cur.next(L);
		if (cur.j != loaded && cur.j < L.nReq) loadReq(L, full);
	}
};

// SourceWalk as the increment source of phaseSpeculateChunk
struct PhaseSrc {
	SourceWalk w;
	const LongStream &L;
	double srD, srInv;
	__device__ PhaseSrc(const LongStream &L_, uint64_t t) : L(L_) {
		srD = (double)L.sampleRate; srInv = 1.0 / srD;
		w.seek(L, t, false);
	}
	__device__ __forceinline__ void tick(double &quot, uint64_t &fixedInc) {
		quot = w.quotOfTick(srD, srInv);
		fixedInc = (uint64_t)cyclesToFixed(quot);
		w.next(L, false);
	}
};

// pass 1: the phase every chunk advances by (fraction of a cycle, 2^-64 fixed point: exact sums, used to LOCATE the anchors)
template <bool MULTI>
__global__ void __launch_bounds__(128)
klatt_long_phase_kernel(LongTable T, uint32_t chunkTicks, uint32_t numChunks, uint64_t *__restrict__ advance) {
	const uint32_t ch = blockIdx.x * blockDim.x + threadIdx.x;
	if (ch >= numChunks) return;
	const uint32_t s = streamOfChunk<MULTI>(T, ch);
	const LongStream &L = streamAt<MULTI>(T, s);
	const uint64_t total = L.start[L.nReq];
	const uint64_t t0 = (uint64_t)(ch - chunkBegin<MULTI>(T, s)) * chunkTicks;
	const uint64_t t1 = (t0 + chunkTicks < total) ? t0 + chunkTicks : total;
	PhaseSrc src(L, t0);
	uint64_t pos = 0, fi;
	double quot;
	for (uint64_t t = t0; t < t1; ++t) {
		src.tick(quot, fi);
		pos += fi;
	}
	advance[ch] = pos;
}

// exclusive scan of the per-chunk phase advances: 64-bit integer sums modulo one cycle, exact.  One block; every thread
// sums a contiguous run, the run totals are scanned with warp shuffles, the runs are replayed from their prefix.  The scan
// runs over the chunks of all streams; a stream's own prefix is this one minus the value at its first chunk (exact mod 2^64).
__global__ void __launch_bounds__(1024)
klatt_long_phase_scan_kernel(const uint64_t *__restrict__ advance, uint32_t numChunks, uint64_t *__restrict__ startPhase) {
	__shared__ uint64_t warpTotal[32];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const uint32_t per = (numChunks + 1023) / 1024;
	const uint32_t c0 = (uint32_t)tid * per < numChunks ? (uint32_t)tid * per : numChunks;
	const uint32_t c1 = c0 + per < numChunks ? c0 + per : numChunks;
	uint64_t run = 0;
	for (uint32_t c = c0; c < c1; ++c) run += advance[c];
	uint64_t inc = run;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		uint64_t up = __shfl_up_sync(0xffffffffu, inc, delta);
		if (lane >= delta) inc += up;
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		uint64_t w = warpTotal[lane];
#pragma unroll
		for (int delta = 1; delta < 32; delta <<= 1) {
			uint64_t up = __shfl_up_sync(0xffffffffu, w, delta);
			if (lane >= delta) w += up;
		}
		warpTotal[lane] = w;
	}
	__syncthreads();
	uint64_t pos = inc - run + (warp > 0 ? warpTotal[warp - 1] : 0);
	for (uint32_t c = c0; c < c1; ++c) {
		startPhase[c] = pos;
		pos += advance[c];
	}
}

// speculative pass: anchors, the two runs per chunk, the offset map of every chunk (klatt_long_phase.cuh)
template <bool MULTI>
__global__ void __launch_bounds__(128)
klatt_long_spec_kernel(LongTable T, uint32_t chunkTicks, uint32_t numChunks, const uint64_t *__restrict__ startPhase,
                       PhaseChunk *__restrict__ chunks, uint32_t *__restrict__ fail) {
	const uint32_t ch = blockIdx.x * blockDim.x + threadIdx.x;
	if (ch >= numChunks) return;
	const uint32_t s = streamOfChunk<MULTI>(T, ch), cb = chunkBegin<MULTI>(T, s);
	const LongStream &L = streamAt<MULTI>(T, s);
	const uint64_t total = L.start[L.nReq];
	PhaseSrc src(L, (uint64_t)(ch - cb) * chunkTicks);
	PhaseChunk pc;
	// a run may extend over up to 15 anchorless chunks (zero pitch, silence); beyond that the stream takes the fallback
	if (!phaseSpeculateChunk(src, ch - cb, chunkTicks, total, startPhase[ch] - startPhase[cb], 16ull * chunkTicks, pc))
		atomicOr(fail + s, 1u);
	chunks[ch] = pc;
}

// exclusive scan of the offset maps in chunk order, restarted at every stream's first chunk: startP[c] = the TRUE phase
// entering tick chunks[c].anchor.  (A restart is not a map of the m -> m + a[m & 3] family, so the scan is SEGMENTED: an
// element is (head, map), and a head discards whatever came before it.  Exact integer arithmetic either way.)
struct SegPhaseMap {
	PhaseMap m;
	int head;  // the segment of this element starts inside it
};
__device__ __forceinline__ SegPhaseMap segCombine(const SegPhaseMap &first, const SegPhaseMap &second) {
	if (second.head) return second;
	SegPhaseMap r;
	r.m = phaseMapCompose(second.m, first.m);
	r.head = first.head;
	return r;
}

template <bool MULTI>
__global__ void __launch_bounds__(1024)
klatt_long_phase_map_scan_kernel(LongTable T, const PhaseChunk *__restrict__ chunks, uint32_t numChunks, double *__restrict__ startP) {
	__shared__ SegPhaseMap warpTotal[32];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const uint32_t per = (numChunks + 1023) / 1024;
	const uint32_t c0 = (uint32_t)tid * per < numChunks ? (uint32_t)tid * per : numChunks;
	const uint32_t c1 = c0 + per < numChunks ? c0 + per : numChunks;
	// the stream of chunk c0; the run then moves on stream by stream (c is a stream's first chunk iff c == chunkBase[s])
	const uint32_t s0 = c0 < numChunks ? streamOfChunk<MULTI>(T, c0) : 0;
	SegPhaseMap run{phaseMapIdentity(), 0};
	for (uint32_t c = c0, s = s0; c < c1; ++c) {
		while (chunkEnd<MULTI>(T, s, numChunks) <= c) ++s;
		run = segCombine(run, SegPhaseMap{chunks[c].map, c == chunkBegin<MULTI>(T, s)});
	}
	auto shfl = [](const SegPhaseMap &m, int delta) {
		SegPhaseMap r;
#pragma unroll
		for (int i = 0; i < kPhaseRuns; ++i) r.m.a[i] = __shfl_up_sync(0xffffffffu, m.m.a[i], delta);
		r.head = __shfl_up_sync(0xffffffffu, m.head, delta);
		return r;
	};
	SegPhaseMap inc = run;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		SegPhaseMap up = shfl(inc, delta);
		if (lane >= delta) inc = segCombine(up, inc);
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		SegPhaseMap w = warpTotal[lane];
#pragma unroll
		for (int delta = 1; delta < 32; delta <<= 1) {
			SegPhaseMap up = shfl(w, delta);
			if (lane >= delta) w = segCombine(up, w);
		}
		warpTotal[lane] = w;
	}
	__syncthreads();
	SegPhaseMap prev = shfl(inc, 1);
	SegPhaseMap pre = lane == 0 ? SegPhaseMap{phaseMapIdentity(), 0} : prev;
	if (warp > 0) pre = segCombine(warpTotal[warp - 1], pre);
	// every stream starts at offset 0 of its first chunk's anchor (phase 0 exactly): the offset at chunk c's anchor is pre(0)
	PhaseMap p = pre.m;
	for (uint32_t c = c0, s = s0; c < c1; ++c) {
		while (chunkEnd<MULTI>(T, s, numChunks) <= c) ++s;
		if (c == chunkBegin<MULTI>(T, s)) p = phaseMapIdentity();
		const PhaseChunk pc = chunks[c];
		startP[c] = pc.anchor == kNoAnchor ? 0.0 : phaseFromOffset(pc.s0, phaseMapApply(p, 0));
		p = phaseMapCompose(pc.map, p);
	}
}

// serial fallback: one thread per stream whose fail flag is set runs the plain recurrence over that whole stream and hands
// every chunk of it its true start (slow: one tick after the other; taken only for a stream whose speculative pass could not
// anchor a chunk or failed its own check).  The other streams' chunks are left as they are.
template <bool MULTI>
__global__ void klatt_long_phase_serial_kernel(LongTable T, uint32_t chunkTicks, uint32_t allChunks, const uint32_t *__restrict__ fail,
                                               PhaseChunk *__restrict__ chunks, double *__restrict__ startP) {
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= T.numStreams || !fail[s]) return;
	const LongStream &L = streamAt<MULTI>(T, s);
	const uint32_t cb = chunkBegin<MULTI>(T, s), numChunks = chunkEnd<MULTI>(T, s, allChunks) - cb;
	const uint64_t total = L.start[L.nReq];
	PhaseSrc src(L, 0);
	double pos = 0.0, quot;
	uint64_t fi;
	for (uint32_t c = 0; c < numChunks; ++c) {
		const uint64_t t0 = (uint64_t)c * chunkTicks, t1 = (t0 + chunkTicks < total) ? t0 + chunkTicks : total;
		PhaseChunk pc;
		pc.anchor = t0; pc.next = t1; pc.s0 = pos; pc.map = phaseMapIdentity();
		chunks[cb + c] = pc;
		startP[cb + c] = pos;
		for (uint64_t t = t0; t < t1; ++t) {
			src.tick(quot, fi);
			pos = phaseStep(pos, quot);
		}
	}
}

// pass 2: the two excitation signals of every tick: cascade input ci (:204, :148) and parallel input pin (:206, :171).
// Chunk ch owns the ticks [anchor, next) of its phase run and renders them from the true start phase; the run must end on
// the next run's start, bit for bit, or `fail` is raised (the construction is verified, not trusted).
template <bool MULTI>
__global__ void __launch_bounds__(128)
klatt_long_source_kernel(LongTable T, uint32_t chunkTicks, uint32_t numChunks, const PhaseChunk *__restrict__ chunks,
                         const double *__restrict__ startP, uint32_t *__restrict__ fail, float *__restrict__ ci,
                         float *__restrict__ pin) {
	const uint32_t ch = blockIdx.x * blockDim.x + threadIdx.x;
	if (ch >= numChunks) return;
	const PhaseChunk pc = chunks[ch];
	if (pc.anchor == kNoAnchor) return;
	const uint32_t s = streamOfChunk<MULTI>(T, ch), cb = chunkBegin<MULTI>(T, s);
	const LongStream &L = streamAt<MULTI>(T, s);
	// the stream's ticks in the signal arrays (the phase runs are in the stream's own ticks)
	ci += (size_t)cb * chunkTicks;
	pin += (size_t)cb * chunkTicks;
	const uint64_t total = L.start[L.nReq];
	const uint64_t t0 = pc.anchor, t1 = pc.next;
	const double srD = (double)L.sampleRate, srInv = 1.0 / srD;
	// warm the two noise colouring filters up on the ticks before the run
	float aspLast = 0.0f, fricLast = 0.0f;
	for (uint64_t g = (t0 > (uint64_t)kWarmTicks ? t0 - kWarmTicks : 0); g < t0; ++g) {
		Philox4 b = noiseBlock(L.seed, L.streamId, g >> 1);
		const uint32_t wA = (g & 1) ? b.w[2] : b.w[0], wF = (g & 1) ? b.w[3] : b.w[1];
		aspLast = fmaf(0.75f, aspLast, bitsToFloat(0x4B000000u | (wA >> 9)) - 8388608.0f);
		fricLast = fmaf(0.75f, fricLast, bitsToFloat(0x4B000000u | (wF >> 9)) - 8388608.0f);
	}
	SourceWalk w;
	w.seek(L, t0, true);
	double pos = startP[ch];
	Philox4 blk;
	blk.w[0] = blk.w[1] = blk.w[2] = blk.w[3] = 0;
	for (uint64_t t = t0; t < t1; ++t) {
		if ((t & 1) == 0 || t == t0) blk = noiseBlock(L.seed, L.streamId, t >> 1);
		const uint32_t wA = (t & 1) ? blk.w[2] : blk.w[0], wF = (t & 1) ? blk.w[3] : blk.w[1];
		const uint32_t c = w.cur.c, F = w.cur.F;
		pos = phaseStep(pos, w.quotOfTick(srD, srInv));
		const float voice = (float)pos;
		aspLast = fmaf(0.75f, aspLast, bitsToFloat(0x4B000000u | (wA >> 9)) - 8388608.0f);
		float asp = aspLast * (0.2f * kDrawScale);
		float turb = asp * w.vta.at(c, F);
		if (voice < w.goq.at(c, F)) turb *= 0.01f;
		float v = (fmaf(voice, 2.0f, -1.0f) + turb) * w.va.at(c, F);
		float src = fmaf(asp, w.aa.at(c, F), v);
		const float halfGain = w.pfg.at(c, F) * 0.5f;
		ci[t] = src * halfGain;
		fricLast = fmaf(0.75f, fricLast, bitsToFloat(0x4B000000u | (wF >> 9)) - 8388608.0f);
		pin[t] = fricLast * (((0.3f * kDrawScale) * w.fa.at(c, F)) * halfGain);
		w.next(L, true);
	}
	if (t1 < total) {  // the chunk whose run starts at t1 must have been handed exactly the value this run arrives with
		const uint32_t nx = cb + (uint32_t)(t1 / chunkTicks);
		if (nx >= chunkEnd<MULTI>(T, s, numChunks) || chunks[nx].anchor != t1 || startP[nx] != pos) atomicOr(fail + s, 1u);
	}
}

// ---------------------------------------------------------------------------------------------------------------
// resonator stages
// ---------------------------------------------------------------------------------------------------------------
enum Stage : int { kStageParallel = 0, kStageNasal = 1, kStageCascade = 2, kStageLast = 3 };

template <int STAGE> struct StageTraits {
	static constexpr int NR = STAGE == kStageParallel ? 6 : 1;  // scanned sections
};

// One chunk of one stage.  PASS 1: from zero state, also accumulate P.  PASS 2: from the scanned start state, write
// the stage's output signal (or, for the last stage, the int16 samples).
//   kStageParallel: in = pin, sections 8..13, out = par (:170-180)
//   kStageNasal   : in = ci, rN0 (FIR) then rNP (section 1), out = x after the caNP mix (:148-150)
//   kStageCascade : in = x, section `res`, out = its output (:151-156)
//   kStageLast    : like kStageCascade for r1, then (x + par) * outputGain * 4000, clamp, truncate (:207-208)
// Memory: thread i of a warp walks chunk (w + i), i.e. addresses chunkTicks * 4 bytes apart -- a warp-wide access to tick t
// of 32 chunks touches 32 different sectors (round 1: 8 x the algorithmic traffic on the stores, long_scoreboard 28 cycles
// per issue).  The signals therefore move through a shared-memory tile per warp: 32 chunks x 32 ticks, loaded and stored as
// 32 coalesced 128-byte rows (row r = 32 consecutive ticks of chunk w + r), read and written by the owning thread along
// its row ([32][33]: conflict-free either way).
constexpr int kStageBlock = 64;   // threads: two warps, one tile each (+ one for the parallel-bank signal in the last stage)
constexpr int kTile = 32;
template <int STAGE, int PASS, bool MULTI>
__global__ void __launch_bounds__(kStageBlock)
klatt_long_stage_kernel(LongTable T, uint32_t chunkTicks, uint32_t numChunks, int res, const float *__restrict__ in,
                        const float *__restrict__ par, Affine *__restrict__ maps, const float2 *__restrict__ startState,
                        float *__restrict__ out, int16_t *__restrict__ pcm) {
	constexpr int NR = StageTraits<STAGE>::NR;
	constexpr bool kHasPar = STAGE == kStageLast && PASS == 2, kHasOut = PASS == 2;
	__shared__ float tIn[kStageBlock / 32][kTile][kTile + 1];
	__shared__ float tPar[kHasPar ? kStageBlock / 32 : 1][kHasPar ? kTile : 1][kTile + 1];
	// (the output tile IS the input tile: a thread overwrites tick q of its own row after it has consumed it -- one tile per
	// warp instead of two lets twice as many warps share an SM, and these kernels are bound by the latency of their recurrences)
	float (*tOut)[kTile][kTile + 1] = tIn;
	// per row of the warp's tiles (= per lane's chunk): ticks in the chunk, and where its tick 0 goes in the int16 output.  A
	// warp may hold chunks of several streams; the signal arrays are addressed in virtual ticks (chunk c at c * chunkTicks).
	__shared__ uint32_t sLen[kStageBlock / 32][kTile];
	__shared__ uint64_t sPcm[kHasPar ? kStageBlock / 32 : 1][kTile];
	const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
	const uint32_t ch = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t warpChunk0 = ch - lane;  // first chunk of this warp
	const bool live = ch < numChunks;
	const uint32_t s = live ? streamOfChunk<MULTI>(T, ch) : 0, cb = chunkBegin<MULTI>(T, s);
	const LongStream &L = streamAt<MULTI>(T, s);
	const uint64_t total = L.start[L.nReq];
	const uint64_t t0 = live ? (uint64_t)(ch - cb) * chunkTicks : 0;  // in the stream's own ticks
	const uint64_t t1 = live ? ((t0 + chunkTicks < total) ? t0 + chunkTicks : total) : 0;
	const bool lastOfStream = live && ch + 1 == chunkEnd<MULTI>(T, s, numChunks);
	if (MULTI) {
		sLen[wib][lane] = (uint32_t)(t1 - t0);
		if (kHasPar) sPcm[kHasPar ? wib : 0][lane] = L.outBase + t0;
		__syncwarp();
	}
	Cursor cur;
	PoleWalk pw[NR], pw0;  // pw0: the FIR anti-resonator of the nasal stage
	DirWalk mix[NR], extra;  // parallel: pa1..6 + bypass; nasal: caNP; last: outputGain
	auto loadDirs = [&]() {
		if (STAGE == kStageParallel) {
#pragma unroll
			for (int k = 0; k < NR; ++k) mix[k].load(L, cur.j, dPa1 + k);
			extra.load(L, cur.j, dParallelBypass);
		} else if (STAGE == kStageNasal) {
			extra.load(L, cur.j, dCaNP);
		} else if (STAGE == kStageLast) {
			extra.load(L, cur.j, dOutputGain);
		}
	};
	uint32_t loaded = 0;
	float y[NR], d[NR];
	float p00[NR], p01[NR], p10[NR], p11[NR];
#pragma unroll
	for (int k = 0; k < NR; ++k) { y[k] = 0.0f; d[k] = 0.0f; p00[k] = 1.0f; p01[k] = 0.0f; p10[k] = 0.0f; p11[k] = 1.0f; }
	float in1 = 0.0f, in2 = 0.0f;  // the FIR section needs the two inputs before the chunk
	if (live) {
		cur.seek(L, t0);
#pragma unroll
		for (int k = 0; k < NR; ++k) pw[k].seek(L, cur.j, cur.c, cur.F, STAGE == kStageParallel ? kResParallel + k : res);
		if (STAGE == kStageNasal) pw0.seek(L, cur.j, cur.c, cur.F, kResN0);
		loadDirs();
		loaded = cur.j;
		if (PASS == 2) {
#pragma unroll
			for (int k = 0; k < NR; ++k) { float2 s = startState[(size_t)ch * NR + k]; y[k] = s.x; d[k] = s.y; }
		}
		if (STAGE == kStageNasal) {
			const size_t v0 = (size_t)cb * chunkTicks + t0;
			if (t0 >= 1) in1 = in[v0 - 1];
			if (t0 >= 2) in2 = in[v0 - 2];
		}
	}
	for (uint32_t tile = 0; tile < chunkTicks; tile += kTile) {
		// ---- tile in: row r = ticks [tile, tile + 32) of chunk warpChunk0 + r ----
#pragma unroll 4
		for (int r = 0; r < kTile; ++r) {
			const uint64_t g = (uint64_t)(warpChunk0 + r) * chunkTicks + tile + lane;
			const bool ok = MULTI ? tile + lane < sLen[wib][r] : (warpChunk0 + r < numChunks && g < total);
			tIn[wib][r][lane] = ok ? in[g] : 0.0f;
			if (kHasPar) tPar[wib][r][lane] = ok ? par[g] : 0.0f;
		}
		__syncwarp();
		if (live) {
			const uint64_t tb = t0 + tile;
			const int qEnd = (tb + kTile <= t1) ? kTile : (tb < t1 ? (int)(t1 - tb) : 0);
			// One tick of the stage with the coefficients of that tick given: the FIR anti-resonator (nasal stage), the scanned
			// sections, the affine map (pass 1), the stage's output (pass 2).
			auto tickWith = [&](int q, const float *a, const float *rho, const float *mixv, float extraV, bool n0Inv, float a0, float rho0) {
				float x = tIn[wib][lane][q];
				const float xin = x;
				if (STAGE == kStageNasal) {  // rN0 on inputs: src/speechWaveGenerator.cpp:129-135 with anti == true
					const float dprev = in1 - in2;
					const float dx = x - in1;
					const float dx1 = fmaf(-rho0, dprev, dprev);
					x = n0Inv ? fmaf(dx - dx1, fastRcp(a0), in1) : fmaf(a0, dx, dx1 + in1);
					in2 = in1;
					in1 = xin;
				}
				float acc = 0.0f;
#pragma unroll
				for (int k = 0; k < NR; ++k) {
					float w = fmaf(-rho[k], d[k], d[k]);
					w = fmaf(-a[k], y[k], w);
					const float dn = fmaf(a[k], x, w);
					d[k] = dn;
					y[k] += dn;
					if (PASS == 1) {  // P <- A P with A = [[1-a, 1-rho], [-a, 1-rho]] acting on (y, d)
						const float g = 1.0f - rho[k];
						const float n10 = fmaf(-a[k], p00[k], g * p10[k]), n11 = fmaf(-a[k], p01[k], g * p11[k]);
						p00[k] += n10; p01[k] += n11;
						p10[k] = n10; p11[k] = n11;
					}
					if (STAGE == kStageParallel) acc = fmaf(y[k] - x, mixv[k], acc);
				}
				if (PASS == 2) {
					float o;
					if (STAGE == kStageParallel) {
						o = fmaf(x - acc, extraV, acc);
					} else if (STAGE == kStageNasal) {
						o = fmaf(y[0] - xin, extraV, xin);
					} else if (STAGE == kStageCascade) {
						o = y[0];
					} else {
						float sgn = (y[0] + tPar[kHasPar ? wib : 0][kHasPar ? lane : 0][q]) * (extraV * 4000.0f);
						sgn = fminf(sgn, 32000.0f);
						sgn = fmaxf(sgn, -32000.0f);
						o = (float)(int)sgn;  // the int16 value, exactly representable
					}
					tOut[wib][lane][q] = o;
				}
			};
			// Events, not branches (as in the batch kernels): a tick that may change something -- the pop tick, the first fade
			// tick, a drift-control point, the landing, the first tick of a tile -- runs the general code; the ticks that follow
			// it inside the same RUN (the rest of a hold: constant coefficients; the fade ticks up to the next multiple of 64:
			// plain pole steps) run a tight loop with no frame-manager logic.  Same operations on the same values per tick.
			int q = 0;
			while (q < qEnd) {
				float a[NR], rho[NR], mixv[NR], a0 = 0.0f, rho0 = 0.0f, extraV = 0.0f;
				bool n0Inv = false;
				{
					const uint32_t j = cur.j, c = cur.c, F = cur.F;
					if (STAGE == kStageNasal) {
						pw0.tick(L, j, c, F, kResN0);
						pw0.coef(a0, rho0);
						n0Inv = n0InvAt(L, j, c, F);
					}
#pragma unroll
					for (int k = 0; k < NR; ++k) {
						pw[k].tick(L, j, c, F, STAGE == kStageParallel ? kResParallel + k : res);
						pw[k].coef(a[k], rho[k]);
						mixv[k] = STAGE == kStageParallel ? mix[k].at(c, F) : 0.0f;
					}
					if (STAGE != kStageCascade) extraV = extra.at(c, F);
					tickWith(q, a, rho, mixv, extraV, n0Inv, a0, rho0);
					++q;
					cur.next(L);
					if (cur.j != loaded && cur.j < L.nReq) { loadDirs(); loaded = cur.j; }
				}
				if (q >= qEnd || cur.j >= L.nReq) continue;
				const uint32_t c = cur.c, F = cur.F;
				if (c > F) {  // inside a hold: nothing moves until the request ends
					uint32_t n = (uint32_t)(qEnd - q);
					if ((uint64_t)n > cur.left) n = (uint32_t)cur.left;
					for (uint32_t i = 0; i < n; ++i) tickWith(q + (int)i, a, rho, mixv, extraV, n0Inv, a0, rho0);
					q += (int)n;
					cur.advance(L, n);
					if (cur.j != loaded && cur.j < L.nReq) { loadDirs(); loaded = cur.j; }
				} else if (c > 1 && c < F && (c & (uint32_t)(kCoarseTicks - 1)) != 0) {  // plain interior fade ticks
					uint32_t n = (uint32_t)(qEnd - q);
					const uint32_t toLanding = F - c, toGrid = (uint32_t)kCoarseTicks - (c & (uint32_t)(kCoarseTicks - 1));
					if (n > toLanding) n = toLanding;
					if (n > toGrid) n = toGrid;
					for (uint32_t i = 0; i < n; ++i) {
						const uint32_t ci = c + i;
						if (STAGE == kStageNasal) { pw0.step(); pw0.coef(a0, rho0); }
#pragma unroll
						for (int k = 0; k < NR; ++k) {
							pw[k].step();
							pw[k].coef(a[k], rho[k]);
							if (STAGE == kStageParallel) mixv[k] = mix[k].at(ci, F);
						}
						if (STAGE != kStageCascade) extraV = extra.at(ci, F);
						tickWith(q + (int)i, a, rho, mixv, extraV, n0Inv, a0, rho0);
					}
					q += (int)n;
					cur.advance(L, n);  // (stays inside the request: n <= F - c < left)
				}
			}
		}
		__syncwarp();
		// ---- tile out ----
		if (PASS == 2) {
#pragma unroll 4
			for (int r = 0; r < kTile; ++r) {
				const uint64_t g = (uint64_t)(warpChunk0 + r) * chunkTicks + tile + lane;
				if (MULTI ? tile + lane < sLen[wib][r] : (warpChunk0 + r < numChunks && g < total)) {
					const float o = tOut[wib][r][lane];
					if (STAGE == kStageLast) pcm[MULTI ? sPcm[kHasPar ? wib : 0][r] + tile + lane : g] = (int16_t)(int)o;
					else out[g] = o;
				}
			}
			__syncwarp();
		}
	}
	if (PASS == 1 && live) {
		// The last chunk of a stream leaves the zero map (P = 0, z = 0): the scan's prefix at the next stream's first chunk is
		// then exactly the zero state it starts from, with no change to the scan.  (Nothing reads a stream's last map otherwise.)
#pragma unroll
		for (int k = 0; k < NR; ++k) {
			Affine m;
			m.p00 = p00[k]; m.p01 = p01[k]; m.p10 = p10[k]; m.p11 = p11[k]; m.zy = y[k]; m.zd = d[k];
			if (lastOfStream) m = Affine{0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
			maps[(size_t)ch * NR + k] = m;
		}
	}
}

// ---------------------------------------------------------------------------------------------------------------
// scan: start state of every chunk = z-part of the composition of all earlier chunks' maps (the stream starts from
// zero state, reference src/speechWaveGenerator.cpp:104-110).  One block: each thread composes a contiguous run of
// chunks, the 1024 run totals are scanned with warp shuffles, then each thread replays its run from its prefix.
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct AffineD {  // composition is done in double: it is cheap and keeps the scan out of the error budget
	double p00, p01, p10, p11, zy, zd;
};
__device__ __forceinline__ AffineD identityMap() { return AffineD{1.0, 0.0, 0.0, 1.0, 0.0, 0.0}; }
__device__ __forceinline__ AffineD toD(const Affine &m) { return AffineD{m.p00, m.p01, m.p10, m.p11, m.zy, m.zd}; }
// `second` after `first`
__device__ __forceinline__ AffineD compose(const AffineD &second, const AffineD &first) {
	AffineD r;
	r.p00 = second.p00 * first.p00 + second.p01 * first.p10;
	r.p01 = second.p00 * first.p01 + second.p01 * first.p11;
	r.p10 = second.p10 * first.p00 + second.p11 * first.p10;
	r.p11 = second.p10 * first.p01 + second.p11 * first.p11;
	r.zy = second.p00 * first.zy + second.p01 * first.zd + second.zy;
	r.zd = second.p10 * first.zy + second.p11 * first.zd + second.zd;
	return r;
}
__device__ __forceinline__ AffineD shflUp(const AffineD &m, int delta) {
	AffineD r;
	r.p00 = __shfl_up_sync(0xffffffffu, m.p00, delta); r.p01 = __shfl_up_sync(0xffffffffu, m.p01, delta);
	r.p10 = __shfl_up_sync(0xffffffffu, m.p10, delta); r.p11 = __shfl_up_sync(0xffffffffu, m.p11, delta);
	r.zy = __shfl_up_sync(0xffffffffu, m.zy, delta); r.zd = __shfl_up_sync(0xffffffffu, m.zd, delta);
	return r;
}
}  // namespace

constexpr int kScanThreads = 1024;

// (round 1 ran this scan in ONE block: every thread composed a run of ~150 chunks out of global memory, twice -- 1.48 ms per
// section, 11.8 ms of a config-4 call.)  Three phases now: every block of 256 chunks scans its own maps (one chunk per
// thread, coalesced loads, Kogge-Stone with warp shuffles) and leaves its total; one block scans the block totals; the blocks
// scan again and write, for every chunk, the z-part of (its exclusive prefix within the block) after (the prefix of the block).
constexpr int kScanBlock = 256;

// inclusive scan of one map per thread across a block of kScanBlock threads; returns the exclusive prefix of the thread too
__device__ __forceinline__ void blockScanAffine(const AffineD &mine, AffineD &inclusive, AffineD &exclusive, AffineD *warpTotal /* smem [8] */) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	AffineD inc = mine;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		AffineD up = shflUp(inc, delta);
		if (lane >= delta) inc = compose(inc, up);
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	AffineD pre = identityMap();  // everything in the warps before this one
	for (int w = 0; w < warp; ++w) pre = compose(warpTotal[w], pre);
	AffineD prevLane = shflUp(inc, 1);
	exclusive = lane == 0 ? pre : compose(prevLane, pre);
	inclusive = compose(inc, pre);
	__syncthreads();
}

template <int PHASE>  // 1: block totals; 3: start states from the scanned block prefixes
__global__ void __launch_bounds__(kScanBlock)
klatt_long_scan_blocks_kernel(const Affine *__restrict__ maps, uint32_t numChunks, int numSections, AffineD *__restrict__ blockTotals,
                              const AffineD *__restrict__ blockPrefix, float2 *__restrict__ startState) {
	__shared__ AffineD warpTotal[kScanBlock / 32];
	const uint32_t c = blockIdx.x * kScanBlock + threadIdx.x;
	for (int k = 0; k < numSections; ++k) {
		const AffineD mine = c < numChunks ? toD(maps[(size_t)c * numSections + k]) : identityMap();
		AffineD inclusive, exclusive;
		blockScanAffine(mine, inclusive, exclusive, warpTotal);
		if (PHASE == 1) {
			if (threadIdx.x == kScanBlock - 1) blockTotals[(size_t)blockIdx.x * numSections + k] = inclusive;
		} else if (c < numChunks) {
			const AffineD pre = compose(exclusive, blockPrefix[(size_t)blockIdx.x * numSections + k]);
			startState[(size_t)c * numSections + k] = make_float2((float)pre.zy, (float)pre.zd);
		}
	}
}

// phase 2: exclusive scan of the block totals in place (one block; every thread takes a run of blocks)
__global__ void __launch_bounds__(kScanThreads)
klatt_long_scan_totals_kernel(AffineD *__restrict__ totals, uint32_t numBlocks, int numSections) {
	__shared__ AffineD warpTotal[32];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const uint32_t per = (numBlocks + kScanThreads - 1) / kScanThreads;
	const uint32_t c0 = (uint32_t)tid * per < numBlocks ? (uint32_t)tid * per : numBlocks;
	const uint32_t c1 = c0 + per < numBlocks ? c0 + per : numBlocks;
	for (int k = 0; k < numSections; ++k) {
		AffineD run = identityMap();
		for (uint32_t c = c0; c < c1; ++c) run = compose(totals[(size_t)c * numSections + k], run);
		AffineD inc = run;
#pragma unroll
		for (int delta = 1; delta < 32; delta <<= 1) {
			AffineD up = shflUp(inc, delta);
			if (lane >= delta) inc = compose(inc, up);
		}
		if (lane == 31) warpTotal[warp] = inc;
		__syncthreads();
		if (warp == 0) {
			AffineD w = warpTotal[lane];
#pragma unroll
			for (int delta = 1; delta < 32; delta <<= 1) {
				AffineD up = shflUp(w, delta);
				if (lane >= delta) w = compose(w, up);
			}
			warpTotal[lane] = w;
		}
		__syncthreads();
		AffineD prev = shflUp(inc, 1);
		AffineD pre = lane == 0 ? identityMap() : prev;
		if (warp > 0) pre = compose(pre, warpTotal[warp - 1]);
		for (uint32_t c = c0; c < c1; ++c) {
			const AffineD m = totals[(size_t)c * numSections + k];
			totals[(size_t)c * numSections + k] = pre;  // exclusive
			pre = compose(m, pre);
		}
		__syncthreads();
	}
}

// maps -> start states of all chunks; blockTotals: scratch of ceil(numChunks / 256) * numSections AffineD
static void launchLongScan(const Affine *maps, uint32_t numChunks, int numSections, void *blockTotals, float2 *startState, cudaStream_t stream) {
	const uint32_t nb = (numChunks + kScanBlock - 1) / kScanBlock;
	AffineD *tot = static_cast<AffineD *>(blockTotals);
	klatt_long_scan_blocks_kernel<1><<<nb, kScanBlock, 0, stream>>>(maps, numChunks, numSections, tot, nullptr, nullptr);
	klatt_long_scan_totals_kernel<<<1, kScanThreads, 0, stream>>>(tot, nb, numSections);
	klatt_long_scan_blocks_kernel<3><<<nb, kScanBlock, 0, stream>>>(maps, numChunks, numSections, nullptr, tot, startState);
}
size_t klattLongScanScratchBytes(uint64_t numChunks) { return sizeof(AffineD) * 6 * (size_t)((numChunks + kScanBlock - 1) / kScanBlock); }

// ---------------------------------------------------------------------------------------------------------------
// ticks of device-resident queues (speechPlayer_synthesizeLongBatchDevice): the occupancy law of timelineTicks (host.h),
// sum over a stream's requests of max(M + 1, max(F, 1) + 2), one block per stream.  Integer sums: exact in any order.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kTicksBlock = 256;
constexpr uint32_t kTicksMaxBlocks = 1u << 20;  // more streams than this: each block takes every kTicksMaxBlocks-th stream

__global__ void __launch_bounds__(kTicksBlock)
klatt_long_ticks_kernel(const int64_t *__restrict__ offsets, uint32_t numStreams, const uint32_t *__restrict__ minDur,
                        const uint32_t *__restrict__ fadeDur, uint64_t *__restrict__ ticks) {
	__shared__ unsigned long long warpSum[kTicksBlock / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (uint32_t s = blockIdx.x; s < numStreams; s += gridDim.x) {
		const int64_t end = offsets[s + 1];
		unsigned long long t = 0;
		for (int64_t j = offsets[s] + threadIdx.x; j < end; j += kTicksBlock) {
			const unsigned long long m = minDur[j], f = fadeDur[j] > 1u ? fadeDur[j] : 1u;
			t += m + 1 > f + 2 ? m + 1 : f + 2;
		}
#pragma unroll
		for (int d = 16; d > 0; d >>= 1) t += __shfl_down_sync(0xffffffffu, t, d);
		if (lane == 0) warpSum[warp] = t;
		__syncthreads();
		if (warp == 0) {
			t = lane < kTicksBlock / 32 ? warpSum[lane] : 0;
#pragma unroll
			for (int d = 16; d > 0; d >>= 1) t += __shfl_down_sync(0xffffffffu, t, d);
			if (lane == 0) ticks[s] = t;
		}
		__syncthreads();  // warpSum is rewritten for the block's next stream
	}
}

// ---------------------------------------------------------------------------------------------------------------
// launchers (launch.h)
// ---------------------------------------------------------------------------------------------------------------
cudaError_t launchKlattLongTicks(const int64_t *offsets, uint32_t numStreams, const uint32_t *minDur, const uint32_t *fadeDur,
                                 uint64_t *ticks, cudaStream_t stream) {
	if (numStreams == 0) return cudaSuccess;
	klatt_long_ticks_kernel<<<numStreams < kTicksMaxBlocks ? numStreams : kTicksMaxBlocks, kTicksBlock, 0, stream>>>(offsets, numStreams, minDur,
	                                                                                                             fadeDur, ticks);
	return cudaGetLastError();
}

cudaError_t launchKlattLongTimeline(const LongTable &T, cudaStream_t stream) {
	if (T.numStreams > 1) klatt_long_timeline_kernel<true><<<T.numStreams, kTimelineTile, 0, stream>>>(T);
	else klatt_long_timeline_kernel<false><<<1, kTimelineTile, 0, stream>>>(T);
	return cudaGetLastError();
}

// The glottal phase of every chunk: the speculative passes (fail[s] is raised for a stream whose chunks could not be
// anchored), or, with `serial`, the plain recurrence on one thread for each stream whose fail[s] is set.
// phase scratch: advance / startPhase [numChunks] u64, chunks [numChunks] PhaseChunk, startP [numChunks] double, fail [numStreams].
template <bool MULTI>
static cudaError_t longPhase(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, uint64_t *advance, uint64_t *startPhase,
                                 PhaseChunk *chunks, double *startP, uint32_t *fail, bool serial, unsigned long long *launchCounter,
                                 cudaStream_t stream) {
	if (numChunks == 0) return cudaSuccess;
	const dim3 grid((numChunks + 127) / 128), block(128);
	if (serial) {
		klatt_long_phase_serial_kernel<MULTI><<<(T.numStreams + 31) / 32, 32, 0, stream>>>(T, chunkTicks, numChunks, fail, chunks, startP);
		if (launchCounter) *launchCounter += 1;
	} else {
		klatt_long_phase_kernel<MULTI><<<grid, block, 0, stream>>>(T, chunkTicks, numChunks, advance);
		klatt_long_phase_scan_kernel<<<1, 1024, 0, stream>>>(advance, numChunks, startPhase);
		klatt_long_spec_kernel<MULTI><<<grid, block, 0, stream>>>(T, chunkTicks, numChunks, startPhase, chunks, fail);
		klatt_long_phase_map_scan_kernel<MULTI><<<1, 1024, 0, stream>>>(T, chunks, numChunks, startP);
		if (launchCounter) *launchCounter += 4;
	}
	return cudaGetLastError();
}

// The source pass (which checks the phase runs and raises fail[s] on a miss) and the resonator stages, into the int16 output.
// signals: five float arrays of numChunks * chunkTicks virtual ticks (+ padding): ci, pin, par, xa, xb.  maps / startState:
// numChunks * 6.  pcm: the packed output, stream s from streams[s].outBase.
template <bool MULTI>
static cudaError_t longSynth(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, const PhaseChunk *chunks,
                                 const double *startP, uint32_t *fail, float *ci, float *pin, float *par, float *xa, float *xb,
                                 Affine *maps, float2 *startState, void *scanScratch, int16_t *pcm, unsigned long long *launchCounter,
                                 cudaStream_t stream) {
	if (numChunks == 0) return cudaSuccess;
	const dim3 grid((numChunks + 127) / 128), block(128);
	const dim3 sgrid((numChunks + kStageBlock - 1) / kStageBlock), sblock(kStageBlock);
	klatt_long_source_kernel<MULTI><<<grid, block, 0, stream>>>(T, chunkTicks, numChunks, chunks, startP, fail, ci, pin);
	// parallel bank
	klatt_long_stage_kernel<kStageParallel, 1, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, 0, pin, nullptr, maps, nullptr, nullptr, nullptr);
	launchLongScan(maps, numChunks, 6, scanScratch, startState, stream);
	klatt_long_stage_kernel<kStageParallel, 2, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, 0, pin, nullptr, nullptr, startState, par, nullptr);
	// rN0 + rNP
	klatt_long_stage_kernel<kStageNasal, 1, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, kResNP, ci, nullptr, maps, nullptr, nullptr, nullptr);
	launchLongScan(maps, numChunks, 1, scanScratch, startState, stream);
	klatt_long_stage_kernel<kStageNasal, 2, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, kResNP, ci, nullptr, nullptr, startState, xa, nullptr);
	// r6 .. r2
	float *src = xa, *dst = xb;
	for (int r = kResCascade; r < kResParallel - 1; ++r) {
		klatt_long_stage_kernel<kStageCascade, 1, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, r, src, nullptr, maps, nullptr, nullptr, nullptr);
		launchLongScan(maps, numChunks, 1, scanScratch, startState, stream);
		klatt_long_stage_kernel<kStageCascade, 2, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, r, src, nullptr, nullptr, startState, dst, nullptr);
		float *tmp = src; src = dst; dst = tmp;
	}
	// r1 + output
	klatt_long_stage_kernel<kStageLast, 1, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, kResParallel - 1, src, par, maps, nullptr, nullptr, nullptr);
	launchLongScan(maps, numChunks, 1, scanScratch, startState, stream);
	klatt_long_stage_kernel<kStageLast, 2, MULTI><<<sgrid, sblock, 0, stream>>>(T, chunkTicks, numChunks, kResParallel - 1, src, par, nullptr, startState, nullptr, pcm);
	if (launchCounter) *launchCounter += 1 + 5 * 8;
	return cudaGetLastError();
}

cudaError_t launchKlattLongPhase(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, uint64_t *advance, uint64_t *startPhase,
                                 PhaseChunk *chunks, double *startP, uint32_t *fail, bool serial, unsigned long long *launchCounter,
                                 cudaStream_t stream) {
	return T.numStreams > 1 ? longPhase<true>(T, numChunks, chunkTicks, advance, startPhase, chunks, startP, fail, serial, launchCounter, stream)
	                        : longPhase<false>(T, numChunks, chunkTicks, advance, startPhase, chunks, startP, fail, serial, launchCounter, stream);
}

cudaError_t launchKlattLongSynth(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, const PhaseChunk *chunks,
                                 const double *startP, uint32_t *fail, float *ci, float *pin, float *par, float *xa, float *xb,
                                 Affine *maps, float2 *startState, void *scanScratch, int16_t *pcm, unsigned long long *launchCounter,
                                 cudaStream_t stream) {
	return T.numStreams > 1
	           ? longSynth<true>(T, numChunks, chunkTicks, chunks, startP, fail, ci, pin, par, xa, xb, maps, startState, scanScratch, pcm, launchCounter, stream)
	           : longSynth<false>(T, numChunks, chunkTicks, chunks, startP, fail, ci, pin, par, xa, xb, maps, startState, scanScratch, pcm, launchCounter, stream);
}

}  // namespace klatt
