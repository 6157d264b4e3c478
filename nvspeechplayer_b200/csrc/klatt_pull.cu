// klatt_pull_kernel: one pull of one player in one thread block, parallel in time (see klatt_pull_core.cuh for the
// scheme and for the per-thread passes; this file adds the block scans and the launcher).
//
// 512 threads; thread i owns ticks [i*L, (i+1)*L) of the pull.  The two signals every stage reads and rewrites in place
// (cascade chain, parallel chain) and the per-tick phase increments live in dynamic shared memory, tick-major ([L][512]: the threads of a warp touch
// consecutive banks).  Affine maps never leave registers: the scans are warp-shuffle scans (the pattern of
// klatt_long_scan_kernel with one chunk per thread) with a 16-entry shared array for the warp totals, seeded with the
// state the player carries from its previous pull.
#include <cuda_runtime.h>
#include "klatt_common.h"
#include "klatt_pull_core.cuh"
#include "launch.h"

namespace klatt {

namespace {

constexpr int kPullWarps = kPullThreads / 32;

__device__ __forceinline__ PullAffineD shflUpD(const PullAffineD &m, int delta) {
	PullAffineD r;
	r.p00 = __shfl_up_sync(0xffffffffu, m.p00, delta); r.p01 = __shfl_up_sync(0xffffffffu, m.p01, delta);
	r.p10 = __shfl_up_sync(0xffffffffu, m.p10, delta); r.p11 = __shfl_up_sync(0xffffffffu, m.p11, delta);
	r.zy = __shfl_up_sync(0xffffffffu, m.zy, delta); r.zd = __shfl_up_sync(0xffffffffu, m.zd, delta);
	return r;
}

// Composition of `seed` and the maps of all threads before this one, in order.  Every thread of the block calls it.
__device__ PullAffineD blockExclusive(const PullAffineD &own, const PullAffineD &seed, PullAffineD *warpTotal) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	PullAffineD inc = own;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		PullAffineD up = shflUpD(inc, delta);
		if (lane >= delta) inc = pullCompose(inc, up);
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		PullAffineD w = lane < kPullWarps ? warpTotal[lane] : pullIdentity();
#pragma unroll
		for (int delta = 1; delta < kPullWarps; delta <<= 1) {
			PullAffineD up = shflUpD(w, delta);
			if (lane >= delta) w = pullCompose(w, up);
		}
		if (lane < kPullWarps) warpTotal[lane] = w;
	}
	__syncthreads();
	// exclusive prefix = (inclusive of the previous lane) after (inclusive total of the earlier warps) after the seed
	PullAffineD prev = shflUpD(inc, 1);
	PullAffineD pre = lane == 0 ? pullIdentity() : prev;
	if (warp > 0) pre = pullCompose(pre, warpTotal[warp - 1]);
	pre = pullCompose(pre, seed);
	__syncthreads();  // warpTotal may be reused; every read of the carried state is behind us
	return pre;
}

__device__ __forceinline__ PullAffineD seedOf(float y, float d) { return pullSeed(y, d); }

// ---- scans of the run decomposition of the phase (phaseMode 1) ----
__device__ __forceinline__ PullRunSum shflUpRun(const PullRunSum &m, int delta) {
	PullRunSum r;
	r.sum = __shfl_up_sync(0xffffffffu, m.sum, delta);
	r.flag = __shfl_up_sync(0xffffffffu, m.flag, delta);
	r.specials = __shfl_up_sync(0xffffffffu, m.specials, delta);
	return r;
}
// exclusive segmented prefix over the block; total = the combination of all 512 elements
__device__ PullRunSum blockExclusiveRuns(const PullRunSum &own, PullRunSum *warpTotal, PullRunSum &total) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const PullRunSum zero{0, 0u, 0u};
	PullRunSum inc = own;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		PullRunSum up = shflUpRun(inc, delta);
		if (lane >= delta) inc = pullRunCombine(up, inc);
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		PullRunSum w = lane < kPullWarps ? warpTotal[lane] : zero;
#pragma unroll
		for (int delta = 1; delta < kPullWarps; delta <<= 1) {
			PullRunSum up = shflUpRun(w, delta);
			if (lane >= delta) w = pullRunCombine(up, w);
		}
		if (lane < kPullWarps) warpTotal[lane] = w;
	}
	__syncthreads();
	PullRunSum prev = shflUpRun(inc, 1);
	PullRunSum pre = lane == 0 ? zero : prev;
	if (warp > 0) pre = pullRunCombine(warpTotal[warp - 1], pre);
	total = warpTotal[kPullWarps - 1];
	__syncthreads();
	return pre;
}
// exclusive sum modulo 2^64 (the approximate phase in 2^-64 cycles: exact and associative)
__device__ uint64_t blockExclusiveU64(uint64_t own, uint64_t *warpSum) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint64_t inc = own;
#pragma unroll
	for (int delta = 1; delta < 32; delta <<= 1) {
		uint64_t up = __shfl_up_sync(0xffffffffu, inc, delta);
		if (lane >= delta) inc += up;
	}
	if (lane == 31) warpSum[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		uint64_t w = lane < kPullWarps ? warpSum[lane] : 0;
#pragma unroll
		for (int delta = 1; delta < kPullWarps; delta <<= 1) {
			uint64_t up = __shfl_up_sync(0xffffffffu, w, delta);
			if (lane >= delta) w += up;
		}
		if (lane < kPullWarps) warpSum[lane] = w;
	}
	__syncthreads();
	const uint64_t pre = inc - own + (warp > 0 ? warpSum[warp - 1] : 0);
	__syncthreads();
	return pre;
}

template <int STAGE>
__device__ __forceinline__ void runStage(const PullCtx &X, uint32_t ch, int res, PullAffineD *warpTotal) {
	constexpr int NR = StageTraits<STAGE>::NR;
	Affine maps[NR];
	PullStart st[NR];
	PoleWalk poles[NR + 1];
	float fir[2] = {0.0f, 0.0f};
	pullStage<STAGE, 1>(X, ch, res, maps, nullptr, fir, poles);
#pragma unroll
	for (int k = 0; k < NR; ++k) {
		const int r = STAGE == kStageParallel ? kResParallel + k : res;
		const PullAffineD pre = blockExclusive(pullToD(maps[k]), seedOf(X.state->y[r], X.state->d[r]), warpTotal);
		st[k].y = (float)pre.zy;
		st[k].d = (float)pre.zd;
	}
	pullStage<STAGE, 2>(X, ch, res, nullptr, st, fir, poles);
}

__device__ __forceinline__ void mark(const PullCtx &X, int slot) {
	if (X.dbg && threadIdx.x == 0) X.dbg[slot] = clock64();
}

}  // namespace

// Shared memory: sigA | sigB | inc | the pull's segments | the pull's samples.  segSrc and pcmOut
// may be pinned host memory (zero-copy): the segments come in and the samples go out in 16-byte words, coalesced, so a
// pull is ONE launch with no copy before or after it.
__device__ __forceinline__ void pullBlock(PullCtx X, const PullSeg *__restrict__ segSrc, int16_t *__restrict__ pcmOut) {
	extern __shared__ __align__(16) unsigned char pullSmem[];
	__shared__ PullAffineD warpTotal[kPullWarps];
	const size_t sigBytes = (size_t)X.L * kPullThreads * sizeof(float);
	X.sigA = reinterpret_cast<float *>(pullSmem);
	X.sigB = reinterpret_cast<float *>(pullSmem + sigBytes);
	X.inc = reinterpret_cast<double *>(pullSmem + 2 * sigBytes);
	PullSeg *segS = reinterpret_cast<PullSeg *>(pullSmem + 4 * sigBytes);
	int16_t *pcmS = reinterpret_cast<int16_t *>(pullSmem + 4 * sigBytes + (size_t)X.nSeg * sizeof(PullSeg));
	X.runI = reinterpret_cast<int64_t *>(pullSmem);         // over sigA + sigB, both dead until source pass 2
	X.runMeta = reinterpret_cast<uint16_t *>(pcmS);         // over the output staging, dead until the last stage
	X.rec = reinterpret_cast<PullPhaseRec *>(pullSmem + 4 * sigBytes + (size_t)X.nSeg * sizeof(PullSeg) +
	                                         (((size_t)X.n * sizeof(int16_t) + 15) & ~(size_t)15));
	const uint32_t ch = threadIdx.x;
	{
		const uint4 *src = reinterpret_cast<const uint4 *>(segSrc);
		uint4 *dst = reinterpret_cast<uint4 *>(segS);
		const uint32_t words = X.nSeg * (uint32_t)(sizeof(PullSeg) / 16);
		for (uint32_t i = ch; i < words; i += kPullThreads) dst[i] = src[i];
	}
	__syncthreads();
	X.segs = segS;
	X.pcm = pcmS;
	if (X.dbg && ch == 0) {
		unsigned long long ns;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
		X.dbg[15] = (long long)ns;
	}
	mark(X, 0);

	// source: phase increments and noise colouring per chunk, the phase recurrence by one thread, then the excitation
	{
		PullSourceSums sums;
		pullSourcePass1(X, ch, sums);
		mark(X, 1);
		const PullAffineD own{sums.decay, 0, 0, sums.decay, sums.zAsp, sums.zFric};
		const PullAffineD pre = blockExclusive(own, seedOf(X.state->aspLast, X.state->fricLast), warpTotal);
		mark(X, 2);
		bool runsDone = false;
		if (X.phaseMode) {  // run decomposition: the serial thread only visits the special ticks
			__shared__ PullRunSum runTotal[kPullWarps];
			__shared__ uint64_t warpSum[kPullWarps];
			const double pos0 = X.state->pitchPos;
			uint64_t fixed0;
			const bool okStart = pullRunsStart(pos0, fixed0);
			const uint64_t startFixed = fixed0 + blockExclusiveU64(sums.phaseFixed, warpSum);
			PullRunSum mine;
			pullRunsClassify(X, ch, startFixed, mine);
			if (ch == 0 && !okStart) mine.specials += kPullMaxSpecial + 1;
			PullRunSum total;
			const PullRunSum before = blockExclusiveRuns(mine, runTotal, total);  // its barriers also publish runMeta / runI
			if (total.specials <= kPullMaxSpecial) {  // uniform
				pullRunsOffsets(X, ch, before);
				__syncthreads();
				if (ch == 0) pullRunsSerial(X, total.specials, pos0);
				__syncthreads();
				pullRunsFinish(X, ch, before.specials, pos0);
				runsDone = true;
			}
		}
		if (!runsDone && ch == 0) pullPhaseSerial(X);
		__syncthreads();
		mark(X, 3);
		pullSourcePass2(X, ch, (float)pre.zy, (float)pre.zd);
	}
	__syncthreads();  // the FIR section of the nasal stage reads its neighbours' last two cascade inputs
	mark(X, 4);

	runStage<kStageParallel>(X, ch, 0, warpTotal);
	mark(X, 5);
	runStage<kStageNasal>(X, ch, kResNP, warpTotal);
	mark(X, 6);
	for (int r = kResCascade; r < kResParallel - 1; ++r) runStage<kStageCascade>(X, ch, r, warpTotal);
	mark(X, 7);
	runStage<kStageLast>(X, ch, kResParallel - 1, warpTotal);

	__syncthreads();
	{
		const uint4 *src = reinterpret_cast<const uint4 *>(pcmS);
		uint4 *dst = reinterpret_cast<uint4 *>(pcmOut);
		const uint32_t words = (X.n * (uint32_t)sizeof(int16_t) + 15u) / 16u;
		for (uint32_t i = ch; i < words; i += kPullThreads) dst[i] = src[i];
	}
	mark(X, 8);
	if (ch == 0) X.state->generated += X.n;
	if (X.dbg && ch == 0) {
		unsigned long long ns;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
		X.dbg[14] = (long long)ns;
	}
}

__global__ void __launch_bounds__(kPullThreads)
klatt_pull_kernel(PullCtx X, const PullSeg *__restrict__ segSrc, int16_t *__restrict__ pcmOut) {
	pullBlock(X, segSrc, pcmOut);
}

// Many interactive players in ONE launch: block b renders the pull of player b (its own segments, carried state, noise and
// output -- nothing is shared between blocks), so 148 players pull at the latency of one.  items may be mapped pinned memory.
__global__ void __launch_bounds__(kPullThreads)
klatt_pull_batch_kernel(const PullBatchItem *__restrict__ items) {
	const PullBatchItem it = items[blockIdx.x];
	if (it.ctx.n == 0) return;  // (uniform per block: this player had nothing to render)
	pullBlock(it.ctx, it.segSrc, it.pcmOut);
}

__global__ void klatt_pull_init_kernel(PullState *s) {
	// src/speechWaveGenerator.cpp:37,49,104-110: phases, noise memories and resonator histories start at zero
	if (threadIdx.x == 0 && blockIdx.x == 0) {
		for (int r = 0; r < kNumResonators; ++r) { s->y[r] = 0.0f; s->d[r] = 0.0f; }
		s->aspLast = 0.0f; s->fricLast = 0.0f; s->pitchPos = 0.0; s->generated = 0;
	}
}

cudaError_t launchKlattPullInit(PullState *state, cudaStream_t stream) {
	klatt_pull_init_kernel<<<1, 32, 0, stream>>>(state);
	return cudaGetLastError();
}

// ctx.sigA / sigB / inc / L / segs / pcm are filled in by the launch; everything else by the caller.  ctx.n <= kPullMaxTicks.
// segSrc: ctx.nSeg segments, pcmOut: room for ctx.n samples rounded up to 8 -- device memory or mapped pinned host memory.
static cudaError_t pullPrepare(PullCtx &ctx, size_t &smem) {
	if (ctx.n > kPullMaxTicks || ctx.nSeg == 0 || ctx.nSeg > kPullMaxSegs) return cudaErrorInvalidValue;
	static bool attrSet[64] = {};
	int dev = 0;
	cudaError_t e = cudaGetDevice(&dev);
	if (e != cudaSuccess) return e;
	constexpr size_t kMaxSmem = 4 * (size_t)kPullMaxTicks * sizeof(float) + kPullMaxSegs * sizeof(PullSeg) +
	                            kPullMaxTicks * sizeof(int16_t) + kPullMaxSpecial * sizeof(PullPhaseRec);
	if (dev >= 0 && dev < 64 && !attrSet[dev]) {
		e = cudaFuncSetAttribute(klatt_pull_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
		if (e != cudaSuccess) return e;
		e = cudaFuncSetAttribute(klatt_pull_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
		if (e != cudaSuccess) return e;
		attrSet[dev] = true;
	}
	ctx.L = pullTicksPerThread(ctx.n);  // 1, 2, 4, 8 or 16: the phase recurrence is unrolled for these
	ctx.sigA = ctx.sigB = nullptr;
	ctx.inc = nullptr;
	ctx.segs = nullptr;
	ctx.pcm = nullptr;
	smem = 4 * (size_t)ctx.L * kPullThreads * sizeof(float) + (size_t)ctx.nSeg * sizeof(PullSeg) +
	       (((size_t)ctx.n * sizeof(int16_t) + 15) & ~(size_t)15) + (ctx.phaseMode ? kPullMaxSpecial * sizeof(PullPhaseRec) : 0);
	ctx.runI = nullptr;
	ctx.runMeta = nullptr;
	ctx.rec = nullptr;
	return cudaSuccess;
}

cudaError_t launchKlattPull(PullCtx ctx, const PullSeg *segSrc, int16_t *pcmOut, cudaStream_t stream) {
	if (ctx.n == 0) return cudaSuccess;
	size_t smem = 0;
	cudaError_t e = pullPrepare(ctx, smem);
	if (e != cudaSuccess) return e;
	klatt_pull_kernel<<<1, kPullThreads, smem, stream>>>(ctx, segSrc, pcmOut);
	return cudaGetLastError();
}

// hItems: host view of `count` items (filled by the caller except what pullPrepare derives), dItems: the same memory as the
// device sees it (mapped pinned) or a device copy made after this call returns... the items are completed IN PLACE, so with a
// device copy the caller copies after launchKlattPullBatchPrepare and launches with launchKlattPullBatch.
cudaError_t launchKlattPullBatch(PullBatchItem *hItems, const PullBatchItem *dItems, uint32_t count, cudaStream_t stream) {
	size_t smemMax = 0;
	bool any = false;
	for (uint32_t i = 0; i < count; ++i) {
		if (hItems[i].ctx.n == 0) continue;
		size_t smem = 0;
		cudaError_t e = pullPrepare(hItems[i].ctx, smem);
		if (e != cudaSuccess) return e;
		if (smem > smemMax) smemMax = smem;
		any = true;
	}
	if (!any) return cudaSuccess;
	klatt_pull_batch_kernel<<<count, kPullThreads, smemMax, stream>>>(dItems);
	return cudaGetLastError();
}

}  // namespace klatt
