// The FP32 production kernels.  One stream per thread; the per-stream working set lives in registers, the frame
// queue and the per-request fade plans are read from HBM only on event ticks, and the int16 output leaves as
// 16-byte stores (out_writer.cuh).  The arithmetic is klatt_f32_core.cuh (compiled with -fmad=false: every fused
// multiply-add is an explicit fmaf, so the two render kernels round identically on a hold tick).
//
//   klatt_plan_kernel        one thread per queued REQUEST: the fade plan (all FP64 transcendentals of the path:
//                            14 x (exp, cos) per frame of reference src/speechWaveGenerator.cpp:113-125, hoisted out
//                            of the per-tick loop) for whole pre-queued batches
//   klatt_partition_kernel   one thread per stream, once per round: which streams have `holdTicks` pure hold ticks
//                            ahead (-> hold list) and which need the frame manager (-> general list)
//   klatt_f32_hold_kernel    `holdTicks` ticks of src/frame.cpp:76-79 + src/speechWaveGenerator.cpp:203-208 with
//                            constant coefficients: no state machine, no coefficient updates
//   klatt_f32_general_kernel up to `genTicks` ticks through the full frame manager (src/frame.cpp:41-80) with
//                            per-tick coefficient recurrences
//   klatt_finalize_kernel    per-stream results of a call made of rounds
//
// Why rounds: lanes of a warp that are in different frame-manager phases would make every tick pay for the fade
// arithmetic (~2x a hold tick).  Re-sorting streams by phase every round keeps warps homogeneous; hold chunks are
// twice as long as general chunks so that both kernels of a round take about the same time (DESIGN.md "Rounds").
#include <cuda_runtime.h>
#include "klatt_common.h"
#include "klatt_f32_core.cuh"
#include "out_writer.cuh"
#include "klatt_f32_pair.cuh"
#include "launch.h"

namespace klatt {

constexpr int kF32Block = 64;
#ifndef KLATT_GEN_MINB
#define KLATT_GEN_MINB 4
#endif


// ---------------------------------------------------------------------------------------------------
// plans for pre-queued batches
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
klatt_plan_kernel(const int64_t *__restrict__ offsets, uint32_t numStreams, const double *__restrict__ frames,
                  const uint32_t *__restrict__ fadeDur, const uint8_t *__restrict__ isNull, int sampleRate,
                  FadePlanF32 *__restrict__ plans) {
	const int64_t total = offsets[numStreams];
	const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= total) return;
	// the stream that owns request g: last s with offsets[s] <= g
	uint32_t lo = 0, hi = numStreams;
	while (hi - lo > 1) {
		uint32_t mid = (lo + hi) >> 1;
		if (offsets[mid] <= g) lo = mid; else hi = mid;
	}
	const int64_t first = offsets[lo];
	const bool curNull = isNull ? (isNull[g] != 0) : false;
	const bool prevNull = (g == first) || (isNull && isNull[g - 1] != 0);
	int64_t p = g - 1;
	while (p >= first && isNull && isNull[p] != 0) --p;
	const double *prevReal = (p >= first && frames) ? frames + (size_t)p * kNumParams : nullptr;
	double o[kNumParams], n[kNumParams];
	plannedFrames(prevReal, prevNull, frames ? frames + (size_t)g * kNumParams : nullptr, curNull || !frames, o, n);
	const uint32_t fd = fadeDur[g];
	planFade(o, n, fd > 1u ? fd : 1u, sampleRate, plans[g]);
}

// ---------------------------------------------------------------------------------------------------
// rounds
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
klatt_partition_kernel(const StreamDesc *__restrict__ descs, uint32_t firstStream, uint32_t numStreams, uint32_t sampleCount,
                       uint32_t holdTicks, uint32_t genTicks, int firstRound, uint32_t *__restrict__ listHold,
                       uint32_t *__restrict__ listGen, uint32_t *__restrict__ counters) {
	const uint32_t s = firstStream + blockIdx.x * blockDim.x + threadIdx.x;
	int cls = 0;  // 0: nothing to do, 1: hold chunk, 2: general chunk
	if (s < firstStream + numStreams) {
		StreamState *st = descs[s].state;
		GenStateF32 &gs = st->gen.f32;
		if (firstRound) { gs.callPos = 0; gs.callDrained = 0; }
		const uint32_t pos = firstRound ? 0u : gs.callPos;
		const bool drained = firstRound ? false : (gs.callDrained != 0);
		if (pos < sampleCount && !drained) {
			const uint32_t left = sampleCount - pos;
			cls = (left >= holdTicks && canHoldF32(*st, holdTicks)) ? 1 : 2;
		}
	}
	const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
	const unsigned mH = __ballot_sync(0xffffffffu, cls == 1), mG = __ballot_sync(0xffffffffu, cls == 2);
	uint32_t baseH = 0, baseG = 0;
	if (lane == 0) {
		if (mH) baseH = atomicAdd(counters + 0, (uint32_t)__popc(mH));
		if (mG) baseG = atomicAdd(counters + 1, (uint32_t)__popc(mG));
	}
	baseH = __shfl_sync(0xffffffffu, baseH, 0);
	baseG = __shfl_sync(0xffffffffu, baseG, 0);
	if (cls == 1) listHold[baseH + __popc(mH & below)] = s;
	if (cls == 2) listGen[baseG + __popc(mG & below)] = s;
}

// descs[numStreams] is a dummy stream (fresh state, empty queue) that the idle lanes of a partially filled warp run
__global__ void __launch_bounds__(kPairBlock, 6)
klatt_f32_hold_kernel(const StreamDesc *__restrict__ descs, const uint32_t *__restrict__ list,
                      const uint32_t *__restrict__ counters, uint32_t numStreams, int sampleRate, uint32_t holdTicks,
                      int16_t *__restrict__ out, size_t rowStride, int16_t *__restrict__ scratchRow, NoiseConfig noise) {
	__shared__ uint4 xbuf[2][2 * kGroupTicks * 32];
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, pair = warp & 1u;
	const uint32_t count = counters[0];
	if (blockIdx.x * kPairStreams + pair * 32 >= count) return;  // the whole warp pair is idle
	const uint32_t slot = blockIdx.x * kPairStreams + pair * 32 + lane;
	const bool valid = slot < count;
	const uint32_t s = valid ? list[slot] : numStreams;
	const StreamDesc &desc = descs[s];
	XchgSmem xc{(uint32_t)__cvta_generic_to_shared(&xbuf[pair][lane]), 1u + pair};
	if (cascadeRole(warp)) {
		// idle lanes render the dummy stream into a scratch row of holdTicks samples
		int16_t *row = valid ? out + (size_t)s * rowStride + desc.state->gen.f32.callPos : scratchRow;
		OutWriter ow;
		ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
		renderHoldF32<kRoleCascadeOsc>(desc, sampleRate, holdTicks, ow, noise, xc);
	} else {
		NullOut no;
		renderHoldF32<kRoleParallelOnly>(desc, sampleRate, holdTicks, no, noise, xc);
	}
}

// a round of the general path: thread pair = stream list[slot], at most genTicks ticks from where the stream stands
__global__ void __launch_bounds__(kPairBlock, KLATT_GEN_MINB)
klatt_f32_general_pair_kernel(const StreamDesc *__restrict__ descs, const uint32_t *__restrict__ list,
                              const uint32_t *__restrict__ counters, uint32_t numStreams, int sampleRate,
                              uint32_t sampleCount, uint32_t genTicks, int16_t *__restrict__ out, size_t rowStride,
                              NoiseConfig noise) {
	__shared__ uint4 xbuf[2][2 * kGroupTicks * 32];
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, pair = warp & 1u;
	const uint32_t count = counters[1];
	if (blockIdx.x * kPairStreams + pair * 32 >= count) return;
	const uint32_t slot = blockIdx.x * kPairStreams + pair * 32 + lane;
	const bool valid = slot < count;
	const uint32_t s = valid ? list[slot] : numStreams;
	const StreamDesc &desc = descs[s];
	const uint32_t pos = desc.state->gen.f32.callPos;
	uint32_t ticks = 0;
	if (valid) {
		ticks = sampleCount - pos;
		if (ticks > genTicks) ticks = genTicks;
	}
	XchgSmem xc{(uint32_t)__cvta_generic_to_shared(&xbuf[pair][lane]), 1u + pair};
	int32_t lastUserIndex;
	uint32_t qHead;
	if (cascadeRole(warp)) {
		int16_t *row = out + (size_t)(valid ? s : 0) * rowStride;
		OutWriter ow;
		ow.init(row + pos, ((reinterpret_cast<uintptr_t>(row + pos) & 15u) == 0));  // idle lanes have no ticks: they never store
		const uint32_t produced = renderGeneralF32<kRoleCascade>(desc, sampleRate, ticks, genTicks, ow, noise, xc, &lastUserIndex, &qHead);
		ow.flush();
		if (produced < ticks) zeroRow(row, pos + produced, sampleCount);  // drained: the rest of the row is silence
	} else {
		NullOut no;
		renderGeneralF32<kRoleParallel>(desc, sampleRate, ticks, genTicks, no, noise, xc, &lastUserIndex, &qHead);
	}
}

// One launch renders the whole call, both sides of a stream in one thread (thread i = stream i; call state reset
// and results written here).  Per-handle API and small batches; plans inline unless the descriptors carry them.
__global__ void __launch_bounds__(kF32Block)
klatt_f32_general_kernel(const StreamDesc *__restrict__ descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                         int16_t *__restrict__ out, size_t rowStride, uint32_t *__restrict__ samplesWritten,
                         StreamResult *__restrict__ results, NoiseConfig noise) {
	const uint32_t s = blockIdx.x * kF32Block + threadIdx.x;
	if (s >= numStreams) return;
	const StreamDesc desc = descs[s];
	GenStateF32 &gs = desc.state->gen.f32;
	gs.callPos = 0;
	gs.callDrained = 0;
	int16_t *row = out + (size_t)s * rowStride;
	OutWriter ow;
	ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
	int32_t lastUserIndex;
	uint32_t qHead;
	XchgSelf xc;
	const uint32_t produced = renderGeneralF32<kRoleBoth>(desc, sampleRate, sampleCount, sampleCount, ow, noise, xc, &lastUserIndex, &qHead);
	ow.flush();
	if (produced < sampleCount) zeroRow(row, produced, sampleCount);  // drained: the rest of the row is silence
	if (samplesWritten) samplesWritten[s] = produced;
	if (results) {
		StreamResult res;
		res.written = produced; res.lastUserIndex = lastUserIndex; res.qHead = qHead; res.pad = 0;
		results[s] = res;
	}
}

__global__ void __launch_bounds__(256)
klatt_finalize_kernel(const StreamDesc *__restrict__ descs, uint32_t numStreams, uint32_t *__restrict__ samplesWritten,
                      StreamResult *__restrict__ results) {
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= numStreams) return;
	const StreamState *st = descs[s].state;
	const uint32_t w = st->gen.f32.callPos;
	if (samplesWritten) samplesWritten[s] = w;
	if (results) {
		StreamResult res;
		res.written = w; res.lastUserIndex = st->fm.lastUserIndex; res.qHead = st->fm.qHead; res.pad = 0;
		results[s] = res;
	}
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
cudaError_t launchKlattFinalize(const StreamDesc *descs, uint32_t numStreams, uint32_t *samplesWritten, StreamResult *results,
                                cudaStream_t stream) {
	klatt_finalize_kernel<<<(numStreams + 255) / 256, 256, 0, stream>>>(descs, numStreams, samplesWritten, results);
	return cudaGetLastError();
}

cudaError_t launchKlattPlan(const int64_t *offsets, uint32_t numStreams, uint64_t totalRequests, const double *frames,
                            const uint32_t *fadeDur, const uint8_t *isNull, int sampleRate, FadePlanF32 *plans,
                            cudaStream_t stream) {
	if (totalRequests == 0) return cudaSuccess;
	const unsigned grid = (unsigned)((totalRequests + 127) / 128);
	klatt_plan_kernel<<<grid, 128, 0, stream>>>(offsets, numStreams, frames, fadeDur, isNull, sampleRate, plans);
	return cudaGetLastError();
}

cudaError_t launchKlattF32(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream) {
	if (numStreams == 0 || sampleCount == 0) return cudaSuccess;
	dim3 grid((numStreams + kF32Block - 1) / kF32Block);
	klatt_f32_general_kernel<<<grid, kF32Block, 0, stream>>>(descs, numStreams, sampleRate, sampleCount, out, rowStride,
	                                                         samplesWritten, results, noise);
	return cudaGetLastError();
}

// One call as rounds of (partition, hold || general).  The streams are split into `numGroups` contiguous groups that
// run their rounds independently, each on its own pair of CUDA streams, so that the tail of one group's round (few
// blocks left, SMs draining) overlaps the other groups' kernels.  lanes[2*g] / lanes[2*g+1] are the two streams of
// group g, evFork / evJoin[g] events owned by the caller.  Everything is ordered after what `stream` holds at the
// time of the call, and `stream` waits for all groups before the results kernel.
// scratch: listHold[numStreams], listGen[numStreams], counters[2 * rounds * numGroups] (zeroed here).  descs holds
// numStreams + 1 entries: the last one is the dummy stream idle lanes run.
cudaError_t launchKlattF32Rounds(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                 uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride,
                                 uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise, uint32_t *listHold,
                                 uint32_t *listGen, uint32_t *counters, int16_t *scratchRow, cudaStream_t stream, uint32_t numGroups,
                                 cudaStream_t *lanes, cudaEvent_t evStart, cudaEvent_t *evFork, cudaEvent_t *evJoin,
                                 unsigned long long *launchCounter) {
	if (numStreams == 0 || sampleCount == 0) return cudaSuccess;
	const uint32_t rounds = (sampleCount + genTicks - 1) / genTicks;
	cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(uint32_t) * 2 * (size_t)rounds * numGroups, stream);
	if (e != cudaSuccess) return e;
	if ((e = cudaEventRecord(evStart, stream)) != cudaSuccess) return e;
	const uint32_t perGroup = ((numStreams + numGroups - 1) / numGroups + kPairStreams - 1) / kPairStreams * kPairStreams;
	for (uint32_t g = 0; g < numGroups; ++g)
		if ((e = cudaStreamWaitEvent(lanes[2 * g], evStart, 0)) != cudaSuccess) return e;
	for (uint32_t r = 0; r < rounds; ++r) {
		for (uint32_t g = 0; g < numGroups; ++g) {
			const uint32_t first = g * perGroup;
			if (first >= numStreams) break;
			const uint32_t n = numStreams - first < perGroup ? numStreams - first : perGroup;
			cudaStream_t main = lanes[2 * g], side = lanes[2 * g + 1];
			uint32_t *cnt = counters + 2 * ((size_t)g * rounds + r);
			const dim3 gridP((n + 255) / 256), gridR((n + kPairStreams - 1) / kPairStreams);
			klatt_partition_kernel<<<gridP, 256, 0, main>>>(descs, first, n, sampleCount, holdTicks, genTicks, r == 0,
			                                                listHold + first, listGen + first, cnt);
			if ((e = cudaEventRecord(evFork[g], main)) != cudaSuccess) return e;
			if ((e = cudaStreamWaitEvent(side, evFork[g], 0)) != cudaSuccess) return e;
			klatt_f32_general_pair_kernel<<<gridR, kPairBlock, 0, side>>>(descs, listGen + first, cnt, numStreams, sampleRate,
			                                                              sampleCount, genTicks, out, rowStride, noise);
			klatt_f32_hold_kernel<<<gridR, kPairBlock, 0, main>>>(descs, listHold + first, cnt, numStreams, sampleRate, holdTicks,
			                                                      out, rowStride, scratchRow, noise);
			if ((e = cudaEventRecord(evJoin[g], side)) != cudaSuccess) return e;
			if ((e = cudaStreamWaitEvent(main, evJoin[g], 0)) != cudaSuccess) return e;
			if (launchCounter) *launchCounter += 3;
		}
	}
	for (uint32_t g = 0; g < numGroups; ++g) {
		if ((e = cudaEventRecord(evJoin[g], lanes[2 * g])) != cudaSuccess) return e;
		if ((e = cudaStreamWaitEvent(stream, evJoin[g], 0)) != cudaSuccess) return e;
	}
	klatt_finalize_kernel<<<(numStreams + 255) / 256, 256, 0, stream>>>(descs, numStreams, samplesWritten, results);
	if (launchCounter) *launchCounter += 1;
	return cudaGetLastError();
}

}  // namespace klatt
