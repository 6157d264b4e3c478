// The block scheduler of the FP32 batch path: the default for large pre-queued batches (klatt_f32_sched.cu's ring scheduler
// serves the smaller ones; NVSP_SCHED=rings / rounds select the older paths).  Same render bodies (klatt_f32_core.cuh), same
// bits.
//
// What the ring scheduler measured (profiles/r02_sched_baseline_*): 81 % of the worker cycles went into GENERAL chunks,
// which ran 61 % of all ticks although only 33 % of the ticks are fade ticks -- a stream had to show 512 pure hold ticks to
// leave the general loop and stayed in it for 640 ticks at a time, because every change of loop cost a trip through two
// device-wide rings (atomics, fences, L1-bypassing loads of a 2.4 KB state block that does not fit the L2 for 65 536
// streams) -- and a general tick cost 3.3 x a hold tick (1535 vs 468 cycles per warp pair): ten branch points per tick,
// event code in the loop, the frame manager's loads on the critical path.
//
// Here a stream belongs to ONE thread block for the whole call (block b owns streams b, b + grid, b + 2 grid, ...), one
// block of 16 warps = 8 workers per SM:
//   * its state lives in a dense array of 560-byte StreamStateLite records (35 MB for 65 536 streams: L2-resident; only the
//     owning SM ever touches a record, so plain cached loads are coherent and a fence.cta orders a hand-over).  A worker
//     copies the 32 records of a cell into shared memory with coalesced 16-byte accesses, the render loops load and store
//     their state THERE, and the records go back the same way (the first version let every lane read its own record word
//     by word: 260 requests x 32 sectors per cell saturated the L1 and made a hold tick 2.4 x slower than under the ring
//     scheduler);
//   * the block sorts its own streams: three queues in shared memory (hold / fade / general), one spin lock, no global
//     atomics, no device-wide fences; a worker pops up to 32 streams of the fullest class, renders ONE CELL of them and
//     pushes them back under the class their state now shows;
//   * cells are short because changing loops is cheap: the hold loop takes 128 pure hold ticks, the new straight-line FADE
//     loop (renderFadeF32T: pole recurrences, coefficients, DSP, no frame manager, no branch) takes 64 interior fade ticks on
//     the 64-sample grid of the drift control, and the general loop -- the only one with the event code -- takes what is left:
//     the 64-sample cells that contain a pop, a landing or a swap, 7-8 % of the ticks of config 3 instead of 61 %.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include "klatt_common.h"
#include "klatt_f32_core.cuh"
#include "out_writer.cuh"
#include "klatt_f32_pair.cuh"
#include "launch.h"

namespace klatt {

constexpr int kBlkThreads = 512, kBlkWorkers = kBlkThreads / 64;
constexpr uint32_t kClsHold = 0, kClsFade = 1, kClsGen = 2, kClsDone = 3, kClsExit = 4;
constexpr uint32_t kCellTicks = kCoarseTicks;  // fade and general cells
constexpr uint32_t kNoStream = 0xffffu;
constexpr uint32_t kRecBytes = sizeof(StreamStateLite), kRecPieces = kRecBytes / 16;  // 560 B = 35 pieces of 16 bytes
constexpr uint32_t kStageStride = kRecBytes + 8;  // bytes between the staged records of neighbouring lanes: 142 words, 2-way conflicts at most
constexpr uint32_t kStageBytes = 32 * kStageStride;  // per worker

struct BlockCtl {
	uint32_t lock;
	uint32_t head[3], count[3];
	uint32_t live;                      // owned streams that still have ticks to render in this call
	uint32_t active[3];                 // workers currently rendering a cell of each class
	uint32_t work[kBlkWorkers][36];     // per worker: 32 local stream indices, class
};

namespace {

__device__ __forceinline__ uint32_t classifyLite(const StreamStateLite &st, uint32_t sampleCount, uint32_t holdTicks) {
	const uint32_t pos = st.f32.callPos;
	if (pos >= sampleCount || st.f32.callDrained != 0) return kClsDone;
	const uint32_t left = sampleCount - pos;
	if (left >= holdTicks && canHoldF32T(st.fm, st.f32, holdTicks)) return kClsHold;
	if (left >= kCellTicks && canFadeF32T(st.fm, st.f32, kCellTicks)) return kClsFade;
	return kClsGen;
}

__device__ __forceinline__ void lockCtl(BlockCtl *ctl) {
	while (atomicCAS(&ctl->lock, 0u, 1u) != 0u) __nanosleep(32);
	__threadfence_block();
}
__device__ __forceinline__ void unlockCtl(BlockCtl *ctl) {
	__threadfence_block();
	atomicExch(&ctl->lock, 0u);
}

// hand-over between the two warps of a worker (klatt_f32_pair.cuh XchgSmem with eight named barriers)
struct XchgBlk {
	uint32_t base;
	uint32_t barId;  // 1..8
	__device__ __forceinline__ void put(uint32_t t, uint32_t wA, float par, float voice) {
		asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %3};" ::"r"(base + (t & 15u) * 512u), "r"(wA), "r"(__float_as_uint(par)),
		             "r"(__float_as_uint(voice)) : "memory");
	}
	__device__ __forceinline__ void get(uint32_t t, uint32_t &wA, float &par, float &voice) const {
		uint32_t p, v, pad;
		asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(wA), "=r"(p), "=r"(v), "=r"(pad) : "r"(base + (t & 15u) * 512u) : "memory");
		par = __uint_as_float(p);
		voice = __uint_as_float(v);
	}
	__device__ __forceinline__ void sync() {  // immediate ids (a register operand makes ptxas reserve all 16 barriers)
		switch (barId) {
			case 1: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
			case 2: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
			case 3: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
			case 4: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
			case 5: asm volatile("bar.sync 5, 64;" ::: "memory"); break;
			case 6: asm volatile("bar.sync 6, 64;" ::: "memory"); break;
			case 7: asm volatile("bar.sync 7, 64;" ::: "memory"); break;
			default: asm volatile("bar.sync 8, 64;" ::: "memory"); break;
		}
	}
};

}  // namespace

// start of a call: the compact copies of every stream's state (and fresh dummy streams for the idle lanes of each worker)
__global__ void __launch_bounds__(256)
klatt_block_import_kernel(const StreamDesc *__restrict__ descs, uint32_t numStreams, uint32_t numDummies, StreamStateLite *__restrict__ lite) {
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= numStreams + numDummies) return;
	StreamStateLite L;
	memset(&L, 0, sizeof L);
	if (s < numStreams) {
		const StreamState *st = descs[s].state;
		const FrameMgrState &fm = st->fm;
		const GenStateF32 &gs = st->gen.f32;
		L.fm.lastUserIndex = fm.lastUserIndex; L.fm.qHead = fm.qHead; L.fm.counter = fm.counter;
		L.fm.hasNew = fm.hasNew; L.fm.curIsNull = fm.curIsNull; L.fm.oldIsNull = fm.oldIsNull; L.fm.newIsNull = fm.newIsNull;
		L.fm.oldM = fm.oldM; L.fm.newM = fm.newM; L.fm.newF = fm.newF; L.fm.purgePending = fm.purgePending;
		L.fm.oldInc = fm.oldInc; L.fm.newInc = fm.newInc;
		L.f32.pitchPos = gs.pitchPos; L.f32.pitch = gs.pitch; L.f32.pitchInc = gs.pitchInc; L.f32.pitchOld = gs.pitchOld; L.f32.pitchNew = gs.pitchNew;
		L.f32.samplesGenerated = gs.samplesGenerated; L.f32.vibratoPos = gs.vibratoPos; L.f32.vibInc = gs.vibInc;
		L.f32.aspLast = gs.aspLast; L.f32.fricLast = gs.fricLast; L.f32.n0Inv = gs.n0Inv; L.f32.holdArmed = gs.holdArmed;
		L.f32.nextEvent = gs.nextEvent; L.f32.coarseAt = gs.coarseAt;
		L.f32.callPos = 0; L.f32.callDrained = 0;
		for (int r = 0; r < kNumResonators; ++r) { L.f32.y[r] = gs.y[r]; L.f32.d[r] = gs.d[r]; L.f32.zre[r] = gs.zre[r]; L.f32.zim[r] = gs.zim[r]; }
		for (int i = 0; i < kNumDirect; ++i) L.f32.dir[i] = gs.dir[i];
		for (int i = 0; i < 2 * kNumResonators; ++i) L.f32.zc[i] = gs.zc[i];
		L.f32.depth = gs.depth;
	} else {  // init_states_kernel's fresh player (host.cu)
		L.fm.lastUserIndex = -1; L.fm.curIsNull = 1; L.fm.oldIsNull = 1;
	}
	lite[s] = L;
}

// end of a call: back into the full state blocks, and the per-stream results
__global__ void __launch_bounds__(256)
klatt_block_export_kernel(const StreamDesc *__restrict__ descs, uint32_t numStreams, const StreamStateLite *__restrict__ lite,
                          uint32_t *__restrict__ samplesWritten, StreamResult *__restrict__ results) {
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= numStreams) return;
	const StreamStateLite L = lite[s];
	StreamState *st = descs[s].state;
	FrameMgrState &fm = st->fm;
	GenStateF32 &gs = st->gen.f32;
	fm.lastUserIndex = L.fm.lastUserIndex; fm.qHead = L.fm.qHead; fm.counter = L.fm.counter;
	fm.hasNew = L.fm.hasNew; fm.curIsNull = L.fm.curIsNull; fm.oldIsNull = L.fm.oldIsNull; fm.newIsNull = L.fm.newIsNull;
	fm.oldM = L.fm.oldM; fm.newM = L.fm.newM; fm.newF = L.fm.newF; fm.purgePending = L.fm.purgePending;
	fm.oldInc = L.fm.oldInc; fm.newInc = L.fm.newInc;
	gs.pitchPos = L.f32.pitchPos; gs.pitch = L.f32.pitch; gs.pitchInc = L.f32.pitchInc; gs.pitchOld = L.f32.pitchOld; gs.pitchNew = L.f32.pitchNew;
	gs.samplesGenerated = L.f32.samplesGenerated; gs.vibratoPos = L.f32.vibratoPos; gs.vibInc = L.f32.vibInc;
	gs.aspLast = L.f32.aspLast; gs.fricLast = L.f32.fricLast; gs.n0Inv = L.f32.n0Inv; gs.holdArmed = L.f32.holdArmed;
	gs.nextEvent = L.f32.nextEvent; gs.coarseAt = L.f32.coarseAt; gs.callPos = L.f32.callPos; gs.callDrained = L.f32.callDrained;
	for (int r = 0; r < kNumResonators; ++r) { gs.y[r] = L.f32.y[r]; gs.d[r] = L.f32.d[r]; gs.zre[r] = L.f32.zre[r]; gs.zim[r] = L.f32.zim[r]; }
	for (int i = 0; i < kNumDirect; ++i) gs.dir[i] = L.f32.dir[i];
	for (int i = 0; i < 2 * kNumResonators; ++i) gs.zc[i] = L.f32.zc[i];
	gs.depth = L.f32.depth;
	if (samplesWritten) samplesWritten[s] = L.f32.callPos;
	if (results) {
		StreamResult res;
		res.written = L.f32.callPos; res.lastUserIndex = L.fm.lastUserIndex; res.qHead = L.fm.qHead; res.pad = 0;
		results[s] = res;
	}
}

// the two conversions as launchers (the ring scheduler's compact-state mode uses them too, klatt_f32_sched.cu)
cudaError_t launchKlattLiteImport(const StreamDesc *descs, uint32_t numStreams, uint32_t numDummies, void *lite, cudaStream_t stream) {
	klatt_block_import_kernel<<<(numStreams + numDummies + 255) / 256, 256, 0, stream>>>(descs, numStreams, numDummies, static_cast<StreamStateLite *>(lite));
	return cudaGetLastError();
}
cudaError_t launchKlattLiteExport(const StreamDesc *descs, uint32_t numStreams, const void *lite, uint32_t *samplesWritten, StreamResult *results,
                                  cudaStream_t stream) {
	klatt_block_export_kernel<<<(numStreams + 255) / 256, 256, 0, stream>>>(descs, numStreams, static_cast<const StreamStateLite *>(lite), samplesWritten, results);
	return cudaGetLastError();
}

#ifdef KLATT_BLOCK_PROFILE
#define BPROF_LAP(acc) { long long t1 = clock64(); acc += t1 - t0; t0 = t1; }
#else
#define BPROF_LAP(acc)
#endif

// dynamic shared memory: [hand-over buffers: 8 workers x 8 KB][staged records: 8 workers x 32 x 552 B][BlockCtl][ring[3][cap] of
// uint16 local stream indices]
__global__ void __launch_bounds__(kBlkThreads, 1)
klatt_f32_block_kernel(const StreamDesc *__restrict__ descs, StreamStateLite *__restrict__ lite, uint32_t numStreams, int sampleRate,
                       uint32_t sampleCount, uint32_t holdTicks, int16_t *__restrict__ out, size_t rowStride,
                       int16_t *__restrict__ scratchRow, NoiseConfig noise, uint32_t cap, uint32_t maxClasses,
                       unsigned long long *__restrict__ prof, uint32_t *__restrict__ fault) {
	extern __shared__ uint4 smem[];
	uint4 *xbuf = smem;
	unsigned char *stageAll = reinterpret_cast<unsigned char *>(smem + kBlkWorkers * 2 * kGroupTicks * 32);
	BlockCtl *ctl = reinterpret_cast<BlockCtl *>(stageAll + kBlkWorkers * kStageBytes);
	uint16_t *ring = reinterpret_cast<uint16_t *>(ctl + 1);
	const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
	const uint32_t worker = warp >> 1;
	// two warps of a worker sit on neighbouring schedulers; the side each runs alternates so that every scheduler of the SM
	// gets two cascade and two parallel warps
	const bool cascade = ((warp & 1u) == 0u) != (((worker >> 1) & 1u) != 0u);
	const uint32_t mask = cap - 1u;
	const uint32_t owned = blockIdx.x < numStreams ? (numStreams - blockIdx.x + gridDim.x - 1u) / gridDim.x : 0u;

	if (tid == 0) {
		ctl->lock = 0;
		for (int c = 0; c < 3; ++c) { ctl->head[c] = 0; ctl->count[c] = 0; ctl->active[c] = 0; }
		ctl->live = 0;
	}
	__syncthreads();
	for (uint32_t l = tid; l < owned; l += kBlkThreads) {
		const uint32_t cls = classifyLite(lite[blockIdx.x + l * gridDim.x], sampleCount, holdTicks);
		if (cls < kClsDone) {
			const uint32_t idx = atomicAdd(&ctl->count[cls], 1u);
			ring[cls * cap + (idx & mask)] = (uint16_t)l;
			atomicAdd(&ctl->live, 1u);
		}
	}
	__syncthreads();

	XchgBlk xc{(uint32_t)__cvta_generic_to_shared(&xbuf[worker * 2 * kGroupTicks * 32 + lane]), 1u + worker};
	uint32_t *work = ctl->work[worker];
	StreamStateLite *dummy = lite + numStreams + (size_t)blockIdx.x * kBlkWorkers + worker;
	unsigned char *stage = stageAll + worker * kStageBytes;
	StreamStateLite *st = reinterpret_cast<StreamStateLite *>(stage + lane * kStageStride);  // this lane's stream while a cell runs
	const uint32_t tw = tid & 63u;  // thread of the worker
#ifdef KLATT_BLOCK_PROFILE
	long long tClaim = 0, tCls[3] = {0, 0, 0}, tPush = 0, nCls[3] = {0, 0, 0}, nLanes = 0;
	long long t0 = clock64();
#endif
	for (;;) {
		if (cascade) {
			uint32_t cls = kClsExit, n = 0, base = 0;
			if (lane == 0) {
				uint32_t idleSpins = 0;
				unsigned long long idleSince = 0;
				for (;;) {
					lockCtl(ctl);
					const uint32_t c0 = ctl->count[0], c1 = ctl->count[1], c2 = ctl->count[2];
					// Which class: at most `maxClasses` different classes are in flight on this SM at any time -- every class is two
					// loops (cascade / parallel side), the SM's instruction cache holds 32 KB, and all six loops together are
					// 36 KB (measured with no limit: 6.9 stall cycles per issue waiting for instructions).  Among the classes that
					// are allowed: a full warp of the RAREST class first (general, then fade, then hold: a stream that waits for 31
					// others of its kind must not also wait behind the majority), else a partial warp of the fullest one.
					const uint32_t a0 = ctl->active[0], a1 = ctl->active[1], a2 = ctl->active[2];
					const uint32_t distinct = (a0 != 0u) + (a1 != 0u) + (a2 != 0u);
					const bool ok0 = a0 != 0u || distinct < maxClasses, ok1 = a1 != 0u || distinct < maxClasses,
					           ok2 = a2 != 0u || distinct < maxClasses;
					const uint32_t e0 = ok0 ? c0 : 0u, e1 = ok1 ? c1 : 0u, e2 = ok2 ? c2 : 0u;
					uint32_t pick;
					if (e2 >= 32u) pick = 2u;
					else if (e1 >= 32u) pick = 1u;
					else if (e0 >= 32u) pick = 0u;
					else pick = (e2 >= e1 && e2 >= e0) ? 2u : (e1 >= e0 ? 1u : 0u);
					if ((pick == 2u ? e2 : (pick == 1u ? e1 : e0)) == 0u) {  // nothing this worker may take right now
						const uint32_t live = ctl->live;
						unlockCtl(ctl);
						if (live == 0u) break;
						__nanosleep(256);
						if ((++idleSpins & 4095u) == 0u) {
							unsigned long long now;
							asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
							if (idleSince == 0) idleSince = now;
							if (now - idleSince > 10ull * 1000 * 1000 * 1000) {
								if (fault) *fault = 1u;
								lockCtl(ctl);
								ctl->live = 0u;
								unlockCtl(ctl);
								break;
							}
						}
						continue;
					}
					const uint32_t have = pick == 2u ? c2 : (pick == 1u ? c1 : c0);
					n = have < 32u ? have : 32u;
					base = ctl->head[pick];
					ctl->head[pick] = base + n;
					ctl->count[pick] = have - n;
					ctl->active[pick] += 1u;
					cls = pick;
					unlockCtl(ctl);
					break;
				}
			}
			cls = __shfl_sync(0xffffffffu, cls, 0);
			n = __shfl_sync(0xffffffffu, n, 0);
			base = __shfl_sync(0xffffffffu, base, 0);
			uint32_t l = kNoStream;
			if (cls < kClsDone && lane < n) l = ring[cls * cap + ((base + lane) & mask)];
			work[lane] = l;
			if (lane == 0) work[32] = cls;
		}
		xc.sync();
		const uint32_t l = work[lane], cls = work[32];
		BPROF_LAP(tClaim)
		if (cls == kClsExit) break;
		const bool valid = l != kNoStream;
		const uint32_t s = valid ? blockIdx.x + l * gridDim.x : numStreams;
		const StreamDesc &desc = descs[s];
		// ---- the records of this cell: global -> shared, both warps, 16 bytes per thread and step, consecutive pieces of a record
		// on consecutive threads (idle lanes get the worker's dummy stream) ----
#pragma unroll 1
		for (uint32_t idx = tw; idx < 32u * kRecPieces; idx += 64u) {
			const uint32_t r = idx / kRecPieces, p = idx - r * kRecPieces;
			const uint32_t lr = work[r];
			const StreamStateLite *src = lr != kNoStream ? lite + (blockIdx.x + lr * gridDim.x) : dummy;
			const uint4 v = reinterpret_cast<const uint4 *>(src)[p];
			uint2 *dst = reinterpret_cast<uint2 *>(stage + r * kStageStride + p * 16u);
			dst[0] = make_uint2(v.x, v.y);
			dst[1] = make_uint2(v.z, v.w);
		}
		xc.sync();
		if (cls == kClsHold) {
			if (cascade) {
				int16_t *row = valid ? out + (size_t)s * rowStride + st->f32.callPos : scratchRow;
				OutWriter ow;
				ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
				renderHoldF32T<kRoleCascadeOsc>(st->fm, st->f32, desc, sampleRate, holdTicks, ow, noise, xc);
			} else {
				NullOut no;
				renderHoldF32T<kRoleParallelOnly>(st->fm, st->f32, desc, sampleRate, holdTicks, no, noise, xc);
			}
		} else if (cls == kClsFade) {
			if (cascade) {
				int16_t *row = valid ? out + (size_t)s * rowStride + st->f32.callPos : scratchRow;
				OutWriter ow;
				ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
				renderFadeF32T<kRoleCascade>(st->fm, st->f32, desc, sampleRate, kCellTicks, ow, noise, xc);
			} else {
				NullOut no;
				renderFadeF32T<kRoleParallel>(st->fm, st->f32, desc, sampleRate, kCellTicks, no, noise, xc);
			}
		} else {
			// the general loop runs a stream up to the next point of the 64-sample grid (or to the end of the call)
			const uint32_t pos = st->f32.callPos;
			uint32_t ticks = 0;
			if (valid) {
				ticks = kCellTicks - (uint32_t)(st->f32.samplesGenerated & (uint64_t)(kCellTicks - 1));
				if (ticks > sampleCount - pos) ticks = sampleCount - pos;
			}
			int32_t lastUserIndex;
			uint32_t qHead;
			if (cascade) {
				int16_t *row = out + (size_t)(valid ? s : 0) * rowStride;
				OutWriter ow;
				ow.init(row + pos, ((reinterpret_cast<uintptr_t>(row + pos) & 15u) == 0));
				const uint32_t produced = renderGeneralF32T<kRoleCascade>(st->fm, st->f32, desc, sampleRate, ticks, kCellTicks, ow, noise, xc,
				                                                           &lastUserIndex, &qHead);
				ow.flush();
				if (produced < ticks) zeroRow(row, pos + produced, sampleCount);  // drained: the rest of the row is silence
			} else {
				NullOut no;
				renderGeneralF32T<kRoleParallel>(st->fm, st->f32, desc, sampleRate, ticks, kCellTicks, no, noise, xc, &lastUserIndex, &qHead);
			}
		}
		xc.sync();  // both halves of every stream of this cell are in the staged records
		uint32_t next = kClsExit;
		if (cascade && valid) next = classifyLite(*st, sampleCount, holdTicks);
		// ---- shared -> global (the idle lanes' dummy is not written back) ----
#pragma unroll 1
		for (uint32_t idx = tw; idx < 32u * kRecPieces; idx += 64u) {
			const uint32_t r = idx / kRecPieces, p = idx - r * kRecPieces;
			const uint32_t lr = work[r];
			if (lr != kNoStream) {
				const uint2 *src = reinterpret_cast<const uint2 *>(stage + r * kStageStride + p * 16u);
				const uint2 a = src[0], b = src[1];
				reinterpret_cast<uint4 *>(lite + (blockIdx.x + lr * gridDim.x))[p] = make_uint4(a.x, a.y, b.x, b.y);
			}
		}
		__threadfence_block();
		xc.sync();  // the records are back in the array: the streams may be handed on
#ifdef KLATT_BLOCK_PROFILE
		BPROF_LAP(tCls[cls])
		nCls[cls]++;
		nLanes += __popc(__ballot_sync(0xffffffffu, valid));
#endif
		if (cascade) {
			const unsigned below = (1u << lane) - 1u;
			const unsigned m0 = __ballot_sync(0xffffffffu, next == kClsHold), m1 = __ballot_sync(0xffffffffu, next == kClsFade);
			const unsigned m2 = __ballot_sync(0xffffffffu, next == kClsGen), mD = __ballot_sync(0xffffffffu, next == kClsDone);
			if (lane == 0) lockCtl(ctl);
			__syncwarp();
			if (next < kClsDone) {
				const unsigned m = next == kClsHold ? m0 : (next == kClsFade ? m1 : m2);
				const uint32_t tail = ctl->head[next] + ctl->count[next];
				ring[next * cap + ((tail + __popc(m & below)) & mask)] = (uint16_t)l;
			}
			__syncwarp();
			if (lane == 0) {
				ctl->count[0] += __popc(m0); ctl->count[1] += __popc(m1); ctl->count[2] += __popc(m2);
				ctl->live -= __popc(mD);
				ctl->active[cls] -= 1u;
				unlockCtl(ctl);
			}
		}
		BPROF_LAP(tPush)
	}
#ifdef KLATT_BLOCK_PROFILE
	if (lane == 0 && prof) {
		unsigned long long *p = prof + (cascade ? 0 : 16);
		atomicAdd(p + 0, (unsigned long long)tClaim); atomicAdd(p + 1, (unsigned long long)tCls[0]);
		atomicAdd(p + 2, (unsigned long long)tCls[1]); atomicAdd(p + 3, (unsigned long long)tCls[2]);
		atomicAdd(p + 4, (unsigned long long)tPush); atomicAdd(p + 5, (unsigned long long)nCls[0]);
		atomicAdd(p + 6, (unsigned long long)nCls[1]); atomicAdd(p + 7, (unsigned long long)nCls[2]);
		atomicAdd(p + 8, (unsigned long long)nLanes);
	}
#endif
}

// bytes of dynamic shared memory for a block that owns up to `cap` streams
static size_t blockSmemBytes(uint32_t cap) {
	return sizeof(uint4) * kBlkWorkers * 2 * kGroupTicks * 32 + (size_t)kBlkWorkers * kStageBytes + sizeof(BlockCtl) +
	       sizeof(uint16_t) * 3 * (size_t)cap;
}

// the block scheduler can take a batch when every block's share fits the 16-bit local indices and the queues fit shared memory
bool klattF32BlockCanTake(uint32_t numStreams, uint32_t numBlocks) {
	if (numBlocks == 0) return false;
	const uint32_t owned = (numStreams + numBlocks - 1) / numBlocks;
	return owned <= 2048u;  // 3 queues of 16-bit indices next to 64 KB of hand-over buffers and 138 KB of staged records
}
size_t klattF32BlockLiteBytes(uint32_t numStreams, uint32_t numBlocks) {
	return sizeof(StreamStateLite) * ((size_t)numStreams + (size_t)numBlocks * kBlkWorkers);
}

// One call through the block scheduler: import, one persistent launch of numBlocks blocks (one per SM), export.
// lite: klattF32BlockLiteBytes() of scratch; descs holds numStreams + 1 entries (the last one the dummy stream's).
cudaError_t launchKlattF32Block(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount, uint32_t holdTicks,
                                int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise,
                                void *liteMem, int16_t *scratchRow, uint32_t numBlocks, void *profMem, uint32_t *hostFault,
                                cudaStream_t stream, unsigned long long *launchCounter) {
	if (numStreams == 0 || sampleCount == 0) return cudaSuccess;
	StreamStateLite *lite = static_cast<StreamStateLite *>(liteMem);
	const uint32_t owned = (numStreams + numBlocks - 1) / numBlocks;
	uint32_t cap = 64;
	while (cap < owned) cap <<= 1;
	const size_t smem = blockSmemBytes(cap);
	static size_t smemSet = 0;
	if (smem > smemSet) {
		cudaError_t e = cudaFuncSetAttribute(klatt_f32_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		if (e != cudaSuccess) return e;
		smemSet = smem;
	}
	const uint32_t numDummies = numBlocks * kBlkWorkers;
	static const uint32_t maxClasses = getenv("NVSP_BLOCK_MAX_CLASSES") ? (uint32_t)atoi(getenv("NVSP_BLOCK_MAX_CLASSES")) : 2u;
	klatt_block_import_kernel<<<(numStreams + numDummies + 255) / 256, 256, 0, stream>>>(descs, numStreams, numDummies, lite);
	klatt_f32_block_kernel<<<numBlocks, kBlkThreads, smem, stream>>>(descs, lite, numStreams, sampleRate, sampleCount, holdTicks, out, rowStride,
	                                                                 scratchRow, noise, cap, maxClasses, static_cast<unsigned long long *>(profMem),
	                                                                 reinterpret_cast<uint32_t *>(static_cast<unsigned long long *>(profMem) + 31));
	// the watchdog's verdict travels to a pinned host word; the engine reads it at its next synchronisation point
	if (hostFault) {
		cudaError_t e = cudaMemcpyAsync(hostFault, static_cast<unsigned long long *>(profMem) + 31, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
		if (e != cudaSuccess) return e;
	}
	klatt_block_export_kernel<<<(numStreams + 255) / 256, 256, 0, stream>>>(descs, numStreams, lite, samplesWritten, results);
	if (launchCounter) *launchCounter += 3;
#ifdef KLATT_BLOCK_PROFILE
	if (profMem) {
		unsigned long long h[32];
		cudaStreamSynchronize(stream);
		cudaMemcpy(h, profMem, sizeof h, cudaMemcpyDeviceToHost);
		cudaMemset(profMem, 0, sizeof h);
		for (int k = 0; k < 2; ++k) {
			const unsigned long long *p = h + 16 * k;
			fprintf(stderr, "[block profile] %s warps: claim %.1f  hold %.1f  fade %.1f  gen %.1f  push %.1f Mcycles; cells hold %llu fade %llu gen %llu; lanes/cell %.2f\n",
			        k ? "parallel" : "cascade ", p[0] / 1e6, p[1] / 1e6, p[2] / 1e6, p[3] / 1e6, p[4] / 1e6, p[5], p[6], p[7],
			        (double)p[8] / (double)(p[5] + p[6] + p[7] + 1));
		}
	}
#endif
	return cudaGetLastError();
}

}  // namespace klatt
