// The persistent stream scheduler of the FP32 batch path: the default for pre-queued batches (NVSP_SCHED=rounds selects
// the round-based launch sequence of klatt_f32.cu instead; DESIGN.md section 5b has the measurements of both).
// Same render bodies as the round kernels (klatt_f32_core.cuh), so the same bits.
//
// This translation unit is compiled with -fmad=false like klatt_f32.cu.  The kernel moves a stream's state between SMs
// without a kernel boundary in between: everything mutable travels in explicit L1-bypassing copies (KLATT_SCHED_LITE
// below; the round-1 layout, KLATT_SCHED_LITE=0, needs -Xptxas -dlcm=cg for the whole unit instead).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <stddef.h>
#include <string.h>
#include "klatt_common.h"
#include "klatt_f32_core.cuh"
#include "out_writer.cuh"
#include "klatt_f32_pair.cuh"
#include "launch.h"

// KLATT_SCHED_LITE (default 1, round 2): the streams of a call live in a dense array of 560-byte StreamStateLite records
// (klatt_common.h; 35 MB for 65 536 streams: L2-resident) instead of the 2.4 KB AoS blocks; a worker copies the 32 records of
// its chunk into shared memory with coalesced 16-byte ld.global.cg, the render loops load and store their state (and the
// drift-control record zc, every 64 fade ticks) THERE, and the records go back with st.global.cg before the fence and the
// push.  Everything mutable that crosses SMs moves through those explicit L1-bypassing copies, so the translation unit no
// longer needs -dlcm=cg: plans, queues and descriptors are read through the L1 like any read-only data.  After a hold chunk
// only the first 256 bytes of a record go back (the pole state, the direct parameters and zc do not move in a hold); the
// output leaves with st.global.cs (out_writer.cuh).  Measured (config 3): 222 -> 200.5 ms per step, DRAM traffic of a step
// 72.1 -> 59.7 GB (algorithmic: 36.6 GB; profiles/r02_sched_ncu_summary.txt, DESIGN.md section 5d, which also has the L2
// residency controls that were tried -- persisting window on the records, evict-last plan rows -- and why they are off).
#ifndef KLATT_SCHED_LITE
#define KLATT_SCHED_LITE 1
#endif

namespace klatt {

#ifdef KLATT_SCHED_PROFILE
#define PROF_LAP(acc) { long long t1 = clock64(); acc += t1 - t0; t0 = t1; }
#else
#define PROF_LAP(acc)
#endif

// ---------------------------------------------------------------------------------------------------
// The stream scheduler: ONE persistent launch renders the whole call.
//
// The rounds above re-sort the streams with a kernel boundary per round: every round ends with a tail (the last blocks
// of the slower kernel run on an emptying GPU), the two kernels of a round are only balanced on average, and a call is
// ~10^4 launches.  Here the sorting is done by the render warps themselves.  Two device-side rings hold the streams that
// are ready for a pure-hold chunk (class 0) or need the frame manager (class 1).  A WORKER is a cascade/parallel warp
// pair; it claims up to 32 streams of one class, renders one chunk of them (the same renderHoldF32 / renderGeneralF32
// as the round kernels: same arithmetic, same bits), classifies each stream's next chunk and pushes it back, until no
// stream of the call has ticks left.  Nothing waits on another worker except through the rings, so the kernel is
// correct for any number of resident blocks; the grid is sized to fill the GPU once.
//
//   ring[c][i & mask] : stream index, kRingEmpty or kRingAbandoned.  Both cursors of a ring only ever move by atomicAdd
//                       (a claim by compare-and-swap collapses when ~10^3 workers arrive within one L2 round trip of
//                       each other: measured 10x slower than the rounds).  Producers reserve [tail, tail+n) and write
//                       their slots; a consumer takes a TICKET [head, head+32) -- possibly ahead of the tail -- and
//                       each of its lanes waits for its own slot to be written, which future pushes do in ticket
//                       order.  A lane that has waited too long abandons its slot (EMPTY -> ABANDONED by CAS; if the
//                       CAS finds a stream, it takes it): the warp then runs with the lanes it has, or picks a ring
//                       again if it has none.  A producer that finds its reserved slot abandoned restores it to
//                       EMPTY and pushes again with a new reservation.  A stream is in at most one ring and tickets
//                       run at most one batch per worker ahead, so a ring of >= 2 x numStreams slots (and far more
//                       than 32 x workers) cannot wrap onto a live entry.
//   state hand-over   : both warps of the pair store their half of the stream state, fence, meet at the pair's
//                       barrier; then the cascade warp pushes.  The consumer fences after taking the slot.  This
//                       translation unit is compiled with -dlcm=cg: global loads bypass L1, so a stream that comes
//                       back to an SM it visited before cannot see a stale line.
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t kRingEmpty = 0xffffffffu, kRingAbandoned = 0xfffffffeu;
constexpr uint32_t kClassHold = 0, kClassGen = 1, kClassFade = 2, kClassExit = 3, kNumRings = 3;
// kClassFade (round 2, on when fadeTicks != 0): streams with fadeTicks INTERIOR fade ticks ahead, starting on the 64-sample
// grid of the drift control: renderFadeF32T's straight-line loop (pole recurrences, coefficients, DSP; no frame manager, no
// branch) renders them; the general loop keeps the ticks around pops, landings and swaps.

struct SchedCtl {  // every hot word on its own 128-byte line
	uint32_t head0, padA[31];
	uint32_t head1, padB[31];
	uint32_t tail0, padC[31];
	uint32_t tail1, padD[31];
	uint32_t remaining, padE[31];  // streams of this call that still have ticks to render
	uint32_t fault, padF[31];      // set by the watchdog: a worker waited kWatchdogNs for work that never came
	uint32_t head2, padG[31];
	uint32_t tail2, padH[31];
	__device__ __forceinline__ uint32_t *head(uint32_t c) { return c == 0 ? &head0 : c == 1 ? &head1 : &head2; }
	__device__ __forceinline__ uint32_t *tail(uint32_t c) { return c == 0 ? &tail0 : c == 1 ? &tail1 : &tail2; }
};

// A worker that has found both rings empty with streams still unaccounted for, for this long, declares the call
// failed: it zeroes `remaining` (every worker then leaves at its next look) and raises `fault`, which the host turns
// into an error.  It cannot fire on a correct run: a chunk takes well under a millisecond.
constexpr unsigned long long kWatchdogNs = 20ull * 1000 * 1000 * 1000;

namespace {

__device__ __forceinline__ unsigned long long globalTimerNs() {
	unsigned long long t;
	asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
	return t;
}

__device__ __forceinline__ uint32_t ldVolatile(const uint32_t *p) { return *reinterpret_cast<const volatile uint32_t *>(p); }
__device__ __forceinline__ void stVolatile(uint32_t *p, uint32_t v) { *reinterpret_cast<volatile uint32_t *>(p) = v; }

// class of a stream's next chunk, or kClassExit when the call is complete for it
template <class FM, class GS>
__device__ __forceinline__ uint32_t classifyNextT(const FM &fm, const GS &gs, uint32_t sampleCount, uint32_t holdTicks, uint32_t fadeTicks) {
	const uint32_t pos = gs.callPos;
	if (pos >= sampleCount || gs.callDrained != 0) return kClassExit;
	if (sampleCount - pos >= holdTicks && canHoldF32T(fm, gs, holdTicks)) return kClassHold;
	if (fadeTicks != 0u && sampleCount - pos >= fadeTicks && canFadeF32T(fm, gs, fadeTicks)) return kClassFade;
	return kClassGen;
}
__device__ __forceinline__ uint32_t classifyNext(const StreamState *st, uint32_t sampleCount, uint32_t holdTicks) {
	return classifyNextT(st->fm, st->gen.f32, sampleCount, holdTicks, 0u);
}
constexpr uint32_t kRecPieces = sizeof(StreamStateLite) / 16, kStageStride = sizeof(StreamStateLite) + 8, kStageBytes = 32 * kStageStride;
constexpr uint32_t kHoldPiecesOut = (uint32_t)(offsetof(StreamStateLite, f32) + offsetof(GenStateF32Lite, zre)) / 16;  // everything before the pole state
static_assert((offsetof(StreamStateLite, f32) + offsetof(GenStateF32Lite, zre)) % 16 == 0, "the hold chunk's write-back ends on a 16-byte piece");

// every lane of the calling warp: push stream s into ring cls (cls == kClassExit: nothing to push, the stream is done)
template <bool SEED>
__device__ __forceinline__ void schedPush(SchedCtl *ctl, uint32_t *ring, uint32_t ringCap, uint32_t cls, uint32_t s, bool valid) {
	const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
	const unsigned mH = __ballot_sync(0xffffffffu, valid && cls == kClassHold);
	const unsigned mG = __ballot_sync(0xffffffffu, valid && cls == kClassGen);
	const unsigned mF = __ballot_sync(0xffffffffu, valid && cls == kClassFade);
	const unsigned mX = __ballot_sync(0xffffffffu, valid && cls == kClassExit);
	uint32_t baseH = 0, baseG = 0, baseF = 0;
	if (lane == 0) {
		if (mH) baseH = atomicAdd(ctl->tail(kClassHold), (uint32_t)__popc(mH));
		if (mG) baseG = atomicAdd(ctl->tail(kClassGen), (uint32_t)__popc(mG));
		if (mF) baseF = atomicAdd(ctl->tail(kClassFade), (uint32_t)__popc(mF));
	}
	baseH = __shfl_sync(0xffffffffu, baseH, 0);
	baseG = __shfl_sync(0xffffffffu, baseG, 0);
	baseF = __shfl_sync(0xffffffffu, baseF, 0);
	const uint32_t mask = ringCap - 1u;
	if (valid && cls != kClassExit) {
		uint32_t *r = ring + cls * ringCap;
		uint32_t idx = cls == kClassHold ? baseH + __popc(mH & below) : cls == kClassGen ? baseG + __popc(mG & below) : baseF + __popc(mF & below);
		if (SEED) {
			stVolatile(r + (idx & mask), s);  // nobody holds a ticket yet
		} else {
			while (atomicCAS(r + (idx & mask), kRingEmpty, s) != kRingEmpty) {  // the ticket of this slot was abandoned
				stVolatile(r + (idx & mask), kRingEmpty);
				idx = atomicAdd(ctl->tail(cls), 1u);
			}
		}
	}
	if (SEED) {  // the seed kernel counts the streams in; the workers count them out
		if (lane == 0 && (mH | mG | mF)) atomicAdd(&ctl->remaining, (uint32_t)__popc(mH | mG | mF));
	} else {
		if (lane == 0 && mX) atomicSub(&ctl->remaining, (uint32_t)__popc(mX));
	}
}

// All 32 lanes of a worker's cascade warp: take a ticket of 32 slots in the ring with the most work waiting (a general or
// a fade chunk costs about as much as two hold chunks) and collect the streams.  Returns the class, or kClassExit when the
// call is complete; s = the lane's stream, or kRingEmpty for a lane that got none.
// Tickets are only taken from a ring that shows a backlog, so consumers run ahead of the producers by at most the
// workers that raced for the same entries; those wait for the next pushes.
// primary: the class this SM's workers take whenever its ring can fill a warp (SM roles with the fade class on: an SM then
// runs ONE loop pair most of the time, which is what its 32 KB instruction cache holds); other rings only when the primary
// one cannot fill a warp and another can, or is empty.  kClassExit = no role.
__device__ __forceinline__ uint32_t schedClaim(SchedCtl *ctl, uint32_t *ring, uint32_t ringCap, uint32_t &s, uint32_t primary) {
	const unsigned lane = threadIdx.x & 31u;
	const uint32_t mask = ringCap - 1u;
	for (;;) {
		uint32_t cls = kClassExit, base = 0;
		if (lane == 0) {
			uint32_t backoff = 128;
			unsigned long long idleSince = 0;
			for (;;) {
				int32_t b0 = (int32_t)(ldVolatile(&ctl->tail0) - ldVolatile(&ctl->head0));
				int32_t b1 = (int32_t)(ldVolatile(&ctl->tail1) - ldVolatile(&ctl->head1));
				int32_t b2 = (int32_t)(ldVolatile(&ctl->tail2) - ldVolatile(&ctl->head2));
				if (b0 > 0 || b1 > 0 || b2 > 0) {
					// most work waiting (general wins a tie with hold, as before); a full warp beats the weights
					uint32_t pick = kClassGen;
					int32_t best = -1;
					bool bestFull = false;
					auto consider = [&](uint32_t c, int32_t backlog, int32_t score) {
						if (backlog <= 0) return;
						const bool full = backlog >= 32;
						if (best < 0 || (full && !bestFull) || (full == bestFull && score > best)) { pick = c; best = score; bestFull = full; }
					};
					consider(kClassGen, b1, 2 * b1);
					consider(kClassFade, b2, 2 * b2);
					consider(kClassHold, b0, b0);
					if (primary < kNumRings) {
						const int32_t bp = primary == kClassHold ? b0 : primary == kClassGen ? b1 : b2;
						if (bp >= 32 || (bp > 0 && !bestFull)) pick = primary;
					}
					cls = pick;
					base = atomicAdd(ctl->head(cls), 32u);
					break;
				}
				if (ldVolatile(&ctl->remaining) == 0u) break;
				__nanosleep(backoff);
				if (backoff < 4096u) {
					backoff *= 2u;
				} else {  // idle at full back-off: watchdog
					const unsigned long long now = globalTimerNs();
					if (idleSince == 0) idleSince = now;
					else if (now - idleSince > kWatchdogNs) {
						stVolatile(&ctl->fault, 1u);
						stVolatile(&ctl->remaining, 0u);
					}
				}
			}
		}
		cls = __shfl_sync(0xffffffffu, cls, 0);
		base = __shfl_sync(0xffffffffu, base, 0);
		if (cls == kClassExit) return kClassExit;
		uint32_t *slot = ring + cls * ringCap + ((base + lane) & mask);
		s = kRingEmpty;
		bool abandoned = false;
		for (uint32_t spins = 0;; ++spins) {
			if (s == kRingEmpty && !abandoned) {
				const uint32_t v = ldVolatile(slot);
				if (v < kRingAbandoned) { s = v; stVolatile(slot, kRingEmpty); }
			}
			const unsigned got = __ballot_sync(0xffffffffu, s != kRingEmpty);
			const unsigned open = __ballot_sync(0xffffffffu, s == kRingEmpty && !abandoned);
			if (open == 0u) {
				if (got) return cls;
				break;  // nothing came: pick a ring again (or find the call complete)
			}
			// Give up on the missing lanes: after ~10 us with streams in hand (they should not wait for stragglers); with
			// none in hand only when the call is over or the other ring has a full warp waiting.
			uint32_t quit = 0;
			if (lane == 0) {
				if (got) quit = spins >= 64u;
				else if ((spins & 15u) == 15u)
				{
					quit = ldVolatile(&ctl->remaining) == 0u;
					for (uint32_t c = 0; c < kNumRings; ++c)
						if (c != cls && (int32_t)(ldVolatile(ctl->tail(c)) - ldVolatile(ctl->head(c))) >= 32) quit = 1u;
				}
			}
			quit = __shfl_sync(0xffffffffu, quit, 0);
			if (quit) {
				if (s == kRingEmpty && !abandoned) {
					const uint32_t v = atomicCAS(slot, kRingEmpty, kRingAbandoned);
					if (v < kRingAbandoned) { s = v; stVolatile(slot, kRingEmpty); }
					else abandoned = true;
				}
			} else {
				__nanosleep(160);
			}
		}
	}
}

}  // namespace

// start of a call: reset the per-call cursors of every stream and seed the rings
__global__ void __launch_bounds__(256)
klatt_sched_seed_kernel(const StreamDesc *__restrict__ descs, const StreamStateLite *__restrict__ lite, uint32_t numStreams,
                        uint32_t sampleCount, uint32_t holdTicks, uint32_t fadeTicks, SchedCtl *ctl, uint32_t *ring, uint32_t ringCap) {
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	const bool valid = s < numStreams;
	uint32_t cls = kClassExit;
	if (valid) {
		if (lite) {  // (the import kernel has reset the per-call cursors)
			cls = classifyNextT(lite[s].fm, lite[s].f32, sampleCount, holdTicks, fadeTicks);
		} else {
			StreamState *st = descs[s].state;
			st->gen.f32.callPos = 0;
			st->gen.f32.callDrained = 0;
			cls = classifyNext(st, sampleCount, holdTicks);
		}
	}
	schedPush<true>(ctl, ring, ringCap, cls, s, valid);
}

#ifndef KLATT_SCHED_MINB
#define KLATT_SCHED_MINB 4
#endif
__global__ void __launch_bounds__(kPairBlock, KLATT_SCHED_MINB)
klatt_f32_sched_kernel(const StreamDesc *__restrict__ descs, StreamStateLite *__restrict__ lite, uint32_t numStreams, int sampleRate,
                       uint32_t sampleCount, uint32_t holdTicks, uint32_t genTicks, int16_t *__restrict__ out, size_t rowStride,
                       int16_t *__restrict__ scratchRow, NoiseConfig noise, SchedCtl *ctl, uint32_t *ring, uint32_t ringCap,
                       uint32_t roleSms, uint32_t holdMax, uint32_t fadeTicks, uint32_t fadeMax) {
	// dynamic shared memory: [hand-over buffers: 2 workers x 8 KB][staged records: 2 workers x 32 x 552 B (KLATT_SCHED_LITE)]
	extern __shared__ uint4 schedSmem[];
	uint4 (*xbuf)[2 * kGroupTicks * 32] = reinterpret_cast<uint4 (*)[2 * kGroupTicks * 32]>(schedSmem);
	__shared__ uint32_t work[2][34];  // per worker: 32 stream indices, class
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, pair = warp & 1u;
	const bool cascade = cascadeRole(warp);
	XchgSmem xc{(uint32_t)__cvta_generic_to_shared(&xbuf[pair][lane]), 1u + pair};
#if KLATT_SCHED_LITE
	unsigned char *stage = reinterpret_cast<unsigned char *>(schedSmem + 2 * 2 * kGroupTicks * 32) + pair * kStageBytes;
	StreamStateLite *st = reinterpret_cast<StreamStateLite *>(stage + lane * kStageStride);  // this lane's stream while a chunk runs
	StreamStateLite *dummy = lite + numStreams + (size_t)blockIdx.x * 2 + pair;
	const uint32_t tw = (warp >> 1) * 32u + lane;  // thread of the worker
#endif
#ifdef KLATT_SCHED_PROFILE
	long long tClaim = 0, tHold = 0, tGen = 0, tFade = 0, tPush = 0, nHold = 0, nGen = 0, nLanes = 0;
	long long t0 = clock64();
#endif
	uint32_t primary = kClassExit;
	if (roleSms) {  // SM roles: (roleSms & 0xff) SMs take hold chunks first, (roleSms >> 8) SMs fade chunks, the rest general chunks; each kind spread evenly over the SM ids
		uint32_t smid, nsm;
		asm("mov.u32 %0, %%smid;" : "=r"(smid));
		asm("mov.u32 %0, %%nsmid;" : "=r"(nsm));
		const uint32_t nH = roleSms & 0xffu, nF = roleSms >> 8;
		if ((smid + 1) * nH / nsm != smid * nH / nsm) {
			primary = kClassHold;
		} else {
			const uint32_t j = smid - smid * nH / nsm, rest = nsm > nH ? nsm - nH : 1u;
			primary = ((j + 1) * nF / rest != j * nF / rest) ? kClassFade : kClassGen;
		}
	}
	for (;;) {
		if (cascade) {
			uint32_t s = kRingEmpty;
			const uint32_t cls = schedClaim(ctl, ring, ringCap, s, primary);
			if (s == kRingEmpty) s = numStreams;  // idle lanes run the dummy stream
			__threadfence();
			work[pair][lane] = s;
			if (lane == 0) work[pair][32] = cls;
		}
		xc.sync();
		const uint32_t s = work[pair][lane], cls = work[pair][32];
		PROF_LAP(tClaim)
		if (cls == kClassExit) break;
		const bool valid = s < numStreams;
		const StreamDesc &desc = descs[s];
#if KLATT_SCHED_LITE
		// the records of this chunk: global -> shared, both warps, 16 bytes per thread and step, L1 bypassed (the stream may have
		// been on another SM a moment ago)
#pragma unroll 1
		for (uint32_t idx = tw; idx < 32u * kRecPieces; idx += 64u) {
			const uint32_t r = idx / kRecPieces, p = idx - r * kRecPieces;
			const uint32_t sr = work[pair][r];
			const StreamStateLite *src = sr < numStreams ? lite + sr : dummy;
			const uint4 v = __ldcg(reinterpret_cast<const uint4 *>(src) + p);
			uint2 *dst = reinterpret_cast<uint2 *>(stage + r * kStageStride + p * 16u);
			dst[0] = make_uint2(v.x, v.y);
			dst[1] = make_uint2(v.z, v.w);
		}
		xc.sync();
		FrameMgrLite &fm = st->fm;
		GenStateF32Lite &gs = st->f32;
#else
		FrameMgrState &fm = desc.state->fm;
		GenStateF32 &gs = desc.state->gen.f32;
#endif
		if (cls == kClassHold) {
			// every stream here can hold for holdTicks (that is what put it into this ring); when ALL 32 can hold longer (steady
			// vowels, sung notes), run as far as the shortest of them allows, up to holdMax: fewer record round trips per tick.
			// Both warps of the pair compute this from the same staged records.
			uint32_t ticks = holdTicks;
#if KLATT_SCHED_LITE
			if (holdMax > holdTicks) {
				uint32_t can = 0xffffffffu;
				if (valid) {
					const uint32_t left = sampleCount - gs.callPos, quiet = fm.oldM - fm.counter;  // (canHoldF32T: counter + ticks <= oldM)
					can = left < quiet ? left : quiet;
				}
				can = __reduce_min_sync(0xffffffffu, can);
				if (can > holdMax) can = holdMax;
				can &= ~63u;
				if (can > ticks) ticks = can;
			}
#endif
			if (cascade) {
				int16_t *row = valid ? out + (size_t)s * rowStride + gs.callPos : scratchRow;
				OutWriter ow;
				ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
				renderHoldF32T<kRoleCascadeOsc>(fm, gs, desc, sampleRate, ticks, ow, noise, xc);
			} else {
				NullOut no;
				renderHoldF32T<kRoleParallelOnly>(fm, gs, desc, sampleRate, ticks, no, noise, xc);
			}
		} else if (cls == kClassFade) {
			// every stream here has fadeTicks interior fade ticks ahead on the 64-sample grid; run as many whole 64-tick cells as
			// the shortest of them allows (canFadeF32T: counter + ticks < newF), up to fadeMax
			uint32_t ticks = fadeTicks;
			if (fadeMax > fadeTicks) {
				uint32_t can = 0xffffffffu;
				if (valid) {
					const uint32_t left = sampleCount - gs.callPos, inside = fm.newF - 1u - fm.counter;
					can = left < inside ? left : inside;
				}
				can = __reduce_min_sync(0xffffffffu, can);
				if (can > fadeMax) can = fadeMax;
				can &= ~63u;
				if (can > ticks) ticks = can;
			}
			if (cascade) {
				int16_t *row = valid ? out + (size_t)s * rowStride + gs.callPos : scratchRow;
				OutWriter ow;
				ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
				renderFadeF32T<kRoleCascade>(fm, gs, desc, sampleRate, ticks, ow, noise, xc);
			} else {
				NullOut no;
				renderFadeF32T<kRoleParallel>(fm, gs, desc, sampleRate, ticks, no, noise, xc);
			}
		} else {
			const uint32_t pos = gs.callPos;
			uint32_t ticks = 0;
			if (valid) {
				ticks = sampleCount - pos;
				if (ticks > genTicks) ticks = genTicks;
				if (fadeTicks != 0u) {  // end on the 64-sample grid of the drift control (the fade class starts there)
					const uint64_t end = gs.samplesGenerated + ticks, grid = end & ~(uint64_t)(kCoarseTicks - 1);
					if (grid > gs.samplesGenerated && pos + ticks < sampleCount) ticks = (uint32_t)(grid - gs.samplesGenerated);
				}
			}
			int32_t lastUserIndex;
			uint32_t qHead;
			if (cascade) {
				int16_t *row = out + (size_t)(valid ? s : 0) * rowStride;
				OutWriter ow;
				ow.init(row + pos, ((reinterpret_cast<uintptr_t>(row + pos) & 15u) == 0));
				const uint32_t produced = renderGeneralF32T<kRoleCascade>(fm, gs, desc, sampleRate, ticks, genTicks, ow, noise, xc, &lastUserIndex, &qHead);
				ow.flush();
				if (produced < ticks) zeroRow(row, pos + produced, sampleCount);
			} else {
				NullOut no;
				renderGeneralF32T<kRoleParallel>(fm, gs, desc, sampleRate, ticks, genTicks, no, noise, xc, &lastUserIndex, &qHead);
			}
		}
#if KLATT_SCHED_LITE
		xc.sync();  // both halves of every stream of this chunk are in the staged records
		const uint32_t next = (cascade && valid) ? classifyNextT(fm, gs, sampleCount, holdTicks, fadeTicks) : kClassExit;
		// (a hold chunk only moves the frame-manager counters, the oscillators, the noise memories and the section memories:
		// the first 256 bytes of a record; the pole state, the direct parameters and the drift-control record are unchanged)
		const uint32_t piecesOut = cls == kClassHold ? kHoldPiecesOut : kRecPieces;
#pragma unroll 1
		for (uint32_t idx = tw; idx < 32u * piecesOut; idx += 64u) {
			const uint32_t r = idx / piecesOut, p = idx - r * piecesOut;
			const uint32_t sr = work[pair][r];
			if (sr < numStreams) {
				const uint2 *src = reinterpret_cast<const uint2 *>(stage + r * kStageStride + p * 16u);
				const uint2 a = src[0], b = src[1];
				__stcg(reinterpret_cast<uint4 *>(lite + sr) + p, make_uint4(a.x, a.y, b.x, b.y));
			}
		}
#endif
		__threadfence();
		xc.sync();  // both halves of every stream of this batch are stored
#ifdef KLATT_SCHED_PROFILE
		if (cls == kClassHold) { PROF_LAP(tHold) nHold++; } else if (cls == kClassFade) { PROF_LAP(tFade) nGen++; } else { PROF_LAP(tGen) nGen++; }
		nLanes += __popc(__ballot_sync(0xffffffffu, valid));
#endif
		if (cascade) {
#if !KLATT_SCHED_LITE
			const uint32_t next = valid ? classifyNext(desc.state, sampleCount, holdTicks) : kClassExit;
#endif
			schedPush<false>(ctl, ring, ringCap, next, s, valid);
		}
		PROF_LAP(tPush)
	}
#ifdef KLATT_SCHED_PROFILE
	if (lane == 0) {
		unsigned long long *p = reinterpret_cast<unsigned long long *>(ctl) + 128 + (cascade ? 0 : 8);
		atomicAdd(p + 0, (unsigned long long)tClaim); atomicAdd(p + 1, (unsigned long long)tHold);
		atomicAdd(p + 2, (unsigned long long)tGen); atomicAdd(p + 3, (unsigned long long)tPush);
		atomicAdd(p + 4, (unsigned long long)nHold); atomicAdd(p + 5, (unsigned long long)nGen);
		atomicAdd(p + 6, (unsigned long long)nLanes); atomicAdd(p + 7, (unsigned long long)tFade);
	}
#endif
}

static size_t schedSmemBytes() {
	return sizeof(uint4) * 2 * 2 * kGroupTicks * 32 + (KLATT_SCHED_LITE ? 2 * (size_t)kStageBytes : 0);
}
bool klattF32SchedUsesLite() { return KLATT_SCHED_LITE != 0; }
size_t klattF32SchedLiteBytes(uint32_t numStreams, uint32_t numBlocks) {
	return sizeof(StreamStateLite) * ((size_t)numStreams + 2 * (size_t)numBlocks);
}

// One call through the stream scheduler: seed the rings, then one persistent launch.  scratch: ring[3 * ringCap]
// (ringCap a power of two >= 2 * numStreams), ctl, scratchRow[max(holdTicks, holdMax, fadeMax)].  descs holds numStreams + 1 entries.
cudaError_t launchKlattF32Sched(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride, uint32_t *samplesWritten,
                                StreamResult *results, NoiseConfig noise, uint32_t *ring, uint32_t ringCap, void *ctlMem,
                                int16_t *scratchRow, uint32_t numBlocks, uint32_t *hostFault, void *liteMem, uint32_t holdMax,
                                uint32_t fadeTicks, uint32_t fadeMax, uint32_t roleSms, cudaStream_t stream, unsigned long long *launchCounter) {
	if (numStreams == 0 || sampleCount == 0) return cudaSuccess;
	SchedCtl *ctl = static_cast<SchedCtl *>(ctlMem);
	StreamStateLite *lite = KLATT_SCHED_LITE ? static_cast<StreamStateLite *>(liteMem) : nullptr;
	static bool attrSet = false;
	if (!attrSet) {
		cudaError_t ea = cudaFuncSetAttribute(klatt_f32_sched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)schedSmemBytes());
		if (ea != cudaSuccess) return ea;
		attrSet = true;
	}
	if (!lite) fadeTicks = 0;  // (the fade loop works on the compact records)
	cudaError_t e = cudaMemsetAsync(ring, 0xff, sizeof(uint32_t) * kNumRings * (size_t)ringCap, stream);
	if (e != cudaSuccess) return e;
	if ((e = cudaMemsetAsync(ctl, 0, 2048, stream)) != cudaSuccess) return e;
	const uint32_t batches = (numStreams + 31) / 32;
	// paired workers: two warps per batch, two batches per block
	const uint32_t blocksWanted = (batches + 1) / 2, grid = blocksWanted < numBlocks ? blocksWanted : numBlocks;
	if (lite && (e = launchKlattLiteImport(descs, numStreams, 2 * grid, lite, stream)) != cudaSuccess) return e;
	klatt_sched_seed_kernel<<<(numStreams + 255) / 256, 256, 0, stream>>>(descs, lite, numStreams, sampleCount, holdTicks, fadeTicks, ctl, ring, ringCap);
	// NVSP_L2_PERSIST=1: pin the record array in the L2 (persisting access-policy window on the launching stream).  Measured
	// (DESIGN.md section 5d): DRAM traffic of a config-3 step 59.7 -> 51.5 GB, but every workload gets SLOWER in warm
	// back-to-back steps (config 3 +1.2 %, config 5 +3.3 %, config 2 -- 190 MB of records against a 79 MB set-aside -- +8 %),
	// so it is off by default.
	static const bool l2Persist = getenv("NVSP_L2_PERSIST") && atoi(getenv("NVSP_L2_PERSIST")) != 0;
	bool windowSet = false;
	if (lite && l2Persist) {
		int dev = 0, maxPersist = 0, maxWindow = 0;
		cudaGetDevice(&dev);
		cudaDeviceGetAttribute(&maxPersist, cudaDevAttrMaxPersistingL2CacheSize, dev);
		cudaDeviceGetAttribute(&maxWindow, cudaDevAttrMaxAccessPolicyWindowSize, dev);
		const size_t bytes = klattF32SchedLiteBytes(numStreams, grid);
		if (maxPersist > 0 && maxWindow > 0) {
			static size_t limitSet = 0;
			const size_t wantLimit = bytes < (size_t)maxPersist ? bytes : (size_t)maxPersist;
			if (wantLimit > limitSet && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, wantLimit) == cudaSuccess) limitSet = wantLimit;
			cudaStreamAttrValue attr;
			memset(&attr, 0, sizeof attr);
			attr.accessPolicyWindow.base_ptr = lite;
			attr.accessPolicyWindow.num_bytes = bytes < (size_t)maxWindow ? bytes : (size_t)maxWindow;
			attr.accessPolicyWindow.hitRatio = limitSet >= bytes ? 1.0f : (float)((double)limitSet / (double)bytes);
			attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
			attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
			windowSet = cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
			if (!windowSet) cudaGetLastError();
		}
	}
	klatt_f32_sched_kernel<<<grid, kPairBlock, schedSmemBytes(), stream>>>(descs, lite, numStreams, sampleRate, sampleCount, holdTicks, genTicks,
	                                                                        out, rowStride, scratchRow, noise, ctl, ring, ringCap, roleSms, holdMax, fadeTicks, fadeMax);
	if (windowSet) {
		cudaStreamAttrValue attr;
		memset(&attr, 0, sizeof attr);
		attr.accessPolicyWindow.num_bytes = 0;
		cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &attr);
	}
	// the watchdog's verdict travels to a pinned host word; the engine reads it at its next synchronisation point
	if (hostFault && (e = cudaMemcpyAsync(hostFault, &ctl->fault, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
	if (lite) {
		if ((e = launchKlattLiteExport(descs, numStreams, lite, samplesWritten, results, stream)) != cudaSuccess) return e;
		if (launchCounter) *launchCounter += 4;  // import, seed, workers, export
	} else {
		if ((e = launchKlattFinalize(descs, numStreams, samplesWritten, results, stream)) != cudaSuccess) return e;
		if (launchCounter) *launchCounter += 3;
	}
#ifdef KLATT_SCHED_PROFILE
	{
		unsigned long long h[16];
		cudaStreamSynchronize(stream);
		cudaMemcpy(h, reinterpret_cast<unsigned long long *>(ctl) + 128, sizeof(h), cudaMemcpyDeviceToHost);
		for (int k = 0; k < 2; ++k)
			fprintf(stderr, "[sched profile] %s warps: claim %.1f  hold %.1f  gen %.1f  fade %.1f  push %.1f Mcycles; batches hold %llu gen+fade %llu; lanes/batch %.2f\n",
			        k ? "parallel" : "cascade ", h[8 * k] / 1e6, h[8 * k + 1] / 1e6, h[8 * k + 2] / 1e6, h[8 * k + 7] / 1e6, h[8 * k + 3] / 1e6, h[8 * k + 4], h[8 * k + 5],
			        (double)h[8 * k + 6] / (double)(h[8 * k + 4] + h[8 * k + 5]));
	}
#endif
	return cudaGetLastError();
}

// resident blocks of the scheduler kernel per SM (occupancy query; the grid is SMs x this)
int klattF32SchedBlocksPerSm() {
	int n = 0;
	cudaFuncSetAttribute(klatt_f32_sched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)schedSmemBytes());
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, klatt_f32_sched_kernel, kPairBlock, schedSmemBytes()) != cudaSuccess) n = 0;
	return n;
}

}  // namespace klatt
