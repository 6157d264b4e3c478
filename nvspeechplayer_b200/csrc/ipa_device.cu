// The device IPA -> frame-queue producer (speechPlayer_ipaFramesDevice, include/speechPlayer_ipa.h): the rules of
// ipa_core.h, compiled for the GPU, bit for bit the host producer (ipa_frames.cpp).  Built with -fmad=false.
//
//   (a) ipa_count_kernel    one thread per text: decode its bytes, run the list builder as a pure counter
//       ipa_scan_kernel     one block: exclusive scan of the counts -> text offsets, and the total
//   (b) ipa_records_kernel  one thread per text: the list builder writing compact records at the text's offset, then
//                           _copyAdjacent, the times and the pitch paths in place, and the text's timeline samples
//   (c) ipa_rows_kernel     grid-stride over rows x 47 parameters (coalesced stores), then the per-row arrays
//
// (a) and (b) hold the table's keys, flags and presence masks in shared memory (binary search on the packed key); (c)
// reads the 47-value rows through L2.  The records go to scratch sized by a bound known before any kernel runs (a code
// point yields at most two entries: a phoneme and either its post-stop aspiration or its pre-stop gap), so the total and
// the count of pitch-factor misses come back to the host in one 16-byte copy after (b): the call's only
// synchronisation.  (c) is left running on the caller's stream.
#include <mutex>
#include <vector>

#include "../../include/speechPlayer_ipa.h"
#include "host.h"
#include "ipa_table.h"

using namespace klatt;

namespace {

constexpr int kTextThreads = 128;

struct DevTable {
	const uint64_t *keys, *present;
	const uint8_t *flags;
	const double *values;
	int n, h;
};

struct Texts {
	const unsigned char *bytes;
	const int64_t *off;  // [n + 1], absolute; text i is bytes [off[i] - base, off[i + 1] - base)
	int64_t base;
	uint32_t n;
	const double *speed, *basePitch;  // or null: 1, 100
	const int32_t *group;             // or null: factor row 0
	const char *clause;               // or null: '.'
	const double *pitchTable;         // ipa::PitchPlan::table
	double trailingMs, perMs;
	__device__ ipa::Utf8 text(uint32_t i) const {
		return ipa::Utf8{bytes + (off[i] - base), bytes + (off[i + 1] - base)};
	}
};

// the keys, flags and presence masks into shared memory (dynamic: n * 17 bytes)
__device__ ipa::TableView stageTable(const DevTable &T, uint64_t *smem) {
	uint64_t *keys = smem, *present = smem + T.n;
	uint8_t *flags = reinterpret_cast<uint8_t *>(smem + 2 * T.n);
	for (int i = threadIdx.x; i < T.n; i += blockDim.x) {
		keys[i] = T.keys[i];
		present[i] = T.present[i];
		flags[i] = T.flags[i];
	}
	__syncthreads();
	return ipa::TableView{keys, flags, present, T.values, T.n, T.h};
}

__global__ void __launch_bounds__(kTextThreads) ipa_count_kernel(DevTable T, Texts X, int64_t *__restrict__ counts) {
	extern __shared__ uint64_t smem[];
	const ipa::TableView tab = stageTable(T, smem);
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= X.n) return;
	counts[i] = ipa::ipaCount(tab, X.text(i), X.trailingMs);
}

// exclusive scan of v[0, n) in place, v[n] = status[0] = the total (every thread sums a run, warp shuffles scan the runs)
__global__ void __launch_bounds__(1024) ipa_scan_kernel(int64_t *__restrict__ v, uint32_t n, unsigned long long *__restrict__ status) {
	__shared__ int64_t warpTotal[32];
	const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const uint32_t per = (n + 1023) / 1024;
	const uint32_t c0 = min(n, tid * per), c1 = min(n, c0 + per);
	int64_t run = 0;
	for (uint32_t c = c0; c < c1; ++c) run += v[c];
	int64_t inc = run;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const int64_t up = __shfl_up_sync(0xffffffffu, inc, d);
		if (lane >= (uint32_t)d) inc += up;
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		int64_t w = warpTotal[lane];
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const int64_t up = __shfl_up_sync(0xffffffffu, w, d);
			if (lane >= (uint32_t)d) w += up;
		}
		warpTotal[lane] = w;
	}
	__syncthreads();
	int64_t pos = inc - run + (warp > 0 ? warpTotal[warp - 1] : 0);
	for (uint32_t c = c0; c < c1; ++c) {
		const int64_t x = v[c];
		v[c] = pos;
		pos += x;
	}
	if (tid == 1023) {
		v[n] = warpTotal[31];
		status[0] = (unsigned long long)warpTotal[31];
	}
}

// 4 blocks an SM: ptxas then gives the rules 74 registers and spills nothing (it spills at its own default of 64)
__global__ void __launch_bounds__(kTextThreads, 4)
ipa_records_kernel(DevTable T, Texts X, const int64_t *__restrict__ offsets, ipa::Rec *__restrict__ recs, uint64_t *__restrict__ timeline,
                   unsigned long long *__restrict__ status) {
	extern __shared__ uint64_t smem[];
	const ipa::TableView tab = stageTable(T, smem);
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= X.n) return;
	const int clause = ipa::clauseIndex(X.clause ? X.clause[i] : '.');
	const ipa::Factors fx{X.pitchTable + (size_t)clause * ipa::kMaxPercents,
	                      X.pitchTable + (size_t)(ipa::kClauseTypes + (X.group ? X.group[i] : 0)) * ipa::kMaxPercents};
	ipa::Rec *out = recs + offsets[i];
	int64_t n = 0;
	if (!ipa::ipaRecords(tab, X.text(i), X.speed ? X.speed[i] : 1.0, X.basePitch ? X.basePitch[i] : 100.0, clause, fx, X.trailingMs,
	                     out, &n))
		atomicAdd(&status[1], 1ull);
	if (timeline) {  // the timeline law: sum of max(M + 1, max(F, 1) + 2)
		uint64_t t = 0;
		for (int64_t j = 0; j < n; ++j) {
			const uint64_t m = ipa::msToSamples(out[j].duration, X.perMs), f0 = ipa::msToSamples(out[j].fade, X.perMs);
			const uint64_t f = f0 > 1 ? f0 : 1;
			t += m + 1 > f + 2 ? m + 1 : f + 2;
		}
		timeline[i] = t;
	}
}

__global__ void __launch_bounds__(256)
ipa_rows_kernel(DevTable T, const ipa::Rec *__restrict__ recs, int64_t total, double perMs, double *__restrict__ frames,
                uint32_t *__restrict__ minDur, uint32_t *__restrict__ fadeDur, uint8_t *__restrict__ isNull, double *__restrict__ durationMs,
                double *__restrict__ fadeMs) {
	const ipa::TableView tab{T.keys, T.flags, T.present, T.values, T.n, T.h};
	const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (frames) {
		const int64_t cells = total * ipa::kParams;
		for (int64_t c = t0; c < cells; c += stride) {
			const int64_t row = c / ipa::kParams;
			frames[c] = ipa::ipaCell(tab, recs[row], (int)(c - row * ipa::kParams));
		}
	}
	for (int64_t r = t0; r < total; r += stride) {
		const ipa::Rec &x = recs[r];
		if (minDur) minDur[r] = ipa::msToSamples(x.duration, perMs);
		if (fadeDur) fadeDur[r] = ipa::msToSamples(x.fade, perMs);
		if (isNull) isNull[r] = (x.deco & ipa::kSilence) ? 1 : 0;
		if (durationMs) durationMs[r] = x.duration;
		if (fadeMs) fadeMs[r] = x.fade;
	}
}

// Grow-only scratch of one device, kept for the life of the process.  Calls on one device are serialised by the mutex;
// `done` orders a call's kernels after the previous call's on whatever streams they were issued.
struct Pool {
	std::mutex mu;
	uint64_t tableId = 0;
	DevBuf tKeys, tPresent, tFlags, tValues;
	DevBuf bytes, textOff, speed, basePitch, group, clause, pitchTable, offsets, recs, timeline, status;
	PinnedBuf hostStatus;
	cudaEvent_t done = nullptr;
};

Pool &poolFor(int dev) {
	static std::mutex mu;
	static std::vector<Pool *> *pools = new std::vector<Pool *>;  // never freed: no CUDA call from a static destructor
	std::lock_guard<std::mutex> lk(mu);
	if ((size_t)dev >= pools->size()) pools->resize(dev + 1, nullptr);
	if (!(*pools)[dev]) (*pools)[dev] = new Pool;
	return *(*pools)[dev];
}

template <class T> bool upload(DevBuf &d, const T *h, size_t n, cudaStream_t s, const char *what) {
	if (!d.reserve(std::max<size_t>(n, 1) * sizeof(T), what)) return false;
	return !n || cudaOk(cudaMemcpyAsync(d.p, h, n * sizeof(T), cudaMemcpyHostToDevice, s), what);
}

}  // namespace

extern "C" {

long long speechPlayer_ipaFramesDevice(const speechPlayer_ipaTable_t *table, const char *text, const int64_t *textOffsets,
                                       unsigned int numTexts, const double *speed, const double *basePitch, const double *inflection,
                                       const char *clauseType, int sampleRate, double trailingSilenceMs, void *dOffsets, void *dFrames,
                                       void *dMinDur, void *dFadeDur, void *dIsNull, void *dDurationMs, void *dFadeMs,
                                       void *dTimelineSamples, unsigned long long capacity, void *cudaStream) {
	g_lastError.clear();
	if (!table) return fail("ipaFramesDevice: null table");
	if (numTexts && (!text || !textOffsets)) return fail("ipaFramesDevice: null text / textOffsets");
	for (unsigned int i = 0; i < numTexts; ++i)
		if (textOffsets[i + 1] < textOffsets[i]) return fail("ipaFramesDevice: textOffsets decrease");
	if ((dMinDur || dFadeDur || dTimelineSamples) && sampleRate <= 0)
		return fail("ipaFramesDevice: sampleRate is required for durations in samples");
	if ((size_t)table->keys.size() * 17 > 48 * 1024) return fail("ipaFramesDevice: the phoneme table does not fit in shared memory");
	int dev = -1, count = 0;
	if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || cudaGetDevice(&dev) != cudaSuccess) {
		cudaGetLastError();
		return fail("ipaFramesDevice: no usable CUDA device (this library has no CPU fallback)");
	}
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	if (numTexts == 0) {
		if (dOffsets) {
			CU(cudaMemsetAsync(dOffsets, 0, sizeof(int64_t), stream));
			CU(cudaStreamSynchronize(stream));
		}
		return 0;
	}
	Pool &P = poolFor(dev);
	std::lock_guard<std::mutex> lk(P.mu);
	if (!P.done) CU(cudaEventCreateWithFlags(&P.done, cudaEventDisableTiming));
	CU(cudaStreamWaitEvent(stream, P.done, 0));  // the previous call's kernels still read the scratch
	const int tn = (int)table->keys.size();
	if (P.tableId != table->id) {
		if (!upload(P.tKeys, table->keys.data(), tn, stream, "ipa table") || !upload(P.tPresent, table->present.data(), tn, stream, "ipa table") ||
		    !upload(P.tFlags, table->flags.data(), tn, stream, "ipa table") ||
		    !upload(P.tValues, table->values.data(), table->values.size(), stream, "ipa table"))
			return -1;
		P.tableId = table->id;
	}
	ipa::PitchPlan plan;
	ipa::planPitches(plan, inflection, clauseType, numTexts);
	const int64_t base = textOffsets[0], numBytes = textOffsets[numTexts] - base;
	if (!upload(P.bytes, reinterpret_cast<const unsigned char *>(text) + base, (size_t)numBytes, stream, "ipa text") ||
	    !upload(P.textOff, textOffsets, (size_t)numTexts + 1, stream, "ipa text offsets") ||
	    !upload(P.pitchTable, plan.table.data(), plan.table.size(), stream, "ipa pitch factors") ||
	    (speed && !upload(P.speed, speed, numTexts, stream, "ipa speed")) ||
	    (basePitch && !upload(P.basePitch, basePitch, numTexts, stream, "ipa basePitch")) ||
	    (clauseType && !upload(P.clause, clauseType, numTexts, stream, "ipa clauseType")) ||
	    (!plan.group.empty() && !upload(P.group, plan.group.data(), numTexts, stream, "ipa pitch groups")))
		return -1;
	// the records bound: two entries per code point (at most one per byte) plus the trailing silence
	const size_t bound = 2 * (size_t)numBytes + numTexts;
	if (!P.offsets.reserve(((size_t)numTexts + 1) * sizeof(int64_t), "ipa offsets") || !P.recs.reserve(bound * sizeof(ipa::Rec), "ipa records") ||
	    !P.status.reserve(2 * sizeof(unsigned long long), "ipa status") ||
	    (dTimelineSamples && !P.timeline.reserve((size_t)numTexts * sizeof(uint64_t), "ipa timeline")))
		return -1;
	CU(P.hostStatus.reserve(2 * sizeof(unsigned long long)));
	const DevTable T{P.tKeys.as<uint64_t>(), P.tPresent.as<uint64_t>(), P.tFlags.as<uint8_t>(), P.tValues.as<double>(), tn, table->h};
	const Texts X{P.bytes.as<unsigned char>(), P.textOff.as<int64_t>(), base, numTexts, speed ? P.speed.as<double>() : nullptr,
	              basePitch ? P.basePitch.as<double>() : nullptr, plan.group.empty() ? nullptr : P.group.as<int32_t>(),
	              clauseType ? P.clause.as<char>() : nullptr, P.pitchTable.as<double>(), trailingSilenceMs, sampleRate / 1000.0};
	const size_t smem = (size_t)tn * 17;
	const unsigned blocks = (numTexts + kTextThreads - 1) / kTextThreads;
	unsigned long long *status = P.status.as<unsigned long long>();
	CU(cudaMemsetAsync(status, 0, 2 * sizeof(unsigned long long), stream));
	ipa_count_kernel<<<blocks, kTextThreads, smem, stream>>>(T, X, P.offsets.as<int64_t>());
	ipa_scan_kernel<<<1, 1024, 0, stream>>>(P.offsets.as<int64_t>(), numTexts, status);
	ipa_records_kernel<<<blocks, kTextThreads, smem, stream>>>(T, X, P.offsets.as<int64_t>(), P.recs.as<ipa::Rec>(),
	                                                          dTimelineSamples ? P.timeline.as<uint64_t>() : nullptr, status);
	CU(cudaGetLastError());
	if (dOffsets)
		CU(cudaMemcpyAsync(dOffsets, P.offsets.p, ((size_t)numTexts + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, stream));
	unsigned long long *hs = P.hostStatus.as<unsigned long long>();
	CU(cudaMemcpyAsync(hs, status, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
	CU(cudaStreamSynchronize(stream));
	const long long total = (long long)hs[0];
	if (hs[1]) return fail("ipaFramesDevice: a pitch percent has no precomputed factor");
	if ((unsigned long long)total > capacity) return total;
	if (total > 0 && (dFrames || dMinDur || dFadeDur || dIsNull || dDurationMs || dFadeMs)) {
		const int64_t work = dFrames ? total * ipa::kParams : total;
		const unsigned grid = (unsigned)std::min<int64_t>((work + 255) / 256, 148 * 16);
		ipa_rows_kernel<<<grid, 256, 0, stream>>>(T, P.recs.as<ipa::Rec>(), total, sampleRate / 1000.0, static_cast<double *>(dFrames),
		                                          static_cast<uint32_t *>(dMinDur), static_cast<uint32_t *>(dFadeDur),
		                                          static_cast<uint8_t *>(dIsNull), static_cast<double *>(dDurationMs),
		                                          static_cast<double *>(dFadeMs));
		CU(cudaGetLastError());
	}
	if (dTimelineSamples)
		CU(cudaMemcpyAsync(dTimelineSamples, P.timeline.p, (size_t)numTexts * sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
	CU(cudaEventRecord(P.done, stream));
	return total;
}

}  // extern "C"
