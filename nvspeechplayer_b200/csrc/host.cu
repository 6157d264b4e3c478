// The out-of-line parts of the host layer (host.h): errors, device selection, queue uploads, and the render pipeline that
// players and batches share -- the FP32 scheduler selection (launchRender) and the device-to-host pipeline (renderToHost).
#include <chrono>
#include <cstdio>
#include <mutex>
#include <vector>

#include "host.h"

using namespace klatt;

// the state speechPlayer_initialize leaves a player in: src/frame.cpp:85-88 (curFrame zeroed, curFrameIsNULL,
// sampleCounter 0, lastUserIndex -1, old request = zeroed NULL request), src/speechWaveGenerator.cpp:37,49,
// 104-110 (phases, noise memory and resonator histories zero).  The memset before this kernel did the zeros.
__global__ void init_states_kernel(StreamState *states, uint32_t n) {
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	states[i].fm.lastUserIndex = -1;
	states[i].fm.curIsNull = 1;
	states[i].fm.oldIsNull = 1;
}

namespace klatt {

// ------------------------------------------------------------------------------------------------
// errors and devices
// ------------------------------------------------------------------------------------------------
thread_local std::string g_lastError;

int fail(const std::string &what) {
	g_lastError = what;
	if (envIs("NVSP_VERBOSE")) fprintf(stderr, "[nvspeechplayer_b200] %s\n", what.c_str());
	return -1;
}
void setLastError(const char *what) { fail(what ? what : "error"); }

bool cudaOk(cudaError_t e, const char *what) {
	if (e == cudaSuccess) return true;
	fail(std::string(what) + ": " + cudaGetErrorString(e));
	return false;
}

int pickDevice() {
	static const int chosen = envNum<int>("NVSP_DEVICE", -1);
	int dev = 0;
	if (chosen >= 0) {
		if (cudaSetDevice(chosen) != cudaSuccess) return -1;
		return chosen;
	}
	if (cudaGetDevice(&dev) != cudaSuccess) return -1;
	return dev;
}

int QueueBufs::upload(const void *hFrames, const uint32_t *hMin, const uint32_t *hFade, const int32_t *hUix, const uint8_t *hNull,
                      size_t n, cudaStream_t stream) {
	const size_t m = std::max<size_t>(n, 1);
	if ((hFrames && !frames.reserve(m * kNumParams * sizeof(double))) || (hMin && !minDur.reserve(m * 4)) ||
	    (hFade && !fadeDur.reserve(m * 4)) || (hUix && !userIndex.reserve(m * 4)) || (hNull && !isNull.reserve(m)))
		return -1;
	if (n == 0) return 0;
	if (hFrames) CU(cudaMemcpyAsync(frames.p, hFrames, n * kNumParams * sizeof(double), cudaMemcpyHostToDevice, stream));
	if (hMin) CU(cudaMemcpyAsync(minDur.p, hMin, n * 4, cudaMemcpyHostToDevice, stream));
	if (hFade) CU(cudaMemcpyAsync(fadeDur.p, hFade, n * 4, cudaMemcpyHostToDevice, stream));
	if (hUix) CU(cudaMemcpyAsync(userIndex.p, hUix, n * 4, cudaMemcpyHostToDevice, stream));
	if (hNull) CU(cudaMemcpyAsync(isNull.p, hNull, n, cudaMemcpyHostToDevice, stream));
	return 0;
}

cudaError_t initStates(StreamState *states, uint32_t n, cudaStream_t stream) {
	cudaError_t e = cudaMemsetAsync(states, 0, sizeof(StreamState) * (size_t)n, stream);
	if (e != cudaSuccess) return e;
	init_states_kernel<<<(n + 255) / 256, 256, 0, stream>>>(states, n);
	return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// FP32 scheduler selection
// ------------------------------------------------------------------------------------------------
bool RoundsCtx::init() {
	if (ok) return true;
	// chunk lengths are multiples of 64: the coarse pole re-basing and the Philox block cadence stay warp-uniform,
	// and every chunk starts on a 16-byte boundary of its output row
	genTicks = std::max<uint32_t>(envNum<uint32_t>("NVSP_GEN_TICKS", 256) & ~63u, 64);
	holdTicks = std::max<uint32_t>(envNum<uint32_t>("NVSP_HOLD_TICKS", 512) & ~63u, 64);
	minStreams = envNum<uint32_t>("NVSP_ROUNDS_MIN_STREAMS", 2048);
	groups = std::min<uint32_t>(std::max<uint32_t>(envNum<uint32_t>("NVSP_GROUPS", 4), 1), kMaxGroups);
	persistent = !envIs("NVSP_SCHED", "rounds");
	blockSched = envIs("NVSP_SCHED", "block");
	blockHoldTicks = std::max<uint32_t>(envNum<uint32_t>("NVSP_BLOCK_HOLD_TICKS", 128) & ~63u, 64);
	blockMinStreams = envNum<uint32_t>("NVSP_BLOCK_MIN_STREAMS", 16384);
	// (round 1, AoS state with L1-bypassing loads: 512 / 640 was the optimum; with the compact staged records a change of
	// loop is cheaper and the optimum is a flat basin around 256 / 384: 200.2 ms vs 207.9 ms at 512 / 640)
	schedGenTicks = std::max<uint32_t>(envNum<uint32_t>("NVSP_SCHED_GEN_TICKS", 384) & ~63u, 64);
	schedHoldTicks = std::max<uint32_t>(envNum<uint32_t>("NVSP_SCHED_HOLD_TICKS", 256) & ~63u, 64);
	// a hold chunk whose 32 streams can all hold longer runs up to this many ticks (steady vowels, sung notes; measured
	// 256 -> 4096: config 2 292 -> 278 ms, config 5 163 -> 155 ms, config 3 unchanged)
	schedHoldMax = std::max<uint32_t>(envNum<uint32_t>("NVSP_SCHED_HOLD_MAX", 4096) & ~63u, schedHoldTicks);
	// the fade class (0: off): streams with this many interior fade ticks ahead on the 64-sample grid take the straight-line
	// fade loop; chunks stretched up to NVSP_SCHED_FADE_MAX.  NVSP_SCHED_HOLD_SMS / NVSP_SCHED_FADE_SMS: that many SMs take
	// hold / fade chunks first, the rest general chunks (SM roles: one loop pair per instruction cache)
	schedFadeTicks = envNum<uint32_t>("NVSP_SCHED_FADE_TICKS", 0) & ~63u;
	schedFadeMax = std::min<uint32_t>(std::max<uint32_t>(envNum<uint32_t>("NVSP_SCHED_FADE_MAX", 512) & ~63u, schedFadeTicks), 4096);
	schedRoleSms = std::min<uint32_t>(envNum<uint32_t>("NVSP_SCHED_HOLD_SMS", 0), 255u) |
	               (std::min<uint32_t>(envNum<uint32_t>("NVSP_SCHED_FADE_SMS", 0), 255u) << 8);
	int dev = 0, sms = 0;
	cudaGetDevice(&dev);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	const int perSm = klattF32SchedBlocksPerSm();
	schedBlocks = envNum<uint32_t>("NVSP_SCHED_BLOCKS", (uint32_t)(sms * std::max(perSm, 1)));
	blockBlocks = std::max<uint32_t>(envNum<uint32_t>("NVSP_BLOCK_BLOCKS", (uint32_t)sms), 1);
	if (envIs("NVSP_VERBOSE"))
		fprintf(stderr, "[nvspeechplayer_b200] scheduler: %d SMs x %d blocks, %u blocks, hold %u / general %u ticks\n", sms, perSm,
		        schedBlocks, schedHoldTicks, schedGenTicks);
	if (!cudaOk(cudaEventCreateWithFlags(&evStart, cudaEventDisableTiming), "cudaEventCreate")) return false;
	for (uint32_t g = 0; g < groups; ++g) {
		if (!cudaOk(cudaStreamCreateWithFlags(&lanes[2 * g], cudaStreamNonBlocking), "cudaStreamCreate")) return false;
		if (!cudaOk(cudaStreamCreateWithFlags(&lanes[2 * g + 1], cudaStreamNonBlocking), "cudaStreamCreate")) return false;
		if (!cudaOk(cudaEventCreateWithFlags(&evFork[g], cudaEventDisableTiming), "cudaEventCreate")) return false;
		if (!cudaOk(cudaEventCreateWithFlags(&evJoin[g], cudaEventDisableTiming), "cudaEventCreate")) return false;
	}
	ok = true;
	return true;
}

cudaError_t RoundsCtx::checkFault() {
	if (!hostFault.p) {
		if (hostFault.reserve(sizeof(uint32_t)) != cudaSuccess) return cudaErrorMemoryAllocation;
		*hostFault.as<uint32_t>() = 0;
	}
	return *hostFault.as<uint32_t>() ? cudaErrorLaunchTimeout : cudaSuccess;
}

RoundsCtx::~RoundsCtx() {
	if (evStart) cudaEventDestroy(evStart);
	for (uint32_t g = 0; g < kMaxGroups; ++g) {
		if (evFork[g]) cudaEventDestroy(evFork[g]);
		if (evJoin[g]) cudaEventDestroy(evJoin[g]);
		if (lanes[2 * g]) cudaStreamDestroy(lanes[2 * g]);
		if (lanes[2 * g + 1]) cudaStreamDestroy(lanes[2 * g + 1]);
	}
}

cudaError_t launchRender(int precision, const StreamDesc *descs, uint32_t n, int sampleRate, uint32_t sampleCount,
                         int16_t *out, size_t rowStride, uint32_t *written, StreamResult *results,
                         NoiseConfig noise, cudaStream_t stream, RoundsCtx *rc, bool planned, unsigned long long *launchCounter) {
	if (precision == kPrecisionF64) {
		if (launchCounter) ++*launchCounter;
		return launchKlattF64(descs, n, sampleRate, sampleCount, out, rowStride, written, results, noise, stream);
	}
	if (rc && planned && rc->init() && rc->blockSched && n >= rc->blockMinStreams && klattF32BlockCanTake(n, rc->blockBlocks)) {
		if (!rc->lite.reserve(klattF32BlockLiteBytes(n, rc->blockBlocks)) ||
		    !rc->scratchRow.reserve(sizeof(int16_t) * (size_t)std::max<uint32_t>(std::max(rc->schedHoldTicks, rc->holdTicks), rc->blockHoldTicks)))
			return cudaErrorMemoryAllocation;
		if (!rc->blockProf.p) {
			if (!rc->blockProf.reserve(256)) return cudaErrorMemoryAllocation;
			cudaMemsetAsync(rc->blockProf.p, 0, 256, stream);
		}
		if (cudaError_t e = rc->checkFault()) return e;
		return launchKlattF32Block(descs, n, sampleRate, sampleCount, rc->blockHoldTicks, out, rowStride, written, results, noise,
		                           rc->lite.p, rc->scratchRow.as<int16_t>(), rc->blockBlocks, rc->blockProf.p, rc->hostFault.as<uint32_t>(),
		                           stream, launchCounter);
	}
	if (rc && planned && rc->init() && rc->persistent && n >= rc->minStreams && sampleCount > rc->schedGenTicks) {
		uint32_t cap = 64;
		while (cap < 2 * n) cap <<= 1;
		if (cudaError_t e = rc->checkFault()) return e;
		if (!rc->ring.reserve(sizeof(uint32_t) * 3 * (size_t)cap) || !rc->ctl.reserve(2048) ||
		    !rc->scratchRow.reserve(sizeof(int16_t) * (size_t)std::max(std::max(std::max(rc->schedHoldTicks, rc->schedHoldMax), rc->holdTicks), rc->schedFadeMax)))
			return cudaErrorMemoryAllocation;
		if (klattF32SchedUsesLite() && !rc->lite.reserve(klattF32SchedLiteBytes(n, rc->schedBlocks))) return cudaErrorMemoryAllocation;
		return launchKlattF32Sched(descs, n, sampleRate, sampleCount, rc->schedHoldTicks, rc->schedGenTicks, out, rowStride, written,
		                           results, noise, rc->ring.as<uint32_t>(), cap, rc->ctl.p, rc->scratchRow.as<int16_t>(),
		                           rc->schedBlocks, rc->hostFault.as<uint32_t>(), rc->lite.p, rc->schedHoldMax, rc->schedFadeTicks,
		                           rc->schedFadeMax, rc->schedRoleSms, stream, launchCounter);
	}
	if (rc && planned && rc->init() && n >= rc->minStreams && sampleCount > rc->genTicks) {
		const uint32_t rounds = (sampleCount + rc->genTicks - 1) / rc->genTicks;
		if (!rc->listHold.reserve(sizeof(uint32_t) * (size_t)n) || !rc->listGen.reserve(sizeof(uint32_t) * (size_t)n) ||
		    !rc->counters.reserve(sizeof(uint32_t) * 2 * (size_t)rounds * rc->groups) ||
		    !rc->scratchRow.reserve(sizeof(int16_t) * (size_t)rc->holdTicks))
			return cudaErrorMemoryAllocation;
		return launchKlattF32Rounds(descs, n, sampleRate, sampleCount, rc->holdTicks, rc->genTicks, out, rowStride, written,
		                            results, noise, rc->listHold.as<uint32_t>(), rc->listGen.as<uint32_t>(),
		                            rc->counters.as<uint32_t>(), rc->scratchRow.as<int16_t>(), stream, rc->groups, rc->lanes, rc->evStart, rc->evFork,
		                            rc->evJoin, launchCounter);
	}
	if (launchCounter) ++*launchCounter;
	return launchKlattF32(descs, n, sampleRate, sampleCount, out, rowStride, written, results, noise, stream);
}

// ------------------------------------------------------------------------------------------------
// device-to-host pipeline
// ------------------------------------------------------------------------------------------------
bool HostPipe::init() {
	if (ok) return true;
	if (!cudaOk(cudaStreamCreateWithFlags(&compute, cudaStreamNonBlocking), "cudaStreamCreate")) return false;
	if (!cudaOk(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking), "cudaStreamCreate")) return false;
	for (int i = 0; i < 2; ++i) {
		if (!cudaOk(cudaEventCreateWithFlags(&kernelDone[i], cudaEventDisableTiming), "cudaEventCreate")) return false;
		if (!cudaOk(cudaEventCreateWithFlags(&copyDone[i], cudaEventDisableTiming), "cudaEventCreate")) return false;
	}
	ok = true;
	return true;
}

HostPipe::~HostPipe() {
	for (int i = 0; i < 2; ++i) {
		if (kernelDone[i]) cudaEventDestroy(kernelDone[i]);
		if (copyDone[i]) cudaEventDestroy(copyDone[i]);
	}
	if (compute) cudaStreamDestroy(compute);
	if (copy) cudaStreamDestroy(copy);
}

static size_t stagingBudgetBytes() {
	// measured on B200 (config 3 e2e): 1024 -> 674 ms, 2048 -> 640 ms, 4096 -> 640 ms per step
	const size_t mb = envNum<size_t>("NVSP_STAGE_MB", 2048);
	return std::max<size_t>(mb, 1) << 20;
}

long long renderToHost(HostPipe &pipe, int precision, const StreamDesc *dDescs, uint32_t n, int sampleRate,
                       uint32_t sampleCount, int16_t *hostOut, uint32_t *perStream, StreamResult *lastResults,
                       NoiseConfig noise, unsigned long long *launchCounter, bool planned) {
	if (!pipe.init()) return -1;
	if (n == 0 || sampleCount == 0) return 0;
	// chunk length in ticks: whole request if it fits the staging budget, else a multiple of 8
	size_t budget = stagingBudgetBytes();
	uint64_t maxTicks = std::max<uint64_t>(budget / ((size_t)n * sizeof(int16_t)), 8);
	uint32_t chunk = (uint32_t)std::min<uint64_t>(sampleCount, maxTicks);
	if (chunk < sampleCount) chunk = chunk >= 64 ? (chunk & ~63u) : (chunk & ~7u);
	size_t stride = ((size_t)chunk + 7) & ~(size_t)7;
	for (int i = 0; i < 2; ++i) {
		if (!pipe.stage[i].reserve(stride * n * sizeof(int16_t))) return -1;
		if (!pipe.res[i].reserve((size_t)n * sizeof(StreamResult))) return -1;
	}
	if (!cudaOk(pipe.hostRes.reserve(sizeof(StreamResult) * (size_t)n * 2), "cudaMallocHost")) return -1;
	StreamResult *hostRes = pipe.hostRes.as<StreamResult>();
	std::vector<uint32_t> total(n, 0);
	// Chunk plan.  The first kernel has no copy to hide behind and the last copy no kernel, so large requests start with
	// a short chunk (~128 MB of output) and double up to the staging size: a copy takes ~2.3x as long as the render of
	// the same ticks (PCIe Gen5 vs. the render rate), so the copy of chunk c still covers the render of chunk c+1.
	std::vector<uint32_t> chunkStart, chunkLen;
	{
		uint32_t len = chunk;
		if ((size_t)n * sampleCount * sizeof(int16_t) > ((size_t)256 << 20)) {
			uint64_t first = (((size_t)128 << 20) / ((size_t)n * sizeof(int16_t))) & ~(uint64_t)63;
			len = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(first, 64), chunk);
		}
		for (uint32_t t = 0; t < sampleCount;) {
			uint32_t l = std::min(len, sampleCount - t);
			chunkStart.push_back(t); chunkLen.push_back(l);
			t += l;
			len = std::min<uint32_t>(len * 2, chunk >= 64 ? (chunk & ~63u) : chunk);  // interior chunk boundaries stay on the 64-tick grid
		}
	}
	const uint32_t numChunks = (uint32_t)chunkStart.size();
	const bool verbose = envIs("NVSP_VERBOSE");
	auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	const double tStart = now();
	auto harvest = [&](uint32_t c) -> bool {  // wait for chunk c's copies and fold its results
		int b = c & 1;
		if (!cudaOk(cudaEventSynchronize(pipe.copyDone[b]), "cudaEventSynchronize")) return false;
		const StreamResult *r = hostRes + (size_t)b * n;
		for (uint32_t s = 0; s < n; ++s) total[s] += r[s].written;
		if (lastResults && c + 1 == numChunks) memcpy(lastResults, r, sizeof(StreamResult) * (size_t)n);
		return true;
	};
	std::vector<cudaEvent_t> tev;
	if (verbose) {
		tev.resize(4 * (size_t)numChunks);
		for (auto &e : tev) cudaEventCreate(&e);
	}
	for (uint32_t c = 0; c < numChunks; ++c) {
		int b = c & 1;
		const uint32_t t0 = chunkStart[c], len = chunkLen[c];
		const double tA = now();
		if (c >= 2 && !harvest(c - 2)) return -1;  // staging buffer b is free again
		const double tB = now();
		if (verbose) cudaEventRecord(tev[4 * c + 0], pipe.compute);
		CU(launchRender(precision, dDescs, n, sampleRate, len, pipe.stage[b].as<int16_t>(), stride, nullptr,
		                pipe.res[b].as<StreamResult>(), noise, pipe.compute, &pipe.rounds, planned, launchCounter));
		if (verbose) cudaEventRecord(tev[4 * c + 1], pipe.compute);
		CU(cudaEventRecord(pipe.kernelDone[b], pipe.compute));
		CU(cudaStreamWaitEvent(pipe.copy, pipe.kernelDone[b], 0));
		if (verbose) cudaEventRecord(tev[4 * c + 2], pipe.copy);
		CU(cudaMemcpy2DAsync(hostOut + t0, (size_t)sampleCount * sizeof(int16_t), pipe.stage[b].p,
		                     stride * sizeof(int16_t), (size_t)len * sizeof(int16_t), n, cudaMemcpyDeviceToHost, pipe.copy));
		CU(cudaMemcpyAsync(hostRes + (size_t)b * n, pipe.res[b].p, sizeof(StreamResult) * (size_t)n,
		                   cudaMemcpyDeviceToHost, pipe.copy));
		if (verbose) cudaEventRecord(tev[4 * c + 3], pipe.copy);
		CU(cudaEventRecord(pipe.copyDone[b], pipe.copy));
		// (the kernel that reuses staging buffer b is chunk c+2: harvest(c) above has waited for this copy on the host by
		// then, so the compute stream needs no wait of its own -- and chunk c+1 must NOT wait for it)
		if (verbose) fprintf(stderr, "[renderToHost] chunk %u/%u len %u: t=%.2f ms, waited %.2f ms for chunk-2, enqueue %.2f ms\n", c, numChunks, len,
		                     tA - tStart, tB - tA, now() - tB);
	}
	for (uint32_t c = (numChunks >= 2 ? numChunks - 2 : 0); c < numChunks; ++c)
		if (!harvest(c)) return -1;
	if (verbose) {
		fprintf(stderr, "[renderToHost] done at t=%.2f ms\n", now() - tStart);
		for (uint32_t c = 0; c < numChunks; ++c) {
			float k0, k1, c0, c1;
			cudaEventElapsedTime(&k0, tev[0], tev[4 * c + 0]); cudaEventElapsedTime(&k1, tev[0], tev[4 * c + 1]);
			cudaEventElapsedTime(&c0, tev[0], tev[4 * c + 2]); cudaEventElapsedTime(&c1, tev[0], tev[4 * c + 3]);
			fprintf(stderr, "[renderToHost]   chunk %u: kernel %.2f..%.2f ms, copy %.2f..%.2f ms\n", c, k0, k1, c0, c1);
		}
		for (auto &e : tev) cudaEventDestroy(e);
	}
	long long sum = 0;
	for (uint32_t s = 0; s < n; ++s) {
		sum += total[s];
		if (perStream) perStream[s] = total[s];
	}
	return sum;
}

}  // namespace klatt
