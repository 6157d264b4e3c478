// Host side of the B200-native Klatt engine: the C-ABI of include/speechPlayer.h and
// include/speechPlayer_batch.h, the handle table, per-player request mirrors, device buffers and launches.
//
// Mapping to the reference (paths relative to the reference checkout):
//   speechPlayer_handleInfo_t + the five exports   src/speechPlayer.cpp:19-53   -> Player, speechPlayer_*()
//   FrameManagerImpl::queueFrame (copy-in, purge)   src/frame.cpp:90-115         -> Player::queue(): the host keeps
//        the not-yet-consumed requests (a purge drops them here); the state-machine half of purge
//        (sampleCounter / snapshot of curFrame, :105-111) runs as the prologue of the next launch
//   LockableObject (queueFrame vs synthesize)        src/lock.h:25-53             -> Player::mu
//   the per-sample loop                              src/speechWaveGenerator.cpp:197-214 -> klatt_f64.cu / klatt_f32.cu
//   SPEECHPLAYER_PRECISION_STREAM handles: the whole FrameManagerImpl runs on the host at request granularity
//        (pull_manager.h) and one pull is one launch of the time-parallel block kernel (klatt_pull.cu)
//
// There is no CPU synthesis path in this library: every sample comes out of a CUDA kernel.
#include <cuda_runtime.h>
#include <chrono>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/speechPlayer.h"
#include "../../include/speechPlayer_batch.h"
#include "glibc_rand.h"
#include "klatt_common.h"
#include "pull_manager.h"
#include "host_pool.h"
#include "klatt_long_phase.cuh"

namespace klatt {
cudaError_t launchKlattF64(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream);
cudaError_t launchKlattF32(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream);
cudaError_t launchKlattF32Rounds(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                 uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride,
                                 uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise, uint32_t *listHold,
                                 uint32_t *listGen, uint32_t *counters, int16_t *scratchRow, cudaStream_t stream, uint32_t numGroups,
                                 cudaStream_t *lanes, cudaEvent_t evStart, cudaEvent_t *evFork, cudaEvent_t *evJoin,
                                 unsigned long long *launchCounter);
cudaError_t launchKlattF32Sched(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride, uint32_t *samplesWritten,
                                StreamResult *results, NoiseConfig noise, uint32_t *ring, uint32_t ringCap, void *ctlMem,
                                int16_t *scratchRow, uint32_t numBlocks, uint32_t *hostFault, void *liteMem, uint32_t holdMax,
                                uint32_t fadeTicks, uint32_t fadeMax, uint32_t roleSms, cudaStream_t stream, unsigned long long *launchCounter);
int klattF32SchedBlocksPerSm();
bool klattF32SchedUsesLite();
size_t klattF32SchedLiteBytes(uint32_t numStreams, uint32_t numBlocks);
cudaError_t launchKlattF32Block(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount, uint32_t holdTicks,
                                int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise,
                                void *liteMem, int16_t *scratchRow, uint32_t numBlocks, void *profMem, uint32_t *hostFault,
                                cudaStream_t stream, unsigned long long *launchCounter);
bool klattF32BlockCanTake(uint32_t numStreams, uint32_t numBlocks);
size_t klattF32BlockLiteBytes(uint32_t numStreams, uint32_t numBlocks);
cudaError_t launchKlattPlan(const int64_t *offsets, uint32_t numStreams, uint64_t totalRequests, const double *frames,
                            const uint32_t *fadeDur, const uint8_t *isNull, int sampleRate, FadePlanF32 *plans,
                            cudaStream_t stream);
struct LongStream {  // klatt_long.cu
	const double *frames;
	const uint32_t *minDur, *fadeDur;
	const uint8_t *isNull;
	const FadePlanF32 *plans;
	uint32_t nReq;
	int sampleRate;
	uint64_t seed, streamId;
	uint64_t cap, outBase;
	uint64_t *start;
	int32_t *prevReal;
	double *pitchPop;
	double *pitchOld, *pitchNew, *pitchInc;
	uint64_t *vibPosStart;
};
struct Affine {
	float p00, p01, p10, p11, zy, zd;
};
cudaError_t launchKlattPullInit(PullState *state, cudaStream_t stream);  // klatt_pull.cu
cudaError_t launchKlattPull(PullCtx ctx, const PullSeg *segSrc, int16_t *pcmOut, cudaStream_t stream);
cudaError_t launchKlattPullBatch(PullBatchItem *hItems, const PullBatchItem *dItems, uint32_t count, cudaStream_t stream);
struct LongTable {
	const LongStream *streams;
	const uint32_t *chunkBase;
	uint32_t numStreams;
	LongStream one;
};
cudaError_t launchKlattLongTimeline(const LongTable &T, cudaStream_t stream);
cudaError_t launchKlattLongPhase(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, uint64_t *advance, uint64_t *startPhase,
                                 PhaseChunk *chunks, double *startP, uint32_t *fail, bool serial, unsigned long long *launchCounter,
                                 cudaStream_t stream);
cudaError_t launchKlattLongSynth(const LongTable &T, uint32_t numChunks, uint32_t chunkTicks, const PhaseChunk *chunks,
                                 const double *startP, uint32_t *fail, float *ci, float *pin, float *par, float *xa, float *xb,
                                 Affine *maps, float2 *startState, void *scanScratch, int16_t *pcm, unsigned long long *launchCounter,
                                 cudaStream_t stream);
size_t klattLongScanScratchBytes(uint64_t numChunks);
}  // namespace klatt

using namespace klatt;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_lastError;

namespace klatt {
void setLastError(const char *what);  // also used by the host-only translation units (ipa_frames.cpp)
}
static int fail(const std::string &what) {
	g_lastError = what;
	if (getenv("NVSP_VERBOSE")) fprintf(stderr, "[nvspeechplayer_b200] %s\n", what.c_str());
	return -1;
}
void klatt::setLastError(const char *what) { fail(what ? what : "error"); }

static bool cudaOk(cudaError_t e, const char *what) {
	if (e == cudaSuccess) return true;
	fail(std::string(what) + ": " + cudaGetErrorString(e));
	return false;
}
#define CU(call) do { if (!cudaOk((call), #call)) return -1; } while (0)
#define CUP(call) do { if (!cudaOk((call), #call)) return nullptr; } while (0)

// ------------------------------------------------------------------------------------------------
// device selection: the calling thread's current device, unless NVSP_DEVICE says otherwise (applied once)
// ------------------------------------------------------------------------------------------------
static int pickDevice() {
	static std::once_flag once;
	static int chosen = -1;
	std::call_once(once, [] {
		const char *e = getenv("NVSP_DEVICE");
		if (e && *e) chosen = atoi(e);
	});
	int dev = 0;
	if (chosen >= 0) {
		if (cudaSetDevice(chosen) != cudaSuccess) return -1;
		return chosen;
	}
	if (cudaGetDevice(&dev) != cudaSuccess) return -1;
	return dev;
}

struct DeviceGuard {
	int prev = -1;
	explicit DeviceGuard(int dev) {
		cudaGetDevice(&prev);
		if (prev != dev) cudaSetDevice(dev);
		else prev = -1;
	}
	~DeviceGuard() {
		if (prev >= 0) cudaSetDevice(prev);
	}
};

// grow-only device buffer
struct DevBuf {
	void *p = nullptr;
	size_t cap = 0;
	bool reserve(size_t bytes) {
		if (bytes <= cap) return true;
		size_t want = std::max(bytes, cap * 2);
		void *np = nullptr;
		if (!cudaOk(cudaMalloc(&np, want), "cudaMalloc")) return false;
		if (p) cudaFree(p);
		p = np; cap = want;
		return true;
	}
	void release() {
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
	}
	template <class T> T *as() const { return static_cast<T *>(p); }
};

// ------------------------------------------------------------------------------------------------
// small device kernels of the host layer
// ------------------------------------------------------------------------------------------------
__global__ void init_states_kernel(StreamState *states, uint32_t n) {
	// the state speechPlayer_initialize leaves a player in: src/frame.cpp:85-88 (curFrame zeroed, curFrameIsNULL,
	// sampleCounter 0, lastUserIndex -1, old request = zeroed NULL request), src/speechWaveGenerator.cpp:37,49,
	// 104-110 (phases, noise memory and resonator histories zero).  The memset before this kernel did the zeros.
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	states[i].fm.lastUserIndex = -1;
	states[i].fm.curIsNull = 1;
	states[i].fm.oldIsNull = 1;
}

// reference nvdaAddon/synthDrivers/nvSpeechPlayer/__init__.py:117-125 (applyVoiceToFrame), one thread per frame value
__global__ void apply_voices_kernel(double *frames, const int64_t *offsets, const uint8_t *isNull, const double *voiceAbs,
                                    const double *voiceMul, const uint32_t *voiceOfStream, uint32_t numVoices, uint32_t numStreams) {
	const uint32_t s = blockIdx.y;
	const int64_t a = offsets[s], b = offsets[s + 1];
	const uint32_t v = voiceOfStream ? voiceOfStream[s] % numVoices : s % numVoices;
	const int64_t cells = (b - a) * kNumParams;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (int64_t)gridDim.x * blockDim.x) {
		const int64_t row = a + i / kNumParams;
		const int p = (int)(i % kNumParams);
		if (isNull && isNull[row]) continue;
		const double ab = voiceAbs[(size_t)v * kNumParams + p];
		const double cur = frames[(size_t)row * kNumParams + p];
		frames[(size_t)row * kNumParams + p] = ((ab != ab) ? cur : ab) * voiceMul[(size_t)v * kNumParams + p];
	}
}

__global__ void build_descs_kernel(StreamDesc *descs, StreamState *states, const int64_t *offsets, const double *frames,
                                   const uint32_t *minDur, const uint32_t *fadeDur, const int32_t *userIndex,
                                   const uint8_t *isNull, const int32_t *replay, uint64_t drawsPerStream,
                                   const uint64_t *streamIds, const FadePlanF32 *plans, uint32_t n) {
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i > n) return;
	StreamDesc d;
	// entry n is the dummy stream (fresh state, empty queue) that idle lanes of the paired kernels run
	int64_t a = (offsets && i < n) ? offsets[i] : 0, b = (offsets && i < n) ? offsets[i + 1] : 0;
	d.state = states + i;
	d.frames = frames ? frames + (size_t)a * kNumParams : nullptr;
	d.minDur = minDur ? minDur + a : nullptr;
	d.fadeDur = fadeDur ? fadeDur + a : nullptr;
	d.userIndex = userIndex ? userIndex + a : nullptr;
	d.isNull = isNull ? isNull + a : nullptr;
	d.replay = (replay && i < n) ? replay + (size_t)i * drawsPerStream : nullptr;
	d.replayLen = (replay && i < n) ? drawsPerStream : 0;
	d.replayBase = 0;
	d.streamId = (streamIds && i < n) ? streamIds[i] : i;
	d.qCount = (uint32_t)(b - a);
	d.qBase = 0;
	d.plans = plans ? plans + a : nullptr;
	descs[i] = d;
}

// Scratch and second stream for round-based FP32 rendering (klatt_f32.cu "rounds"); owned by a batch or a pipe.
struct RoundsCtx {
	static constexpr uint32_t kMaxGroups = 8;
	DevBuf listHold, listGen, counters, scratchRow;
	DevBuf ring, ctl;            // stream scheduler (persistent kernel, klatt_f32_sched.cu)
	bool persistent = true;      // NVSP_SCHED=rounds selects the round-based launch sequence instead
	// block scheduler (klatt_f32_block.cu), NVSP_SCHED=block: an experiment of round 2 that is correct (bit-identical, tested) but
	// slower than the ring scheduler -- its code does not fit the SM's 32 KB instruction cache (DESIGN.md section 5c)
	DevBuf lite, blockProf;
	bool blockSched = false;
	uint32_t blockHoldTicks = 128, blockMinStreams = 16384, blockBlocks = 0;
	uint32_t *hostFault = nullptr;  // pinned: the scheduler watchdog's verdict of the last call
	uint32_t schedHoldTicks = 256, schedGenTicks = 384, schedHoldMax = 4096, schedFadeTicks = 0, schedFadeMax = 512, schedRoleSms = 0, schedBlocks = 0;
	cudaStream_t lanes[2 * kMaxGroups] = {};
	cudaEvent_t evStart = nullptr, evFork[kMaxGroups] = {}, evJoin[kMaxGroups] = {};
	uint32_t holdTicks = 512, genTicks = 256, minStreams = 2048, groups = 4;
	bool ok = false;
	bool init() {
		if (ok) return true;
		auto envU = [](const char *name, uint32_t dflt) {
			const char *e = getenv(name);
			return (e && *e) ? (uint32_t)strtoul(e, nullptr, 0) : dflt;
		};
		// chunk lengths are multiples of 64: the coarse pole re-basing and the Philox block cadence stay warp-uniform,
		// and every chunk starts on a 16-byte boundary of its output row
		genTicks = std::max<uint32_t>(envU("NVSP_GEN_TICKS", 256) & ~63u, 64);
		holdTicks = std::max<uint32_t>(envU("NVSP_HOLD_TICKS", 512) & ~63u, 64);
		minStreams = envU("NVSP_ROUNDS_MIN_STREAMS", 2048);
		groups = std::min<uint32_t>(std::max<uint32_t>(envU("NVSP_GROUPS", 4), 1), kMaxGroups);
		{
			const char *e = getenv("NVSP_SCHED");
			persistent = !(e && strcmp(e, "rounds") == 0);
			blockSched = e && strcmp(e, "block") == 0;
			blockHoldTicks = std::max<uint32_t>(envU("NVSP_BLOCK_HOLD_TICKS", 128) & ~63u, 64);
			blockMinStreams = envU("NVSP_BLOCK_MIN_STREAMS", 16384);
			// (round 1, AoS state with L1-bypassing loads: 512 / 640 was the optimum; with the compact staged records a change of
			// loop is cheaper and the optimum is a flat basin around 256 / 384: 200.2 ms vs 207.9 ms at 512 / 640)
			schedGenTicks = std::max<uint32_t>(envU("NVSP_SCHED_GEN_TICKS", 384) & ~63u, 64);
			schedHoldTicks = std::max<uint32_t>(envU("NVSP_SCHED_HOLD_TICKS", 256) & ~63u, 64);
			// a hold chunk whose 32 streams can all hold longer runs up to this many ticks (steady vowels, sung notes; measured
			// 256 -> 4096: config 2 292 -> 278 ms, config 5 163 -> 155 ms, config 3 unchanged)
			schedHoldMax = std::max<uint32_t>(envU("NVSP_SCHED_HOLD_MAX", 4096) & ~63u, schedHoldTicks);
			// the fade class (0: off): streams with this many interior fade ticks ahead on the 64-sample grid take the straight-line
			// fade loop; chunks stretched up to NVSP_SCHED_FADE_MAX.  NVSP_SCHED_HOLD_SMS / NVSP_SCHED_FADE_SMS: that many SMs take
			// hold / fade chunks first, the rest general chunks (SM roles: one loop pair per instruction cache)
			schedFadeTicks = envU("NVSP_SCHED_FADE_TICKS", 0) & ~63u;
			schedFadeMax = std::min<uint32_t>(std::max<uint32_t>(envU("NVSP_SCHED_FADE_MAX", 512) & ~63u, schedFadeTicks), 4096);
			schedRoleSms = std::min<uint32_t>(envU("NVSP_SCHED_HOLD_SMS", 0), 255u) | (std::min<uint32_t>(envU("NVSP_SCHED_FADE_SMS", 0), 255u) << 8);
			int dev = 0, sms = 0;
			cudaGetDevice(&dev);
			cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
			const int perSm = klattF32SchedBlocksPerSm();
			schedBlocks = envU("NVSP_SCHED_BLOCKS", (uint32_t)(sms * std::max(perSm, 1)));
			blockBlocks = std::max<uint32_t>(envU("NVSP_BLOCK_BLOCKS", (uint32_t)sms), 1);
			if (getenv("NVSP_VERBOSE"))
				fprintf(stderr, "[nvspeechplayer_b200] scheduler: %d SMs x %d blocks, %u blocks, hold %u / general %u ticks\n", sms, perSm,
				        schedBlocks, schedHoldTicks, schedGenTicks);
		}
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
	void destroy() {
		listHold.release(); listGen.release(); counters.release(); scratchRow.release(); ring.release(); ctl.release();
		lite.release(); blockProf.release();
		if (hostFault) cudaFreeHost(hostFault);
		hostFault = nullptr;
		if (evStart) cudaEventDestroy(evStart);
		for (uint32_t g = 0; g < kMaxGroups; ++g) {
			if (evFork[g]) cudaEventDestroy(evFork[g]);
			if (evJoin[g]) cudaEventDestroy(evJoin[g]);
			if (lanes[2 * g]) cudaStreamDestroy(lanes[2 * g]);
			if (lanes[2 * g + 1]) cudaStreamDestroy(lanes[2 * g + 1]);
			evFork[g] = evJoin[g] = nullptr;
			lanes[2 * g] = lanes[2 * g + 1] = nullptr;
		}
		evStart = nullptr;
		ok = false;
	}
};

// planned: the descriptors carry precomputed fade plans (pre-queued batches) -> FP32 renders may run as rounds
static cudaError_t launchRender(int precision, const StreamDesc *descs, uint32_t n, int sampleRate, uint32_t sampleCount,
                                int16_t *out, size_t rowStride, uint32_t *written, StreamResult *results,
                                NoiseConfig noise, cudaStream_t stream, RoundsCtx *rc = nullptr, bool planned = false,
                                unsigned long long *launchCounter = nullptr) {
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
		if (!rc->hostFault) {
			if (cudaMallocHost((void **)&rc->hostFault, sizeof(uint32_t)) != cudaSuccess) return cudaErrorMemoryAllocation;
			*rc->hostFault = 0;
		}
		if (*rc->hostFault) return cudaErrorLaunchTimeout;  // an earlier call of this batch tripped the watchdog
		return launchKlattF32Block(descs, n, sampleRate, sampleCount, rc->blockHoldTicks, out, rowStride, written, results, noise,
		                           rc->lite.p, rc->scratchRow.as<int16_t>(), rc->blockBlocks, rc->blockProf.p, rc->hostFault, stream,
		                           launchCounter);
	}
	if (rc && planned && rc->init() && rc->persistent && n >= rc->minStreams && sampleCount > rc->schedGenTicks) {
		uint32_t cap = 64;
		while (cap < 2 * n) cap <<= 1;
		if (!rc->hostFault) {
			if (cudaMallocHost((void **)&rc->hostFault, sizeof(uint32_t)) != cudaSuccess) return cudaErrorMemoryAllocation;
			*rc->hostFault = 0;
		}
		if (*rc->hostFault) return cudaErrorLaunchTimeout;  // an earlier call of this batch tripped the watchdog
		if (!rc->ring.reserve(sizeof(uint32_t) * 3 * (size_t)cap) || !rc->ctl.reserve(2048) ||
		    !rc->scratchRow.reserve(sizeof(int16_t) * (size_t)std::max(std::max(std::max(rc->schedHoldTicks, rc->schedHoldMax), rc->holdTicks), rc->schedFadeMax)))
			return cudaErrorMemoryAllocation;
		if (klattF32SchedUsesLite() && !rc->lite.reserve(klattF32SchedLiteBytes(n, rc->schedBlocks))) return cudaErrorMemoryAllocation;
		return launchKlattF32Sched(descs, n, sampleRate, sampleCount, rc->schedHoldTicks, rc->schedGenTicks, out, rowStride, written,
		                           results, noise, rc->ring.as<uint32_t>(), cap, rc->ctl.p, rc->scratchRow.as<int16_t>(),
		                           rc->schedBlocks, rc->hostFault, rc->lite.p, rc->schedHoldMax, rc->schedFadeTicks, rc->schedFadeMax, rc->schedRoleSms, stream,
		                           launchCounter);
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

static cudaError_t initStates(StreamState *states, uint32_t n, cudaStream_t stream) {
	cudaError_t e = cudaMemsetAsync(states, 0, sizeof(StreamState) * (size_t)n, stream);
	if (e != cudaSuccess) return e;
	init_states_kernel<<<(n + 255) / 256, 256, 0, stream>>>(states, n);
	return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Chunked render into HOST memory: kernel(chunk c) overlaps the D2H copy of chunk c-1 (two staging buffers,
// compute stream + copy stream).  hostOut is [n][sampleCount]; rows are gathered with a 2-D copy.
// ------------------------------------------------------------------------------------------------
struct HostPipe {
	cudaStream_t compute = nullptr, copy = nullptr;
	cudaEvent_t kernelDone[2] = {nullptr, nullptr}, copyDone[2] = {nullptr, nullptr};
	DevBuf stage[2], res[2];
	RoundsCtx rounds;
	StreamResult *hostRes = nullptr;  // pinned, [2][n]
	size_t hostResCap = 0;
	bool ok = false;
	bool init() {
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
	void destroy() {
		if (!ok) return;
		for (int i = 0; i < 2; ++i) {
			stage[i].release(); res[i].release();
			cudaEventDestroy(kernelDone[i]); cudaEventDestroy(copyDone[i]);
		}
		rounds.destroy();
		if (hostRes) cudaFreeHost(hostRes);
		cudaStreamDestroy(compute); cudaStreamDestroy(copy);
		ok = false;
	}
};

static size_t stagingBudgetBytes() {
	const char *e = getenv("NVSP_STAGE_MB");
	size_t mb = (e && *e) ? (size_t)atoll(e) : 2048;  // measured on B200 (config 3 e2e): 1024 -> 674 ms, 2048 -> 640 ms, 4096 -> 640 ms per step
	return std::max<size_t>(mb, 1) << 20;
}

// returns total samples written, or -1.  perStream (host, [n]) and lastResults (host, [n]) are optional outputs.
static long long renderToHost(HostPipe &pipe, int precision, const StreamDesc *dDescs, uint32_t n, int sampleRate,
                              uint32_t sampleCount, int16_t *hostOut, uint32_t *perStream, StreamResult *lastResults,
                              NoiseConfig noise, unsigned long long *launchCounter, bool planned = false) {
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
	if (pipe.hostResCap < (size_t)n * 2) {
		if (pipe.hostRes) cudaFreeHost(pipe.hostRes);
		pipe.hostRes = nullptr;
		if (!cudaOk(cudaMallocHost((void **)&pipe.hostRes, sizeof(StreamResult) * (size_t)n * 2), "cudaMallocHost")) return -1;
		pipe.hostResCap = (size_t)n * 2;
	}
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
	const bool verbose = getenv("NVSP_VERBOSE") != nullptr;
	auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	const double tStart = now();
	auto harvest = [&](uint32_t c) -> bool {  // wait for chunk c's copies and fold its results
		int b = c & 1;
		if (!cudaOk(cudaEventSynchronize(pipe.copyDone[b]), "cudaEventSynchronize")) return false;
		const StreamResult *r = pipe.hostRes + (size_t)b * n;
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
		CU(cudaMemcpyAsync(pipe.hostRes + (size_t)b * n, pipe.res[b].p, sizeof(StreamResult) * (size_t)n,
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

// ------------------------------------------------------------------------------------------------
// process-global glibc-compatible noise (reference: libc rand() shared by every player)
// ------------------------------------------------------------------------------------------------
static std::mutex g_noiseMu;
static GlibcRand g_noise;

// ------------------------------------------------------------------------------------------------
// Player: one reference "speechPlayer_handleInfo_t"
// ------------------------------------------------------------------------------------------------
struct Player {
	std::mutex mu;
	int device = 0, sampleRate = 0, precision = kPrecisionF64, noiseMode = kNoiseGlibc;
	uint64_t seed = 0, streamId = 0;
	StreamState *dState = nullptr;
	// host mirror of the requests the device has not consumed yet (src/frame.cpp:33 frameRequestQueue)
	std::vector<double> frames;
	std::vector<uint32_t> minDur, fadeDur;
	std::vector<int32_t> userIndex;
	std::vector<uint8_t> isNull;
	uint32_t qBase = 0;       // absolute index of mirror[0] == requests consumed so far
	bool mirrorDirty = false; // device copy of the mirror is stale
	bool purgePending = false;
	DevBuf dFrames, dMin, dFade, dUix, dNull, dReplay, dDesc;
	std::vector<int32_t> replayHost;  // kNoiseReplay: user-provided draws
	bool replayDirty = false;
	uint64_t generated = 0;   // samples generated so far (== draws/2)
	int lastIndex = -1;
	HostPipe pipe;
	std::vector<int16_t> hostScratch;  // rows of the last synthesize call before the written prefixes are handed out
	// SPEECHPLAYER_PRECISION_STREAM: host frame manager, carried device state, staging for one launch
	PullManager *pull = nullptr;
	PullState *dPull = nullptr;
	DevBuf dSegs, dPullPcm, dDraws, dPullDbg;
	unsigned char *hPullStage = nullptr;  // pinned and mapped: [segments | pcm | draws]
	unsigned char *dPullStage = nullptr;  // the same memory as the device sees it (zero-copy)
	std::vector<PullSeg> pullSegs;
	uint64_t pullLaunches = 0;
	static constexpr size_t kStageSegs = sizeof(PullSeg) * kPullMaxSegs, kStagePcm = sizeof(int16_t) * kPullMaxTicks,
	                        kStageDraws = sizeof(int32_t) * 2 * kPullMaxTicks;

	size_t pending() const { return minDur.size(); }

	void push(const speechPlayer_frame_t *frame, unsigned m, unsigned f, int ux, bool null) {
		size_t at = frames.size();
		frames.resize(at + kNumParams, 0.0);
		if (frame && !null) memcpy(&frames[at], frame, sizeof(double) * kNumParams);
		minDur.push_back(m);
		fadeDur.push_back(f);
		userIndex.push_back(ux);
		isNull.push_back((null || !frame) ? 1 : 0);
		mirrorDirty = true;
	}
	void clearQueue() {
		frames.clear(); minDur.clear(); fadeDur.clear(); userIndex.clear(); isNull.clear();
		mirrorDirty = true;
	}
	void dropConsumed(uint32_t newHead) {
		uint32_t k = newHead - qBase;
		if (k == 0) return;
		k = (uint32_t)std::min<size_t>(k, pending());
		frames.erase(frames.begin(), frames.begin() + (size_t)k * kNumParams);
		minDur.erase(minDur.begin(), minDur.begin() + k);
		fadeDur.erase(fadeDur.begin(), fadeDur.begin() + k);
		userIndex.erase(userIndex.begin(), userIndex.begin() + k);
		isNull.erase(isNull.begin(), isNull.begin() + k);
		qBase = newHead;
		mirrorDirty = true;
	}
	// upload what changed and fill the descriptor for the next launch (on `stream`)
	int prepare(StreamDesc &d, uint32_t sampleCount, cudaStream_t stream) {
		if (mirrorDirty) {
			size_t n = pending();
			if (n) {
				if (!dFrames.reserve(n * kNumParams * sizeof(double)) || !dMin.reserve(n * 4) || !dFade.reserve(n * 4) ||
				    !dUix.reserve(n * 4) || !dNull.reserve(n))
					return -1;
				CU(cudaMemcpyAsync(dFrames.p, frames.data(), n * kNumParams * sizeof(double), cudaMemcpyHostToDevice, stream));
				CU(cudaMemcpyAsync(dMin.p, minDur.data(), n * 4, cudaMemcpyHostToDevice, stream));
				CU(cudaMemcpyAsync(dFade.p, fadeDur.data(), n * 4, cudaMemcpyHostToDevice, stream));
				CU(cudaMemcpyAsync(dUix.p, userIndex.data(), n * 4, cudaMemcpyHostToDevice, stream));
				CU(cudaMemcpyAsync(dNull.p, isNull.data(), n, cudaMemcpyHostToDevice, stream));
			}
			mirrorDirty = false;
		}
		if (purgePending) {
			static const uint32_t one = 1;
			CU(cudaMemcpyAsync(&dState->fm.purgePending, &one, 4, cudaMemcpyHostToDevice, stream));
			purgePending = false;
		}
		d.state = dState;
		d.frames = dFrames.as<double>();
		d.minDur = dMin.as<uint32_t>();
		d.fadeDur = dFade.as<uint32_t>();
		d.userIndex = dUix.as<int32_t>();
		d.isNull = dNull.as<uint8_t>();
		d.qCount = (uint32_t)pending();
		d.qBase = qBase;
		d.streamId = streamId;
		d.plans = nullptr;  // per-handle queues grow and get purged: fades are planned inline at the pop tick
		d.replay = nullptr; d.replayLen = 0; d.replayBase = 0;
		if (noiseMode == kNoiseGlibc) {
			// draws for the worst case (every tick generates); the caller rewinds the generator afterwards
			size_t n = (size_t)sampleCount * 2;
			std::vector<int32_t> draws(n);
			g_noise.fill(draws.data(), n);
			if (!dReplay.reserve(n * 4)) return -1;
			CU(cudaMemcpyAsync(dReplay.p, draws.data(), n * 4, cudaMemcpyHostToDevice, stream));
			CU(cudaStreamSynchronize(stream));  // `draws` dies at scope exit
			d.replay = dReplay.as<int32_t>(); d.replayLen = n; d.replayBase = generated * 2;
		} else if (noiseMode == kNoiseReplay) {
			if (replayDirty) {
				if (!dReplay.reserve(std::max<size_t>(replayHost.size(), 1) * 4)) return -1;
				CU(cudaMemcpyAsync(dReplay.p, replayHost.data(), replayHost.size() * 4, cudaMemcpyHostToDevice, stream));
				replayDirty = false;
			}
			d.replay = dReplay.as<int32_t>(); d.replayLen = replayHost.size(); d.replayBase = 0;
		}
		return 0;
	}
	void absorb(const StreamResult &r, uint32_t written) {
		generated += written;
		lastIndex = r.lastUserIndex;
		dropConsumed(r.qHead);
	}
	void destroy() {
		DeviceGuard g(device);
		pipe.destroy();
		dFrames.release(); dMin.release(); dFade.release(); dUix.release(); dNull.release(); dReplay.release(); dDesc.release();
		dSegs.release(); dPullPcm.release(); dDraws.release(); dPullDbg.release();
		if (hPullStage) cudaFreeHost(hPullStage);
		hPullStage = nullptr;
		if (dPull) cudaFree(dPull);
		dPull = nullptr;
		delete pull;
		pull = nullptr;
		if (dState) cudaFree(dState);
		dState = nullptr;
	}
};

// handle table: handles are small integers (index+1) cast to void*, so they survive a round trip through a C int
static std::mutex g_tableMu;
static std::vector<Player *> g_players;

static Player *lookup(speechPlayer_handle_t h) {
	uintptr_t v = reinterpret_cast<uintptr_t>(h);
	std::lock_guard<std::mutex> lk(g_tableMu);
	if (v == 0 || v > g_players.size()) return nullptr;
	return g_players[v - 1];
}

static int envPrecision() {
	const char *e = getenv("NVSP_PRECISION");
	if (e && (!strcmp(e, "fp32") || !strcmp(e, "f32") || !strcmp(e, "FP32"))) return kPrecisionF32;
	if (e && (!strcmp(e, "stream") || !strcmp(e, "pull"))) return kPrecisionStream;
	return kPrecisionF64;
}
static int envNoise() {
	const char *e = getenv("NVSP_NOISE");
	if (e && !strcmp(e, "philox")) return kNoisePhilox;
	return kNoiseGlibc;
}
static uint64_t envSeed() {
	const char *e = getenv("NVSP_SEED");
	return (e && *e) ? strtoull(e, nullptr, 0) : 0xB200ull;
}

// ------------------------------------------------------------------------------------------------
// C-ABI: per-handle API
// ------------------------------------------------------------------------------------------------
extern "C" {

const char *speechPlayer_lastError(void) { return g_lastError.c_str(); }
const char *speechPlayer_version(void) { return "nvspeechplayer_b200 0.1 sm_100a"; }

speechPlayer_handle_t speechPlayer_initializeEx(int sampleRate, int precision, int noiseMode, uint64_t seed,
                                                uint64_t streamId) {
	g_lastError.clear();
	if (sampleRate <= 0) { fail("sampleRate must be positive"); return nullptr; }
	if (precision != kPrecisionF64 && precision != kPrecisionF32 && precision != kPrecisionStream) {
		fail("unknown precision");
		return nullptr;
	}
	if (noiseMode < kNoisePhilox || noiseMode > kNoiseReplay) { fail("unknown noise mode"); return nullptr; }
	int dev = pickDevice();
	if (dev < 0) { fail("no usable CUDA device (this library has no CPU fallback)"); return nullptr; }
	Player *p = new Player;
	p->device = dev; p->sampleRate = sampleRate; p->precision = precision; p->noiseMode = noiseMode;
	p->seed = seed; p->streamId = streamId;
	DeviceGuard g(dev);
	if (!cudaOk(cudaMalloc((void **)&p->dState, sizeof(StreamState)), "cudaMalloc(state)") ||
	    !cudaOk(initStates(p->dState, 1, nullptr), "init state") ||
	    !cudaOk(cudaStreamSynchronize(nullptr), "init state sync")) {
		delete p;
		return nullptr;
	}
	if (precision == kPrecisionStream) {
		p->pull = new PullManager(sampleRate);
		if (!cudaOk(cudaMalloc((void **)&p->dPull, sizeof(PullState)), "cudaMalloc(pull state)") ||
		    !cudaOk(launchKlattPullInit(p->dPull, nullptr), "init pull state") ||
		    !cudaOk(cudaStreamSynchronize(nullptr), "init pull state sync") ||
		    !cudaOk(cudaHostAlloc((void **)&p->hPullStage, Player::kStageSegs + Player::kStagePcm + Player::kStageDraws,
		                          cudaHostAllocMapped), "cudaHostAlloc(pull staging)") ||
		    !cudaOk(cudaHostGetDevicePointer((void **)&p->dPullStage, p->hPullStage, 0), "cudaHostGetDevicePointer") ||
		    !p->dSegs.reserve(Player::kStageSegs) || !p->dPullPcm.reserve(Player::kStagePcm)) {
			p->destroy();
			delete p;
			return nullptr;
		}
	}
	std::lock_guard<std::mutex> lk(g_tableMu);
	for (size_t i = 0; i < g_players.size(); ++i)
		if (!g_players[i]) {
			g_players[i] = p;
			return reinterpret_cast<speechPlayer_handle_t>(i + 1);
		}
	g_players.push_back(p);
	return reinterpret_cast<speechPlayer_handle_t>(g_players.size());
}

speechPlayer_handle_t speechPlayer_initialize(int sampleRate) {
	// Philox stream ids of the five-symbol API come from a process-wide counter, not from the handle table: slots are reused
	// after terminate, and two live players must never share (seed, streamId)
	static std::atomic<uint64_t> nextStreamId{0};
	const uint64_t sid = nextStreamId.fetch_add(1);
	return speechPlayer_initializeEx(sampleRate, envPrecision(), envNoise(), envSeed(), sid);
}

void speechPlayer_queueFrame(speechPlayer_handle_t playerHandle, speechPlayer_frame_t *framePtr,
                             unsigned int minFrameDuration, unsigned int fadeDuration, int userIndex, bool purgeQueue) {
	Player *p = lookup(playerHandle);
	if (!p) return;
	std::lock_guard<std::mutex> lk(p->mu);
	if (p->pull) {
		p->pull->queueFrame(reinterpret_cast<const double *>(framePtr), minFrameDuration, fadeDuration, userIndex, purgeQueue);
		return;
	}
	if (purgeQueue) {  // src/frame.cpp:103-112: drop everything still queued; the rest happens on the device
		p->clearQueue();
		p->purgePending = true;
	}
	p->push(framePtr, minFrameDuration, fadeDuration, userIndex, framePtr == nullptr);
}

int speechPlayer_queueFrames(speechPlayer_handle_t playerHandle, const speechPlayer_frame_t *frames,
                             const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                             const int *userIndex, const unsigned char *isNull, unsigned int n) {
	Player *p = lookup(playerHandle);
	if (!p) return fail("bad handle");
	if (n && (!minFrameDuration || !fadeDuration)) return fail("durations missing");
	std::lock_guard<std::mutex> lk(p->mu);
	for (unsigned i = 0; i < n; ++i) {
		bool null = (isNull && isNull[i]) || !frames;
		if (p->pull) {
			p->pull->queueFrame(null ? nullptr : reinterpret_cast<const double *>(frames + i), minFrameDuration[i], fadeDuration[i],
			                    userIndex ? userIndex[i] : -1, false);
			continue;
		}
		p->push(frames ? frames + i : nullptr, minFrameDuration[i], fadeDuration[i], userIndex ? userIndex[i] : -1, null);
	}
	return 0;
}

int speechPlayer_setNoiseReplay(speechPlayer_handle_t playerHandle, const int32_t *draws, size_t numDraws) {
	Player *p = lookup(playerHandle);
	if (!p) return fail("bad handle");
	std::lock_guard<std::mutex> lk(p->mu);
	if (p->noiseMode != kNoiseReplay) return fail("handle was not created with SPEECHPLAYER_NOISE_REPLAY");
	p->replayHost.assign(draws, draws + numDraws);
	p->replayDirty = true;
	return 0;
}

void speechPlayer_seedNoise(unsigned int seed) {
	std::lock_guard<std::mutex> lk(g_noiseMu);
	g_noise.seed(seed);
}

// Stage one launch of a SPEECHPLAYER_PRECISION_STREAM player: the host manager has described the next `got` ticks in
// p->pullSegs (src/frame.cpp:41-80 in closed form); copy the segments into the player's pinned staging, fetch the noise draws,
// fill the launch context.  The kernel reads the segments from and writes the samples to the pinned staging itself
// (zero-copy, the default), so a pull is one launch and one synchronize; NVSP_PULL_ZEROCOPY=0 goes through device buffers.
static bool pullZeroCopy() {
	static const bool zc = !(getenv("NVSP_PULL_ZEROCOPY") && atoi(getenv("NVSP_PULL_ZEROCOPY")) == 0);
	return zc;
}
static bool pullDebugPhases() {
	static const bool dbg = getenv("NVSP_PULL_DEBUG") != nullptr;
	return dbg;
}
static int pullStage(Player *p, uint32_t got, PullCtx &X, const PullSeg *&segSrc, int16_t *&pcmOut, bool &zeroCopy, cudaStream_t stream) {
	zeroCopy = pullZeroCopy();
	PullSeg *hSegs = reinterpret_cast<PullSeg *>(p->hPullStage);
	int32_t *hDraws = reinterpret_cast<int32_t *>(p->hPullStage + Player::kStageSegs + Player::kStagePcm);
	if (p->noiseMode == kNoiseReplay && p->replayDirty) {
		if (!p->dReplay.reserve(std::max<size_t>(p->replayHost.size(), 1) * 4)) return -1;
		CU(cudaMemcpyAsync(p->dReplay.p, p->replayHost.data(), p->replayHost.size() * 4, cudaMemcpyHostToDevice, stream));
		CU(cudaStreamSynchronize(stream));
		p->replayDirty = false;
	}
	const size_t nSeg = p->pullSegs.size();
	memcpy(hSegs, p->pullSegs.data(), nSeg * sizeof(PullSeg));
	segSrc = reinterpret_cast<const PullSeg *>(p->dPullStage);
	pcmOut = reinterpret_cast<int16_t *>(p->dPullStage + Player::kStageSegs);
	if (!zeroCopy) {
		CU(cudaMemcpyAsync(p->dSegs.p, hSegs, nSeg * sizeof(PullSeg), cudaMemcpyHostToDevice, stream));
		segSrc = p->dSegs.as<PullSeg>();
		pcmOut = p->dPullPcm.as<int16_t>();
	}
	memset(&X, 0, sizeof X);
	X.nSeg = (uint32_t)nSeg; X.n = got; X.sampleRate = p->sampleRate;
	X.state = p->dPull; X.noiseMode = p->noiseMode; X.seed = p->seed; X.streamId = p->streamId;
	if (p->noiseMode == kNoiseGlibc) {  // the reference consumes exactly two rand() calls per generated sample
		{
			std::lock_guard<std::mutex> nl(g_noiseMu);
			g_noise.fill(hDraws, (size_t)got * 2);
		}
		if (!p->dDraws.reserve(Player::kStageDraws)) return -1;
		CU(cudaMemcpyAsync(p->dDraws.p, hDraws, (size_t)got * 2 * 4, cudaMemcpyHostToDevice, stream));
		X.draws = p->dDraws.as<int32_t>(); X.drawBase = p->generated * 2; X.drawLen = (uint64_t)got * 2;
	} else if (p->noiseMode == kNoiseReplay) {
		X.draws = p->dReplay.as<int32_t>(); X.drawBase = 0; X.drawLen = p->replayHost.size();
	}
	// the glottal-phase recurrence: run decomposition (klatt_pull_core.cuh pullRuns*; bit-identical to the serial loop,
	// 280 k -> 48 k cycles of an 8192-tick launch on B200) unless NVSP_PULL_PHASE=serial asks for the plain loop
	static const bool phaseSerial = getenv("NVSP_PULL_PHASE") && !strcmp(getenv("NVSP_PULL_PHASE"), "serial");
	X.phaseMode = phaseSerial ? 0 : 1;
	if (pullDebugPhases() && p->dPullDbg.reserve(16 * sizeof(long long))) X.dbg = p->dPullDbg.as<long long>();
	return 0;
}

// One pull of a SPEECHPLAYER_PRECISION_STREAM player: one launch of klatt_pull_kernel per kPullMaxTicks, the samples come back
// through pinned memory.
static long long synthesizePull(Player *p, unsigned int sampleCount, int16_t *out) {
	std::lock_guard<std::mutex> lk(p->mu);
	DeviceGuard g(p->device);
	if (!p->pipe.init()) return -1;
	cudaStream_t stream = p->pipe.compute;
	int16_t *hPcm = reinterpret_cast<int16_t *>(p->hPullStage + Player::kStageSegs);
	unsigned int total = 0;
	while (total < sampleCount) {
		const uint32_t want = std::min<uint32_t>(sampleCount - total, kPullMaxTicks);
		p->pullSegs.clear();
		bool drained = false;
		const uint32_t got = p->pull->advance(want, 0, kPullMaxSegs, p->pullSegs, drained);
		if (got) {
			PullCtx X;
			const PullSeg *segSrc;
			int16_t *pcmOut;
			bool zeroCopy;
			if (pullStage(p, got, X, segSrc, pcmOut, zeroCopy, stream) != 0) return -1;
			CU(launchKlattPull(X, segSrc, pcmOut, stream));
			if (!zeroCopy) CU(cudaMemcpyAsync(hPcm, pcmOut, (size_t)got * sizeof(int16_t), cudaMemcpyDeviceToHost, stream));
			CU(cudaStreamSynchronize(stream));
			memcpy(out + total, hPcm, (size_t)got * sizeof(int16_t));
			if (X.dbg) {  // SM cycles between the phase boundaries of the launch (tools/latency_probe.py reads these lines)
				long long c[16];
				CU(cudaMemcpy(c, X.dbg, sizeof c, cudaMemcpyDeviceToHost));
				fprintf(stderr, "[pull] n=%u segs=%zu cycles: src1 %lld noise-scan %lld phase %lld src2 %lld parallel %lld nasal %lld "
				        "r6-r2 %lld r1+out %lld total %lld in %lld ns\n", got, p->pullSegs.size(), c[1] - c[0], c[2] - c[1], c[3] - c[2], c[4] - c[3],
				        c[5] - c[4], c[6] - c[5], c[7] - c[6], c[8] - c[7], c[8] - c[0], c[14] - c[15]);
			}
			++p->pullLaunches;
			p->generated += got;
		}
		total += got;
		if (drained) break;
	}
	p->lastIndex = p->pull->lastIndex();
	return (long long)total;
}

// speechPlayer_synthesizeBatch over SPEECHPLAYER_PRECISION_STREAM handles: ONE launch per kPullMaxTicks for all players, one
// block per player (klatt_pull_batch_kernel) -- 148 interactive players at the latency of one.  Each row is what the player's
// own speechPlayer_synthesize would have produced (same kernel body, same carried state).  With the process-global glibc noise
// the players draw in handle order, as sequential calls would.
static std::mutex g_pullBatchMu;
static PullBatchItem *g_pullItemsHost = nullptr, *g_pullItemsDev = nullptr;
static size_t g_pullItemsCap = 0;
static int g_pullItemsDevice = -1;

static long long synthesizePullBatch(std::vector<Player *> &ps, unsigned int sampleCount, int16_t *out, unsigned int *samplesWritten) {
	const size_t n = ps.size();
	std::vector<Player *> order(ps);
	std::sort(order.begin(), order.end());
	for (Player *p : order) p->mu.lock();
	struct Unlock {
		std::vector<Player *> &o;
		~Unlock() { for (Player *p : o) p->mu.unlock(); }
	} unlock{order};
	std::lock_guard<std::mutex> bl(g_pullBatchMu);
	Player *lead = ps[0];
	DeviceGuard g(lead->device);
	if (!lead->pipe.init()) return -1;
	cudaStream_t stream = lead->pipe.compute;
	if (g_pullItemsCap < n || g_pullItemsDevice != lead->device) {
		if (g_pullItemsHost) cudaFreeHost(g_pullItemsHost);
		g_pullItemsHost = nullptr; g_pullItemsCap = 0;
		const size_t cap = std::max<size_t>(n, 256);
		CU(cudaHostAlloc((void **)&g_pullItemsHost, cap * sizeof(PullBatchItem), cudaHostAllocMapped));
		CU(cudaHostGetDevicePointer((void **)&g_pullItemsDev, g_pullItemsHost, 0));
		g_pullItemsCap = cap; g_pullItemsDevice = lead->device;
	}
	std::vector<unsigned int> total(n, 0);
	std::vector<uint32_t> got(n, 0);
	std::vector<char> done(n, 0), zero(n, 1);
	// The per-player host work runs on the helper threads when it touches no shared state and makes no CUDA call: zero-copy
	// staging, no process-global rand() sequence (its draws are handed out in player order), no replay upload pending.
	bool parallel = pullZeroCopy() && !pullDebugPhases() && n >= 8 && HostPool::get().helpers() > 0;
	for (size_t i = 0; i < n && parallel; ++i)
		if (ps[i]->noiseMode == kNoiseGlibc || (ps[i]->noiseMode == kNoiseReplay && ps[i]->replayDirty)) parallel = false;
	const size_t grain = parallel ? std::max<size_t>(1, n / (4 * (HostPool::get().helpers() + 1))) : n;
	auto forEach = [&](const std::function<void(size_t)> &fn) {
		if (parallel) HostPool::get().parallelFor(n, grain, fn);
		else
			for (size_t i = 0; i < n; ++i) fn(i);
	};
	for (;;) {
		std::atomic<int> any{0}, failed{0};
		auto prepare = [&](size_t i) {
			Player *p = ps[i];
			PullBatchItem &it = g_pullItemsHost[i];
			memset(&it, 0, sizeof it);
			got[i] = 0;
			if (done[i] || total[i] >= sampleCount) return;
			const uint32_t want = std::min<uint32_t>(sampleCount - total[i], kPullMaxTicks);
			p->pullSegs.clear();
			bool drained = false;
			got[i] = p->pull->advance(want, 0, kPullMaxSegs, p->pullSegs, drained);
			if (drained) done[i] = 1;
			if (!got[i]) return;
			bool zc;
			if (pullStage(p, got[i], it.ctx, it.segSrc, it.pcmOut, zc, stream) != 0) {
				failed.store(1);
				return;
			}
			zero[i] = zc ? 1 : 0;
			any.store(1);
		};
		static const bool timing = getenv("NVSP_PULL_TIMING") != nullptr;  // host-side phases of a batched pull, one line per launch
		const auto t0 = std::chrono::steady_clock::now();
		forEach(prepare);
		if (failed.load()) return -1;
		if (!any.load()) break;
		const auto t1 = std::chrono::steady_clock::now();
		CU(launchKlattPullBatch(g_pullItemsHost, g_pullItemsDev, (uint32_t)n, stream));
		for (size_t i = 0; i < n; ++i)
			if (got[i] && !zero[i])
				CU(cudaMemcpyAsync(ps[i]->hPullStage + Player::kStageSegs, g_pullItemsHost[i].pcmOut, (size_t)got[i] * sizeof(int16_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		const auto t2 = std::chrono::steady_clock::now();
		forEach([&](size_t i) {
			if (!got[i]) return;
			memcpy(out + i * (size_t)sampleCount + total[i], ps[i]->hPullStage + Player::kStageSegs, (size_t)got[i] * sizeof(int16_t));
			++ps[i]->pullLaunches;
			ps[i]->generated += got[i];
			total[i] += got[i];
		});
		if (timing) {
			const auto t3 = std::chrono::steady_clock::now();
			auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
				return std::chrono::duration<double, std::micro>(b - a).count();
			};
			fprintf(stderr, "[pull batch] %zu players, %s: prepare %.0f us, launch + sync %.0f us, copy out %.0f us\n", n,
			        parallel ? "helpers" : "serial", us(t0, t1), us(t1, t2), us(t2, t3));
		}
	}
	long long sum = 0;
	for (size_t i = 0; i < n; ++i) {
		ps[i]->lastIndex = ps[i]->pull->lastIndex();
		if (samplesWritten) samplesWritten[i] = total[i];
		sum += total[i];
	}
	return sum;
}

long long speechPlayer_synthesizeBatch(speechPlayer_handle_t *handles, unsigned int numHandles, unsigned int sampleCount,
                                       sample *sampleBuf, unsigned int *samplesWritten) {
	g_lastError.clear();
	if (numHandles == 0 || sampleCount == 0) return 0;
	if (!handles || !sampleBuf) return fail("null argument");
	std::vector<Player *> ps(numHandles);
	bool anyPull = false;
	for (unsigned i = 0; i < numHandles; ++i) {
		ps[i] = lookup(handles[i]);
		if (!ps[i]) return fail("bad handle in batch");
		anyPull = anyPull || ps[i]->pull != nullptr;
	}
	if (anyPull) {  // low-latency players: one block per player, one launch for all of them
		std::vector<Player *> uniq(ps);
		std::sort(uniq.begin(), uniq.end());
		if (std::adjacent_find(uniq.begin(), uniq.end()) != uniq.end()) return fail("duplicate handle in batch");
		for (unsigned i = 0; i < numHandles; ++i)
			if (!ps[i]->pull || ps[i]->device != ps[0]->device)
				return fail("handles of one batch must share device and precision");
		if (numHandles == 1) {
			long long w = synthesizePull(ps[0], sampleCount, reinterpret_cast<int16_t *>(sampleBuf));
			if (w >= 0 && samplesWritten) samplesWritten[0] = (unsigned int)w;
			return w;
		}
		return synthesizePullBatch(ps, sampleCount, reinterpret_cast<int16_t *>(sampleBuf), samplesWritten);
	}
	for (unsigned i = 0; i < numHandles; ++i) {
		if (ps[i]->precision != ps[0]->precision || ps[i]->sampleRate != ps[0]->sampleRate ||
		    ps[i]->device != ps[0]->device || ps[i]->noiseMode != ps[0]->noiseMode || ps[i]->seed != ps[0]->seed)
			return fail("handles of one batch must share device, sample rate, precision and noise mode");
	}
	// lock in address order; a handle may appear only once
	std::vector<Player *> order(ps);
	std::sort(order.begin(), order.end());
	if (std::adjacent_find(order.begin(), order.end()) != order.end()) return fail("duplicate handle in batch");
	for (Player *p : order) p->mu.lock();
	struct Unlock {
		std::vector<Player *> &o;
		~Unlock() { for (Player *p : o) p->mu.unlock(); }
	} unlock{order};

	Player *lead = ps[0];
	DeviceGuard g(lead->device);
	if (!lead->pipe.init()) return -1;
	cudaStream_t stream = lead->pipe.compute;
	std::unique_lock<std::mutex> noiseLock(g_noiseMu, std::defer_lock);
	GlibcRand checkpoint;
	if (lead->noiseMode == kNoiseGlibc) {
		noiseLock.lock();
		checkpoint = g_noise;
	}
	std::vector<StreamDesc> descs(numHandles);
	for (unsigned i = 0; i < numHandles; ++i)
		if (ps[i]->prepare(descs[i], sampleCount, stream) != 0) return -1;
	if (!lead->dDesc.reserve(sizeof(StreamDesc) * (size_t)numHandles)) return -1;
	CU(cudaMemcpyAsync(lead->dDesc.p, descs.data(), sizeof(StreamDesc) * (size_t)numHandles, cudaMemcpyHostToDevice, stream));
	CU(cudaStreamSynchronize(stream));
	std::vector<uint32_t> written(numHandles);
	std::vector<StreamResult> results(numHandles);
	NoiseConfig nc{lead->noiseMode, lead->seed};
	// The reference's generate() returns the count and leaves sampleBuf[count..] untouched (src/speechWaveGenerator.cpp:210),
	// so the rows land in a scratch buffer first and only the written prefix of each row is handed to the caller.
	std::vector<int16_t> &scratch = lead->hostScratch;
	scratch.resize((size_t)numHandles * sampleCount);
	long long total = renderToHost(lead->pipe, lead->precision, lead->dDesc.as<StreamDesc>(), numHandles, lead->sampleRate,
	                               sampleCount, scratch.data(), written.data(), results.data(), nc, nullptr);
	if (total < 0) return -1;
	for (unsigned i = 0; i < numHandles; ++i) {
		ps[i]->absorb(results[i], written[i]);
		if (samplesWritten) samplesWritten[i] = written[i];
		memcpy(reinterpret_cast<int16_t *>(sampleBuf) + (size_t)i * sampleCount, scratch.data() + (size_t)i * sampleCount,
		       sizeof(int16_t) * (size_t)written[i]);
	}
	if (lead->noiseMode == kNoiseGlibc && numHandles == 1) {
		// the reference consumes exactly two rand() calls per generated sample: rewind to that point
		g_noise = checkpoint;
		g_noise.skip((uint64_t)written[0] * 2);
	}
	return total;
}

int speechPlayer_synthesize(speechPlayer_handle_t playerHandle, unsigned int sampleCount, sample *sampleBuf) {
	unsigned int written = 0;
	long long r = speechPlayer_synthesizeBatch(&playerHandle, 1, sampleCount, sampleBuf, &written);
	if (r < 0) return -1;
	return (int)written;
}

int speechPlayer_getLastIndex(speechPlayer_handle_t playerHandle) {
	Player *p = lookup(playerHandle);
	return p ? p->lastIndex : -1;  // read without the lock, like src/frame.cpp:117-119
}

void speechPlayer_terminate(speechPlayer_handle_t playerHandle) {
	uintptr_t v = reinterpret_cast<uintptr_t>(playerHandle);
	Player *p = nullptr;
	{
		std::lock_guard<std::mutex> lk(g_tableMu);
		if (v == 0 || v > g_players.size()) return;
		p = g_players[v - 1];
		g_players[v - 1] = nullptr;
	}
	if (!p) return;
	{ std::lock_guard<std::mutex> lk(p->mu); }
	p->destroy();
	delete p;
}

unsigned long long speechPlayer_timelineSamples(const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                                unsigned int n) {
	unsigned long long t = 0;
	for (unsigned i = 0; i < n; ++i) {
		unsigned long long m = minFrameDuration[i], f = fadeDuration[i] > 1 ? fadeDuration[i] : 1;
		t += std::max(m + 1, f + 2);
	}
	return t;
}

// Measured FP32 roofline denominator: a register-resident FFMA loop (16 independent chains per thread, 3-register
// form) timed with CUDA events on the current device; returns TFLOP/s (2 flops per FMA), <0 on error.  bench.py
// reports the render kernel's counted flops against this number and against SMs x 128 lanes x 2 x clock.
__global__ void fp32_peak_kernel(float *out, int iters, float x, float y) {
	float a[16];
#pragma unroll
	for (int j = 0; j < 16; ++j) a[j] = (float)(threadIdx.x + j) * 1e-3f;
	for (int i = 0; i < iters; ++i) {
#pragma unroll
		for (int j = 0; j < 16; ++j) a[j] = fmaf(a[j], x, y);
	}
	float sum = 0;
#pragma unroll
	for (int j = 0; j < 16; ++j) sum += a[j];
	out[blockIdx.x * blockDim.x + threadIdx.x] = sum;
}

extern "C" double speechPlayer_debugFp32PeakTflops(void) {
	int dev = 0, sms = 0;
	if (cudaGetDevice(&dev) != cudaSuccess) return -1;
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	const int threads = 256, blocks = sms * 8, iters = 1 << 15;
	float *out = nullptr;
	if (cudaMalloc(&out, sizeof(float) * threads * blocks) != cudaSuccess) return -1;
	cudaEvent_t e0, e1;
	cudaEventCreate(&e0); cudaEventCreate(&e1);
	double best = -1;
	for (int rep = 0; rep < 5; ++rep) {
		cudaEventRecord(e0);
		fp32_peak_kernel<<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
		cudaEventRecord(e1);
		if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1; break; }
		float ms = 0;
		cudaEventElapsedTime(&ms, e0, e1);
		double tf = 2.0 * 16.0 * iters * (double)threads * blocks / (ms * 1e-3) / 1e12;
		if (rep > 0 && tf > best) best = tf;
	}
	cudaEventDestroy(e0); cudaEventDestroy(e1);
	cudaFree(out);
	return best;
}

// test hook: the first n values of the glibc-compatible generator after seed(s)
void speechPlayer_debugGlibcRand(unsigned int seed, unsigned int n, int32_t *out) {
	GlibcRand r;
	r.seed(seed);
	r.fill(out, n);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// C-ABI: batch API
// ------------------------------------------------------------------------------------------------
struct speechPlayer_batch {
	int device = 0, sampleRate = 0, precision = kPrecisionF32, noiseMode = kNoisePhilox;
	uint64_t seed = 0;
	uint32_t n = 0;
	StreamState *dStates = nullptr;
	StreamDesc *dDescs = nullptr;
	uint64_t *dStreamIds = nullptr;
	// current queue arrays (borrowed device pointers, or the owned copies below)
	const int64_t *dOffsets = nullptr;
	const double *dFrames = nullptr;
	const uint32_t *dMin = nullptr, *dFade = nullptr;
	const int32_t *dUix = nullptr;
	const uint8_t *dNull = nullptr;
	const int32_t *dReplay = nullptr;
	uint64_t drawsPerStream = 0;
	DevBuf ownOffsets, ownFrames, ownMin, ownFade, ownUix, ownNull;
	DevBuf voiceTables;        // speechPlayer_batchApplyVoices: abs | mul | voiceOfStream
	DevBuf plans;              // FadePlanF32 per queued request (FP32 precision)
	bool plansDirty = false;   // frames changed since the plans were made
	uint64_t totalRequests = 0;
	HostPipe pipe;
	RoundsCtx rounds;
	unsigned long long launches = 0, ticks = 0;
	std::mutex mu;

	int rebuildDescs(cudaStream_t stream, bool withPlans) {
		build_descs_kernel<<<(n + 256) / 256, 256, 0, stream>>>(dDescs, dStates, dOffsets, dFrames, dMin, dFade, dUix, dNull,
		                                                        dReplay, drawsPerStream, dStreamIds,
		                                                        withPlans ? plans.as<FadePlanF32>() : nullptr, n);
		CU(cudaGetLastError());
		++launches;
		return 0;
	}
	bool planned() const { return precision == kPrecisionF32 && dOffsets != nullptr && !plansDirty; }
	// FP32: (re)make the fade plans of every queued request; runs inside the first synthesize after SetFrames, on
	// the synthesize stream, so the work is part of the rendered step
	int ensurePlans(cudaStream_t stream) {
		if (precision != kPrecisionF32 || !dOffsets || !plansDirty) return 0;
		if (!plans.reserve(std::max<uint64_t>(totalRequests, 1) * sizeof(FadePlanF32))) return -1;
		CU(launchKlattPlan(dOffsets, n, totalRequests, dFrames, dFade, dNull, sampleRate, plans.as<FadePlanF32>(), stream));
		++launches;
		plansDirty = false;
		return rebuildDescs(stream, true);
	}
};

extern "C" {

speechPlayer_batch_t *speechPlayer_batchCreate(int sampleRate, unsigned int numStreams, int precision, int noiseMode,
                                               uint64_t seed, const uint64_t *streamIds) {
	g_lastError.clear();
	if (sampleRate <= 0 || numStreams == 0) { fail("bad sampleRate / numStreams"); return nullptr; }
	if (precision != kPrecisionF64 && precision != kPrecisionF32) {
		fail(precision == kPrecisionStream ? "SPEECHPLAYER_PRECISION_STREAM is a per-handle mode (speechPlayer_initializeEx)" : "unknown precision");
		return nullptr;
	}
	if (noiseMode != kNoisePhilox && noiseMode != kNoiseReplay) { fail("batch noise mode must be PHILOX or REPLAY"); return nullptr; }
	int dev = pickDevice();
	if (dev < 0) { fail("no usable CUDA device (this library has no CPU fallback)"); return nullptr; }
	DeviceGuard g(dev);
	speechPlayer_batch *b = new speechPlayer_batch;
	b->device = dev; b->sampleRate = sampleRate; b->precision = precision; b->noiseMode = noiseMode; b->seed = seed;
	b->n = numStreams;
	bool ok = cudaOk(cudaMalloc((void **)&b->dStates, sizeof(StreamState) * ((size_t)numStreams + 1)), "cudaMalloc(states)") &&
	          cudaOk(cudaMalloc((void **)&b->dDescs, sizeof(StreamDesc) * ((size_t)numStreams + 1)), "cudaMalloc(descs)") &&
	          cudaOk(cudaMalloc((void **)&b->dStreamIds, sizeof(uint64_t) * (size_t)numStreams), "cudaMalloc(ids)");
	if (ok) {
		std::vector<uint64_t> ids(numStreams);
		for (uint32_t i = 0; i < numStreams; ++i) ids[i] = streamIds ? streamIds[i] : i;
		ok = cudaOk(cudaMemcpy(b->dStreamIds, ids.data(), sizeof(uint64_t) * (size_t)numStreams, cudaMemcpyHostToDevice), "ids H2D") &&
		     cudaOk(initStates(b->dStates, numStreams + 1, nullptr), "init states") && b->rebuildDescs(nullptr, false) == 0 &&
		     cudaOk(cudaStreamSynchronize(nullptr), "sync");
	}
	if (!ok) {
		speechPlayer_batchDestroy(b);
		return nullptr;
	}
	return b;
}

void speechPlayer_batchDestroy(speechPlayer_batch_t *b) {
	if (!b) return;
	DeviceGuard g(b->device);
	cudaDeviceSynchronize();
	b->pipe.destroy();
	b->rounds.destroy();
	b->plans.release();
	b->voiceTables.release();
	b->ownOffsets.release(); b->ownFrames.release(); b->ownMin.release(); b->ownFade.release(); b->ownUix.release(); b->ownNull.release();
	if (b->dStates) cudaFree(b->dStates);
	if (b->dDescs) cudaFree(b->dDescs);
	if (b->dStreamIds) cudaFree(b->dStreamIds);
	delete b;
}

int speechPlayer_batchReset(speechPlayer_batch_t *b, void *cudaStream) {
	if (!b) return fail("null batch");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	CU(initStates(b->dStates, b->n + 1, static_cast<cudaStream_t>(cudaStream)));
	b->launches += 1;
	return 0;
}

int speechPlayer_batchSetFramesDevice(speechPlayer_batch_t *b, const void *dOffsets, const void *dFrames, const void *dMinDur,
                                      const void *dFadeDur, const void *dUserIndex, const void *dIsNull, void *cudaStream) {
	if (!b) return fail("null batch");
	if (!dOffsets || !dMinDur || !dFadeDur) return fail("offsets and durations are required");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	b->dOffsets = static_cast<const int64_t *>(dOffsets);
	b->dFrames = static_cast<const double *>(dFrames);
	b->dMin = static_cast<const uint32_t *>(dMinDur);
	b->dFade = static_cast<const uint32_t *>(dFadeDur);
	b->dUix = static_cast<const int32_t *>(dUserIndex);
	b->dNull = static_cast<const uint8_t *>(dIsNull);
	// new queues start on fresh players (the batch equivalent of initialize + queueFrame x n)
	CU(initStates(b->dStates, b->n + 1, stream));
	b->launches += 1;
	if (b->precision == kPrecisionF32) {
		// the plan buffer is sized from the total request count: one 8-byte read-back
		int64_t total = 0;
		CU(cudaMemcpyAsync(&total, b->dOffsets + b->n, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		if (total < 0) return fail("offsets[numStreams] is negative");
		b->totalRequests = (uint64_t)total;
		b->plansDirty = true;
	}
	return b->rebuildDescs(stream, false);
}

int speechPlayer_batchSetFramesHost(speechPlayer_batch_t *b, const int64_t *offsets, const speechPlayer_frame_t *frames,
                                    const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                    const int *userIndex, const unsigned char *isNull, void *cudaStream) {
	if (!b) return fail("null batch");
	if (!offsets || !minFrameDuration || !fadeDuration) return fail("offsets and durations are required");
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	size_t total = (size_t)offsets[b->n];
	{
		std::lock_guard<std::mutex> lk(b->mu);
		DeviceGuard g(b->device);
		if (!b->ownOffsets.reserve(sizeof(int64_t) * ((size_t)b->n + 1)) ||
		    !b->ownFrames.reserve(std::max<size_t>(total, 1) * sizeof(speechPlayer_frame_t)) ||
		    !b->ownMin.reserve(std::max<size_t>(total, 1) * 4) || !b->ownFade.reserve(std::max<size_t>(total, 1) * 4) ||
		    !b->ownUix.reserve(std::max<size_t>(total, 1) * 4) || !b->ownNull.reserve(std::max<size_t>(total, 1)))
			return -1;
		CU(cudaMemcpyAsync(b->ownOffsets.p, offsets, sizeof(int64_t) * ((size_t)b->n + 1), cudaMemcpyHostToDevice, stream));
		if (total) {
			if (frames) CU(cudaMemcpyAsync(b->ownFrames.p, frames, total * sizeof(speechPlayer_frame_t), cudaMemcpyHostToDevice, stream));
			CU(cudaMemcpyAsync(b->ownMin.p, minFrameDuration, total * 4, cudaMemcpyHostToDevice, stream));
			CU(cudaMemcpyAsync(b->ownFade.p, fadeDuration, total * 4, cudaMemcpyHostToDevice, stream));
			if (userIndex) CU(cudaMemcpyAsync(b->ownUix.p, userIndex, total * 4, cudaMemcpyHostToDevice, stream));
			if (isNull) CU(cudaMemcpyAsync(b->ownNull.p, isNull, total, cudaMemcpyHostToDevice, stream));
		}
	}
	int r = speechPlayer_batchSetFramesDevice(b, b->ownOffsets.p, frames ? b->ownFrames.p : nullptr, b->ownMin.p, b->ownFade.p,
	                                          userIndex ? b->ownUix.p : nullptr, isNull ? b->ownNull.p : nullptr, cudaStream);
	if (r != 0) return r;
	DeviceGuard g(b->device);
	CU(cudaStreamSynchronize(stream));  // the caller's host arrays may be reused now
	return 0;
}

int speechPlayer_batchApplyVoices(speechPlayer_batch_t *b, const double *voiceAbs, const double *voiceMul,
                                  const unsigned int *voiceOfStream, unsigned int numVoices, void *cudaStream) {
	if (!b) return fail("null batch");
	if (!voiceAbs || !voiceMul || numVoices == 0) return fail("voice tables are required");
	std::lock_guard<std::mutex> lk(b->mu);
	if (!b->dOffsets || !b->dFrames) return fail("no frames queued (call SetFrames first)");
	DeviceGuard g(b->device);
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	const size_t tableBytes = sizeof(double) * (size_t)numVoices * kNumParams;
	if (!b->voiceTables.reserve(2 * tableBytes + sizeof(uint32_t) * (size_t)b->n)) return -1;
	char *base = b->voiceTables.as<char>();
	CU(cudaMemcpyAsync(base, voiceAbs, tableBytes, cudaMemcpyHostToDevice, stream));
	CU(cudaMemcpyAsync(base + tableBytes, voiceMul, tableBytes, cudaMemcpyHostToDevice, stream));
	if (voiceOfStream) CU(cudaMemcpyAsync(base + 2 * tableBytes, voiceOfStream, sizeof(uint32_t) * (size_t)b->n, cudaMemcpyHostToDevice, stream));
	apply_voices_kernel<<<dim3(4, b->n), 128, 0, stream>>>(const_cast<double *>(b->dFrames), b->dOffsets, b->dNull,
	                                                      reinterpret_cast<const double *>(base), reinterpret_cast<const double *>(base + tableBytes),
	                                                      voiceOfStream ? reinterpret_cast<const uint32_t *>(base + 2 * tableBytes) : nullptr, numVoices, b->n);
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(stream));  // the host tables may be reused
	b->launches += 1;
	if (b->precision == kPrecisionF32) b->plansDirty = true;
	return 0;
}

int speechPlayer_batchSetNoiseReplayDevice(speechPlayer_batch_t *b, const void *dDraws, size_t drawsPerStream) {
	if (!b) return fail("null batch");
	if (b->noiseMode != kNoiseReplay) return fail("batch was not created with SPEECHPLAYER_NOISE_REPLAY");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	b->dReplay = static_cast<const int32_t *>(dDraws);
	b->drawsPerStream = drawsPerStream;
	// the entry has no stream argument: the descriptor rewrite runs on the legacy default stream and is complete on return,
	// so a synthesize on any (also non-blocking) stream afterwards sees whole descriptors
	if (b->rebuildDescs(nullptr, b->planned()) != 0) return -1;
	CU(cudaStreamSynchronize(nullptr));
	return 0;
}

int speechPlayer_batchSynthesizeDevice(speechPlayer_batch_t *b, unsigned int sampleCount, void *dOut, size_t rowStride,
                                       void *dSamplesWritten, void *cudaStream) {
	if (!b) return fail("null batch");
	if (!dOut) return fail("null output");
	if (rowStride < sampleCount) return fail("rowStride < sampleCount");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	NoiseConfig nc{b->noiseMode, b->seed};
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	if (b->ensurePlans(stream) != 0) return -1;
	CU(launchRender(b->precision, b->dDescs, b->n, b->sampleRate, sampleCount, static_cast<int16_t *>(dOut), rowStride,
	                static_cast<uint32_t *>(dSamplesWritten), nullptr, nc, stream, &b->rounds, b->planned(), &b->launches));
	b->ticks += (unsigned long long)b->n * sampleCount;
	return 0;
}

long long speechPlayer_batchSynthesizeHost(speechPlayer_batch_t *b, unsigned int sampleCount, sample *out,
                                           unsigned int *samplesWritten) {
	if (!b) return fail("null batch");
	if (!out) return fail("null output");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	CU(cudaDeviceSynchronize());  // frames / resets enqueued on other streams must have landed
	NoiseConfig nc{b->noiseMode, b->seed};
	if (!b->pipe.init()) return -1;
	if (b->ensurePlans(b->pipe.compute) != 0) return -1;
	long long r = renderToHost(b->pipe, b->precision, b->dDescs, b->n, b->sampleRate, sampleCount,
	                           reinterpret_cast<int16_t *>(out), samplesWritten, nullptr, nc, &b->launches, b->planned());
	if (r >= 0) b->ticks += (unsigned long long)b->n * sampleCount;
	return r;
}

// ---- output sinks on the device (include/speechPlayer_batch.h) ----
}  // extern "C"

// int16 -> float32 as reference lavPlayer.py:17 does it: (double)sample / 32767.0, then rounded to float.  HBM-bound: 2 bytes
// in, 4 bytes out per sample; one thread converts 8 samples (one 16-byte load, two 16-byte stores) when the rows allow it.
__global__ void __launch_bounds__(256)
pcm_to_float32_kernel(const int16_t *__restrict__ pcm, size_t rowStride, uint32_t sampleCount, float *__restrict__ out, size_t outStride,
                      bool vec) {
	const uint32_t s = blockIdx.y;
	const int16_t *row = pcm + (size_t)s * rowStride;
	float *orow = out + (size_t)s * outStride;
	auto conv = [](int v) { return (float)((double)v / 32767.0); };
	if (vec) {
		const uint32_t groups = sampleCount / 8;
		for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += gridDim.x * blockDim.x) {
			const uint4 w = reinterpret_cast<const uint4 *>(row)[g];
			const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
			float f[8];
#pragma unroll
			for (int k = 0; k < 4; ++k) { f[2 * k] = conv((int16_t)(ww[k] & 0xffffu)); f[2 * k + 1] = conv((int16_t)(ww[k] >> 16)); }
			reinterpret_cast<float4 *>(orow)[2 * g] = make_float4(f[0], f[1], f[2], f[3]);
			reinterpret_cast<float4 *>(orow)[2 * g + 1] = make_float4(f[4], f[5], f[6], f[7]);
		}
		for (uint32_t i = groups * 8 + blockIdx.x * blockDim.x + threadIdx.x; i < sampleCount; i += gridDim.x * blockDim.x) orow[i] = conv(row[i]);
	} else {
		for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < sampleCount; i += gridDim.x * blockDim.x) orow[i] = conv(row[i]);
	}
}

// exclusive prefix sum of the per-stream sample counts (one block; numStreams is at most a few million)
__global__ void __launch_bounds__(1024)
concat_offsets_kernel(const uint32_t *__restrict__ written, uint32_t sampleCount, uint32_t n, int64_t *__restrict__ offsets) {
	__shared__ int64_t warpTotal[32];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const uint32_t per = (n + 1023) / 1024;
	const uint32_t c0 = (uint32_t)tid * per < n ? (uint32_t)tid * per : n, c1 = c0 + per < n ? c0 + per : n;
	int64_t run = 0;
	for (uint32_t c = c0; c < c1; ++c) run += written ? (int64_t)(written[c] < sampleCount ? written[c] : sampleCount) : (int64_t)sampleCount;
	int64_t inc = run;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		int64_t up = __shfl_up_sync(0xffffffffu, inc, d);
		if (lane >= d) inc += up;
	}
	if (lane == 31) warpTotal[warp] = inc;
	__syncthreads();
	if (warp == 0) {
		int64_t w = warpTotal[lane];
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			int64_t up = __shfl_up_sync(0xffffffffu, w, d);
			if (lane >= d) w += up;
		}
		warpTotal[lane] = w;
	}
	__syncthreads();
	int64_t pos = inc - run + (warp > 0 ? warpTotal[warp - 1] : 0);
	for (uint32_t c = c0; c < c1; ++c) {
		offsets[c] = pos;
		pos += written ? (int64_t)(written[c] < sampleCount ? written[c] : sampleCount) : (int64_t)sampleCount;
	}
	if (tid == 1023) offsets[n] = warpTotal[31];
}

// one block row per stream: its first offsets[s+1]-offsets[s] samples go to packed + offsets[s] (destinations are 2-byte
// aligned only; 32-bit stores from the first even destination index on)
__global__ void __launch_bounds__(256)
concat_gather_kernel(const int16_t *__restrict__ pcm, size_t rowStride, const int64_t *__restrict__ offsets, int16_t *__restrict__ packed) {
	const uint32_t s = blockIdx.y;
	const int64_t o0 = offsets[s], cnt = offsets[s + 1] - o0;
	const int16_t *row = pcm + (size_t)s * rowStride;
	int16_t *dst = packed + o0;
	const int64_t head = (o0 & 1) ? 1 : 0;  // samples before the first 4-byte aligned destination
	if (blockIdx.x == 0 && threadIdx.x == 0 && head && cnt > 0) dst[0] = row[0];
	const int64_t pairs = (cnt - head) / 2;
	for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (int64_t)gridDim.x * blockDim.x) {
		const uint32_t lo = (uint16_t)row[head + 2 * i], hi = (uint16_t)row[head + 2 * i + 1];
		*reinterpret_cast<uint32_t *>(dst + head + 2 * i) = lo | (hi << 16);
	}
	if (blockIdx.x == 0 && threadIdx.x == 0 && ((cnt - head) & 1) && cnt > head) dst[cnt - 1] = row[cnt - 1];
}

extern "C" {

int speechPlayer_batchToFloat32Device(const void *dPcm, size_t rowStride, unsigned int numStreams, unsigned int sampleCount,
                                      void *dOutFloat, size_t outStride, void *cudaStream) {
	if (!dPcm || !dOutFloat) return fail("null argument");
	if (rowStride < sampleCount || outStride < sampleCount) return fail("stride < sampleCount");
	if (numStreams == 0 || sampleCount == 0) return 0;
	const bool vec = (reinterpret_cast<uintptr_t>(dPcm) & 15u) == 0 && (reinterpret_cast<uintptr_t>(dOutFloat) & 15u) == 0 &&
	                 rowStride % 8 == 0 && outStride % 4 == 0;
	const unsigned gx = (unsigned)std::min<size_t>(((size_t)sampleCount / 8 + 255) / 256 + 1, 64);
	for (unsigned s0 = 0; s0 < numStreams; s0 += 65535u) {
		const unsigned ny = std::min(numStreams - s0, 65535u);
		pcm_to_float32_kernel<<<dim3(gx, ny), 256, 0, static_cast<cudaStream_t>(cudaStream)>>>(
		    static_cast<const int16_t *>(dPcm) + (size_t)s0 * rowStride, rowStride, sampleCount, static_cast<float *>(dOutFloat) + (size_t)s0 * outStride,
		    outStride, vec);
	}
	CU(cudaGetLastError());
	return 0;
}

int speechPlayer_batchConcatenateDevice(const void *dPcm, size_t rowStride, unsigned int numStreams, unsigned int sampleCount,
                                        const void *dSamplesWritten, void *dOffsets, void *dOutPacked, void *cudaStream) {
	if (!dPcm || !dOffsets || !dOutPacked) return fail("null argument");
	if (rowStride < sampleCount) return fail("rowStride < sampleCount");
	if (numStreams == 0) return 0;
	cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
	concat_offsets_kernel<<<1, 1024, 0, stream>>>(static_cast<const uint32_t *>(dSamplesWritten), sampleCount, numStreams, static_cast<int64_t *>(dOffsets));
	const unsigned gx = (unsigned)std::min<size_t>(((size_t)sampleCount / 2 + 255) / 256 + 1, 32);
	for (unsigned s0 = 0; s0 < numStreams; s0 += 65535u) {
		const unsigned ny = std::min(numStreams - s0, 65535u);
		concat_gather_kernel<<<dim3(gx, ny), 256, 0, stream>>>(static_cast<const int16_t *>(dPcm) + (size_t)s0 * rowStride, rowStride,
		                                                       static_cast<const int64_t *>(dOffsets) + s0, static_cast<int16_t *>(dOutPacked));
	}
	CU(cudaGetLastError());
	return 0;
}

int speechPlayer_batchGetLastIndices(speechPlayer_batch_t *b, int *lastIndex) {
	if (!b || !lastIndex) return fail("null argument");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	CU(cudaDeviceSynchronize());
	// lastUserIndex is the first word of every state block
	CU(cudaMemcpy2D(lastIndex, sizeof(int), b->dStates, sizeof(StreamState), sizeof(int), b->n, cudaMemcpyDeviceToHost));
	return 0;
}

int speechPlayer_batchGetLaunchStats(speechPlayer_batch_t *b, unsigned long long *kernelLaunches,
                                     unsigned long long *ticksRequested) {
	if (!b) return fail("null batch");
	if (kernelLaunches) *kernelLaunches = b->launches;
	if (ticksRequested) *ticksRequested = b->ticks;
	return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// C-ABI: several GPUs of one box (include/speechPlayer_batch.h): shards = per-device batches, one host thread each
// ------------------------------------------------------------------------------------------------
struct speechPlayer_multiBatch {
	int sampleRate = 0, precision = kPrecisionF32, noiseMode = kNoisePhilox;
	uint64_t seed = 0;
	uint32_t n = 0;
	std::vector<uint64_t> streamIds;
	std::vector<int> devices;
	std::vector<uint32_t> first;                  // [numDevices + 1]
	std::vector<speechPlayer_batch_t *> shards;   // per device (nullptr while the shard is empty)
	std::mutex mu;
};

// run fn(d) for every shard on its own thread with the shard's device current; returns false if any failed
template <class Fn>
static bool forEachShard(speechPlayer_multiBatch *mb, Fn fn, std::string &err) {
	const size_t nd = mb->devices.size();
	std::vector<std::thread> th;
	std::vector<int> ok(nd, 1);
	std::vector<std::string> errs(nd);
	for (size_t d = 0; d < nd; ++d)
		th.emplace_back([&, d] {
			if (cudaSetDevice(mb->devices[d]) != cudaSuccess) { ok[d] = 0; errs[d] = "cudaSetDevice failed"; return; }
			if (!fn(d)) { ok[d] = 0; errs[d] = g_lastError; }
		});
	for (auto &t : th) t.join();
	for (size_t d = 0; d < nd; ++d)
		if (!ok[d]) { err = "shard " + std::to_string(d) + " (device " + std::to_string(mb->devices[d]) + "): " + errs[d]; return false; }
	return true;
}

extern "C" {

speechPlayer_multiBatch_t *speechPlayer_multiBatchCreate(int sampleRate, unsigned int numStreams, int precision, int noiseMode,
                                                         uint64_t seed, const uint64_t *streamIds, const int *devices,
                                                         unsigned int numDevices) {
	g_lastError.clear();
	if (sampleRate <= 0 || numStreams == 0 || numDevices == 0 || !devices) { fail("bad sampleRate / numStreams / devices"); return nullptr; }
	int have = 0;
	if (cudaGetDeviceCount(&have) != cudaSuccess || have <= 0) { fail("no usable CUDA device (this library has no CPU fallback)"); return nullptr; }
	for (unsigned d = 0; d < numDevices; ++d)
		if (devices[d] < 0 || devices[d] >= have) { fail("device ordinal out of range"); return nullptr; }
	speechPlayer_multiBatch *mb = new speechPlayer_multiBatch;
	mb->sampleRate = sampleRate; mb->precision = precision; mb->noiseMode = noiseMode; mb->seed = seed; mb->n = numStreams;
	mb->streamIds.resize(numStreams);
	for (uint32_t i = 0; i < numStreams; ++i) mb->streamIds[i] = streamIds ? streamIds[i] : i;
	mb->devices.assign(devices, devices + numDevices);
	mb->shards.assign(numDevices, nullptr);
	// until queues are known: equal counts (sizes differ by at most one)
	mb->first.resize(numDevices + 1);
	for (unsigned d = 0; d <= numDevices; ++d) mb->first[d] = (uint32_t)((uint64_t)numStreams * d / numDevices);
	return mb;
}

void speechPlayer_multiBatchDestroy(speechPlayer_multiBatch_t *mb) {
	if (!mb) return;
	for (size_t d = 0; d < mb->shards.size(); ++d)
		if (mb->shards[d]) speechPlayer_batchDestroy(mb->shards[d]);
	delete mb;
}

int speechPlayer_multiBatchSetFramesHost(speechPlayer_multiBatch_t *mb, const int64_t *offsets, const speechPlayer_frame_t *frames,
                                         const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                         const int *userIndex, const unsigned char *isNull) {
	if (!mb) return fail("null batch");
	if (!offsets || !minFrameDuration || !fadeDuration) return fail("offsets and durations are required");
	std::lock_guard<std::mutex> lk(mb->mu);
	const size_t nd = mb->devices.size();
	// contiguous ranges balanced by the ticks every stream yields: cut where the running sum passes k / nd of the total
	std::vector<uint64_t> upto(mb->n + 1, 0);
	for (uint32_t s = 0; s < mb->n; ++s)
		upto[s + 1] = upto[s] + speechPlayer_timelineSamples(minFrameDuration + offsets[s], fadeDuration + offsets[s],
		                                                     (unsigned int)(offsets[s + 1] - offsets[s])) + 1;  // (+1: empty queues still cost a lane)
	std::vector<uint32_t> first(nd + 1, 0);
	first[nd] = mb->n;
	for (size_t d = 1; d < nd; ++d) {
		const uint64_t want = upto[mb->n] / nd * d + upto[mb->n] % nd * d / nd;
		first[d] = (uint32_t)(std::lower_bound(upto.begin(), upto.end(), want) - upto.begin());
		if (first[d] < first[d - 1]) first[d] = first[d - 1];
		if (first[d] > mb->n) first[d] = mb->n;
	}
	std::string err;
	const bool ok = forEachShard(mb, [&](size_t d) -> bool {
		const uint32_t a = first[d], b = first[d + 1], cnt = b - a;
		if (mb->shards[d] && (mb->first[d] != a || mb->first[d + 1] != b)) {  // the shard moved: new per-device buffers
			speechPlayer_batchDestroy(mb->shards[d]);
			mb->shards[d] = nullptr;
		}
		if (cnt == 0) return true;
		if (!mb->shards[d]) {
			mb->shards[d] = speechPlayer_batchCreate(mb->sampleRate, cnt, mb->precision, mb->noiseMode, mb->seed, mb->streamIds.data() + a);
			if (!mb->shards[d]) return false;
		}
		std::vector<int64_t> off(cnt + 1);
		for (uint32_t i = 0; i <= cnt; ++i) off[i] = offsets[a + i] - offsets[a];
		const size_t o = (size_t)offsets[a];
		return speechPlayer_batchSetFramesHost(mb->shards[d], off.data(), frames ? frames + o : nullptr, minFrameDuration + o, fadeDuration + o,
		                                       userIndex ? userIndex + o : nullptr, isNull ? isNull + o : nullptr, nullptr) == 0;
	}, err);
	if (!ok) return fail(err);
	mb->first = first;
	return 0;
}

long long speechPlayer_multiBatchSynthesizeHost(speechPlayer_multiBatch_t *mb, unsigned int sampleCount, sample *out,
                                                unsigned int *samplesWritten) {
	if (!mb) return fail("null batch");
	if (!out) return fail("null output");
	std::lock_guard<std::mutex> lk(mb->mu);
	std::vector<long long> got(mb->devices.size(), 0);
	std::string err;
	const bool ok = forEachShard(mb, [&](size_t d) -> bool {
		const uint32_t a = mb->first[d], b = mb->first[d + 1];
		if (a == b) return true;
		if (!mb->shards[d]) { g_lastError = "no frames queued (call SetFramesHost first)"; return false; }
		got[d] = speechPlayer_batchSynthesizeHost(mb->shards[d], sampleCount, out + (size_t)a * sampleCount, samplesWritten ? samplesWritten + a : nullptr);
		return got[d] >= 0;
	}, err);
	if (!ok) return fail(err);
	long long total = 0;
	for (long long g : got) total += g;
	return total;
}

int speechPlayer_multiBatchGetShards(speechPlayer_multiBatch_t *mb, unsigned int *firstStream) {
	if (!mb || !firstStream) return fail("null argument");
	std::lock_guard<std::mutex> lk(mb->mu);
	for (size_t d = 0; d < mb->first.size(); ++d) firstStream[d] = mb->first[d];
	return 0;
}

int speechPlayer_multiBatchGetLastIndices(speechPlayer_multiBatch_t *mb, int *lastIndex) {
	if (!mb || !lastIndex) return fail("null argument");
	std::lock_guard<std::mutex> lk(mb->mu);
	std::string err;
	const bool ok = forEachShard(mb, [&](size_t d) -> bool {
		const uint32_t a = mb->first[d], b = mb->first[d + 1];
		if (a == b || !mb->shards[d]) { for (uint32_t s = a; s < b; ++s) lastIndex[s] = -1; return true; }
		return speechPlayer_batchGetLastIndices(mb->shards[d], lastIndex + a) == 0;
	}, err);
	return ok ? 0 : fail(err);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// C-ABI: long-utterance path (klatt_long.cu)
// ------------------------------------------------------------------------------------------------
static std::atomic<unsigned long long> g_longSerialFallbacks{0};
// how many streams rendered by the long path in this process had to take the serial phase fallback (tests, bench); for
// speechPlayer_synthesizeLong a stream is a call
extern "C" unsigned long long speechPlayer_debugLongSerialFallbacks(void) { return g_longSerialFallbacks.load(); }

// One call of the long path: numStreams pre-queued streams (host arrays in the layout of speechPlayer_batchSetFramesHost),
// already validated, with the output offsets from the timeline law.
struct LongCall {
	int sampleRate;
	uint32_t numStreams;
	const int64_t *offsets;                 // [numStreams + 1]
	const speechPlayer_frame_t *frames;     // null: every request is a NULL request
	const unsigned int *minDur, *fadeDur;
	const unsigned char *isNull;            // may be null
	uint64_t seed;
	const uint64_t *streamIds;              // [numStreams]
	uint32_t chunkTicks;                    // 0: chosen per group (batch default)
	const int64_t *outOffsets;              // [numStreams + 1]: stream s renders outOffsets[s + 1] - outOffsets[s] samples
	int16_t *out;
	bool outOnDevice;
	unsigned char *serialPhase;             // [numStreams] or null
};

// Below this many chunks a group of the batch entry halves its default chunk length (1024), down to 64: fewer chunks than
// this leave SMs idle in the stage kernels (one thread per chunk).  Measured on a B200 by tools/long_batch_bench.py.
static constexpr uint64_t kLongFillChunks = 65536;

static long long renderLong(const LongCall &C, double *renderMs, unsigned long long *kernelLaunches) {
	int dev = pickDevice();
	if (dev < 0) return fail("no usable CUDA device (this library has no CPU fallback)");
	DeviceGuard g(dev);
	auto envU64 = [](const char *name, uint64_t dflt) {
		const char *e = getenv(name);
		return (e && *e) ? (uint64_t)strtoull(e, nullptr, 0) : dflt;
	};
	// streams are rendered in consecutive groups of at most this many ticks (one launch sequence each; a stream longer than
	// that is a group of its own).  The scratch is ~22 bytes per tick (five float signals, the int16 output, the chunk maps): 6 GB at the default.
	static const uint64_t groupTicks = std::max<uint64_t>(envU64("NVSP_LONG_BATCH_TICKS", 1ull << 28), 1);
	// Scratch of the long path: grow-only buffers kept per device between calls (a config-4 call needs ~5 GB of stage signals;
	// allocating and freeing them inside every call cost 10-20 ms of a 40 ms render).  One long render at a time per process.
	struct LongScratch {
		DevBuf dFrames, dMin, dFade, dNull, dOff, dPlans, dStart, dPrev, dPitch, dVib, dTable, dChunkBase;
		DevBuf sig, maps, st, ph, pcm, phChunks, phStart, phFail, scanTmp;
	};
	static std::mutex longMu;
	static LongScratch pool[16];
	std::lock_guard<std::mutex> longLock(longMu);
	LongScratch local;
	static const bool usePool = !(getenv("NVSP_LONG_POOL") && atoi(getenv("NVSP_LONG_POOL")) == 0);
	LongScratch &S = (usePool && dev >= 0 && dev < 16) ? pool[dev] : local;
	struct Cleanup {
		std::vector<DevBuf *> bufs;
		cudaEvent_t e0 = nullptr, e1 = nullptr;
		~Cleanup() {
			for (DevBuf *b : bufs) b->release();
			if (e0) cudaEventDestroy(e0);
			if (e1) cudaEventDestroy(e1);
		}
	} cleanup;
	if (&S == &local) cleanup.bufs = {&S.dFrames, &S.dMin, &S.dFade, &S.dNull, &S.dOff, &S.dPlans, &S.dStart, &S.dPrev, &S.dPitch, &S.dVib,
	                                  &S.dTable, &S.dChunkBase, &S.sig, &S.maps, &S.st, &S.ph, &S.pcm, &S.phChunks, &S.phStart, &S.phFail,
	                                  &S.scanTmp};
	CU(cudaEventCreate(&cleanup.e0));
	CU(cudaEventCreate(&cleanup.e1));
	cudaStream_t stream = nullptr;
	// The glottal phase is the reference's FP64 recurrence, parallel in time by speculation + verification
	// (klatt_long_phase.cuh).  The streams whose check failed -- or all, with NVSP_LONG_PHASE=serial -- are rendered again
	// with the plain recurrence on one thread per stream: slow, exact by definition.
	static const bool forceSerial = getenv("NVSP_LONG_PHASE") && !strcmp(getenv("NVSP_LONG_PHASE"), "serial");
	unsigned long long launches = 0;
	double ms = 0.0;
	const uint32_t N = C.numStreams;
	std::vector<uint64_t> ticks(N);
	for (uint32_t s = 0; s < N; ++s) ticks[s] = (uint64_t)(C.outOffsets[s + 1] - C.outOffsets[s]);
	for (uint32_t g0 = 0, g1; g0 < N; g0 = g1) {
		uint64_t sum = ticks[g0];
		for (g1 = g0 + 1; g1 < N && sum + ticks[g1] <= groupTicks; ++g1) sum += ticks[g1];
		const uint32_t G = g1 - g0;
		const int64_t reqBase = C.offsets[g0];
		const size_t n = (size_t)(C.offsets[g1] - reqBase);
		uint32_t chunkTicks = C.chunkTicks;
		if (chunkTicks == 0) {  // the batch default: 1024 ticks, shorter while the group has too few chunks to fill the GPU
			auto chunksAt = [&](uint64_t L) { uint64_t c = 0; for (uint32_t s = g0; s < g1; ++s) c += (ticks[s] + L - 1) / L; return c; };
			chunkTicks = 1024;
			while (chunkTicks > 64 && chunksAt(chunkTicks) < kLongFillChunks) chunkTicks >>= 1;
		}
		chunkTicks = std::max(chunkTicks, 64u) & ~31u;  // whole 32-tick tiles (klatt_long.cu stage kernels)
		std::vector<uint32_t> chunkBase(G + 1, 0);
		for (uint32_t k = 0; k < G; ++k) {
			const uint64_t c = chunkBase[k] + (ticks[g0 + k] + chunkTicks - 1) / chunkTicks;
			if (c > 0x7fffffffull) return fail("stream too long for one call");
			chunkBase[k + 1] = (uint32_t)c;
		}
		const uint32_t numChunks = chunkBase[G];
		if (!S.dFrames.reserve(n * sizeof(speechPlayer_frame_t)) || !S.dMin.reserve(n * 4) || !S.dFade.reserve(n * 4) || !S.dNull.reserve(n) ||
		    !S.dOff.reserve((G + 1) * 8) || !S.dPlans.reserve(n * sizeof(FadePlanF32)) || !S.dStart.reserve((n + G) * 8) ||
		    !S.dPrev.reserve(n * 4) || !S.dPitch.reserve(n * 8 * 4) || !S.dVib.reserve(n * 8) || !S.dTable.reserve(G * sizeof(LongStream)) ||
		    !S.dChunkBase.reserve((G + 1) * 4))
			return -1;
		const unsigned char *isNull = C.isNull ? C.isNull + reqBase : nullptr;
		std::vector<unsigned char> allNull;
		if (!C.frames) { allNull.assign(n, 1); isNull = allNull.data(); }
		if (n) {
			if (C.frames) CU(cudaMemcpyAsync(S.dFrames.p, C.frames + reqBase, n * sizeof(speechPlayer_frame_t), cudaMemcpyHostToDevice, stream));
			else CU(cudaMemsetAsync(S.dFrames.p, 0, n * sizeof(speechPlayer_frame_t), stream));
			CU(cudaMemcpyAsync(S.dMin.p, C.minDur + reqBase, n * 4, cudaMemcpyHostToDevice, stream));
			CU(cudaMemcpyAsync(S.dFade.p, C.fadeDur + reqBase, n * 4, cudaMemcpyHostToDevice, stream));
			if (isNull) CU(cudaMemcpyAsync(S.dNull.p, isNull, n, cudaMemcpyHostToDevice, stream));
		}
		std::vector<int64_t> off(G + 1);
		for (uint32_t k = 0; k <= G; ++k) off[k] = C.offsets[g0 + k] - reqBase;
		CU(cudaMemcpyAsync(S.dOff.p, off.data(), (G + 1) * 8, cudaMemcpyHostToDevice, stream));
		// the stream table: stream k's requests at off[k] of the flat arrays, its start ticks at off[k] + k (nReq + 1 each)
		const double *dFrames = S.dFrames.as<double>();
		double *dPitch = S.dPitch.as<double>();
		std::vector<LongStream> table(G);
		for (uint32_t k = 0; k < G; ++k) {
			LongStream &L = table[k];
			const size_t a = (size_t)off[k];
			L.frames = dFrames + a * kNumParams; L.minDur = S.dMin.as<uint32_t>() + a; L.fadeDur = S.dFade.as<uint32_t>() + a;
			L.isNull = isNull ? S.dNull.as<uint8_t>() + a : nullptr;
			L.plans = S.dPlans.as<FadePlanF32>() + a; L.nReq = (uint32_t)(off[k + 1] - off[k]); L.sampleRate = C.sampleRate;
			L.seed = C.seed; L.streamId = C.streamIds[g0 + k];
			L.cap = ticks[g0 + k]; L.outBase = (uint64_t)(C.outOffsets[g0 + k] - C.outOffsets[g0]);
			L.start = S.dStart.as<uint64_t>() + a + k; L.prevReal = S.dPrev.as<int32_t>() + a;
			L.pitchPop = dPitch + a; L.pitchOld = dPitch + n + a; L.pitchNew = dPitch + 2 * n + a; L.pitchInc = dPitch + 3 * n + a;
			L.vibPosStart = S.dVib.as<uint64_t>() + a;
		}
		CU(cudaMemcpyAsync(S.dTable.p, table.data(), G * sizeof(LongStream), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(S.dChunkBase.p, chunkBase.data(), (G + 1) * 4, cudaMemcpyHostToDevice, stream));
		CU(cudaEventRecord(cleanup.e0, stream));
		CU(launchKlattPlan(S.dOff.as<int64_t>(), G, n, dFrames, S.dFade.as<uint32_t>(), isNull ? S.dNull.as<uint8_t>() : nullptr,
		                   C.sampleRate, S.dPlans.as<FadePlanF32>(), stream));
		LongTable T;
		T.streams = S.dTable.as<LongStream>(); T.chunkBase = S.dChunkBase.as<uint32_t>(); T.numStreams = G; T.one = table[0];
		CU(launchKlattLongTimeline(T, stream));
		launches += 2;
		if (numChunks == 0) continue;
		// signals in virtual ticks: stream k's tick t at chunkBase[k] * chunkTicks + t
		const size_t pad = (size_t)numChunks * chunkTicks + 64;
		if (!S.sig.reserve(5 * pad * sizeof(float)) || !S.maps.reserve((size_t)numChunks * 6 * sizeof(Affine)) ||
		    !S.st.reserve((size_t)numChunks * 6 * sizeof(float2)) || !S.ph.reserve((size_t)numChunks * 2 * sizeof(double)) ||
		    !S.phChunks.reserve((size_t)numChunks * sizeof(PhaseChunk)) || !S.scanTmp.reserve(klattLongScanScratchBytes(numChunks)) ||
		    !S.phStart.reserve((size_t)numChunks * sizeof(double)) || !S.phFail.reserve(std::max<size_t>(16, (size_t)G * 4)))
			return -1;
		int16_t *dPcm = C.out + C.outOffsets[g0];
		if (!C.outOnDevice) {
			if (!S.pcm.reserve((sum + 64) * sizeof(int16_t))) return -1;
			dPcm = S.pcm.as<int16_t>();
		}
		float *f = S.sig.as<float>();
		uint32_t *dFail = S.phFail.as<uint32_t>();
		uint64_t *advance = S.ph.as<uint64_t>();
		auto synth = [&]() {
			return launchKlattLongSynth(T, numChunks, chunkTicks, S.phChunks.as<PhaseChunk>(), S.phStart.as<double>(), dFail, f, f + pad,
			                            f + 2 * pad, f + 3 * pad, f + 4 * pad, S.maps.as<Affine>(), S.st.as<float2>(), S.scanTmp.p, dPcm,
			                            &launches, stream);
		};
		CU(cudaMemsetAsync(dFail, forceSerial ? 0xff : 0, (size_t)G * 4, stream));
		CU(launchKlattLongPhase(T, numChunks, chunkTicks, advance, advance + numChunks, S.phChunks.as<PhaseChunk>(), S.phStart.as<double>(),
		                        dFail, forceSerial, &launches, stream));
		CU(synth());
		CU(cudaEventRecord(cleanup.e1, stream));
		std::vector<uint32_t> failed(G, 0);
		CU(cudaMemcpyAsync(failed.data(), dFail, (size_t)G * 4, cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		uint32_t nFailed = 0;
		for (uint32_t k = 0; k < G; ++k) nFailed += failed[k] && ticks[g0 + k] ? 1 : 0;
		if (nFailed && !forceSerial) {
			if (getenv("NVSP_VERBOSE"))
				fprintf(stderr, "[nvspeechplayer_b200] long path: speculative phase of %u stream(s) not verified, serial fallback\n", nFailed);
			// only the failed streams' chunks get new phases; the source and stage passes run again for all
			CU(launchKlattLongPhase(T, numChunks, chunkTicks, advance, advance + numChunks, S.phChunks.as<PhaseChunk>(), S.phStart.as<double>(),
			                        dFail, true, &launches, stream));
			CU(synth());
			CU(cudaEventRecord(cleanup.e1, stream));
			g_longSerialFallbacks += nFailed;
		}
		if (C.serialPhase)
			for (uint32_t k = 0; k < G; ++k) C.serialPhase[g0 + k] = (failed[k] && ticks[g0 + k]) ? 1 : 0;
		if (!C.outOnDevice) CU(cudaMemcpyAsync(C.out + C.outOffsets[g0], dPcm, sum * sizeof(int16_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		float groupMs = 0;
		CU(cudaEventElapsedTime(&groupMs, cleanup.e0, cleanup.e1));
		ms += groupMs;
	}
	if (renderMs) *renderMs = ms;
	if (kernelLaunches) *kernelLaunches = launches;
	return C.outOffsets[N];
}

extern "C" long long speechPlayer_synthesizeLong(int sampleRate, const speechPlayer_frame_t *frames,
                                                 const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                                 const unsigned char *isNull, unsigned int numFrames, uint64_t seed,
                                                 uint64_t streamId, unsigned int chunkTicks, sample *out,
                                                 unsigned long long maxSamples, int outOnDevice, double *renderMs,
                                                 unsigned long long *kernelLaunches) {
	g_lastError.clear();
	if (sampleRate <= 0) return fail("sampleRate must be positive");
	if (numFrames && (!minFrameDuration || !fadeDuration)) return fail("durations missing");
	if (numFrames == 0) return 0;
	if (chunkTicks == 0) {
		const char *e = getenv("NVSP_LONG_CHUNK");
		chunkTicks = (e && *e) ? (unsigned)strtoul(e, nullptr, 0) : 1024u;
	}
	const int64_t offsets[2] = {0, (int64_t)numFrames};
	const int64_t outOffsets[2] = {0, (int64_t)std::min<unsigned long long>(speechPlayer_timelineSamples(minFrameDuration, fadeDuration, numFrames),
	                                                                          maxSamples)};
	LongCall C;
	C.sampleRate = sampleRate; C.numStreams = 1; C.offsets = offsets; C.frames = frames; C.minDur = minFrameDuration;
	C.fadeDur = fadeDuration; C.isNull = isNull; C.seed = seed; C.streamIds = &streamId; C.chunkTicks = std::max(chunkTicks, 64u);
	C.outOffsets = outOffsets; C.out = reinterpret_cast<int16_t *>(out); C.outOnDevice = outOnDevice != 0; C.serialPhase = nullptr;
	return renderLong(C, renderMs, kernelLaunches);
}

extern "C" long long speechPlayer_synthesizeLongBatch(int sampleRate, unsigned int numStreams, const int64_t *offsets,
                                                      const speechPlayer_frame_t *frames, const unsigned int *minFrameDuration,
                                                      const unsigned int *fadeDuration, const unsigned char *isNull, uint64_t seed,
                                                      const uint64_t *streamIds, unsigned int chunkTicks,
                                                      const unsigned long long *maxSamples, sample *out, int64_t *outOffsets,
                                                      int outOnDevice, unsigned char *serialPhase, double *renderMs,
                                                      unsigned long long *kernelLaunches) {
	g_lastError.clear();
	// everything is checked, and the output sized, on the host: a size query needs no device
	if (sampleRate <= 0) return fail("sampleRate must be positive");
	if (numStreams == 0) return fail("numStreams must be positive");
	if (!offsets) return fail("null offsets");
	if (!outOffsets) return fail("null outOffsets");
	if (offsets[0] != 0) return fail("offsets[0] must be 0");
	for (unsigned s = 0; s < numStreams; ++s) {
		if (offsets[s + 1] < offsets[s]) return fail("offsets must be non-decreasing");
		if (offsets[s + 1] - offsets[s] > (int64_t)0xffffffffll) return fail("too many requests in one stream");
	}
	const int64_t total = offsets[numStreams];
	if (total && (!minFrameDuration || !fadeDuration)) return fail("durations missing");
	outOffsets[0] = 0;
	for (unsigned s = 0; s < numStreams; ++s) {
		unsigned long long t = speechPlayer_timelineSamples(minFrameDuration + offsets[s], fadeDuration + offsets[s],
		                                                    (unsigned)(offsets[s + 1] - offsets[s]));
		if (maxSamples) t = std::min(t, maxSamples[s]);
		outOffsets[s + 1] = outOffsets[s] + (int64_t)t;
	}
	if (serialPhase) memset(serialPhase, 0, numStreams);
	if (renderMs) *renderMs = 0;
	if (kernelLaunches) *kernelLaunches = 0;
	if (!out || outOffsets[numStreams] == 0) return outOffsets[numStreams];
	std::vector<uint64_t> ids;
	if (!streamIds) {
		ids.resize(numStreams);
		for (unsigned s = 0; s < numStreams; ++s) ids[s] = s;
		streamIds = ids.data();
	}
	LongCall C;
	C.sampleRate = sampleRate; C.numStreams = numStreams; C.offsets = offsets; C.frames = frames; C.minDur = minFrameDuration;
	C.fadeDur = fadeDuration; C.isNull = isNull; C.seed = seed; C.streamIds = streamIds; C.chunkTicks = chunkTicks;
	C.outOffsets = outOffsets; C.out = reinterpret_cast<int16_t *>(out); C.outOnDevice = outOnDevice != 0; C.serialPhase = serialPhase;
	return renderLong(C, renderMs, kernelLaunches);
}
