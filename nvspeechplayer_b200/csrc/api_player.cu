// The per-handle C-ABI of include/speechPlayer.h (and speechPlayer_synthesizeBatch of include/speechPlayer_batch.h): the
// handle table, per-player request mirrors, the low-latency pull path, and the debug hooks.
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
#include <atomic>
#include <chrono>
#include <cstdio>
#include <functional>
#include <memory>
#include <mutex>
#include <vector>

#include "../../include/speechPlayer.h"
#include "../../include/speechPlayer_batch.h"
#include "glibc_rand.h"
#include "host.h"
#include "host_pool.h"
#include "pull_manager.h"

using namespace klatt;

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
	DevBuf dState;  // StreamState
	// host mirror of the requests the device has not consumed yet (src/frame.cpp:33 frameRequestQueue)
	std::vector<double> frames;
	std::vector<uint32_t> minDur, fadeDur;
	std::vector<int32_t> userIndex;
	std::vector<uint8_t> isNull;
	uint32_t qBase = 0;       // absolute index of mirror[0] == requests consumed so far
	bool mirrorDirty = false; // device copy of the mirror is stale
	bool purgePending = false;
	QueueBufs queue;
	DevBuf dReplay, dDesc;
	std::vector<int32_t> replayHost;  // kNoiseReplay: user-provided draws
	bool replayDirty = false;
	uint64_t generated = 0;   // samples generated so far (== draws/2)
	int lastIndex = -1;
	HostPipe pipe;
	std::vector<int16_t> hostScratch;  // rows of the last synthesize call before the written prefixes are handed out
	// SPEECHPLAYER_PRECISION_STREAM: host frame manager, carried device state, staging for one launch
	std::unique_ptr<PullManager> pull;
	DevBuf dPull;  // PullState
	DevBuf dSegs, dPullPcm, dDraws, dPullDbg;
	PinnedBuf hPullStage;                 // pinned and mapped: [segments | pcm | draws]
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
			if (n && queue.upload(frames.data(), minDur.data(), fadeDur.data(), userIndex.data(), isNull.data(), n, stream) != 0) return -1;
			mirrorDirty = false;
		}
		if (purgePending) {
			static const uint32_t one = 1;
			CU(cudaMemcpyAsync(&dState.as<StreamState>()->fm.purgePending, &one, 4, cudaMemcpyHostToDevice, stream));
			purgePending = false;
		}
		d.state = dState.as<StreamState>();
		d.frames = queue.frames.as<double>();
		d.minDur = queue.minDur.as<uint32_t>();
		d.fadeDur = queue.fadeDur.as<uint32_t>();
		d.userIndex = queue.userIndex.as<int32_t>();
		d.isNull = queue.isNull.as<uint8_t>();
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
};

// Locks a set of players in address order, the one order every multi-player call takes them in; a handle may appear only
// once.  Taken before g_noiseMu / g_pullBatchMu.
struct PlayerLocks {
	std::vector<Player *> order;
	bool lock(const std::vector<Player *> &ps) {
		order = ps;
		std::sort(order.begin(), order.end());
		if (std::adjacent_find(order.begin(), order.end()) != order.end()) {
			order.clear();
			return false;
		}
		for (Player *p : order) p->mu.lock();
		return true;
	}
	~PlayerLocks() {
		for (Player *p : order) p->mu.unlock();
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
	if (envIs("NVSP_PRECISION", "fp32") || envIs("NVSP_PRECISION", "f32") || envIs("NVSP_PRECISION", "FP32")) return kPrecisionF32;
	if (envIs("NVSP_PRECISION", "stream") || envIs("NVSP_PRECISION", "pull")) return kPrecisionStream;
	return kPrecisionF64;
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
	if (!p->dState.reserve(sizeof(StreamState), "cudaMalloc(state)") ||
	    !cudaOk(initStates(p->dState.as<StreamState>(), 1, nullptr), "init state") ||
	    !cudaOk(cudaStreamSynchronize(nullptr), "init state sync")) {
		delete p;
		return nullptr;
	}
	if (precision == kPrecisionStream) {
		p->pull.reset(new PullManager(sampleRate));
		if (!p->dPull.reserve(sizeof(PullState), "cudaMalloc(pull state)") ||
		    !cudaOk(launchKlattPullInit(p->dPull.as<PullState>(), nullptr), "init pull state") ||
		    !cudaOk(cudaStreamSynchronize(nullptr), "init pull state sync") ||
		    !cudaOk(p->hPullStage.reserve(Player::kStageSegs + Player::kStagePcm + Player::kStageDraws, cudaHostAllocMapped),
		            "cudaHostAlloc(pull staging)") ||
		    !cudaOk(cudaHostGetDevicePointer((void **)&p->dPullStage, p->hPullStage.p, 0), "cudaHostGetDevicePointer") ||
		    !p->dSegs.reserve(Player::kStageSegs) || !p->dPullPcm.reserve(Player::kStagePcm)) {
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
	return speechPlayer_initializeEx(sampleRate, envPrecision(), envIs("NVSP_NOISE", "philox") ? kNoisePhilox : kNoiseGlibc,
	                                 envNum<uint64_t>("NVSP_SEED", 0xB200ull), sid);
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
	static const bool zc = envNum<uint64_t>("NVSP_PULL_ZEROCOPY", 1) != 0;
	return zc;
}
static bool pullDebugPhases() {
	static const bool dbg = envIs("NVSP_PULL_DEBUG");
	return dbg;
}
static int pullStage(Player *p, uint32_t got, PullCtx &X, const PullSeg *&segSrc, int16_t *&pcmOut, bool &zeroCopy, cudaStream_t stream) {
	zeroCopy = pullZeroCopy();
	PullSeg *hSegs = p->hPullStage.as<PullSeg>();
	int32_t *hDraws = reinterpret_cast<int32_t *>(p->hPullStage.as<unsigned char>() + Player::kStageSegs + Player::kStagePcm);
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
	X.state = p->dPull.as<PullState>(); X.noiseMode = p->noiseMode; X.seed = p->seed; X.streamId = p->streamId;
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
	static const bool phaseSerial = envIs("NVSP_PULL_PHASE", "serial");
	X.phaseMode = phaseSerial ? 0 : 1;
	if (pullDebugPhases() && p->dPullDbg.reserve(16 * sizeof(long long))) X.dbg = p->dPullDbg.as<long long>();
	return 0;
}

// One pull of a SPEECHPLAYER_PRECISION_STREAM player: one launch of klatt_pull_kernel per kPullMaxTicks, the samples come back
// through pinned memory.  The caller holds p->mu.
static long long synthesizePull(Player *p, unsigned int sampleCount, int16_t *out) {
	DeviceGuard g(p->device);
	if (!p->pipe.init()) return -1;
	cudaStream_t stream = p->pipe.compute;
	int16_t *hPcm = reinterpret_cast<int16_t *>(p->hPullStage.as<unsigned char>() + Player::kStageSegs);
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
// own speechPlayer_synthesize would have produced (same kernel body, same carried state).  Players with the process-global
// glibc noise never come here: speechPlayer_synthesizeBatch renders them one after another.
static std::mutex g_pullBatchMu;
static PullBatchItem *g_pullItemsHost = nullptr, *g_pullItemsDev = nullptr;
static size_t g_pullItemsCap = 0;
static int g_pullItemsDevice = -1;

// The caller holds the players' locks.
static long long synthesizePullBatch(std::vector<Player *> &ps, unsigned int sampleCount, int16_t *out, unsigned int *samplesWritten) {
	const size_t n = ps.size();
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
	// staging, no replay upload pending.
	bool parallel = pullZeroCopy() && !pullDebugPhases() && n >= 8 && HostPool::get().helpers() > 0;
	for (size_t i = 0; i < n && parallel; ++i)
		if (ps[i]->noiseMode == kNoiseReplay && ps[i]->replayDirty) parallel = false;
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
		static const bool timing = envIs("NVSP_PULL_TIMING");  // host-side phases of a batched pull, one line per launch
		const auto t0 = std::chrono::steady_clock::now();
		forEach(prepare);
		if (failed.load()) return -1;
		if (!any.load()) break;
		const auto t1 = std::chrono::steady_clock::now();
		CU(launchKlattPullBatch(g_pullItemsHost, g_pullItemsDev, (uint32_t)n, stream));
		for (size_t i = 0; i < n; ++i)
			if (got[i] && !zero[i])
				CU(cudaMemcpyAsync(ps[i]->hPullStage.as<unsigned char>() + Player::kStageSegs, g_pullItemsHost[i].pcmOut, (size_t)got[i] * sizeof(int16_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		const auto t2 = std::chrono::steady_clock::now();
		forEach([&](size_t i) {
			if (!got[i]) return;
			memcpy(out + i * (size_t)sampleCount + total[i], ps[i]->hPullStage.as<unsigned char>() + Player::kStageSegs, (size_t)got[i] * sizeof(int16_t));
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

// One launch for the FP64 / FP32 handles ps[0..n) (the caller holds their locks and has checked that they share device, sample
// rate, precision, noise mode and seed).
static long long synthesizeHandles(Player *const *ps, unsigned int n, unsigned int sampleCount, sample *sampleBuf,
                                   unsigned int *samplesWritten) {
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
	std::vector<StreamDesc> descs(n);
	for (unsigned i = 0; i < n; ++i)
		if (ps[i]->prepare(descs[i], sampleCount, stream) != 0) return -1;
	if (!lead->dDesc.reserve(sizeof(StreamDesc) * (size_t)n)) return -1;
	CU(cudaMemcpyAsync(lead->dDesc.p, descs.data(), sizeof(StreamDesc) * (size_t)n, cudaMemcpyHostToDevice, stream));
	CU(cudaStreamSynchronize(stream));
	std::vector<uint32_t> written(n);
	std::vector<StreamResult> results(n);
	NoiseConfig nc{lead->noiseMode, lead->seed};
	// The reference's generate() returns the count and leaves sampleBuf[count..] untouched (src/speechWaveGenerator.cpp:210),
	// so the rows land in a scratch buffer first and only the written prefix of each row is handed to the caller.
	std::vector<int16_t> &scratch = lead->hostScratch;
	scratch.resize((size_t)n * sampleCount);
	long long total = renderToHost(lead->pipe, lead->precision, lead->dDesc.as<StreamDesc>(), n, lead->sampleRate,
	                               sampleCount, scratch.data(), written.data(), results.data(), nc, nullptr);
	if (total < 0) return -1;
	for (unsigned i = 0; i < n; ++i) {
		ps[i]->absorb(results[i], written[i]);
		if (samplesWritten) samplesWritten[i] = written[i];
		memcpy(reinterpret_cast<int16_t *>(sampleBuf) + (size_t)i * sampleCount, scratch.data() + (size_t)i * sampleCount,
		       sizeof(int16_t) * (size_t)written[i]);
	}
	if (lead->noiseMode == kNoiseGlibc) {
		// the reference consumes exactly two rand() calls per generated sample: rewind to that point (one handle only, see
		// speechPlayer_synthesizeBatch)
		g_noise = checkpoint;
		g_noise.skip((uint64_t)written[0] * 2);
	}
	return total;
}

long long speechPlayer_synthesizeBatch(speechPlayer_handle_t *handles, unsigned int numHandles, unsigned int sampleCount,
                                       sample *sampleBuf, unsigned int *samplesWritten) {
	g_lastError.clear();
	if (numHandles == 0 || sampleCount == 0) return 0;
	if (!handles || !sampleBuf) return fail("null argument");
	std::vector<Player *> ps(numHandles);
	bool anyPull = false, anyGlibc = false;
	for (unsigned i = 0; i < numHandles; ++i) {
		ps[i] = lookup(handles[i]);
		if (!ps[i]) return fail("bad handle in batch");
		anyPull = anyPull || ps[i]->pull != nullptr;
		anyGlibc = anyGlibc || ps[i]->noiseMode == kNoiseGlibc;
	}
	if (!anyPull)
		for (unsigned i = 0; i < numHandles; ++i) {
			if (ps[i]->precision != ps[0]->precision || ps[i]->sampleRate != ps[0]->sampleRate ||
			    ps[i]->device != ps[0]->device || ps[i]->noiseMode != ps[0]->noiseMode || ps[i]->seed != ps[0]->seed)
				return fail("handles of one batch must share device, sample rate, precision and noise mode");
		}
	PlayerLocks locks;
	if (!locks.lock(ps)) return fail("duplicate handle in batch");
	// The process-global glibc sequence is handed out in call order: a player takes two draws per sample it generates, and
	// how many it generates is known only once it has rendered.  So with glibc noise the handles render one after another, in
	// handle order, each exactly as its own speechPlayer_synthesize would.
	const bool oneByOne = anyGlibc && numHandles > 1;
	if (anyPull) {  // low-latency players: one block per player, one launch for all of them
		for (unsigned i = 0; i < numHandles; ++i)
			if (!ps[i]->pull || ps[i]->device != ps[0]->device)
				return fail("handles of one batch must share device and precision");
		if (numHandles > 1 && !oneByOne) return synthesizePullBatch(ps, sampleCount, reinterpret_cast<int16_t *>(sampleBuf), samplesWritten);
		long long total = 0;
		for (unsigned i = 0; i < numHandles; ++i) {
			long long w = synthesizePull(ps[i], sampleCount, reinterpret_cast<int16_t *>(sampleBuf) + (size_t)i * sampleCount);
			if (w < 0) return -1;
			if (samplesWritten) samplesWritten[i] = (unsigned int)w;
			total += w;
		}
		return total;
	}
	if (!oneByOne) return synthesizeHandles(ps.data(), numHandles, sampleCount, sampleBuf, samplesWritten);
	long long total = 0;
	for (unsigned i = 0; i < numHandles; ++i) {
		long long w = synthesizeHandles(&ps[i], 1, sampleCount, sampleBuf + (size_t)i * sampleCount, samplesWritten ? samplesWritten + i : nullptr);
		if (w < 0) return -1;
		total += w;
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
	DeviceGuard g(p->device);
	delete p;
}

unsigned long long speechPlayer_timelineSamples(const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                                unsigned int n) {
	return timelineTicks(minFrameDuration, fadeDuration, n);
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
