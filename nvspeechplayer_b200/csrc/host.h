// The host layer shared by the C-ABI units (api_player.cu, api_batch.cu, api_long.cu): errors, device selection,
// owning device / pinned buffers, environment knobs, the timeline law, and the render pipeline that players and batches
// both use (launchRender, renderToHost; out-of-line parts in host.cu).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/speechPlayer.h"
#include "klatt_common.h"
#include "launch.h"

namespace klatt {

static_assert(sizeof(speechPlayer_frame_t) == sizeof(double) * kNumParams, "a queued frame is kNumParams doubles");

// ------------------------------------------------------------------------------------------------
// errors: fail() records the message for speechPlayer_lastError (per thread) and returns -1
// ------------------------------------------------------------------------------------------------
extern thread_local std::string g_lastError;
int fail(const std::string &what);
void setLastError(const char *what);  // also used by the host-only translation units (ipa_frames.cpp)
bool cudaOk(cudaError_t e, const char *what);
#define CU(call) do { if (!cudaOk((call), #call)) return -1; } while (0)

// ------------------------------------------------------------------------------------------------
// environment knobs (INTEGRATION.md section 5): an unset or empty variable takes the default; numbers parse with base 0
// ------------------------------------------------------------------------------------------------
template <class T = uint64_t> T envNum(const char *name, T dflt) {
	const char *e = getenv(name);
	return (e && *e) ? (T)strtoull(e, nullptr, 0) : dflt;
}
// the variable is set to `value`, or (value == nullptr) set at all
inline bool envIs(const char *name, const char *value = nullptr) {
	const char *e = getenv(name);
	return e && *e && (!value || strcmp(e, value) == 0);
}

// ------------------------------------------------------------------------------------------------
// devices: the calling thread's current device, unless NVSP_DEVICE says otherwise (applied once)
// ------------------------------------------------------------------------------------------------
int pickDevice();

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

// ------------------------------------------------------------------------------------------------
// owning buffers: freed by the destructor, on whatever device is current then (owners destroy under a DeviceGuard)
// ------------------------------------------------------------------------------------------------
// grow-only device buffer
struct DevBuf {
	void *p = nullptr;
	size_t cap = 0;
	DevBuf() = default;
	DevBuf(const DevBuf &) = delete;
	DevBuf &operator=(const DevBuf &) = delete;
	DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
	DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
	~DevBuf() {
		if (p) cudaFree(p);
	}
	bool reserve(size_t bytes, const char *what = "cudaMalloc") {
		if (bytes <= cap) return true;
		size_t want = std::max(bytes, cap * 2);
		void *np = nullptr;
		if (!cudaOk(cudaMalloc(&np, want), what)) return false;
		if (p) cudaFree(p);
		p = np; cap = want;
		return true;
	}
	template <class T> T *as() const { return static_cast<T *>(p); }
};

// pinned host memory of exactly the size last asked for (a larger request replaces it; the contents are not kept)
struct PinnedBuf {
	void *p = nullptr;
	size_t cap = 0;
	PinnedBuf() = default;
	PinnedBuf(const PinnedBuf &) = delete;
	PinnedBuf &operator=(const PinnedBuf &) = delete;
	~PinnedBuf() {
		if (p) cudaFreeHost(p);
	}
	cudaError_t reserve(size_t bytes, unsigned flags = cudaHostAllocDefault) {
		if (bytes <= cap) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr; cap = 0;
		cudaError_t e = cudaHostAlloc(&p, bytes, flags);
		if (e == cudaSuccess) cap = bytes;
		else p = nullptr;
		return e;
	}
	template <class T> T *as() const { return static_cast<T *>(p); }
};

// The five device arrays of a request queue (frames [n][kNumParams], minDur, fadeDur, userIndex, isNull), grow-only.
// upload() sizes and copies the arrays whose host pointer is given (at least one element, so a present array is never
// null) and skips the others.
struct QueueBufs {
	DevBuf frames, minDur, fadeDur, userIndex, isNull;
	int upload(const void *hFrames, const uint32_t *hMin, const uint32_t *hFade, const int32_t *hUix, const uint8_t *hNull, size_t n,
	           cudaStream_t stream);
};

// ------------------------------------------------------------------------------------------------
// the timeline law: ticks a queue yields, sum of max(M + 1, max(F, 1) + 2) (reference src/frame.cpp:41-80)
// ------------------------------------------------------------------------------------------------
inline unsigned long long timelineTicks(const unsigned int *minDur, const unsigned int *fadeDur, size_t n) {
	unsigned long long t = 0;
	for (size_t i = 0; i < n; ++i) {
		unsigned long long m = minDur[i], f = fadeDur[i] > 1 ? fadeDur[i] : 1;
		t += std::max(m + 1, f + 2);
	}
	return t;
}

// ------------------------------------------------------------------------------------------------
// the render pipeline of players and batches (host.cu)
// ------------------------------------------------------------------------------------------------
cudaError_t initStates(StreamState *states, uint32_t n, cudaStream_t stream);

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
	PinnedBuf hostFault;         // uint32_t: the scheduler watchdog's verdict of the last call
	uint32_t schedHoldTicks = 256, schedGenTicks = 384, schedHoldMax = 4096, schedFadeTicks = 0, schedFadeMax = 512, schedRoleSms = 0, schedBlocks = 0;
	cudaStream_t lanes[2 * kMaxGroups] = {};
	cudaEvent_t evStart = nullptr, evFork[kMaxGroups] = {}, evJoin[kMaxGroups] = {};
	uint32_t holdTicks = 512, genTicks = 256, minStreams = 2048, groups = 4;
	bool ok = false;
	bool init();
	// the watchdog flag, allocated on first use: cudaErrorLaunchTimeout once an earlier call of this batch tripped the watchdog
	cudaError_t checkFault();
	~RoundsCtx();
};

// planned: the descriptors carry precomputed fade plans (pre-queued batches) -> FP32 renders may run as rounds
cudaError_t launchRender(int precision, const StreamDesc *descs, uint32_t n, int sampleRate, uint32_t sampleCount,
                         int16_t *out, size_t rowStride, uint32_t *written, StreamResult *results,
                         NoiseConfig noise, cudaStream_t stream, RoundsCtx *rc = nullptr, bool planned = false,
                         unsigned long long *launchCounter = nullptr);

// Chunked render into HOST memory: kernel(chunk c) overlaps the D2H copy of chunk c-1 (two staging buffers,
// compute stream + copy stream).  hostOut is [n][sampleCount]; rows are gathered with a 2-D copy.
struct HostPipe {
	cudaStream_t compute = nullptr, copy = nullptr;
	cudaEvent_t kernelDone[2] = {nullptr, nullptr}, copyDone[2] = {nullptr, nullptr};
	DevBuf stage[2], res[2];
	RoundsCtx rounds;
	PinnedBuf hostRes;  // StreamResult [2][n]
	bool ok = false;
	bool init();
	~HostPipe();
};

// returns total samples written, or -1.  perStream (host, [n]) and lastResults (host, [n]) are optional outputs.
long long renderToHost(HostPipe &pipe, int precision, const StreamDesc *dDescs, uint32_t n, int sampleRate,
                       uint32_t sampleCount, int16_t *hostOut, uint32_t *perStream, StreamResult *lastResults,
                       NoiseConfig noise, unsigned long long *launchCounter, bool planned = false);

}  // namespace klatt
