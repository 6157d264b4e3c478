// The long-utterance C-ABI (speechPlayer_synthesizeLong, speechPlayer_synthesizeLongBatch and
// speechPlayer_synthesizeLongBatchDevice of include/speechPlayer_batch.h): the host side of kernel (b), klatt_long.cu.
#include <atomic>
#include <cstdio>
#include <mutex>
#include <vector>

#include "../../include/speechPlayer_batch.h"
#include "host.h"
#include "klatt_long_phase.cuh"

using namespace klatt;

static std::atomic<unsigned long long> g_longSerialFallbacks{0};
// how many streams rendered by the long path in this process had to take the serial phase fallback (tests, bench); for
// speechPlayer_synthesizeLong a stream is a call
extern "C" unsigned long long speechPlayer_debugLongSerialFallbacks(void) { return g_longSerialFallbacks.load(); }

// One call of the long path: numStreams pre-queued streams in the layout of speechPlayer_batchSetFramesHost, already
// validated, with the output offsets from the timeline law.  The queue arrays (frames, minDur, fadeDur, isNull) are host
// arrays, or with queuesOnDevice device arrays of the current device that are read in place; the others are host arrays.
struct LongCall {
	int sampleRate;
	uint32_t numStreams;
	const int64_t *offsets;                 // [numStreams + 1]
	const speechPlayer_frame_t *frames;     // null: every request is a NULL request (host queues only)
	const unsigned int *minDur, *fadeDur;
	const unsigned char *isNull;            // may be null
	uint64_t seed;
	const uint64_t *streamIds;              // [numStreams], or null: 0..numStreams-1
	uint32_t chunkTicks;                    // 0: chosen per group (batch default)
	const int64_t *outOffsets;              // [numStreams + 1]: stream s renders outOffsets[s + 1] - outOffsets[s] samples
	int16_t *out;
	bool outOnDevice;
	unsigned char *serialPhase;             // [numStreams] or null
	bool queuesOnDevice = false;
	cudaStream_t stream = nullptr;          // every copy, event and launch of the call
};

// Below this many chunks a group of the batch entry halves its default chunk length (1024), down to 64: fewer chunks than
// this leave SMs idle in the stage kernels (one thread per chunk).  Measured on a B200 by tools/long_batch_bench.py.
static constexpr uint64_t kLongFillChunks = 65536;

// Scratch of the long path: grow-only buffers kept per device between calls (a config-4 call needs ~5 GB of stage signals;
// allocating and freeing them inside every call cost 10-20 ms of a 40 ms render).
struct LongScratch {
	QueueBufs q;  // frames, minDur, fadeDur, isNull
	DevBuf dOff, dPlans, dStart, dPrev, dPitch, dVib, dTable, dChunkBase;
	DevBuf sig, maps, st, ph, pcm, phChunks, phStart, phFail, scanTmp;
	DevBuf dTicks;  // device queues: each stream's ticks
};

// fn(dev, scratch) on the calling thread's device, with the long path's lock held: one long call at a time per process.
// The scratch is the device's pool (it lives as long as the process and is never destroyed: no CUDA call at exit), or with
// NVSP_LONG_POOL=0 this call's own, freed on return.
template <class Fn> static long long withLongScratch(Fn &&fn) {
	int dev = pickDevice();
	if (dev < 0) return fail("no usable CUDA device (this library has no CPU fallback)");
	DeviceGuard g(dev);
	static std::mutex longMu;
	static LongScratch *const pool = new LongScratch[16];
	std::lock_guard<std::mutex> longLock(longMu);
	LongScratch local;
	static const bool usePool = envNum<uint64_t>("NVSP_LONG_POOL", 1) != 0;
	return fn(dev, (usePool && dev < 16) ? pool[dev] : local);
}

static long long renderLong(const LongCall &C, LongScratch &S, double *renderMs, unsigned long long *kernelLaunches) {
	// streams are rendered in consecutive groups of at most this many ticks (one launch sequence each; a stream longer than
	// that is a group of its own).  The scratch is ~22 bytes per tick (five float signals, the int16 output, the chunk maps): 6 GB at the default.
	static const uint64_t groupTicks = std::max<uint64_t>(envNum<uint64_t>("NVSP_LONG_BATCH_TICKS", 1ull << 28), 1);
	struct Events {
		cudaEvent_t e0 = nullptr, e1 = nullptr;
		~Events() {
			if (e0) cudaEventDestroy(e0);
			if (e1) cudaEventDestroy(e1);
		}
	} ev;
	CU(cudaEventCreate(&ev.e0));
	CU(cudaEventCreate(&ev.e1));
	const cudaStream_t stream = C.stream;
	// The glottal phase is the reference's FP64 recurrence, parallel in time by speculation + verification
	// (klatt_long_phase.cuh).  The streams whose check failed -- or all, with NVSP_LONG_PHASE=serial -- are rendered again
	// with the plain recurrence on one thread per stream: slow, exact by definition.
	static const bool forceSerial = envIs("NVSP_LONG_PHASE", "serial");
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
		// the group's queues: the caller's device arrays from its first request on, or an upload of its host arrays
		const double *dFrames;
		const uint32_t *dMin, *dFade;
		const uint8_t *dNull;
		std::vector<unsigned char> allNull;
		if (C.queuesOnDevice) {
			dFrames = reinterpret_cast<const double *>(C.frames + reqBase);
			dMin = C.minDur + reqBase;
			dFade = C.fadeDur + reqBase;
			dNull = C.isNull ? C.isNull + reqBase : nullptr;
		} else {
			const unsigned char *isNull = C.isNull ? C.isNull + reqBase : nullptr;
			if (!C.frames) {  // every request is a NULL request: zero frames
				allNull.assign(n, 1);
				isNull = allNull.data();
				if (!S.q.frames.reserve(n * sizeof(speechPlayer_frame_t))) return -1;
				if (n) CU(cudaMemsetAsync(S.q.frames.p, 0, n * sizeof(speechPlayer_frame_t), stream));
			}
			if (S.q.upload(C.frames ? C.frames + reqBase : nullptr, C.minDur + reqBase, C.fadeDur + reqBase, nullptr, isNull, n, stream) != 0)
				return -1;
			dFrames = S.q.frames.as<double>();
			dMin = S.q.minDur.as<uint32_t>();
			dFade = S.q.fadeDur.as<uint32_t>();
			dNull = isNull ? S.q.isNull.as<uint8_t>() : nullptr;
		}
		if (!S.dOff.reserve((G + 1) * 8) || !S.dPlans.reserve(n * sizeof(FadePlanF32)) || !S.dStart.reserve((n + G) * 8) ||
		    !S.dPrev.reserve(n * 4) || !S.dPitch.reserve(n * 8 * 4) || !S.dVib.reserve(n * 8) || !S.dTable.reserve(G * sizeof(LongStream)) ||
		    !S.dChunkBase.reserve((G + 1) * 4))
			return -1;
		std::vector<int64_t> off(G + 1);
		for (uint32_t k = 0; k <= G; ++k) off[k] = C.offsets[g0 + k] - reqBase;
		CU(cudaMemcpyAsync(S.dOff.p, off.data(), (G + 1) * 8, cudaMemcpyHostToDevice, stream));
		// the stream table: stream k's requests at off[k] of the flat arrays, its start ticks at off[k] + k (nReq + 1 each)
		double *dPitch = S.dPitch.as<double>();
		std::vector<LongStream> table(G);
		for (uint32_t k = 0; k < G; ++k) {
			LongStream &L = table[k];
			const size_t a = (size_t)off[k];
			L.frames = dFrames + a * kNumParams; L.minDur = dMin + a; L.fadeDur = dFade + a;
			L.isNull = dNull ? dNull + a : nullptr;
			L.plans = S.dPlans.as<FadePlanF32>() + a; L.nReq = (uint32_t)(off[k + 1] - off[k]); L.sampleRate = C.sampleRate;
			L.seed = C.seed; L.streamId = C.streamIds ? C.streamIds[g0 + k] : g0 + k;
			L.cap = ticks[g0 + k]; L.outBase = (uint64_t)(C.outOffsets[g0 + k] - C.outOffsets[g0]);
			L.start = S.dStart.as<uint64_t>() + a + k; L.prevReal = S.dPrev.as<int32_t>() + a;
			L.pitchPop = dPitch + a; L.pitchOld = dPitch + n + a; L.pitchNew = dPitch + 2 * n + a; L.pitchInc = dPitch + 3 * n + a;
			L.vibPosStart = S.dVib.as<uint64_t>() + a;
		}
		CU(cudaMemcpyAsync(S.dTable.p, table.data(), G * sizeof(LongStream), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(S.dChunkBase.p, chunkBase.data(), (G + 1) * 4, cudaMemcpyHostToDevice, stream));
		CU(cudaEventRecord(ev.e0, stream));
		CU(launchKlattPlan(S.dOff.as<int64_t>(), G, n, dFrames, dFade, dNull, C.sampleRate, S.dPlans.as<FadePlanF32>(), stream));
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
		CU(cudaEventRecord(ev.e1, stream));
		std::vector<uint32_t> failed(G, 0);
		CU(cudaMemcpyAsync(failed.data(), dFail, (size_t)G * 4, cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		uint32_t nFailed = 0;
		for (uint32_t k = 0; k < G; ++k) nFailed += failed[k] && ticks[g0 + k] ? 1 : 0;
		if (nFailed && !forceSerial) {
			if (envIs("NVSP_VERBOSE"))
				fprintf(stderr, "[nvspeechplayer_b200] long path: speculative phase of %u stream(s) not verified, serial fallback\n", nFailed);
			// only the failed streams' chunks get new phases; the source and stage passes run again for all
			CU(launchKlattLongPhase(T, numChunks, chunkTicks, advance, advance + numChunks, S.phChunks.as<PhaseChunk>(), S.phStart.as<double>(),
			                        dFail, true, &launches, stream));
			CU(synth());
			CU(cudaEventRecord(ev.e1, stream));
			g_longSerialFallbacks += nFailed;
		}
		if (C.serialPhase)
			for (uint32_t k = 0; k < G; ++k) C.serialPhase[g0 + k] = (failed[k] && ticks[g0 + k]) ? 1 : 0;
		if (!C.outOnDevice) CU(cudaMemcpyAsync(C.out + C.outOffsets[g0], dPcm, sum * sizeof(int16_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		float groupMs = 0;
		CU(cudaEventElapsedTime(&groupMs, ev.e0, ev.e1));
		ms += groupMs;
	}
	if (renderMs) *renderMs = ms;
	if (kernelLaunches) *kernelLaunches = launches;
	return C.outOffsets[N];
}

// The rules of a batch's offsets (a host array, or the host copy of a device array): checked before any queue is read.
static int checkOffsets(const int64_t *offsets, unsigned numStreams) {
	if (offsets[0] != 0) return fail("offsets[0] must be 0");
	for (unsigned s = 0; s < numStreams; ++s) {
		if (offsets[s + 1] < offsets[s]) return fail("offsets must be non-decreasing");
		if (offsets[s + 1] - offsets[s] > (int64_t)0xffffffffll) return fail("too many requests in one stream");
	}
	return 0;
}

// A batch call's outputs before it renders: outOffsets from each stream's ticks, ticksOf(s), capped by maxSamples;
// serialPhase, renderMs and kernelLaunches zeroed.  Returns the total samples.
template <class TicksOf>
static int64_t sizeLongBatch(unsigned numStreams, TicksOf ticksOf, const unsigned long long *maxSamples, int64_t *outOffsets,
                             unsigned char *serialPhase, double *renderMs, unsigned long long *kernelLaunches) {
	outOffsets[0] = 0;
	for (unsigned s = 0; s < numStreams; ++s) {
		unsigned long long t = ticksOf(s);
		if (maxSamples) t = std::min(t, maxSamples[s]);
		outOffsets[s + 1] = outOffsets[s] + (int64_t)t;
	}
	if (serialPhase) memset(serialPhase, 0, numStreams);
	if (renderMs) *renderMs = 0;
	if (kernelLaunches) *kernelLaunches = 0;
	return outOffsets[numStreams];
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
	if (chunkTicks == 0) chunkTicks = envNum<unsigned>("NVSP_LONG_CHUNK", 1024u);
	const int64_t offsets[2] = {0, (int64_t)numFrames};
	const int64_t outOffsets[2] = {0, (int64_t)std::min<unsigned long long>(timelineTicks(minFrameDuration, fadeDuration, numFrames),
	                                                                          maxSamples)};
	LongCall C;
	C.sampleRate = sampleRate; C.numStreams = 1; C.offsets = offsets; C.frames = frames; C.minDur = minFrameDuration;
	C.fadeDur = fadeDuration; C.isNull = isNull; C.seed = seed; C.streamIds = &streamId; C.chunkTicks = std::max(chunkTicks, 64u);
	C.outOffsets = outOffsets; C.out = reinterpret_cast<int16_t *>(out); C.outOnDevice = outOnDevice != 0; C.serialPhase = nullptr;
	return withLongScratch([&](int, LongScratch &S) { return renderLong(C, S, renderMs, kernelLaunches); });
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
	if (checkOffsets(offsets, numStreams) != 0) return -1;
	if (offsets[numStreams] && (!minFrameDuration || !fadeDuration)) return fail("durations missing");
	const int64_t samples = sizeLongBatch(
		numStreams, [&](unsigned s) { return timelineTicks(minFrameDuration + offsets[s], fadeDuration + offsets[s], (size_t)(offsets[s + 1] - offsets[s])); },
		maxSamples, outOffsets, serialPhase, renderMs, kernelLaunches);
	if (!out || samples == 0) return samples;
	LongCall C;
	C.sampleRate = sampleRate; C.numStreams = numStreams; C.offsets = offsets; C.frames = frames; C.minDur = minFrameDuration;
	C.fadeDur = fadeDuration; C.isNull = isNull; C.seed = seed; C.streamIds = streamIds; C.chunkTicks = chunkTicks;
	C.outOffsets = outOffsets; C.out = reinterpret_cast<int16_t *>(out); C.outOnDevice = outOnDevice != 0; C.serialPhase = serialPhase;
	return withLongScratch([&](int, LongScratch &S) { return renderLong(C, S, renderMs, kernelLaunches); });
}

// p is device (or managed) memory of device dev
static bool onDevice(const void *p, int dev) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		cudaGetLastError();
		return false;
	}
	return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == dev;
}

extern "C" long long speechPlayer_synthesizeLongBatchDevice(int sampleRate, unsigned int numStreams, const void *dOffsets,
                                                            const void *dFrames, const void *dMinDur, const void *dFadeDur,
                                                            const void *dIsNull, uint64_t seed, const uint64_t *streamIds,
                                                            unsigned int chunkTicks, const unsigned long long *maxSamples, sample *out,
                                                            int64_t *outOffsets, int outOnDevice, unsigned char *serialPhase,
                                                            double *renderMs, unsigned long long *kernelLaunches, void *cudaStream) {
	g_lastError.clear();
	if (sampleRate <= 0) return fail("sampleRate must be positive");
	if (numStreams == 0) return fail("numStreams must be positive");
	if (!dOffsets) return fail("null offsets");
	if (!outOffsets) return fail("null outOffsets");
	return withLongScratch([&](int dev, LongScratch &S) -> long long {
		const cudaStream_t stream = static_cast<cudaStream_t>(cudaStream);
		const size_t N = numStreams;
		if (!onDevice(dOffsets, dev)) return fail("offsets are not device memory of the current device");
		// the offsets, checked on the host before any kernel reads the queues
		std::vector<int64_t> offsets(N + 1);
		CU(cudaMemcpyAsync(offsets.data(), dOffsets, (N + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		if (checkOffsets(offsets.data(), numStreams) != 0) return -1;
		if (offsets[N]) {
			if (!dMinDur || !dFadeDur) return fail("durations missing");
			if (!dFrames) return fail("null frames (device queues carry every request's frame row)");
			const void *queue[] = {dFrames, dMinDur, dFadeDur, dIsNull};
			for (const void *p : queue)
				if (p && !onDevice(p, dev)) return fail("queue arrays are not device memory of the current device");
		}
		// each stream's ticks, for the output offsets and the grouping
		if (!S.dTicks.reserve(N * sizeof(uint64_t))) return -1;
		CU(launchKlattLongTicks(static_cast<const int64_t *>(dOffsets), numStreams, static_cast<const uint32_t *>(dMinDur),
		                        static_cast<const uint32_t *>(dFadeDur), S.dTicks.as<uint64_t>(), stream));
		std::vector<uint64_t> ticks(N);
		CU(cudaMemcpyAsync(ticks.data(), S.dTicks.p, N * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
		CU(cudaStreamSynchronize(stream));
		const int64_t samples = sizeLongBatch(numStreams, [&](unsigned s) { return ticks[s]; }, maxSamples, outOffsets, serialPhase, renderMs,
		                                      kernelLaunches);
		long long r = samples;
		if (out && samples) {
			LongCall C;
			C.sampleRate = sampleRate; C.numStreams = numStreams; C.offsets = offsets.data();
			C.frames = static_cast<const speechPlayer_frame_t *>(dFrames); C.minDur = static_cast<const unsigned int *>(dMinDur);
			C.fadeDur = static_cast<const unsigned int *>(dFadeDur); C.isNull = static_cast<const unsigned char *>(dIsNull);
			C.seed = seed; C.streamIds = streamIds; C.chunkTicks = chunkTicks; C.outOffsets = outOffsets;
			C.out = reinterpret_cast<int16_t *>(out); C.outOnDevice = outOnDevice != 0; C.serialPhase = serialPhase;
			C.queuesOnDevice = true; C.stream = stream;
			r = renderLong(C, S, renderMs, kernelLaunches);
		}
		if (r >= 0 && kernelLaunches) *kernelLaunches += 1;  // the ticks kernel
		return r;
	});
}
