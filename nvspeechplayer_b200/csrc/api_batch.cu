// The batch C-ABI of include/speechPlayer_batch.h: pre-queued batches (speechPlayer_batch*), the device-side output sinks,
// and batches over several GPUs of one box (speechPlayer_multiBatch*).
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/speechPlayer_batch.h"
#include "host.h"

using namespace klatt;

// ------------------------------------------------------------------------------------------------
// C-ABI: batch API
// ------------------------------------------------------------------------------------------------
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

struct speechPlayer_batch {
	int device = 0, sampleRate = 0, precision = kPrecisionF32, noiseMode = kNoisePhilox;
	uint64_t seed = 0;
	uint32_t n = 0;
	DevBuf dStates;     // StreamState [n + 1]
	DevBuf dDescs;      // StreamDesc [n + 1]
	DevBuf dStreamIds;  // uint64_t [n]
	// current queue arrays (borrowed device pointers, or the owned copies below)
	const int64_t *dOffsets = nullptr;
	const double *dFrames = nullptr;
	const uint32_t *dMin = nullptr, *dFade = nullptr;
	const int32_t *dUix = nullptr;
	const uint8_t *dNull = nullptr;
	const int32_t *dReplay = nullptr;
	uint64_t drawsPerStream = 0;
	DevBuf ownOffsets;
	QueueBufs own;
	DevBuf voiceTables;        // speechPlayer_batchApplyVoices: abs | mul | voiceOfStream
	DevBuf plans;              // FadePlanF32 per queued request (FP32 precision)
	bool plansDirty = false;   // frames changed since the plans were made
	uint64_t totalRequests = 0;
	HostPipe pipe;
	RoundsCtx rounds;
	unsigned long long launches = 0, ticks = 0;
	std::mutex mu;

	int rebuildDescs(cudaStream_t stream, bool withPlans) {
		build_descs_kernel<<<(n + 256) / 256, 256, 0, stream>>>(dDescs.as<StreamDesc>(), dStates.as<StreamState>(), dOffsets, dFrames, dMin, dFade, dUix, dNull,
		                                                        dReplay, drawsPerStream, dStreamIds.as<uint64_t>(),
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
	bool ok = b->dStates.reserve(sizeof(StreamState) * ((size_t)numStreams + 1), "cudaMalloc(states)") &&
	          b->dDescs.reserve(sizeof(StreamDesc) * ((size_t)numStreams + 1), "cudaMalloc(descs)") &&
	          b->dStreamIds.reserve(sizeof(uint64_t) * (size_t)numStreams, "cudaMalloc(ids)");
	if (ok) {
		std::vector<uint64_t> ids(numStreams);
		for (uint32_t i = 0; i < numStreams; ++i) ids[i] = streamIds ? streamIds[i] : i;
		ok = cudaOk(cudaMemcpy(b->dStreamIds.p, ids.data(), sizeof(uint64_t) * (size_t)numStreams, cudaMemcpyHostToDevice), "ids H2D") &&
		     cudaOk(initStates(b->dStates.as<StreamState>(), numStreams + 1, nullptr), "init states") && b->rebuildDescs(nullptr, false) == 0 &&
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
	delete b;
}

int speechPlayer_batchReset(speechPlayer_batch_t *b, void *cudaStream) {
	if (!b) return fail("null batch");
	std::lock_guard<std::mutex> lk(b->mu);
	DeviceGuard g(b->device);
	CU(initStates(b->dStates.as<StreamState>(), b->n + 1, static_cast<cudaStream_t>(cudaStream)));
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
	CU(initStates(b->dStates.as<StreamState>(), b->n + 1, stream));
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
		if (!b->ownOffsets.reserve(sizeof(int64_t) * ((size_t)b->n + 1))) return -1;
		CU(cudaMemcpyAsync(b->ownOffsets.p, offsets, sizeof(int64_t) * ((size_t)b->n + 1), cudaMemcpyHostToDevice, stream));
		if (b->own.upload(frames, minFrameDuration, fadeDuration, userIndex, isNull, total, stream) != 0) return -1;
	}
	int r = speechPlayer_batchSetFramesDevice(b, b->ownOffsets.p, frames ? b->own.frames.p : nullptr, b->own.minDur.p, b->own.fadeDur.p,
	                                          userIndex ? b->own.userIndex.p : nullptr, isNull ? b->own.isNull.p : nullptr, cudaStream);
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
	CU(launchRender(b->precision, b->dDescs.as<StreamDesc>(), b->n, b->sampleRate, sampleCount, static_cast<int16_t *>(dOut), rowStride,
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
	long long r = renderToHost(b->pipe, b->precision, b->dDescs.as<StreamDesc>(), b->n, b->sampleRate, sampleCount,
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
	CU(cudaMemcpy2D(lastIndex, sizeof(int), b->dStates.p, sizeof(StreamState), sizeof(int), b->n, cudaMemcpyDeviceToHost));
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
	// the shards are made at the first SetFrames: refuse here what speechPlayer_batchCreate would refuse there, and REPLAY, for
	// which a multi-batch has no entry that takes the draws
	if (precision != kPrecisionF64 && precision != kPrecisionF32) {
		fail(precision == kPrecisionStream ? "SPEECHPLAYER_PRECISION_STREAM is a per-handle mode (speechPlayer_initializeEx)" : "unknown precision");
		return nullptr;
	}
	if (noiseMode != kNoisePhilox) { fail("multi-batch noise mode must be PHILOX"); return nullptr; }
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
		upto[s + 1] = upto[s] + timelineTicks(minFrameDuration + offsets[s], fadeDuration + offsets[s],
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
