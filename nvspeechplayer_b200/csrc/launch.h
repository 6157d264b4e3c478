// The host interface of the kernel units: every host-callable function that one translation unit defines and another
// calls, and the records the host fills for the long-utterance kernels.  Each unit that defines or calls one of them
// includes this header, so a declaration and its definition cannot drift apart unnoticed.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "klatt_common.h"

namespace klatt {

struct PullState;      // klatt_pull_core.cuh
struct PullCtx;
struct PullSeg;
struct PullBatchItem;
struct PhaseChunk;     // klatt_long_phase.cuh

// ---- klatt_f64.cu ----
cudaError_t launchKlattF64(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream);

// ---- klatt_f32.cu ----
cudaError_t launchKlattF32(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream);
cudaError_t launchKlattF32Rounds(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                 uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride,
                                 uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise, uint32_t *listHold,
                                 uint32_t *listGen, uint32_t *counters, int16_t *scratchRow, cudaStream_t stream, uint32_t numGroups,
                                 cudaStream_t *lanes, cudaEvent_t evStart, cudaEvent_t *evFork, cudaEvent_t *evJoin,
                                 unsigned long long *launchCounter);
cudaError_t launchKlattFinalize(const StreamDesc *descs, uint32_t numStreams, uint32_t *samplesWritten, StreamResult *results,
                                cudaStream_t stream);
cudaError_t launchKlattPlan(const int64_t *offsets, uint32_t numStreams, uint64_t totalRequests, const double *frames,
                            const uint32_t *fadeDur, const uint8_t *isNull, int sampleRate, FadePlanF32 *plans,
                            cudaStream_t stream);

// ---- klatt_f32_sched.cu ----
cudaError_t launchKlattF32Sched(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                                uint32_t holdTicks, uint32_t genTicks, int16_t *out, size_t rowStride, uint32_t *samplesWritten,
                                StreamResult *results, NoiseConfig noise, uint32_t *ring, uint32_t ringCap, void *ctlMem,
                                int16_t *scratchRow, uint32_t numBlocks, uint32_t *hostFault, void *liteMem, uint32_t holdMax,
                                uint32_t fadeTicks, uint32_t fadeMax, uint32_t roleSms, cudaStream_t stream, unsigned long long *launchCounter);
int klattF32SchedBlocksPerSm();
bool klattF32SchedUsesLite();
size_t klattF32SchedLiteBytes(uint32_t numStreams, uint32_t numBlocks);

// ---- klatt_f32_block.cu ----
cudaError_t launchKlattF32Block(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount, uint32_t holdTicks,
                                int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results, NoiseConfig noise,
                                void *liteMem, int16_t *scratchRow, uint32_t numBlocks, void *profMem, uint32_t *hostFault,
                                cudaStream_t stream, unsigned long long *launchCounter);
bool klattF32BlockCanTake(uint32_t numStreams, uint32_t numBlocks);
size_t klattF32BlockLiteBytes(uint32_t numStreams, uint32_t numBlocks);
cudaError_t launchKlattLiteImport(const StreamDesc *descs, uint32_t numStreams, uint32_t numDummies, void *lite, cudaStream_t stream);
cudaError_t launchKlattLiteExport(const StreamDesc *descs, uint32_t numStreams, const void *lite, uint32_t *samplesWritten, StreamResult *results,
                                  cudaStream_t stream);

// ---- klatt_pull.cu ----
cudaError_t launchKlattPullInit(PullState *state, cudaStream_t stream);
cudaError_t launchKlattPull(PullCtx ctx, const PullSeg *segSrc, int16_t *pcmOut, cudaStream_t stream);
cudaError_t launchKlattPullBatch(PullBatchItem *hItems, const PullBatchItem *dItems, uint32_t count, cudaStream_t stream);

// ---- klatt_long.cu ----
// One stream of a launch: pointers into the flat arrays of all the launch's requests at this stream's offset.
struct LongStream {
	const double *frames;      // [nReq][47]
	const uint32_t *minDur, *fadeDur;
	const uint8_t *isNull;     // may be null
	const FadePlanF32 *plans;  // [nReq]
	uint32_t nReq;
	int sampleRate;
	uint64_t seed, streamId;
	uint64_t cap;              // ticks rendered: the timeline is cut here (start[nReq] = min(ticks the queue yields, cap))
	uint64_t outBase;          // where the stream's tick 0 goes in the launch's packed int16 output
	// made by klatt_long_timeline_kernel
	uint64_t *start;        // [nReq+1] tick of each request's pop tick; start[nReq] = ticks rendered
	int32_t *prevReal;      // [nReq] last non-NULL request before j, or -1
	double *pitchPop;       // [nReq] cur.voicePitch on the pop tick (stale value)
	double *pitchOld, *pitchNew, *pitchInc;  // [nReq] fade end points and hold glide
	uint64_t *vibPosStart;  // [nReq] vibrato phase before the pop tick
};

// The streams of one launch.  Stream s owns the chunks [chunkBase[s], chunkBase[s+1]) (chunkBase: exclusive scan of
// ceil(ticks_s / L)); its tick t lives at VIRTUAL tick chunkBase[s] * L + t of the signal arrays, so every chunk starts on
// a multiple of L as it does for one stream, and the gap between two streams is under L ticks.
struct LongTable {
	const LongStream *streams;   // [numStreams]
	const uint32_t *chunkBase;   // [numStreams + 1]
	uint32_t numStreams;
	LongStream one;              // streams[0] by value: a one-stream launch reads its stream from the parameter bank
};

// affine map of one section over one chunk, (y, d)_end = P (y, d)_start + z, row-major P
struct Affine {
	float p00, p01, p10, p11, zy, zd;
};

// Launchers: everything device-resident, scratch sized by the caller (api_long.cu).
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
