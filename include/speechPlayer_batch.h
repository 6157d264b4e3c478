/*
 * Batched / device-resident entry points of the B200-native Klatt engine.
 *
 * A batch is N independent players ("streams") whose frame queues, state blocks and
 * (optionally) output live in HBM.  It is the same engine as the per-handle API of
 * speechPlayer.h -- one stream of a batch behaves exactly like one reference player
 * (reference src/frame.cpp:41-115 frame manager + src/speechWaveGenerator.cpp:197-214
 * generate loop) -- but all streams advance in ONE kernel launch, and frames can be
 * handed over in bulk, either from host memory or as device pointers (no copies).
 *
 * Plain C: device pointers and the CUDA stream travel as void* (a cudaStream_t is a
 * pointer; pass NULL for the default stream, or e.g. torch.cuda.current_stream().cuda_stream).
 * All calls return 0 on success, -1 on failure (speechPlayer_lastError() has the reason).
 */
#ifndef NVSP_B200_SPEECHPLAYER_BATCH_H
#define NVSP_B200_SPEECHPLAYER_BATCH_H

#include "speechPlayer.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct speechPlayer_batch speechPlayer_batch_t;

/* streamIds: HOST array [numStreams] of noise-stream ids (Philox counter words 2,3), or NULL for 0..N-1.
 * The batch lives on the calling thread's current CUDA device (NVSP_DEVICE / LOCAL_RANK / 0 on first use). */
speechPlayer_batch_t *speechPlayer_batchCreate(int sampleRate, unsigned int numStreams, int precision,
                                               int noiseMode, uint64_t seed, const uint64_t *streamIds);
void speechPlayer_batchDestroy(speechPlayer_batch_t *batch);

/* Put every stream back into the state speechPlayer_initialize leaves it in and rewind the queue cursors
 * (the queued frames stay).  Asynchronous on cudaStream. */
int speechPlayer_batchReset(speechPlayer_batch_t *batch, void *cudaStream);

/* Replace the frame queues of all streams.  Stream s owns requests [offsets[s], offsets[s+1]) of the flat
 * arrays, in queue order (the batch equivalent of calling speechPlayer_queueFrame that many times on a fresh
 * player; fadeDuration 0 counts as 1).  userIndex / isNull may be NULL.
 * Setting new queues also puts every stream back into the freshly initialised state, and (FP32) makes the next
 * synthesize call re-plan every fade (klatt_plan_kernel) before it renders.
 *   ...Host:   all pointers are HOST memory; contents are copied to the device (async on cudaStream when the
 *              memory is pinned) before the call returns control of them.
 *   ...Device: all pointers are DEVICE memory that must stay valid and unchanged until the next
 *              SetFrames / Destroy; nothing is copied.  This is the HBM-resident path of bench.py's `value`. */
int speechPlayer_batchSetFramesHost(speechPlayer_batch_t *batch, const int64_t *offsets,
                                    const speechPlayer_frame_t *frames, const unsigned int *minFrameDuration,
                                    const unsigned int *fadeDuration, const int *userIndex,
                                    const unsigned char *isNull, void *cudaStream);
int speechPlayer_batchSetFramesDevice(speechPlayer_batch_t *batch, const void *dOffsets /* int64[N+1] */,
                                      const void *dFrames /* double[total][47] */, const void *dMinDur /* u32 */,
                                      const void *dFadeDur /* u32 */, const void *dUserIndex /* i32 or NULL */,
                                      const void *dIsNull /* u8 or NULL */, void *cudaStream);

/* Voices (SURVEY.md section 8f rank 2; reference nvdaAddon/synthDrivers/nvSpeechPlayer/__init__.py:86-125,
 * applyVoiceToFrame): rewrite the queued frames of every stream with its voice, on the device, in place:
 *     value = isnan(voiceAbs[v][p]) ? frame[p] : voiceAbs[v][p];   frame[p] = value * voiceMul[v][p]
 * for each of the 47 params p, v = voiceOfStream[s] -- the reference's "absolute override, then _mul factor" per
 * parameter, in double, so a voiced batch renders exactly what uploading host-rewritten frames would.
 *   voiceAbs, voiceMul : HOST double [numVoices][47]  (voiceAbs: NaN = no override; voiceMul: 1.0 = none)
 *   voiceOfStream      : HOST u32 [numStreams], or NULL = stream s uses voice s % numVoices
 * Call after SetFramesHost (the batch's own copy is rewritten) or SetFramesDevice (the CALLER'S frame array is
 * rewritten).  NULL-request rows are left alone.  Fade plans are re-made by the next synthesize call. */
int speechPlayer_batchApplyVoices(speechPlayer_batch_t *batch, const double *voiceAbs, const double *voiceMul,
                                  const unsigned int *voiceOfStream, unsigned int numVoices, void *cudaStream);

/* SPEECHPLAYER_NOISE_REPLAY: device int32 [numStreams][drawsPerStream]; draw d of stream s is at [s][d]. */
int speechPlayer_batchSetNoiseReplayDevice(speechPlayer_batch_t *batch, const void *dDraws, size_t drawsPerStream);

/* Advance every stream by up to sampleCount ticks (one kernel launch on cudaStream).
 *   dOut             device int16, row s starts at dOut + s*rowStride (rowStride in samples, >= sampleCount;
 *                    a multiple of 8 with a 16-byte aligned base enables 16-byte stores)
 *   dSamplesWritten  device u32 [numStreams] or NULL: per-stream count, < sampleCount iff that queue drained
 * Returns immediately after enqueueing (asynchronous). */
int speechPlayer_batchSynthesizeDevice(speechPlayer_batch_t *batch, unsigned int sampleCount, void *dOut,
                                       size_t rowStride, void *dSamplesWritten, void *cudaStream);

/* Same, into HOST memory [numStreams][sampleCount] (row-major, no padding); blocks until the samples have
 * landed.  samplesWritten (host u32 [numStreams]) may be NULL.  Returns total samples or -1. */
long long speechPlayer_batchSynthesizeHost(speechPlayer_batch_t *batch, unsigned int sampleCount, sample *out,
                                           unsigned int *samplesWritten);

/* Output sinks on the device (SURVEY.md section 8f rank 4): what the reference's consumers do with the int16 buffers, without
 * leaving HBM.  Both read the [numStreams][rowStride] int16 output of speechPlayer_batchSynthesizeDevice (or any int16 rows)
 * and are asynchronous on cudaStream.
 *   ...ToFloat32Device : sample / 32767.0 rounded to float32 -- exactly what reference lavPlayer.py:17 feeds its audio graph
 *                        (numpy int16 / 32767.0, taken as float32).  dOutFloat: device float [numStreams][outStride].
 *   ...ConcatenateDevice: the ragged rows packed back to back in stream order (reference nvdaAddon/synthDrivers/nvSpeechPlayer/
 *                        __init__.py:70-73 appends every buffer it pulls to one audio stream): stream s contributes its first
 *                        dSamplesWritten[s] samples (device u32 [numStreams]; NULL = sampleCount each).  dOffsets: device
 *                        int64 [numStreams + 1], filled with the exclusive prefix sum (dOffsets[numStreams] = total samples);
 *                        dOutPacked: device int16, at least the sum of the counts (numStreams * sampleCount always suffices). */
int speechPlayer_batchToFloat32Device(const void *dPcm, size_t rowStride, unsigned int numStreams, unsigned int sampleCount,
                                      void *dOutFloat, size_t outStride, void *cudaStream);
int speechPlayer_batchConcatenateDevice(const void *dPcm, size_t rowStride, unsigned int numStreams, unsigned int sampleCount,
                                        const void *dSamplesWritten, void *dOffsets, void *dOutPacked, void *cudaStream);

/* getLastIndex of every stream (host int32 [numStreams]); synchronises with the batch's last launch. */
int speechPlayer_batchGetLastIndices(speechPlayer_batch_t *batch, int *lastIndex);

/* Counters of the launches issued so far by this batch: kernels launched, ticks requested (streams x sampleCount). */
int speechPlayer_batchGetLaunchStats(speechPlayer_batch_t *batch, unsigned long long *kernelLaunches,
                                     unsigned long long *ticksRequested);

/* ---- several GPUs of one box, in-library (SURVEY.md section 8e) --------------------------------------------------------
 * Streams are independent, so a job shards by stream with NO collective: contiguous ranges of stream indices per device,
 * balanced by the ticks each stream's queue yields (occupancy law sum_j max(M+1, F+2), capped at nothing: whole queues), one
 * host thread and one per-device batch (its own CUDA streams) per shard, and SynthesizeHost gathers into disjoint row ranges
 * of ONE caller buffer [numStreams][sampleCount] (pinned memory makes the copies asynchronous).
 *   devices     : CUDA device ordinals, one shard each (an ordinal may repeat: two shards on one GPU); numDevices >= 1
 *   SetFramesHost: same arguments as speechPlayer_batchSetFramesHost; (re)partitions the streams and uploads every shard's
 *                 queues from its own thread
 *   GetShards   : firstStream[numDevices + 1] -- shard d owns streams [firstStream[d], firstStream[d + 1])
 *   Create refuses what speechPlayer_batchCreate refuses (STREAM precision, GLIBC noise), and REPLAY noise too: a
 *                 multi-batch has no entry that takes replay draws.  precision is FP64 or FP32, noiseMode PHILOX.
 * Everything a single batch guarantees holds per stream (same kernels, same bits as one batch on one GPU). */
typedef struct speechPlayer_multiBatch speechPlayer_multiBatch_t;
speechPlayer_multiBatch_t *speechPlayer_multiBatchCreate(int sampleRate, unsigned int numStreams, int precision, int noiseMode,
                                                         uint64_t seed, const uint64_t *streamIds, const int *devices,
                                                         unsigned int numDevices);
void speechPlayer_multiBatchDestroy(speechPlayer_multiBatch_t *mb);
int speechPlayer_multiBatchSetFramesHost(speechPlayer_multiBatch_t *mb, const int64_t *offsets, const speechPlayer_frame_t *frames,
                                         const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                         const int *userIndex, const unsigned char *isNull);
long long speechPlayer_multiBatchSynthesizeHost(speechPlayer_multiBatch_t *mb, unsigned int sampleCount, sample *out,
                                                unsigned int *samplesWritten);
int speechPlayer_multiBatchGetShards(speechPlayer_multiBatch_t *mb, unsigned int *firstStream);
int speechPlayer_multiBatchGetLastIndices(speechPlayer_multiBatch_t *mb, int *lastIndex);

/* Long-utterance path: ONE pre-queued stream rendered with parallelism in TIME (nvspeechplayer_b200/csrc/klatt_long.cu):
 * the stream is cut into chunks of chunkTicks ticks (0 = default 1024) that are rendered concurrently; the glottal
 * phase each chunk starts from comes from a scan of per-chunk phase advances, the state each two-pole section starts
 * from comes from a parallel scan (warp shuffles) over the per-chunk 2x2 affine maps of that section.  FP32
 * arithmetic, Philox noise keyed (seed, streamId); same audio as a fresh FP32 player fed the same queue, within the
 * FP32 tolerance (not bit for bit: the scan re-associates).
 *   frames / minFrameDuration / fadeDuration / isNull : HOST arrays, the stream's queueFrame calls in order
 *   out          : int16 [maxSamples], HOST memory, or DEVICE memory when outOnDevice != 0
 *   renderMs     : (optional) device time from the first to the last kernel of the call, in milliseconds
 * Returns the number of samples written = min(maxSamples, sum max(M+1, F+2)), or -1 on error. */
long long speechPlayer_synthesizeLong(int sampleRate, const speechPlayer_frame_t *frames,
                                      const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                                      const unsigned char *isNull, unsigned int numFrames, uint64_t seed,
                                      uint64_t streamId, unsigned int chunkTicks, sample *out,
                                      unsigned long long maxSamples, int outOnDevice, double *renderMs,
                                      unsigned long long *kernelLaunches);

/* Many pre-queued streams rendered with parallelism in time (the long-utterance path above), all streams' chunks in one
 * launch sequence (streams are taken in consecutive groups of at most NVSP_LONG_BATCH_TICKS ticks, default 2^28).
 * Inputs are HOST arrays in the layout of speechPlayer_batchSetFramesHost: stream s owns requests [offsets[s], offsets[s+1]).
 * Stream s renders what speechPlayer_synthesizeLong(sampleRate, <its requests>, seed, streamIds[s], chunkTicks,
 * maxSamples[s]) renders (Philox noise keyed (seed, streamIds[s]); streamIds NULL = 0..N-1).  Its glottal phase and its
 * excitation are bit for bit the same; the start state of a resonator chunk comes from a double-precision scan whose
 * association depends on where the stream sits among the scan's blocks, so a sample may in rare cases differ by a last-bit
 * rounding from the solo render.  That is the only source of difference.
 *   chunkTicks   : 0 = 1024, halved (down to 64) while a group has too few chunks to fill the GPU
 *   maxSamples   : HOST u64 [numStreams] cap per stream, or NULL = the whole queue
 *   outOffsets   : HOST int64 [numStreams + 1], filled: stream s's samples are out[outOffsets[s] .. outOffsets[s+1])
 *   out          : packed int16 (HOST, or DEVICE when outOnDevice); NULL = size query only (no device work, no device needed)
 *   serialPhase  : HOST u8 [numStreams] or NULL: 1 where that stream's glottal phase took the serial fallback
 *   renderMs     : (optional) device time of the groups' launch sequences, summed
 * Returns the total samples written (= outOffsets[numStreams]) or -1 (speechPlayer_lastError()). */
long long speechPlayer_synthesizeLongBatch(int sampleRate, unsigned int numStreams, const int64_t *offsets,
                                           const speechPlayer_frame_t *frames, const unsigned int *minFrameDuration,
                                           const unsigned int *fadeDuration, const unsigned char *isNull, uint64_t seed,
                                           const uint64_t *streamIds, unsigned int chunkTicks,
                                           const unsigned long long *maxSamples, sample *out, int64_t *outOffsets,
                                           int outOnDevice, unsigned char *serialPhase, double *renderMs,
                                           unsigned long long *kernelLaunches);

/* The same call for queues that are already in device memory, e.g. written by speechPlayer_ipaFramesDevice or by a model on
 * the GPU: stream s renders exactly what speechPlayer_synthesizeLongBatch renders for the same queues, bit for bit, and
 * outOffsets and serialPhase are the same.  Nothing of the queues is uploaded; they are read in place.
 *   dOffsets, dFrames, dMinDur, dFadeDur, dIsNull : DEVICE pointers of the current device, in the layout of
 *                  speechPlayer_batchSetFramesDevice (int64 [N+1], double [total][47], u32, u32, u8 or NULL).  dFrames,
 *                  dMinDur and dFadeDur are required when the queues hold any request.  The arrays are only read, and must
 *                  stay valid and unchanged until the call returns.
 *   the others   : as for speechPlayer_synthesizeLongBatch (host arrays; out is HOST, or DEVICE when outOnDevice)
 *   cudaStream   : every copy, event and launch of the call goes on it, so the call is ordered after work already queued
 *                  there (the producer of the queues) without synchronisation by the caller; NULL = the default stream
 * The offsets are copied back and checked by the host entry's rules before any kernel reads the queues, then one kernel
 * counts each stream's ticks (the occupancy law) and they are copied back: out = NULL is still a size query, but it needs
 * the device.  kernelLaunches counts that kernel too.  The call synchronises cudaStream before it returns.
 * Returns the total samples written (= outOffsets[numStreams]) or -1 (speechPlayer_lastError()). */
long long speechPlayer_synthesizeLongBatchDevice(int sampleRate, unsigned int numStreams, const void *dOffsets, const void *dFrames,
                                                 const void *dMinDur, const void *dFadeDur, const void *dIsNull, uint64_t seed,
                                                 const uint64_t *streamIds, unsigned int chunkTicks,
                                                 const unsigned long long *maxSamples, sample *out, int64_t *outOffsets,
                                                 int outOnDevice, unsigned char *serialPhase, double *renderMs,
                                                 unsigned long long *kernelLaunches, void *cudaStream);

/* Pure host helper (no device needed): samples a fully pre-queued stream yields,
 * sum_j max(M_j+1, max(F_j,1)+2)  -- the occupancy law of the reference frame manager (src/frame.cpp:41-80). */
unsigned long long speechPlayer_timelineSamples(const unsigned int *minFrameDuration,
                                                const unsigned int *fadeDuration, unsigned int n);

/* Library / build identification: "nvspeechplayer_b200 <ver> sm_100a". */
const char *speechPlayer_version(void);

#ifdef __cplusplus
}
#endif
#endif
