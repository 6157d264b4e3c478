/*
 * NV Speech Player C-ABI, served by the B200-native Klatt engine (libspeechPlayer.so).
 *
 * The first five entry points are the drop-in boundary: they are exactly what the
 * reference's Python binding (reference speechPlayer.py:48-65) and any other FFI user
 * bind, with the same argument meaning, units and return conventions as the
 * reference's own header (reference src/speechPlayer.h:25-31, export list
 * src/speechPlayer.def:1-6).  The remaining entry points are additions named by the
 * project's north star (batched synthesis) plus the knobs a GPU engine needs
 * (precision / noise mode / device-resident buffers); see speechPlayer_batch.h.
 *
 * Everything here is plain C: pointers, sizes, integers.  No CUDA or torch types.
 * There is no CPU fallback: without a usable CUDA device speechPlayer_initialize
 * returns NULL and speechPlayer_lastError() says why.
 */
#ifndef NVSP_B200_SPEECHPLAYER_H
#define NVSP_B200_SPEECHPLAYER_H

#include <stdint.h>
#include <stddef.h>
#ifndef __cplusplus
#include <stdbool.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* 47 doubles, ABI order == reference src/frame.h:20-47 (speechPlayer.py:20-40 mirrors it). */
typedef double speechPlayer_frameParam_t;
typedef struct {
	speechPlayer_frameParam_t voicePitch;               /* Hz */
	speechPlayer_frameParam_t vibratoPitchOffset;       /* fraction of a semitone */
	speechPlayer_frameParam_t vibratoSpeed;             /* Hz */
	speechPlayer_frameParam_t voiceTurbulenceAmplitude; /* 0..1 breathiness */
	speechPlayer_frameParam_t glottalOpenQuotient;      /* 0..1 */
	speechPlayer_frameParam_t voiceAmplitude;           /* 0..1 */
	speechPlayer_frameParam_t aspirationAmplitude;      /* 0..1 */
	speechPlayer_frameParam_t cf1, cf2, cf3, cf4, cf5, cf6, cfN0, cfNP; /* cascade formant / nasal zero / nasal pole, Hz */
	speechPlayer_frameParam_t cb1, cb2, cb3, cb4, cb5, cb6, cbN0, cbNP; /* their bandwidths, Hz */
	speechPlayer_frameParam_t caNP;                     /* 0..1 nasal pole mix */
	speechPlayer_frameParam_t fricationAmplitude;       /* 0..1 */
	speechPlayer_frameParam_t pf1, pf2, pf3, pf4, pf5, pf6; /* parallel formants, Hz */
	speechPlayer_frameParam_t pb1, pb2, pb3, pb4, pb5, pb6; /* bandwidths, Hz */
	speechPlayer_frameParam_t pa1, pa2, pa3, pa4, pa5, pa6; /* amplitudes 0..1 */
	speechPlayer_frameParam_t parallelBypass;           /* 0..1 */
	speechPlayer_frameParam_t preFormantGain;           /* 0..1 */
	speechPlayer_frameParam_t outputGain;               /* master volume */
	speechPlayer_frameParam_t endVoicePitch;            /* Hz at the end of the frame */
} speechPlayer_frame_t;
#define SPEECHPLAYER_FRAME_NUM_PARAMS 47

/* reference src/sample.h:18-22 */
typedef short sampleVal;
typedef struct { sampleVal value; } sample;

/* Opaque.  Values are small positive integers cast to a pointer, so they survive the
 * reference wrapper's untyped ctypes round trip through a C int (reference
 * speechPlayer.py:49 leaves restype unset). */
typedef void *speechPlayer_handle_t;

/* ---- the reference's five exports (drop-in) ---------------------------------------------- */

/* reference src/speechPlayer.cpp:25-32.  NULL on failure (no CUDA device / allocation). */
speechPlayer_handle_t speechPlayer_initialize(int sampleRate);

/* reference src/speechPlayer.cpp:34-37 + src/frame.cpp:90-115.  framePtr==NULL queues a silence
 * request; durations are in SAMPLES; fadeDuration 0 is treated as 1; userIndex -1 = none; the frame
 * is copied, the caller may reuse it at once.  May be called from any thread while another thread
 * is inside speechPlayer_synthesize on the same handle. */
void speechPlayer_queueFrame(speechPlayer_handle_t playerHandle, speechPlayer_frame_t *framePtr,
                             unsigned int minFrameDuration, unsigned int fadeDuration, int userIndex,
                             bool purgeQueue);

/* reference src/speechPlayer.cpp:39-41 + src/speechWaveGenerator.cpp:197-214.  Writes up to sampleCount
 * int16 samples into caller-owned HOST memory; returns how many were written (< sampleCount exactly when
 * the queue drained, 0 when idle).  Returns -1 only on a CUDA failure (the reference has no error path). */
int speechPlayer_synthesize(speechPlayer_handle_t playerHandle, unsigned int sampleCount, sample *sampleBuf);

/* reference src/speechPlayer.cpp:43-46 + src/frame.cpp:117-119: userIndex of the last popped request
 * that carried one; -1 initially. */
int speechPlayer_getLastIndex(speechPlayer_handle_t playerHandle);

/* reference src/speechPlayer.cpp:48-53 */
void speechPlayer_terminate(speechPlayer_handle_t playerHandle);

/* ---- additions ---------------------------------------------------------------------------- */

enum { /* arithmetic the render kernel runs in */
	SPEECHPLAYER_PRECISION_FP64 = 0, /* reference evaluation order in double: bit-exact int16 parity mode */
	SPEECHPLAYER_PRECISION_FP32 = 1, /* production: FP32 DSP, FP64 pitch/phase */
	SPEECHPLAYER_PRECISION_STREAM = 2 /* low-latency pulls: the FP32 arithmetic, one pull rendered parallel in time by one
	                                    * thread block with the player's state carried over (per-handle API only) */
};
enum { /* source of the two uniform draws per generated sample (reference rand(), speechWaveGenerator.cpp:40) */
	SPEECHPLAYER_NOISE_PHILOX = 0, /* counter-based Philox4x32-10 keyed by (seed, stream id) */
	SPEECHPLAYER_NOISE_GLIBC = 1,  /* process-global replica of glibc rand() (TYPE_3 additive feedback), replayed */
	SPEECHPLAYER_NOISE_REPLAY = 2  /* caller-supplied draw sequence (speechPlayer_setNoiseReplay) */
};

/* Like speechPlayer_initialize with explicit modes.  speechPlayer_initialize itself reads the environment:
 * NVSP_PRECISION=fp64|fp32|stream (default fp64: faithful drop-in), NVSP_NOISE=glibc|philox (default glibc),
 * NVSP_SEED, NVSP_DEVICE (CUDA ordinal; default LOCAL_RANK or 0). */
speechPlayer_handle_t speechPlayer_initializeEx(int sampleRate, int precision, int noiseMode, uint64_t seed,
                                                uint64_t streamId);

/* Bulk form of speechPlayer_queueFrame (no purge): n requests in one call.  isNull[i]!=0 queues a silence
 * request and frames[i] is ignored; userIndex / isNull may be NULL (-1 / all real). */
int speechPlayer_queueFrames(speechPlayer_handle_t playerHandle, const speechPlayer_frame_t *frames,
                             const unsigned int *minFrameDuration, const unsigned int *fadeDuration,
                             const int *userIndex, const unsigned char *isNull, unsigned int n);

/* Render numHandles independent players at once (one launch).  sampleBuf is HOST memory,
 * [numHandles][sampleCount] row-major; samplesWritten[i] (may be NULL) receives what
 * speechPlayer_synthesize would have returned for handles[i].  All handles must share precision and
 * sample rate.  Returns the total number of samples written, or -1 on error.
 * With SPEECHPLAYER_NOISE_GLIBC the handles are not rendered in parallel: they render one after another, in
 * handle order, so each row and the process-global generator end up exactly as the same speechPlayer_synthesize
 * calls made one by one would leave them (the reference's shared rand() is sequential by nature). */
long long speechPlayer_synthesizeBatch(speechPlayer_handle_t *handles, unsigned int numHandles,
                                       unsigned int sampleCount, sample *sampleBuf, unsigned int *samplesWritten);

/* SPEECHPLAYER_NOISE_REPLAY: the draw sequence (values 0..2^31-1, aspiration then frication per generated
 * sample) of this handle, indexed from its first sample: the g-th sample the handle generates since it was
 * created reads draws[2g] and draws[2g+1], also when the sequence is set after the handle has rendered.  Draws
 * past numDraws are 0.  Copied to the device. */
int speechPlayer_setNoiseReplay(speechPlayer_handle_t playerHandle, const int32_t *draws, size_t numDraws);

/* SPEECHPLAYER_NOISE_GLIBC: reseed the process-global generator (what srand() is to the reference). */
void speechPlayer_seedNoise(unsigned int seed);

/* Human-readable reason for the last failure on this thread ("" if none). */
const char *speechPlayer_lastError(void);

#ifdef __cplusplus
}
#endif
#endif
