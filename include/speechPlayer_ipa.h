/*
 * Bulk frame producer (SURVEY.md section 8f, rank 1): IPA text -> queues of Klatt frames, natively and for many
 * utterances at once.  It produces exactly what the reference's Python pipeline produces, value for value:
 *
 *   reference ipa.py:336-353  generateFramesAndTiming(ipaText, speed, basePitch, inflection, clauseType)
 *             ipa.py:39-82    _IPAToPhonemesHelper   (stress marks, tie bars, length marks, table look-up)
 *             ipa.py:84-121   IPAToPhonemes          (syllable starts, post-stop aspiration, pre-stop gaps)
 *             ipa.py:123-135  correctHPhonemes       (_copyAdjacent)
 *             ipa.py:137-189  calculatePhonemeTimes
 *             ipa.py:191-211  applyPitchPath,  ipa.py:213-275 intonationParamTable,  ipa.py:277-334 calculatePhonemePitches
 *   reference speechPlayer.py:51-53  queueFrame: milliseconds -> samples, int(ms * (sampleRate / 1000.0))
 *
 * The reference spends ~1 us per frame in ctypes calls alone and renders ~5e3 audio-seconds per second per core through
 * this pipeline (SURVEY.md 8f); the arrays this producer fills are the ones speechPlayer_batchSetFramesHost takes.
 * The table calls and speechPlayer_ipaFrames are host code only: no CUDA device is needed for them.
 * speechPlayer_ipaFramesDevice runs the same rules on the GPU and fills the arrays speechPlayer_batchSetFramesDevice takes.
 */
#ifndef NVSP_B200_SPEECHPLAYER_IPA_H
#define NVSP_B200_SPEECHPLAYER_IPA_H

#include "speechPlayer.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct speechPlayer_ipaTable speechPlayer_ipaTable_t;

/* phoneme flags of the reference's data.py ('_isNasal', ... ) as a bit mask */
#define SPEECHPLAYER_IPA_NASAL 1u
#define SPEECHPLAYER_IPA_STOP 2u
#define SPEECHPLAYER_IPA_LIQUID 4u
#define SPEECHPLAYER_IPA_VOWEL 8u
#define SPEECHPLAYER_IPA_VOICED 16u
#define SPEECHPLAYER_IPA_AFRICATE 32u
#define SPEECHPLAYER_IPA_COPY_ADJACENT 64u
#define SPEECHPLAYER_IPA_SEMIVOWEL 128u

/* The phoneme table (the numeric content of the reference's data.py):
 *   keys    [n][3]  Unicode code points of each phoneme's key, zero padded (keys have 1..3 code points)
 *   values  [n][47] parameter values in frame order; present [n][47]: 1 where the phoneme's entry holds that parameter
 *   flags   [n]     SPEECHPLAYER_IPA_* bits
 * The table must contain the key "h" (post-stop aspiration is a copy of it, ipa.py:104).  Returns NULL on bad input. */
speechPlayer_ipaTable_t *speechPlayer_ipaTableCreate(const unsigned int *keys, const double *values,
                                                     const unsigned char *present, const unsigned int *flags,
                                                     unsigned int n);
void speechPlayer_ipaTableDestroy(speechPlayer_ipaTable_t *table);

/* IPA texts -> frame queues.  texts[i] is NUL-terminated UTF-8 (one clause; leading / trailing blanks are the caller's
 * business, the reference's callers strip them).  speed / basePitch / inflection / clauseType are per-text arrays or NULL
 * (defaults 1, 100, 0.5, '.'; clauseType 0 also means '.').  trailingSilenceMs >= 0 appends queueFrame(None, ms, 0) after
 * each text (reference test_speakIpa.py:26 uses 150).
 *
 * Outputs (any of them may be NULL; arrays are written only when capacity >= the total frame count):
 *   offsets [numTexts+1]  text i owns frames [offsets[i], offsets[i+1])            -- always written when non-NULL
 *   frames / minDur / fadeDur / isNull [capacity]  what speechPlayer_batchSetFramesHost takes (durations in SAMPLES;
 *                         rows of silence requests are zero and flagged in isNull)
 *   durationMs / fadeMs [capacity]   the generator's own units, as ipa.generateFramesAndTiming yields them
 * Returns the total number of frames, or -1 (speechPlayer_lastError()).  numThreads 0 = one per hardware thread. */
long long speechPlayer_ipaFrames(const speechPlayer_ipaTable_t *table, const char *const *texts, unsigned int numTexts,
                                 const double *speed, const double *basePitch, const double *inflection,
                                 const char *clauseType, int sampleRate, double trailingSilenceMs, long long *offsets,
                                 speechPlayer_frame_t *frames, unsigned int *minDur, unsigned int *fadeDur,
                                 unsigned char *isNull, double *durationMs, double *fadeMs,
                                 unsigned long long capacity, unsigned int numThreads);

/* The same producer on the calling thread's current CUDA device, bit for bit speechPlayer_ipaFrames.  Only the UTF-8
 * bytes and the per-text parameters cross PCIe; the frames are written in device memory.
 *
 * Inputs are HOST memory and the caller's to reuse once the call returns:
 *   text + textOffsets [numTexts+1]  packed UTF-8: text i is the bytes [textOffsets[i], textOffsets[i+1]) of text, ending
 *                                    early at its first NUL byte (offsets must not decrease)
 *   speed / basePitch / inflection / clauseType, sampleRate, trailingSilenceMs: as speechPlayer_ipaFrames
 * Outputs are DEVICE memory on the current device; any may be NULL:
 *   dOffsets [numTexts+1] int64                                        -- always written when non-NULL
 *   dFrames [capacity][47] double, dMinDur / dFadeDur [capacity] uint32, dIsNull [capacity] uint8,
 *   dDurationMs / dFadeMs [capacity] double, dTimelineSamples [numTexts] uint64 (samples each text yields, the sum of
 *   max(M + 1, max(F, 1) + 2) that speechPlayer_timelineSamples computes)  -- written only when capacity >= the total
 * The call synchronises once (to learn the total) and returns with the rows still being written on cudaStream, so a
 * speechPlayer_batchSetFramesDevice on the same stream may follow without a synchronisation.  Returns the total number
 * of frames, or -1 (speechPlayer_lastError()): bad arguments, no device (there is no CPU fallback), or a pitch percent
 * without a precomputed factor. */
long long speechPlayer_ipaFramesDevice(const speechPlayer_ipaTable_t *table, const char *text, const int64_t *textOffsets,
                                       unsigned int numTexts, const double *speed, const double *basePitch,
                                       const double *inflection, const char *clauseType, int sampleRate,
                                       double trailingSilenceMs, void *dOffsets, void *dFrames, void *dMinDur,
                                       void *dFadeDur, void *dIsNull, void *dDurationMs, void *dFadeMs,
                                       void *dTimelineSamples, unsigned long long capacity, void *cudaStream);

#ifdef __cplusplus
}
#endif
#endif
