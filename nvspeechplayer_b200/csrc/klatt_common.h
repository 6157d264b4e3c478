// Shared definitions of the B200-native Klatt engine: parameter slots, per-stream device state,
// stream descriptors.  Header-only, usable from host C++ and from CUDA.
//
// Parameter order is the ABI of speechPlayer_frame_t (reference src/frame.h:20-47).
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define KLATT_HD __host__ __device__ __forceinline__
#else
#define KLATT_HD inline
#endif

namespace klatt {

enum Param : int {
	kVoicePitch = 0, kVibratoPitchOffset, kVibratoSpeed, kVoiceTurbulenceAmplitude, kGlottalOpenQuotient,
	kVoiceAmplitude, kAspirationAmplitude,
	kCf1, kCf2, kCf3, kCf4, kCf5, kCf6, kCfN0, kCfNP,
	kCb1, kCb2, kCb3, kCb4, kCb5, kCb6, kCbN0, kCbNP,
	kCaNP, kFricationAmplitude,
	kPf1, kPf2, kPf3, kPf4, kPf5, kPf6,
	kPb1, kPb2, kPb3, kPb4, kPb5, kPb6,
	kPa1, kPa2, kPa3, kPa4, kPa5, kPa6,
	kParallelBypass, kPreFormantGain, kOutputGain, kEndVoicePitch,
	kNumParams
};
static_assert(kNumParams == 47, "frame ABI is 47 doubles");

// The 14 two-pole sections in the order the engine numbers them:
//   0 rN0 (anti), 1 rNP, 2..7 cascade r6..r1 (order of use, reference speechWaveGenerator.cpp:149-156),
//   8..13 parallel r1..r6 (reference :172-177).
constexpr int kNumResonators = 14;
constexpr int kResN0 = 0, kResNP = 1, kResCascade = 2, kResParallel = 8;

// frame slot holding the centre frequency / bandwidth of resonator r
KLATT_HD constexpr int resFreqParam(int r) {
	return r == kResN0 ? kCfN0 : r == kResNP ? kCfNP : r < kResParallel ? (kCf6 - (r - kResCascade)) : (kPf1 + (r - kResParallel));
}
KLATT_HD constexpr int resBwParam(int r) {
	return r == kResN0 ? kCbN0 : r == kResNP ? kCbNP : r < kResParallel ? (kCb6 - (r - kResCascade)) : (kPb1 + (r - kResParallel));
}

// kPrecisionStream: per-handle API only -- FP32 arithmetic rendered one pull at a time by the time-parallel block
// kernel (klatt_pull.cu) with the frame manager on the host (pull_manager.h): the low-latency path
enum Precision : int { kPrecisionF64 = 0, kPrecisionF32 = 1, kPrecisionStream = 2 };
enum NoiseMode : int { kNoisePhilox = 0, kNoiseGlibc = 1, kNoiseReplay = 2 };

// ---------------------------------------------------------------------------------------------
// Frame-manager state of one stream: the members of the reference's FrameManagerImpl
// (src/frame.cpp:30-39) plus the queue cursor.  Lives in HBM between launches; precision-independent.
// ---------------------------------------------------------------------------------------------
struct FrameMgrState {
	// first 16 bytes are what the host reads back after a launch
	int32_t lastUserIndex;   // frame.cpp:39
	uint32_t qHead;          // requests consumed so far (absolute count)
	uint32_t counter;        // sampleCounter, frame.cpp:38
	uint8_t hasNew;          // newFrameRequest != NULL
	uint8_t curIsNull;       // frame.cpp:37
	uint8_t oldIsNull;       // oldFrameRequest->NULLFrame
	uint8_t newIsNull;
	uint32_t oldM;           // oldFrameRequest->minNumSamples
	uint32_t newM, newF;     // of the request being faded in
	uint32_t purgePending;   // host-set: a purgeQueue=true request arrived since the last launch (frame.cpp:103-112);
	                         // the next launch applies the purge prologue and clears it
	double oldInc, newInc;   // voicePitchInc of old / new
	double oldFrame[kNumParams];
	double newFrame[kNumParams];
	double curFrame[kNumParams];
};

// Generator state, FP64 parity kernel: members of SpeechWaveGeneratorImpl and its parts
// (src/speechWaveGenerator.cpp:34,49,93-101,184-192).  Coefficients are a pure function of curFrame and are
// recomputed on entry, so the reference's setOnce/frequency/bandwidth cache needs no storage.
struct GenStateF64 {
	double pitchPos, vibratoPos;   // FrequencyGenerator::lastCyclePos x2
	double aspLast, fricLast;      // NoiseGenerator::lastValue x2
	double p1[kNumResonators], p2[kNumResonators];
	uint64_t samplesGenerated;     // == rand() draws consumed / 2
};

// Generator state, FP32 production kernels (DESIGN.md "FP32 formulation").
constexpr int kNumDirect = 16;   // frame params used directly by the DSP each tick (not via coefficients / phase increments)

// Everything the FP32 kernels need to walk one fade (request j faded in from its predecessor) without
// transcendental functions in the per-tick path.  Computed in double by planFade() -- by klatt_plan_kernel for
// whole pre-queued batches, or inline at the pop tick when the predecessor is only known at run time
// (per-handle API, purge).
//   direct params : value at fade start, per-tick increment, value after the fade
//   resonators    : zeta = 1 - pole (pole = r*exp(i*theta), r = exp(-pi*bw/sr), theta = 2*pi*f/sr) at fade start
//                   and end, plus the per-tick complex ratio of the pole written as 1 - omega.  A linear fade of
//                   (f, bw) makes the pole a complex geometric sequence.  Only SMALL quantities are stored (zeta,
//                   omega), never b~2, c~-1;  a = |zeta|^2 and rho = 1-|pole|^2 = 2*Re(zeta) - a follow per tick.
//   vibrato       : phase increment per tick as 2^-64-cycle fixed point (start, per-tick change, end), and the depth
//                   0.06 * vibratoPitchOffset (start, per-tick change, end) in double: a depth rounded to FP32 is a
//                   constant pitch error of up to 2^-24 relative for the whole request, which the FP64 glottal phase
//                   integrates and never forgets -- after minutes a sawtooth wrap lands on the neighbouring tick
constexpr int kCoarseTicks = 64;  // drift control: every 64 samples the per-tick pole recurrence is re-based on a
                                   // 64-tick recurrence, so rounding bias accumulates over F/64 + 127 steps, not F
struct alignas(16) FadePlanF32 {
	float z0re[kNumResonators], z0im[kNumResonators];
	float zFre[kNumResonators], zFim[kNumResonators];
	float wre[kNumResonators], wim[kNumResonators];
	float Wre[kNumResonators], Wim[kNumResonators];  // the same ratio over kCoarseTicks ticks at once
	float dir0[kNumDirect], dirStep[kNumDirect], dirFinal[kNumDirect];
	int64_t vibInc0, vibIncStep, vibIncFinal;
	double depth0, depthStep, depthFinal;
	uint32_t n0InvFade, n0InvFinal;  // anti-resonator inverted (cfN0 != 0, reference speechWaveGenerator.cpp:120) during / after the fade
};
static_assert(sizeof(FadePlanF32) % 16 == 0, "plan records are read with 16-byte loads");

// affine map of one two-pole section over a run of ticks, (y, d)_end = P (y, d)_start + z, row-major P: what pass 1 of a
// time-parallel stage leaves for the scan (klatt_tick_core.cuh)
struct Affine {
	float p00, p01, p10, p11, zy, zd;
};

struct GenStateF32 {
	double pitchPos;               // glottal phase in cycles, FP64 and accumulated exactly like the reference does
	double pitch;                  // cur.voicePitch
	double pitchInc;               // its per-tick increment in force: fade step, hold glide, or 0 (pop / swap / landing tick)
	double pitchOld, pitchNew;     // end points of the fade in progress (the landing tick evaluates old+(new-old)*1.0)
	uint64_t samplesGenerated;
	uint64_t vibratoPos;           // vibrato phase, 2^-64 cycles (exact integer accumulation)
	int64_t vibInc;                // its current per-tick increment (vibratoSpeed/sampleRate)
	float aspLast, fricLast;       // coloured-noise memories, in units of 2^-23
	uint32_t n0Inv;                // anti-resonator currently inverted
	uint32_t holdArmed;            // holding with pitchInc == oldInc and nextEvent == oldM+1 (pure-hold chunks allowed)
	uint32_t nextEvent;            // sampleCounter value at which the frame manager has something to do
	uint32_t coarseAt;             // fade tick at which zc[] was last in sync (0x80000000: not yet)
	uint32_t callPos;              // ticks of the current synthesize call already rendered (round-based execution)
	uint32_t callDrained;          // the queue drained during the current call
	float y[kNumResonators];       // delta-form state: last output (rN0: last input)
	float d[kNumResonators];       //                   last output difference (rN0: last input difference)
	float zre[kNumResonators];     // zeta = 1 - pole, tracked through fades
	float zim[kNumResonators];
	float dir[kNumDirect];         // current value of the directly used params
	float zc[2 * kNumResonators];  // coarse-recurrence state (zeta re/im) of the fade in progress
	double depth;                  // current vibrato depth, 0.06 * vibratoPitchOffset (FadePlanF32: in double)
	FadePlanF32 plan;              // plan of the fade in progress when it was made inline (no precomputed plans)
};

// The same two blocks WITHOUT what a pre-queued (planned) FP32 stream never touches -- the three 47-double frames of the
// frame manager and the inline fade plan: 560 bytes instead of 2.4 KB.  The block scheduler (klatt_f32_block.cu) keeps the
// streams of a call in a dense array of these (65 536 streams: 31 MB, resident in the 126 MB L2) and switches a stream
// between the hold, fade and general loops every 64..128 ticks; members keep the names of the full structures so the
// render bodies of klatt_f32_core.cuh work on either.
struct FrameMgrLite {
	int32_t lastUserIndex;
	uint32_t qHead, counter;
	uint8_t hasNew, curIsNull, oldIsNull, newIsNull;
	uint32_t oldM, newM, newF, purgePending;
	double oldInc, newInc;
};
struct GenStateF32Lite {
	double pitchPos, pitch, pitchInc, pitchOld, pitchNew;
	uint64_t samplesGenerated, vibratoPos;
	int64_t vibInc;
	float aspLast, fricLast;
	uint32_t n0Inv, holdArmed, nextEvent, coarseAt, callPos, callDrained;
	float y[kNumResonators], d[kNumResonators], zre[kNumResonators], zim[kNumResonators];
	float dir[kNumDirect];
	float zc[2 * kNumResonators];
	double depth;
	uint32_t pad[2];
};
struct alignas(8) StreamStateLite {  // (8, not 16: the copies staged in shared memory sit on an 8-byte aligned stride)
	FrameMgrLite fm;
	GenStateF32Lite f32;
};

static_assert(sizeof(StreamStateLite) % 16 == 0, "records are copied with 16-byte accesses");

struct StreamState {
	FrameMgrState fm;
	union {
		GenStateF64 f64;
		GenStateF32 f32;
	} gen;
};

// What a render kernel needs to know about one stream.  Built on the host (per-handle API) or by
// build_descs_kernel (batch API) and read once per launch.
struct StreamDesc {
	StreamState *state;
	const double *frames;        // [qCount][47], queue order; rows of NULL requests are ignored
	const uint32_t *minDur;      // [qCount]
	const uint32_t *fadeDur;     // [qCount]  (0 means 1, reference speechPlayer.cpp:36)
	const int32_t *userIndex;    // [qCount] or nullptr (-1)
	const uint8_t *isNull;       // [qCount] or nullptr (all real)
	const int32_t *replay;       // noise draws for kNoiseGlibc / kNoiseReplay, else nullptr
	uint64_t replayLen;
	uint64_t replayBase;         // draw index of replay[0] (draws consumed before this buffer)
	uint64_t streamId;           // Philox counter words 2,3
	uint32_t qCount;             // requests available in the arrays (absolute index qBase + i)
	uint32_t qBase;              // absolute index of frames[0]
	const FadePlanF32 *plans;    // [qCount] precomputed fade plans (FP32 kernels), or nullptr: plan inline at the pop tick
};

// Per-stream outcome of one launch (optional output of the render kernels).
struct StreamResult {
	uint32_t written;        // samples produced by this launch (what speechPlayer_synthesize returns)
	int32_t lastUserIndex;   // getLastIndex() after the launch
	uint32_t qHead;          // absolute count of requests consumed so far
	uint32_t pad;
};

struct NoiseConfig {
	int mode;
	uint64_t seed;
};

}  // namespace klatt
