// FP32 production formulation of the Klatt hot path (one stream, serial in time).
//
// renderGeneralF32() and renderHoldF32() below ARE the bodies of the two batch kernels (klatt_f32.cu calls them
// once per thread); they are written against plain pointers so that the very same arithmetic can also be compiled
// for the host by the numerics study under tests/hostsim/ (test infrastructure; the product never runs it on a CPU).
// Every multiply-add that is meant to be fused is an explicit fmaf(); the translation unit is compiled with
// -fmad=false (host: -ffp-contract=off), so both functions round identically on a hold tick and a stream may
// switch between them at any chunk boundary without changing a single output bit.
//
// What they compute is the reference's per-sample loop (reference src/speechWaveGenerator.cpp:197-214 driven by
// the frame manager of src/frame.cpp:41-80), reformulated so that FP32 is accurate enough (DESIGN.md
// "FP32 formulation" has the derivations and the measured SNR):
//
//  * frame manager: same tick state machine (pop / fade / swap / hold, NULL-frame rewrites, userIndex, drain),
//    run as EVENTS: a stream only enters the state machine on the ticks where something changes (first fade
//    tick, landing tick, swap tick, first hold tick, pop tick); every other tick is the same straight-line
//    update with per-tick INCREMENTS that are zero outside fades.  The increments of a fade are prepared once
//    per request by planFade() in double.
//  * pitch and glottal phase stay FP64 (src/speechWaveGenerator.cpp:55,74): the sawtooth turns phase error into
//    full-scale error (a wrap that lands one sample early rings through every resonator), FP32 phase gives
//    ~11 dB SNR.  Vibrato phase and its increment are 64-bit fixed point: exact accumulation, no drift.  The
//    vibrato depth (0.06 * vibratoPitchOffset, lerped through fades) is FP64 too: the phase is never reset, so it
//    integrates a constant pitch error for as long as the stream lives, and a depth rounded to FP32 (2^-24 relative)
//    moved wraps to the neighbouring tick after 2-3 minutes of audio (61 dB SNR over 10 minutes, 92 dB in FP64).
//    Only the vibrato sine is FP32: its gain is divided out of the depth (vibratoDepth), and its rounding changes from tick
//    to tick and does not add up.
//  * two-pole sections run in DELTA FORM:  d' = (1-rho)*d + a*(x - y);  y' = y + d'
//    (a = |1-pole|^2, rho = 1-|pole|^2), algebraically the reference's  y' = a*x + b*y + c*y1  (b = 2 - rho - a,
//    c = rho - 1; src :116-131) but only the SMALL quantities a, rho, d are represented, instead of cancelling
//    b ~ 2 against c ~ -1.
//  * coefficients during a fade: a linear fade of (f, bw) moves the pole along a complex geometric sequence,
//    so zeta = 1 - pole is advanced by  zeta' = zeta + omega - zeta*omega  (6 flops) and a = |zeta|^2,
//    rho = 2*Re(zeta) - a follow (3 flops), instead of 14 x (exp + cos) per tick (src :113-125).
//  * noise, source shaping, mixes, gain, clamp and truncation follow src :40, :72-86, :150, :172-179, :207-208.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <type_traits>
#include "klatt_common.h"
#include "philox.cuh"

#if defined(__GNUC__) || defined(__CUDACC__)
#define KLATT_UNLIKELY(x) __builtin_expect(!!(x), 0)
#else
#define KLATT_UNLIKELY(x) (x)
#endif

namespace klatt {

// slots of GenStateF32::dir (dVibratoPitchOffset keeps the pair layout; the render paths carry the vibrato depth in
// double instead: GenStateF32::depth, FadePlanF32::depth*)
enum Direct : int {
	dVibratoPitchOffset = 0, dVoiceTurbulenceAmplitude, dGlottalOpenQuotient, dVoiceAmplitude,
	dAspirationAmplitude, dCaNP, dPa1, dPa2, dPa3, dPa4, dPa5, dPa6, dFricationAmplitude, dParallelBypass,
	dPreFormantGain, dOutputGain  // (pa1, pa2) (pa3, pa4) (pa5, pa6) sit in pairs 3..5: they multiply resonator pairs
};
static_assert(dOutputGain + 1 == kNumDirect, "direct slots");

KLATT_HD constexpr int directParam(int i) {
	return i == dVibratoPitchOffset ? kVibratoPitchOffset
	     : i == dVoiceTurbulenceAmplitude ? kVoiceTurbulenceAmplitude : i == dGlottalOpenQuotient ? kGlottalOpenQuotient
	     : i == dVoiceAmplitude ? kVoiceAmplitude : i == dAspirationAmplitude ? kAspirationAmplitude
	     : i == dCaNP ? kCaNP : i == dFricationAmplitude ? kFricationAmplitude
	     : (i >= dPa1 && i <= dPa6) ? (kPa1 + (i - dPa1))
	     : i == dParallelBypass ? kParallelBypass : i == dPreFormantGain ? kPreFormantGain : kOutputGain;
}

// ---------------------------------------------------------------------------------------------------
// planFade: everything a fade from frame `o` to frame `n` over F ticks needs (double precision, once per request).
// `o`/`n` are what the reference holds in oldFrameRequest->frame / newFrameRequest->frame after the pop-tick
// rewrites (src/frame.cpp:59-71).  NaN in a target keeps the old value (src/utils.h:21).  voicePitch is not
// part of the plan (it is tracked in FP64 by the render kernels).
// ---------------------------------------------------------------------------------------------------
// 1 - exp(x + i*th) as (re, im), cancellation-free: 1 - r cos(th) = -expm1(x) + 2 r sin^2(th/2), r sin(th) = 2 r sin(th/2) cos(th/2).
// One expm1 and one sincos (the plan kernel spends all its time in these: 4 per resonator per request).
KLATT_HD void oneMinusExpD(double x, double th, double &re, double &im) {
	double em1 = expm1(x);  // r - 1
	double r = 1.0 + em1;
	double sh, ch;
	sincos(0.5 * th, &sh, &ch);
	re = -em1 + 2.0 * r * sh * sh;
	im = -r * (2.0 * sh * ch);
}
KLATT_HD void oneMinusExp(double x, double th, float &re, float &im) {
	double dre, dim;
	oneMinusExpD(x, th, dre, dim);
	re = (float)dre;
	im = (float)dim;
}
KLATT_HD void poleTerms(double f, double bw, double srInv, float &zre, float &zim) {
	const double PI = 3.14159265358979323846;
	oneMinusExp(-PI * bw * srInv /* log of the pole radius */, 2.0 * PI * f * srInv /* pole angle */, zre, zim);
}

// vibratoSpeed (Hz) -> phase increment per tick in 2^-64 cycles
KLATT_HD int64_t vibratoIncrement(double speed, double srInv) {
	double t = speed * srInv;  // cycles per tick
	if (t != t) t = 0.0;
	if (!(t > -0.49 && t < 0.49)) t = fmod(t, 1.0);  // absurd speeds: only the fraction of a cycle matters
	if (t >= 0.5) t -= 1.0;
	if (t < -0.5) t += 1.0;
	return (int64_t)(t * 18446744073709551616.0);
}

// vibratoPitchOffset -> the depth the FP32 vibrato sine is multiplied by: pitch * (1 + sinTurns(t) * depth) is the reference's
// pitch * (1 + sin(2*pi*t) * 0.06 * vibratoPitchOffset) (src/speechWaveGenerator.cpp:73).  The float coefficients of sinTurns
// (2*pi itself is 2.8e-8 high in FP32) make its fundamental 3.861e-8 larger than sin's, and a gain error of the vibrato is a
// pitch error the glottal phase integrates like a wrong depth (tests/test_long_stream_numerics_cpu.py measures the gain of
// the compiled sinTurns); the depth divides it out.
constexpr double kSinTurnsGain = 1.0 + 3.861e-8;
KLATT_HD double vibratoDepth(double vibratoPitchOffset) { return vibratoPitchOffset * (0.06 / kSinTurnsGain); }

KLATT_HD void planFade(const double *o, const double *n, uint32_t F, int sampleRate, FadePlanF32 &p) {
	const double srInv = 1.0 / (double)sampleRate;
	const double invF = 1.0 / (double)F;
	{
		double v0 = o[kVibratoSpeed], v1 = n[kVibratoSpeed];
		if (v1 != v1) v1 = v0;
		p.vibInc0 = vibratoIncrement(v0, srInv);
		p.vibIncFinal = vibratoIncrement(v0 + ((v1 - v0) * 1.0), srInv);
		p.vibIncStep = (p.vibIncFinal - p.vibInc0) / (int64_t)F;
		double d0 = o[kVibratoPitchOffset], d1 = n[kVibratoPitchOffset];
		if (d1 != d1) d1 = d0;
		p.depth0 = vibratoDepth(d0);
		p.depthStep = vibratoDepth((d1 - d0) * invF);
		p.depthFinal = vibratoDepth(d0 + ((d1 - d0) * 1.0));
	}
	for (int i = 0; i < kNumDirect; ++i) {
		double a = o[directParam(i)], b = n[directParam(i)];
		if (b != b) b = a;  // NaN target: keep
		p.dir0[i] = (float)a;
		p.dirStep[i] = (float)((b - a) * invF);
		p.dirFinal[i] = (float)(a + ((b - a) * 1.0));
	}
	for (int r = 0; r < kNumResonators; ++r) {
		double f0 = o[resFreqParam(r)], f1 = n[resFreqParam(r)];
		double b0 = o[resBwParam(r)], b1 = n[resBwParam(r)];
		if (f1 != f1) f1 = f0;
		if (b1 != b1) b1 = b0;
		poleTerms(f0, b0, srInv, p.z0re[r], p.z0im[r]);
		poleTerms(f0 + ((f1 - f0) * 1.0), b0 + ((b1 - b0) * 1.0), srInv, p.zFre[r], p.zFim[r]);
		// per-tick ratio of the pole: q*exp(i*dth) = 1 - omega
		const double PI = 3.14159265358979323846;
		double xs = -PI * (b1 - b0) * invF * srInv;
		double dth = 2.0 * PI * (f1 - f0) * invF * srInv;
		double wr, wi;
		oneMinusExpD(xs, dth, wr, wi);
		p.wre[r] = (float)wr; p.wim[r] = (float)wi;
		// the same pole ratio over kCoarseTicks = 2^6 ticks: (1 - w)^2 = 1 - w(2 - w), six times, in double (cancellation-free like
		// the one-tick form, ~1e-15 relative; a quarter of the plan kernel's transcendentals less)
		static_assert(kCoarseTicks == 64, "six squarings");
#pragma unroll
		for (int k = 0; k < 6; ++k) {
			const double ar = 2.0 - wr, ai = -wi;
			const double nr = wr * ar - wi * ai, ni = wr * ai + wi * ar;
			wr = nr; wi = ni;
		}
		p.Wre[r] = (float)wr; p.Wim[r] = (float)wi;
		if (r == kResN0) {
			p.n0InvFade = !(f0 == 0 && f1 == 0);
			p.n0InvFinal = (f0 + ((f1 - f0) * 1.0)) != 0;
		}
	}
}

// The frames a pre-queued request fades between, without running the stream (klatt_plan_kernel): request j of a
// queue whose predecessors are all known.  prevReal = the last non-NULL request before j (nullptr: none, the
// zero-initialised oldFrameRequest of src/frame.cpp:86), prevIsNull = request j-1 was a NULL request (or j is
// the first request of a fresh player: the initial old request is NULL, src/frame.cpp:87).
//   NULL request : new = old with preFormantGain 0                          (src/frame.cpp:59-63)
//   real after NULL : old = new with preFormantGain 0                       (src/frame.cpp:64-67)
KLATT_HD void plannedFrames(const double *prevReal, bool prevIsNull, const double *cur, bool curIsNull, double *o, double *n) {
	for (int i = 0; i < kNumParams; ++i) o[i] = prevReal ? prevReal[i] : 0.0;
	if (prevIsNull) o[kPreFormantGain] = 0;
	if (curIsNull) {
		for (int i = 0; i < kNumParams; ++i) n[i] = o[i];
		n[kPreFormantGain] = 0;
	} else {
		for (int i = 0; i < kNumParams; ++i) n[i] = cur[i];
		if (prevIsNull) {
			for (int i = 0; i < kNumParams; ++i) o[i] = n[i];
			o[kPreFormantGain] = 0;
		}
	}
}

// ---------------------------------------------------------------------------------------------------
// Roles.  A stream's tick splits into two halves that only meet in the final mix (reference
// src/speechWaveGenerator.cpp:203-207):
//   cascade side  : aspiration, glottal shaping, rN0, rNP, r6..r1          (resonators 0..7)  -> x, and the sample
//   parallel side : noise draws, frication, the six parallel sections      (resonators 8..13) -> par,
//                   and the two oscillators with their FP64 arithmetic: vibrato, pitch glide, glottal phase -> voice
//                   (they feed the cascade side, but depend on nothing the cascade side computes; the cascade
//                   side is a long dependent chain, the parallel side has independent work to hide them behind)
// kRoleBoth runs both in one thread (per-handle API, host numerics build).  The batch kernels give each side its
// own thread in a different warp of the block (half the registers per thread, twice the warps per SM); the
// parallel side hands (aspiration noise word, par, sawtooth value) over through shared memory 8 ticks at a time.  Every role
// executes the same operations on the same values, so all of them produce the same bits.
// ---------------------------------------------------------------------------------------------------
// kRoleCascade / kRoleParallel: the general kernel's split (oscillators on the parallel side: its cascade side is the
// longer dependent chain).  kRoleCascadeOsc / kRoleParallelOnly: the hold kernel's split (straight-line code: the
// oscillators overlap with the cascade chain there, and the parallel side carries the Philox generator).
enum Role : int { kRoleBoth = 0, kRoleCascade = 1, kRoleParallel = 2, kRoleCascadeOsc = 3, kRoleParallelOnly = 4 };
constexpr int kGroupTicks = 8;  // hand-over granularity, and one 16-byte output store
#ifndef KLATT_HOLD_UNROLL
#define KLATT_HOLD_UNROLL 1
#endif
constexpr int kHoldUnroll = KLATT_HOLD_UNROLL;  // tick PAIRS of a hold group per loop body.  1, not the whole group (4): the hold loops
                                                // were 21 KB of straight-line code and ncu showed 10 % of the stall samples waiting for
                                                // instructions; measured 225.8 -> 221.9 ms (config 3), 175.0 -> 163.6 ms (config 5)

template <int ROLE> struct RoleTraits {
	static constexpr bool hasC = ROLE == kRoleBoth || ROLE == kRoleCascade || ROLE == kRoleCascadeOsc;      // cascade side
	static constexpr bool hasP = ROLE == kRoleBoth || ROLE == kRoleParallel || ROLE == kRoleParallelOnly;   // noise + parallel bank
	static constexpr bool hasO = ROLE == kRoleBoth || ROLE == kRoleParallel || ROLE == kRoleCascadeOsc;     // the two oscillators
	static constexpr int R0 = hasC ? 0 : kResParallel;
	static constexpr int R1 = hasP ? kNumResonators : kResParallel;
};
// direct params each side reads
KLATT_HD constexpr bool directOfCascade(int i) {
	return i == dVoiceTurbulenceAmplitude || i == dGlottalOpenQuotient || i == dVoiceAmplitude ||
	       i == dAspirationAmplitude || i == dCaNP || i == dPreFormantGain || i == dOutputGain;
}
KLATT_HD constexpr bool directOfParallel(int i) {
	return i == dFricationAmplitude || (i >= dPa1 && i <= dPa6) || i == dParallelBypass || i == dPreFormantGain;
}
template <int ROLE> KLATT_HD constexpr bool roleUsesDirect(int i) {
	return (RoleTraits<ROLE>::hasC && directOfCascade(i)) || (RoleTraits<ROLE>::hasP && directOfParallel(i));
}

// hand-over between the two sides when they share a thread: plain members
struct XchgSelf {
	uint32_t wA_;
	float par_, voice_;
	KLATT_HD void put(uint32_t, uint32_t wA, float par, float voice) { wA_ = wA; par_ = par; voice_ = voice; }
	KLATT_HD void get(uint32_t, uint32_t &wA, float &par, float &voice) const { wA = wA_; par = par_; voice = voice_; }
	KLATT_HD void sync() {}
};

// ---------------------------------------------------------------------------------------------------
// Packed pairs.  sm_100a issues fma/mul/add/sub.rn.f32x2 (SASS FFMA2 / FMUL2 / FADD2): two independent IEEE FP32
// operations on an aligned register pair in ONE issue slot, with the dependent latency of a scalar FFMA (measured on
// B200, tools/ubench/ffma2.cu: 4.5 cycles; half the issue rate, so the same FP32 peak).  The render kernels are
// bound by issue slots and dependent latency, not by the FMA pipe (ncu: pipe_fma ~33 % busy), so everything that
// comes in independent pairs is computed in pairs: the pole recurrences, the coefficients and the memory part of the
// sections of resonators 2k and 2k+1, the whole parallel bank (three pairs), and the direct parameters.  Each half is
// exactly the scalar operation (the host build below IS the scalar operation), so pairing changes no bit.
// f32x2 has no operand negation, so the working set is kept in the signs that need none:
//   nz  = -zeta   (u = -Re zeta, v = -Im zeta)          ny = -y (negated section output)
//   nrho = -(1 - |pole|^2)                               npar accumulates -par
// Negation commutes with IEEE rounding, so every value is the exact negative of the one the scalar formulation had.
// ---------------------------------------------------------------------------------------------------
struct F2 { float lo, hi; };
KLATT_HD F2 f2(float lo, float hi) { F2 r; r.lo = lo; r.hi = hi; return r; }
KLATT_HD F2 f2s(float x) { F2 r; r.lo = x; r.hi = x; return r; }
KLATT_HD F2 fma2(F2 a, F2 b, F2 c) {
	F2 r;
#ifdef __CUDA_ARCH__
	asm("{ .reg .b64 pa, pb, pc, pd; mov.b64 pa, {%2, %3}; mov.b64 pb, {%4, %5}; mov.b64 pc, {%6, %7}; "
	    "fma.rn.f32x2 pd, pa, pb, pc; mov.b64 {%0, %1}, pd; }"
	    : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi), "f"(c.lo), "f"(c.hi));
#else
	r.lo = fmaf(a.lo, b.lo, c.lo); r.hi = fmaf(a.hi, b.hi, c.hi);
#endif
	return r;
}
KLATT_HD F2 mul2(F2 a, F2 b) {
	F2 r;
#ifdef __CUDA_ARCH__
	asm("{ .reg .b64 pa, pb, pd; mov.b64 pa, {%2, %3}; mov.b64 pb, {%4, %5}; mul.rn.f32x2 pd, pa, pb; mov.b64 {%0, %1}, pd; }"
	    : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi));
#else
	r.lo = a.lo * b.lo; r.hi = a.hi * b.hi;
#endif
	return r;
}
KLATT_HD F2 add2(F2 a, F2 b) {
	F2 r;
#ifdef __CUDA_ARCH__
	asm("{ .reg .b64 pa, pb, pd; mov.b64 pa, {%2, %3}; mov.b64 pb, {%4, %5}; add.rn.f32x2 pd, pa, pb; mov.b64 {%0, %1}, pd; }"
	    : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi));
#else
	r.lo = a.lo + b.lo; r.hi = a.hi + b.hi;
#endif
	return r;
}
KLATT_HD F2 sub2(F2 a, F2 b) {
	F2 r;
#ifdef __CUDA_ARCH__
	asm("{ .reg .b64 pa, pb, pd; mov.b64 pa, {%2, %3}; mov.b64 pb, {%4, %5}; sub.rn.f32x2 pd, pa, pb; mov.b64 {%0, %1}, pd; }"
	    : "=f"(r.lo), "=f"(r.hi) : "f"(a.lo), "f"(a.hi), "f"(b.lo), "f"(b.hi));
#else
	r.lo = a.lo - b.lo; r.hi = a.hi - b.hi;
#endif
	return r;
}
// half r&1 of pair r>>1 (r is a compile-time constant everywhere: the loops are fully unrolled)
KLATT_HD float &half(F2 *arr, int r) { return (r & 1) ? arr[r >> 1].hi : arr[r >> 1].lo; }
KLATT_HD const float &half(const F2 *arr, int r) { return (r & 1) ? arr[r >> 1].hi : arr[r >> 1].lo; }

constexpr int kNumPairs = kNumResonators / 2;       // (rN0, rNP) (r6, r5) (r4, r3) (r2, r1) | (p1, p2) (p3, p4) (p5, p6)
constexpr int kNumDirectPairs = kNumDirect / 2;     // direct params 2k and 2k+1
static_assert(kResCascade % 2 == 0 && kResParallel % 2 == 0, "role boundaries fall between pairs");
template <int ROLE> struct PairTraits {
	static constexpr int P0 = RoleTraits<ROLE>::R0 / 2, P1 = RoleTraits<ROLE>::R1 / 2;
};
template <int ROLE> KLATT_HD constexpr bool roleUsesDirectPair(int k) {
	return roleUsesDirect<ROLE>(2 * k) || roleUsesDirect<ROLE>(2 * k + 1);
}

// ---------------------------------------------------------------------------------------------------
// per-stream working set (registers on the device).  Arrays are indexed with compile-time constants only
// (every loop below is fully unrolled), so a role never materialises the elements it does not touch.
// ---------------------------------------------------------------------------------------------------
struct DspState {  // what every tick reads AND writes
	F2 ny[kNumPairs];  // NEGATED last output of each section; ny[0].lo is rN0's last INPUT, not negated (it stores inputs)
	F2 d[kNumPairs];   // last output difference (rN0: last input difference)
	float aspLast, fricLast;
	uint64_t vibratoPos;
	int64_t vibInc;
	double pitchPos;         // glottal phase in cycles, FP64 like the reference's (parallel side)
	double pitch, pitchInc;  // cur.voicePitch and its per-tick increment (parallel side)
	double depth;            // vibrato depth 0.06 * cur.vibratoPitchOffset (the oscillators' side)
};

struct CoefF32 {  // what a tick only reads: a pure function of (zeta, direct params)
	F2 a[kNumPairs], nrho[kNumPairs];  // |1 - pole|^2 and -(1 - |pole|^2)
	float invA0;  // 1/a of the anti-resonator
	float vta, goq, va, aa, caNP, bypass;
	F2 pa[3];
	float halfGain, fricGain, og4000;
	bool n0Inv;
};

KLATT_HD float fastRcp(float x) {
#ifdef __CUDA_ARCH__
	float r;
	asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // one MUFU.RCP
	return r;
#else
	return 1.0f / x;
#endif
}

constexpr float kDrawScale = 1.0f / 8388608.0f;  // noise draws enter as 23-bit integers

// nz = -zeta as pairs (u = -Re, v = -Im); dir = the direct params as pairs
template <int ROLE>
KLATT_HD void buildCoef(CoefF32 &C, const F2 *u, const F2 *v, const F2 *dir, bool n0Inv) {
	using T = RoleTraits<ROLE>;
	using P = PairTraits<ROLE>;
#pragma unroll
	for (int k = P::P0; k < P::P1; ++k) {
		F2 a = fma2(u[k], u[k], mul2(v[k], v[k]));  // |1 - pole|^2
		C.a[k] = a;
		C.nrho[k] = fma2(f2s(2.0f), u[k], a);        // -(2 Re zeta - a) = -(1 - |pole|^2)
	}
	C.halfGain = half(dir, dPreFormantGain) * 0.5f;
	if (T::hasC) {
		C.invA0 = fastRcp(C.a[0].lo);
		C.vta = half(dir, dVoiceTurbulenceAmplitude); C.goq = half(dir, dGlottalOpenQuotient);
		C.va = half(dir, dVoiceAmplitude); C.aa = half(dir, dAspirationAmplitude); C.caNP = half(dir, dCaNP);
		C.og4000 = half(dir, dOutputGain) * 4000.0f;
		C.n0Inv = n0Inv;
	}
	if (T::hasP) {
		static_assert(dPa1 % 2 == 0, "the parallel amplitudes are whole pairs of the direct params");
#pragma unroll
		for (int k = 0; k < 3; ++k) C.pa[k] = dir[dPa1 / 2 + k];
		C.bypass = half(dir, dParallelBypass);
		C.fricGain = ((0.3f * kDrawScale) * half(dir, dFricationAmplitude)) * C.halfGain;
	}
}

// one tick of the pole recurrences: zeta' = zeta + omega - zeta*omega (a no-op when omega == 0), on nz = -zeta:
//   tr = fma(-zr, wr, wr);  tr = fma(zi, wi, tr);  ti = fma(-zr, wi, wi);  ti = fma(-zi, wr, ti);  nz' = nz - (tr, ti)
template <int ROLE>
KLATT_HD void stepPoles(F2 *u, F2 *v, const F2 *wr, const F2 *wi) {
	using P = PairTraits<ROLE>;
#pragma unroll
	for (int k = P::P0; k < P::P1; ++k) {
		F2 zi = mul2(v[k], f2s(-1.0f));
		F2 tr = fma2(u[k], wr[k], wr[k]);
		tr = fma2(zi, wi[k], tr);
		F2 ti = fma2(u[k], wi[k], wi[k]);
		ti = fma2(v[k], wr[k], ti);
		u[k] = sub2(u[k], tr);
		v[k] = sub2(v[k], ti);
	}
}

// delta-form two-pole section, scalar (the cascade chain): w = (1-rho)*d - a*y has been prepared (memory part);
// returns the new output
KLATT_HD float sectionOut(float &ny, float &d, float a, float w, float x) {
	float dn = fmaf(a, x, w);
	d = dn;
	ny = ny - dn;
	return -ny;
}
// memory part of two sections at once: (1-rho)*d - a*y
KLATT_HD F2 sectionMemory(const DspState &S, const CoefF32 &C, int k) {
	F2 w = fma2(C.nrho[k], S.d[k], S.d[k]);
	return fma2(C.a[k], S.ny[k], w);
}

// sin(2*pi*t) for |t| <= 0.5: fold to |t| <= 0.25, then t*(c0 + u*Q(u)), u = t^2 (odd degree-11 least-squares fit on
// Chebyshev nodes; the fit is good to 1.3e-11, the FP32 evaluation to ~1 ulp).  Same code on host and device, so the
// CPU numerics tests see the kernel's vibrato bit for bit.
KLATT_HD float sinTurns(float t) {
	if (t > 0.25f) t = 0.5f - t;
	if (t < -0.25f) t = -0.5f - t;
	const float u = t * t;
	float q = fmaf(u, -14.3368558883667f, 41.999961853027344f);
	q = fmaf(u, q, -76.70366668701172f);
	q = fmaf(u, q, 81.60520935058594f);
	q = fmaf(u, q, -41.34170150756836f);
	return fmaf(t * u, q, t * 6.2831854820251465f);
}

KLATT_HD float bitsToFloat(uint32_t u) {
#ifdef __CUDA_ARCH__
	return __uint_as_float(u);
#else
	float f;
	memcpy(&f, &u, 4);
	return f;
#endif
}

// phase increment in cycles -> 2^-64-cycle fixed point (|x| < 0.5, i.e. |pitch| < sampleRate/2; saturates beyond).
// Used by the time-parallel path (klatt_long.cu), where the phase must be summed associatively.
KLATT_HD int64_t cyclesToFixed(double x) {
#ifdef __CUDA_ARCH__
	return __double2ll_rn(x * 18446744073709551616.0);
#else
	double y = x * 18446744073709551616.0;
	if (y != y) return (int64_t)0x8000000000000000ull;
	if (y >= 9223372036854775807.0) return 0x7fffffffffffffffll;
	if (y <= -9223372036854775808.0) return (int64_t)0x8000000000000000ull;
	return (int64_t)nearbyint(y);
#endif
}

// x - trunc(x): the reference's fmod(x, 1) (src/speechWaveGenerator.cpp:55); exact for |x| < 2^31.  |x| < 2 whenever
// |pitch| < sampleRate: trunc(x) is then -1, 0 or 1 and two compares replace the double->int->double round trip
// through the conversion unit (which sits on the loop-carried chain of the phase: ~40 cycles per tick).
KLATT_HD double fracRef(double x) {
#ifdef __CUDA_ARCH__
	if (fabs(x) < 2.0) {
		double t = x >= 1.0 ? 1.0 : 0.0;
		t = x <= -1.0 ? -1.0 : t;
		return x - t;
	}
	return x - (double)__double2int_rz(x);
#else
	double t = (x != x) ? 0.0 : (x >= 2147483647.0 ? 2147483647.0 : (x <= -2147483648.0 ? -2147483648.0 : (double)(int32_t)x));
	return x - t;
#endif
}

// n successive FP64 additions  p = p + inc  (round to nearest even), bit for bit, in O(binades crossed) steps: the reference's
// hold glide `curFrame.voicePitch += oldFrameRequest->voicePitchInc` once per tick (src/frame.cpp:77), needed in the middle of
// a hold by the time-parallel paths.  While p stays inside one binade every value it takes lies on that binade's grid (ulp
// u), so RN(p + inc) = p + RN_u(inc): a constant step (a tie inc/u = k + 1/2 rounds to even once and is stationary from the
// second addition on).  Two real additions give the stationary step, whole-grid integer arithmetic covers the rest of the
// binade (stopping one step short of either edge, where the ulp changes), and the crossing is done with real additions again.
KLATT_HD double glideExact(double p, double inc, uint64_t n) {
	if (n == 0) return p;
	if (!(inc == inc) || !(p == p) || inc == 0.0) return p + inc;  // NaN propagates; +0 is the identity (the sign of zero never matters here)
	while (n > 0) {
		// three real additions: p1 may still come from the neighbouring binade's grid; p2 = RN(p1 + inc) is then a value this
		// binade's rounding produced (even after a tie), so p2 -> p3 is the stationary step
		const double p1 = p + inc;
		if (--n == 0) return p1;
		const double p2 = p1 + inc;
		if (--n == 0) return p2;
		const double p3 = p2 + inc;
		--n;
		p = p3;
		if (n == 0) return p3;
		const double step = p3 - p2;  // exact (neighbouring values)
		if (step == 0.0) return p3;   // inc is below half an ulp from here on: every further addition is the identity
		const double a1 = p1 < 0 ? -p1 : p1, a2 = p2 < 0 ? -p2 : p2, a3 = p3 < 0 ? -p3 : p3;
		if (!(a3 >= 1e-290 && a3 <= 1e290) || !(a2 >= 1e-290) || !(a1 >= 1e-290)) continue;  // zero, denormal, huge, inf: plain additions
		int e1, e2, e3;
		(void)frexp(a1, &e1);
		(void)frexp(a2, &e2);
		const double f3 = frexp(a3, &e3);  // a3 = f3 * 2^e3, f3 in [0.5, 1)
		if (e1 != e3 || e2 != e3 || (p1 < 0) != (p3 < 0) || (p2 < 0) != (p3 < 0)) continue;  // straddles a binade edge (or zero)
		// grid units: P = a3 / u in [2^52, 2^53), S = signed step of |p| per addition
		const int64_t P = (int64_t)ldexp(f3, 53);
		const double sMag = ldexp(step, 53 - e3);  // exact integer: step is a multiple of u
		const int64_t S = (p3 < 0) ? -(int64_t)sMag : (int64_t)sMag;
		if (S == 0) continue;
		const int64_t lo = (int64_t)1 << 52, hi = (int64_t)1 << 53;
		int64_t room = S > 0 ? (hi - P) / S : (P - lo) / (-S);
		room -= 1;  // stay one step clear of the edge: the addition that reaches it is a real one
		if (room <= 0) continue;
		const uint64_t k = (uint64_t)room < n ? (uint64_t)room : n;
		const double mag = ldexp((double)(P + (int64_t)k * S), e3 - 53);
		p = (p3 < 0) ? -mag : mag;
		n -= k;
	}
	return p;
}

// parallel side of one generated sample (reference src/speechWaveGenerator.cpp:205-206, :170-180): wF is the
// frication noise word (the reference's rand() value is word>>1; the top 23 bits are used).  The six sections run as
// three pairs; the weighted sum is accumulated per half and folded at the end.
KLATT_HD float parallelSide(DspState &S, const CoefF32 &C, uint32_t wF) {
	float uF = bitsToFloat(0x4B000000u | (wF >> 9)) - 8388608.0f;  // exact integer 0..2^23-1
	S.fricLast = fmaf(0.75f, S.fricLast, uF);
	float pin = S.fricLast * C.fricGain;
	const F2 pin2 = f2s(pin);
	F2 nacc = f2s(0.0f);  // -(sum of (y_k - pin) * pa_k), per half
#pragma unroll
	for (int k = 0; k < 3; ++k) {
		const int p = kResParallel / 2 + k;
		F2 dn = fma2(C.a[p], pin2, sectionMemory(S, C, p));
		S.d[p] = dn;
		S.ny[p] = sub2(S.ny[p], dn);
		nacc = fma2(add2(S.ny[p], pin2), C.pa[k], nacc);  // (ny + pin) = -(y - pin)
	}
	float par = -(nacc.lo + nacc.hi);
	return fmaf(pin - par, C.bypass, par);
}

// the two oscillators (reference src/speechWaveGenerator.cpp:73-74, :54-58): vibrato, pitch glide, glottal phase;
// returns the sawtooth value in [0, 1).  The phase is accumulated exactly like the reference does it --
// fmod((pitch*vibrato)/sampleRate + pos, 1) in double, with a true division -- because a pitch whose period is a whole
// number of samples (150 Hz at 22 050 Hz) makes the wrap instant a matter of the last bit of that sum, and a wrap
// that lands one sample apart from the reference's is a full-scale error once per period.
// x / sr, correctly rounded, from the correctly rounded reciprocal (Markstein): q = RN(x*y), r = x - q*sr exactly (FMA),
// RN(q + r*y) is the IEEE quotient.  Three FP64 instructions instead of a division sequence.
KLATT_HD double divideBySampleRate(double x, double srD, double srInv) {
	double q = x * srInv;
	double r = fma(-q, srD, x);
	return fma(r, srInv, q);
}

// The oscillators of one tick as SEGMENTS of one dependent chain (~16 operations through the FP64 and conversion
// units, ~200 cycles end to end).  ptxas keeps close to source order, and the SM issues in order: a warp only keeps
// issuing while the NEXT instruction is independent.  The general kernel therefore threads these segments between
// its other phases (pole recurrences, coefficients, the parallel bank), which do not depend on them; oscillatorSide()
// below is the same segments back to back -- same operations, same bits.
struct OscChain {
	float t, u, q;
	double m, quot, pos;
	KLATT_HD void seg1(DspState &S) {  // vibrato phase -> folded quarter-period argument
		S.vibratoPos += (uint64_t)S.vibInc;
		// cycles in [-0.5, 0.5), rounded to nearest: a truncated phase is a systematic pitch error while a slow vibrato
		// sits inside one quantisation step
		t = (float)(int32_t)(uint32_t)(S.vibratoPos >> 32) * 2.3283064365386963e-10f;
		if (t > 0.25f) t = 0.5f - t;
		if (t < -0.25f) t = -0.5f - t;
		u = t * t;
	}
	KLATT_HD void seg2() {  // the sine polynomial (sinTurns)
		q = fmaf(u, -14.3368558883667f, 41.999961853027344f);
		q = fmaf(u, q, -76.70366668701172f);
		q = fmaf(u, q, 81.60520935058594f);
		q = fmaf(u, q, -41.34170150756836f);
		q = fmaf(t * u, q, t * 6.2831854820251465f);
	}
	KLATT_HD void seg3(DspState &S) {  // pitch glide, pitch * (1 + vibrato), the vibrato in FP64 from the FP32 sine
		S.pitch += S.pitchInc;
		m = S.pitch * fma((double)q, S.depth, 1.0);
	}
	KLATT_HD void seg4(double srD, double srInv) { quot = divideBySampleRate(m, srD, srInv); }
	KLATT_HD void seg5(DspState &S) {
		pos = fracRef(quot + S.pitchPos);
		S.pitchPos = pos;
	}
	KLATT_HD float seg6() const { return (float)pos; }
};

KLATT_HD float oscillatorSide(DspState &S, const CoefF32 &C, double srD, double srInv) {
	OscChain o;
	o.seg1(S); o.seg2(); o.seg3(S); o.seg4(srD, srInv); o.seg5(S);
	return o.seg6();
}

// cascade side (reference src/speechWaveGenerator.cpp:203-204, :72-86, :147-158) and the final mix (:207-208), as
// stages: source -> nasal pair -> six sections -> output.
// ---- aspiration noise + turbulence + glottal shaping (:40, :75-80), returns the cascade input (:147) ----
KLATT_HD float stageSource(DspState &S, const CoefF32 &C, uint32_t wA, float voice) {
	float uA = bitsToFloat(0x4B000000u | (wA >> 9)) - 8388608.0f;
	S.aspLast = fmaf(0.75f, S.aspLast, uA);
	float asp = S.aspLast * (0.2f * kDrawScale);
	float turb = asp * C.vta;
	if (voice < C.goq) turb *= 0.01f;
	float v = (fmaf(voice, 2.0f, -1.0f) + turb) * C.va;
	float src = fmaf(asp, C.aa, v);
	return src * C.halfGain;
}
// ---- rN0 (anti-resonator: memories hold INPUTS, :133), rNP, caNP mix (:148-150) ----
KLATT_HD float stageNasal(DspState &S, const CoefF32 &C, float ci) {
	float dx = ci - S.ny[0].lo;
	float dx1 = fmaf(C.nrho[0].lo, S.d[0].lo, S.d[0].lo);  // (1-rho) * previous input difference
	float n0 = C.n0Inv ? fmaf(dx - dx1, C.invA0, S.ny[0].lo)
	                   : fmaf(C.a[0].lo, dx, dx1 + S.ny[0].lo);
	S.d[0].lo = dx;
	S.ny[0].lo = ci;
	float wNP = fmaf(C.nrho[0].hi, S.d[0].hi, S.d[0].hi);
	wNP = fmaf(C.a[0].hi, S.ny[0].hi, wNP);
	float np = sectionOut(S.ny[0].hi, S.d[0].hi, C.a[0].hi, wNP, n0);
	return fmaf(np - ci, C.caNP, ci);
}
// ---- section q = 0..5 (r6..r1, :151-156); w = its memory part ----
KLATT_HD float stageSection(DspState &S, const CoefF32 &C, int q, float w, float x) {
	const int r = kResCascade + q;
	return sectionOut(half(S.ny, r), half(S.d, r), half(C.a, r), w, x);
}
// ---- mix, gain, clamp with the Win32 macro NaN behaviour (NaN -> +32000), truncate (:207-208) ----
KLATT_HD int stageOut(const CoefF32 &C, float x, float par) {
	float s = (x + par) * C.og4000;
	s = fminf(s, 32000.0f);  // fminf(NaN, 32000) == 32000
	s = fmaxf(s, -32000.0f);
	return (int)s;
}

KLATT_HD int cascadeSide(DspState &S, const CoefF32 &C, uint32_t wA, float par, float voice) {
	float ci = stageSource(S, C, wA, voice);
	F2 w[3];
#pragma unroll
	for (int p = 0; p < 3; ++p) w[p] = sectionMemory(S, C, 1 + p);  // r6 r5 | r4 r3 | r2 r1
	float x = stageNasal(S, C, ci);
#pragma unroll
	for (int q = 0; q < 6; ++q) x = stageSection(S, C, q, half(w, q), x);
	return stageOut(C, x, par);
}

// the two noise words of generated sample `gen` (Philox mode caches the 4-word block of samples 2b, 2b+1)
struct NoiseSource {
	Philox4 blk;
	uint64_t blkIndex;
	KLATT_HD void init() { blk.w[0] = blk.w[1] = blk.w[2] = blk.w[3] = 0; blkIndex = ~0ull; }
	KLATT_HD void draw(const NoiseConfig &noise, const StreamDesc &desc, uint64_t streamId, uint64_t gen, uint32_t &wA, uint32_t &wF) {
		if (noise.mode == kNoisePhilox) {
			uint64_t b = gen >> 1;
			if (b != blkIndex) { blk = noiseBlock(noise.seed, streamId, b); blkIndex = b; }
			bool odd = (gen & 1ull) != 0;
			wA = odd ? blk.w[2] : blk.w[0];
			wF = odd ? blk.w[3] : blk.w[1];
		} else {  // replayed rand() values (31 bits): shift into word position
			uint64_t d0 = 2 * gen - desc.replayBase;
			wA = (d0 < desc.replayLen) ? ((uint32_t)desc.replay[d0] << 1) : 0u;
			wF = (d0 + 1 < desc.replayLen) ? ((uint32_t)desc.replay[d0 + 1] << 1) : 0u;
		}
	}
};

template <int ROLE, class GS>
KLATT_HD void loadDspState(DspState &S, const GS &gs) {
	using T = RoleTraits<ROLE>;
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { half(S.ny, r) = (r == kResN0) ? gs.y[r] : -gs.y[r]; half(S.d, r) = gs.d[r]; }
	if (T::hasC) S.aspLast = gs.aspLast;
	if (T::hasP) S.fricLast = gs.fricLast;
	if (T::hasO) {
		S.vibratoPos = gs.vibratoPos; S.vibInc = gs.vibInc;
		S.pitchPos = gs.pitchPos; S.pitch = gs.pitch; S.pitchInc = gs.pitchInc; S.depth = gs.depth;
	}
}
template <int ROLE, class GS>
KLATT_HD void storeDspState(GS &gs, const DspState &S) {
	using T = RoleTraits<ROLE>;
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { gs.y[r] = (r == kResN0) ? half(S.ny, r) : -half(S.ny, r); gs.d[r] = half(S.d, r); }
	if (T::hasC) gs.aspLast = S.aspLast;
	if (T::hasP) gs.fricLast = S.fricLast;
	if (T::hasO) {
		gs.vibratoPos = S.vibratoPos; gs.vibInc = S.vibInc;
		gs.pitchPos = S.pitchPos; gs.pitch = S.pitch; gs.pitchInc = S.pitchInc; gs.depth = S.depth;
	}
}

// ---------------------------------------------------------------------------------------------------
// renderHoldF32: `ticks` PURE HOLD ticks of one stream (reference src/frame.cpp:76-79: only the pitch glides).
// The caller guarantees (canHoldF32) that no frame-manager event falls inside: coefficients are built once.
// `ticks` is a multiple of kGroupTicks.  Only the cascade side owns the frame-manager counters.
// ---------------------------------------------------------------------------------------------------
template <class FM, class GS>
KLATT_HD bool canHoldF32T(const FM &fm, const GS &gs, uint32_t ticks) {
	return !fm.hasNew && !fm.curIsNull && !fm.purgePending && gs.holdArmed && (uint64_t)fm.counter + ticks <= (uint64_t)fm.oldM;
}
KLATT_HD bool canHoldF32(const StreamState &st, uint32_t ticks) { return canHoldF32T(st.fm, st.gen.f32, ticks); }
// `ticks` ticks ahead are all INTERIOR fade ticks (frame.cpp:49-52 with 1 <= sampleCounter < fade length, no event among
// them) and the first of them falls on the 64-sample grid of the drift control
template <class FM, class GS>
KLATT_HD bool canFadeF32T(const FM &fm, const GS &gs, uint32_t ticks) {
	return fm.hasNew && !fm.purgePending && fm.counter >= 1 && (uint64_t)fm.counter + ticks < (uint64_t)fm.newF &&
	       (gs.samplesGenerated & (uint64_t)(kCoarseTicks - 1)) == 0;
}
// ... and the stream's noise is Philox: renderFadeF32T may run them.  The fade loop draws Philox noise only, so a stream under
// any other noise mode takes the general loop for its interior fades.  Every caller that picks the loop for a stream asks this.
template <class FM, class GS>
KLATT_HD bool canFadeF32T(const FM &fm, const GS &gs, uint32_t ticks, const NoiseConfig &noise) {
	return noise.mode == kNoisePhilox && canFadeF32T(fm, gs, ticks);
}

template <int ROLE, class Out, class Xchg, class FM, class GS>
KLATT_HD void renderHoldF32T(FM &fm, GS &gs, const StreamDesc &desc, int sampleRate, uint32_t ticks, Out &out, const NoiseConfig &noise,
                             Xchg &xc) {
	using T = RoleTraits<ROLE>;
	const double srD = (double)sampleRate, srInv = 1.0 / (double)sampleRate;
	DspState S;
	loadDspState<ROLE>(S, gs);
	CoefF32 C;
	{
		F2 u[kNumPairs], v[kNumPairs], dir[kNumDirectPairs];
#pragma unroll
		for (int r = T::R0; r < T::R1; ++r) { half(u, r) = -gs.zre[r]; half(v, r) = -gs.zim[r]; }
#pragma unroll
		for (int i = 0; i < kNumDirect; ++i)
			if (roleUsesDirectPair<ROLE>(i / 2)) half(dir, i) = roleUsesDirect<ROLE>(i) ? gs.dir[i] : 0.0f;
		buildCoef<ROLE>(C, u, v, dir, gs.n0Inv != 0);
	}
	uint64_t gen = gs.samplesGenerated;
	const uint64_t streamId = desc.streamId;
	NoiseSource ns;
	ns.init();
	const bool evenPhilox = noise.mode == kNoisePhilox && (gen & 1ull) == 0;
	for (uint32_t t = 0; t < ticks; t += kGroupTicks) {
		if (T::hasC && !T::hasP) xc.sync();  // the parallel side has finished this group
		if (!T::hasP || evenPhilox) {  // straight-line group: one Philox block per two ticks
#pragma unroll(kHoldUnroll)
			for (int k = 0; k < kGroupTicks; k += 2) {
				Philox4 blk;
				if (T::hasP) blk = noiseBlock(noise.seed, streamId, (gen + k) >> 1);
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					uint32_t wA = 0;
					float par = 0.0f, voice = 0.0f;
					if (T::hasP) {
						wA = blk.w[2 * h];
						par = parallelSide(S, C, blk.w[2 * h + 1]);
						if (T::hasO && !T::hasC) voice = oscillatorSide(S, C, srD, srInv);
						if (!T::hasC) xc.put(t + k + h, wA, par, voice);
					}
					if (T::hasC) {
						if (!T::hasP) xc.get(t + k + h, wA, par, voice);
						if (T::hasO) voice = oscillatorSide(S, C, srD, srInv);
						out.push(cascadeSide(S, C, wA, par, voice));
					}
				}
			}
		} else {
			for (int k = 0; k < kGroupTicks; ++k) {
				uint32_t wA, wF;
				ns.draw(noise, desc, streamId, gen + k, wA, wF);
				float par = parallelSide(S, C, wF), voice = 0.0f;
				if (T::hasO) voice = oscillatorSide(S, C, srD, srInv);
				if (!T::hasC) xc.put(t + k, wA, par, voice);
				if (T::hasC) out.push(cascadeSide(S, C, wA, par, voice));
			}
		}
		gen += kGroupTicks;
		if (T::hasP && !T::hasC) xc.sync();  // hand the group over
	}
	storeDspState<ROLE>(gs, S);
	if (T::hasC) {
		gs.samplesGenerated = gen;
		fm.counter += ticks;
		gs.callPos += ticks;
	}
}
template <int ROLE, class Out, class Xchg>
KLATT_HD void renderHoldF32(const StreamDesc &desc, int sampleRate, uint32_t ticks, Out &out, const NoiseConfig &noise, Xchg &xc) {
	renderHoldF32T<ROLE>(desc.state->fm, desc.state->gen.f32, desc, sampleRate, ticks, out, noise, xc);
}

// ---------------------------------------------------------------------------------------------------
// renderGeneralF32: advance one stream by up to myTicks ticks through the full frame manager.
// Returns the number of samples produced (< myTicks iff the queue drained).  loopTicks >= myTicks is the trip
// count every thread of a cascade/parallel warp pair shares (hand-over barriers are warp-wide).
// desc.plans (may be null, kRoleBoth only) holds precomputed FadePlanF32 for requests [qBase, qBase+qCount);
// without it the plan is made inline at the pop tick from the frame manager's own frames (per-handle API, purge).
// ---------------------------------------------------------------------------------------------------
template <int ROLE, class Out, class Xchg, class FM, class GS>
KLATT_HD uint32_t renderGeneralF32T(FM &fm, GS &gs, const StreamDesc &desc, int sampleRate, uint32_t myTicks, uint32_t loopTicks, Out &out,
                                    const NoiseConfig &noise, Xchg &xc, int32_t *lastUserIndexOut, uint32_t *qHeadOut) {
	using T = RoleTraits<ROLE>;
	// inline planning (per-handle API, purge) needs the frame manager's three frames and the plan slot of the full state
	constexpr bool kInline = ROLE == kRoleBoth && std::is_same<FM, FrameMgrState>::value;
	const double srD = (double)sampleRate, srInv = 1.0 / (double)sampleRate;
	const bool planned = desc.plans != nullptr;  // always true for the split roles

	uint32_t counter = fm.counter, qHead = fm.qHead;
	uint32_t oldM = fm.oldM, newM = fm.newM, newF = fm.newF;
	int32_t lastUserIndex = fm.lastUserIndex;
	bool hasNew = fm.hasNew, curIsNull = fm.curIsNull, oldIsNull = fm.oldIsNull, newIsNull = fm.newIsNull;
	// (fm.oldInc / fm.newInc / gs.pitchOld / gs.pitchNew are only touched on event ticks, by the parallel side: they stay
	// in memory instead of occupying eight registers)
	uint32_t nextEvent = gs.nextEvent;
	bool holdArmed = gs.holdArmed != 0;
	bool n0Inv = gs.n0Inv != 0;

	DspState S;
	loadDspState<ROLE>(S, gs);
	using P = PairTraits<ROLE>;
	F2 u[kNumPairs], v[kNumPairs], wr[kNumPairs], wi[kNumPairs];  // -zeta and omega, as pairs of resonators
	F2 dir0[kNumDirectPairs], dstep[kNumDirectPairs];
	float kf = 0.0f, kfStep = 0.0f;
	int64_t vibIncStep = 0;
	double depthStep = 0.0;  // S.depth advances by it on every tick (an FP64 sum: ~F ulps off the lerp, far below FP32's 2^-24)
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { half(u, r) = -gs.zre[r]; half(v, r) = -gs.zim[r]; half(wr, r) = 0.0f; half(wi, r) = 0.0f; }
#pragma unroll
	for (int i = 0; i < kNumDirect; ++i)
		if (roleUsesDirectPair<ROLE>(i / 2)) { half(dir0, i) = roleUsesDirect<ROLE>(i) ? gs.dir[i] : 0.0f; half(dstep, i) = 0.0f; }
	uint64_t gen = gs.samplesGenerated;
	const uint64_t streamId = desc.streamId;

	// purge prologue, src/frame.cpp:103-112 (the dropped requests were removed on the host).  fm.curFrame is kept
	// current at every exit in inline mode, so the snapshot is available here; the working set simply stays where
	// the interrupted fade left it.
	if constexpr (kInline) {
		if (fm.purgePending) {
			fm.purgePending = 0;
			counter = oldM;
			if (hasNew) {
				oldIsNull = newIsNull;
				for (int i = 0; i < kNumParams; ++i) fm.oldFrame[i] = fm.curFrame[i];
				hasNew = false;
			}
			S.pitchInc = 0.0;
			holdArmed = false;
			nextEvent = oldM + 1;
		}
	}
	const FadePlanF32 *plan = nullptr;
	if (hasNew) {
		if constexpr (kInline) plan = planned ? desc.plans + (qHead - 1 - desc.qBase) : &gs.plan;
		else plan = desc.plans + (qHead - 1 - desc.qBase);
		if (counter >= 1 && counter < newF) {  // resuming in the middle of a fade: the increments are in force
#pragma unroll
			for (int r = T::R0; r < T::R1; ++r) { half(wr, r) = plan->wre[r]; half(wi, r) = plan->wim[r]; }
#pragma unroll
			for (int i = 0; i < kNumDirect; ++i)
				if (roleUsesDirect<ROLE>(i)) { half(dir0, i) = plan->dir0[i]; half(dstep, i) = plan->dirStep[i]; }
			kf = (float)counter;
			kfStep = 1.0f;
			vibIncStep = plan->vibIncStep;
			depthStep = plan->depthStep;
		}
	}
	uint32_t coarseAt = hasNew ? gs.coarseAt : 0x80000000u;

	NoiseSource ns;
	ns.init();

	uint32_t produced = 0;
	bool active = myTicks > 0;
	for (uint32_t tg = 0; tg < loopTicks; tg += kGroupTicks) {
	if (T::hasC && !T::hasP) xc.sync();  // the parallel side has finished this group
	for (uint32_t t = tg; t < tg + kGroupTicks && t < loopTicks; ++t) {
		if (active) {
			// ================= frame manager, src/frame.cpp:41-80, entered only on event ticks =================
			counter++;
			if (KLATT_UNLIKELY(counter >= nextEvent)) {
				if (hasNew) {
					if (counter > newF) {  // :44-47 the fade is over: new becomes old; cur keeps its ratio-1 value
						if constexpr (kInline) {
							if (!planned)
								for (int i = 0; i < kNumParams; ++i) fm.oldFrame[i] = fm.newFrame[i];
						}
						oldM = newM; oldIsNull = newIsNull;
						if (T::hasO) fm.oldInc = fm.newInc;
						hasNew = false;
						S.pitchInc = 0.0;
						nextEvent = counter + 1;  // next tick: first hold tick, or the next pop
					} else if (counter == 1 && newF > 1) {  // :49-52 first fade tick: start from the (possibly rewritten) old frame
#pragma unroll
						for (int r = T::R0; r < T::R1; ++r) {
							half(u, r) = -plan->z0re[r]; half(v, r) = -plan->z0im[r]; half(wr, r) = plan->wre[r]; half(wi, r) = plan->wim[r];
						}
#pragma unroll
						for (int i = 0; i < kNumDirect; ++i)
							if (roleUsesDirect<ROLE>(i)) { half(dir0, i) = plan->dir0[i]; half(dstep, i) = plan->dirStep[i]; }
						kf = 0.0f; kfStep = 1.0f;
						if (T::hasO) {
							S.vibInc = plan->vibInc0; vibIncStep = plan->vibIncStep;
							S.depth = plan->depth0; depthStep = plan->depthStep;
							const double pitchOld = gs.pitchOld, pitchNew = gs.pitchNew;
							S.pitch = pitchOld;
							S.pitchInc = (pitchNew != pitchNew) ? 0.0 : (pitchNew - pitchOld) / (double)newF;
						}
						if (T::hasC) n0Inv = plan->n0InvFade != 0;
						coarseAt = 0x80000000u;
						nextEvent = newF;
					} else {  // counter == newF, ratio == 1: land exactly on the planned end values
#pragma unroll
						for (int r = T::R0; r < T::R1; ++r) {
							half(u, r) = -plan->zFre[r]; half(v, r) = -plan->zFim[r]; half(wr, r) = 0.0f; half(wi, r) = 0.0f;
						}
#pragma unroll
						for (int i = 0; i < kNumDirect; ++i)
							if (roleUsesDirect<ROLE>(i)) { half(dir0, i) = plan->dirFinal[i]; half(dstep, i) = 0.0f; }
						kf = 0.0f; kfStep = 0.0f;
						if (T::hasC) n0Inv = plan->n0InvFinal != 0;
						if (T::hasO) {
							const double pitchOld = gs.pitchOld, pitchNew = gs.pitchNew;
							S.pitch = (pitchNew != pitchNew) ? pitchOld : pitchOld + ((pitchNew - pitchOld) * 1.0);
							S.pitchInc = 0.0;
							S.vibInc = plan->vibIncFinal; vibIncStep = 0;
							S.depth = plan->depthFinal; depthStep = 0.0;
						}
						nextEvent = newF + 1;
					}
				} else if (counter > oldM) {  // :54
					uint32_t rel = qHead - desc.qBase;
					if (rel < desc.qCount) {  // :55-72
						curIsNull = false;
						// the working set is where the previous request left it and stays frozen for this tick (cur is
						// untouched on the pop tick, so this tick still renders with the stale values)
						newM = desc.minDur[rel];
						uint32_t fd = desc.fadeDur[rel];
						newF = fd > 1u ? fd : 1u;  // src/speechPlayer.cpp:36
						newIsNull = desc.isNull ? (desc.isNull[rel] != 0) : false;
						int32_t ux = desc.userIndex ? desc.userIndex[rel] : -1;
						qHead++;
						hasNew = true;
						double pitchOld = S.pitch, pitchNew, newInc;  // old.frame.voicePitch follows the glide (:78)
						if constexpr (kInline) {
							if (!planned) {
								fm.oldFrame[kVoicePitch] = S.pitch;
								for (int i = 0; i < kNumParams; ++i) fm.curFrame[i] = fm.oldFrame[i];
							}
						}
						if (newIsNull) {  // :59-63
							if constexpr (kInline) {
								if (!planned) {
									for (int i = 0; i < kNumParams; ++i) fm.newFrame[i] = fm.oldFrame[i];
									fm.newFrame[kPreFormantGain] = 0;
								}
							}
							pitchNew = S.pitch;
							newInc = 0;
						} else {
							const double *fr = desc.frames + (size_t)rel * kNumParams;
							pitchNew = fr[kVoicePitch];
							newInc = (fr[kEndVoicePitch] - fr[kVoicePitch]) / (double)newM;  // src/frame.cpp:98
							if constexpr (kInline) {
								if (!planned)
									for (int i = 0; i < kNumParams; ++i) fm.newFrame[i] = fr[i];
							}
							if (oldIsNull) {  // :64-67
								pitchOld = pitchNew;
								if constexpr (kInline) {
									if (!planned) {
										for (int i = 0; i < kNumParams; ++i) fm.oldFrame[i] = fm.newFrame[i];
										fm.oldFrame[kPreFormantGain] = 0;
									}
								}
							}
						}
						if (ux != -1) lastUserIndex = ux;  // :69
						counter = 0;                       // :70
						pitchNew += (newInc * (double)newF);  // :71
						if (T::hasO) { gs.pitchOld = pitchOld; gs.pitchNew = pitchNew; fm.newInc = newInc; }
						if (planned) {
							plan = desc.plans + rel;
						} else {
							if constexpr (kInline) {  // plan the fade here (double precision, once per request)
								fm.newFrame[kVoicePitch] = pitchNew;
								fm.oldFrame[kVoicePitch] = pitchOld;
								planFade(fm.oldFrame, fm.newFrame, newF, sampleRate, gs.plan);
								plan = &gs.plan;
							}
						}
						S.pitchInc = 0.0;
						holdArmed = false;
						nextEvent = 1;
					} else {
						curIsNull = true;  // :73-75
					}
				} else {  // :76-79 first hold tick: only the pitch glides from here on
					if (T::hasO) S.pitchInc = fm.oldInc;
					holdArmed = true;
					nextEvent = oldM + 1;
				}
				if (curIsNull) active = false;  // src/speechWaveGenerator.cpp:210
			}
		}
		if (active) {
			// ================= the straight-line per-tick update (all increments are zero outside fades) ===========
			// Order matters for speed, not for the result: the noise block (every other tick, a chain of ten dependent
			// rounds) is drawn first so that the rest is one basic block, and the oscillator chain is threaded through
			// the phases that do not depend on it.
			uint32_t wA = 0, wF = 0;
			if (T::hasP) ns.draw(noise, desc, streamId, gen, wA, wF);
			const bool oscHere = T::hasO && !T::hasC;  // the parallel warp of a pair carries the oscillators
			OscChain osc;
			kf += kfStep;
			if (T::hasO) { S.vibInc += vibIncStep; S.depth += depthStep; }
			if (KLATT_UNLIKELY((gen & (uint64_t)(kCoarseTicks - 1)) == 0 && kfStep != 0.0f)) {
				// drift control, on a grid of ABSOLUTE sample indices (identical for every chunking of the render, and
				// the same loop iteration for every lane of a batch that started together): the poles of this tick come
				// from the coarse recurrence instead of the per-tick one
				if (counter - coarseAt == (uint32_t)kCoarseTicks) {
#pragma unroll
					for (int r = T::R0; r < T::R1; ++r) {
						float zr = gs.zc[r], zi = gs.zc[kNumResonators + r], Wr = plan->Wre[r], Wi = plan->Wim[r];
						float tr = fmaf(-zr, Wr, Wr);
						tr = fmaf(zi, Wi, tr);
						float ti = fmaf(-zr, Wi, Wi);
						ti = fmaf(-zi, Wr, ti);
						half(u, r) = -(zr + tr);
						half(v, r) = -(zi + ti);
					}
				} else {
					stepPoles<ROLE>(u, v, wr, wi);
				}
#pragma unroll
				for (int r = T::R0; r < T::R1; ++r) { gs.zc[r] = -half(u, r); gs.zc[kNumResonators + r] = -half(v, r); }
				coarseAt = counter;
			} else {
				stepPoles<ROLE>(u, v, wr, wi);
			}
			// (one basic block from here to the end of the tick)
			if (oscHere) { osc.seg1(S); osc.seg2(); }
			CoefF32 C;
			{
				F2 dir[kNumDirectPairs];
				const F2 kf2 = f2s(kf);
#pragma unroll
				for (int k = 0; k < kNumDirectPairs; ++k)
					if (roleUsesDirectPair<ROLE>(k)) dir[k] = fma2(kf2, dstep[k], dir0[k]);
				if (oscHere) osc.seg3(S);
				buildCoef<ROLE>(C, u, v, dir, n0Inv);
			}
			if (oscHere) osc.seg4(srD, srInv);
			// ================= the DSP =================
			float par = 0.0f, voice = 0.0f;
			if (T::hasP) {
				if (oscHere) osc.seg5(S);
				par = parallelSide(S, C, wF);
				if (oscHere) voice = osc.seg6();
				if (!T::hasC) xc.put(t, wA, par, voice);
			}
			gen++;
			if (T::hasC) {
				if (!T::hasP) xc.get(t, wA, par, voice);
				if (T::hasO) voice = oscillatorSide(S, C, srD, srInv);
				out.push(cascadeSide(S, C, wA, par, voice));
			}
			produced++;
			if (produced == myTicks) active = false;
		}
	}
	if (T::hasP && !T::hasC) xc.sync();  // hand the group over
	}

	// ---- store the stream back ----
	if constexpr (kInline) {
		if (!planned) {  // keep fm.curFrame / fm.oldFrame meaningful for purge and for the next inline plan
			if (hasNew) {
				if (counter >= 1) {
					double ratio = (double)counter / (double)newF;
					for (int i = 0; i < kNumParams; ++i) {
						double o = fm.oldFrame[i], n = fm.newFrame[i];
						fm.curFrame[i] = (n != n) ? o : o + ((n - o) * ratio);
					}
				}
			} else {
				for (int i = 0; i < kNumParams; ++i) fm.curFrame[i] = fm.oldFrame[i];
				fm.oldFrame[kVoicePitch] = S.pitch;
			}
			fm.curFrame[kVoicePitch] = S.pitch;
		}
	}
	storeDspState<ROLE>(gs, S);
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { gs.zre[r] = -half(u, r); gs.zim[r] = -half(v, r); }
#pragma unroll
	for (int i = 0; i < kNumDirect; ++i)
		if (roleUsesDirect<ROLE>(i) && (T::hasC || i != dPreFormantGain)) gs.dir[i] = fmaf(kf, half(dstep, i), half(dir0, i));
	if (T::hasC) {
		fm.counter = counter; fm.qHead = qHead; fm.oldM = oldM; fm.newM = newM; fm.newF = newF;
		fm.lastUserIndex = lastUserIndex;
		fm.hasNew = hasNew; fm.curIsNull = curIsNull; fm.oldIsNull = oldIsNull; fm.newIsNull = newIsNull;
		gs.n0Inv = n0Inv ? 1u : 0u;
		gs.holdArmed = holdArmed ? 1u : 0u;
		gs.nextEvent = nextEvent;
		gs.samplesGenerated = gen;
		gs.coarseAt = coarseAt;
		gs.callPos += produced;
		if (produced < myTicks) gs.callDrained = 1;
	}
	*lastUserIndexOut = lastUserIndex;
	*qHeadOut = qHead;
	return produced;
}
template <int ROLE, class Out, class Xchg>
KLATT_HD uint32_t renderGeneralF32(const StreamDesc &desc, int sampleRate, uint32_t myTicks, uint32_t loopTicks, Out &out,
                                   const NoiseConfig &noise, Xchg &xc, int32_t *lastUserIndexOut, uint32_t *qHeadOut) {
	return renderGeneralF32T<ROLE>(desc.state->fm, desc.state->gen.f32, desc, sampleRate, myTicks, loopTicks, out, noise, xc,
	                               lastUserIndexOut, qHeadOut);
}

// ---------------------------------------------------------------------------------------------------
// renderFadeF32T: `ticks` INTERIOR fade ticks of one pre-queued stream (reference src/frame.cpp:49-52 feeding
// src/speechWaveGenerator.cpp:113-125 on every tick), straight-line: the caller guarantees (canFadeF32T) that no
// frame-manager event falls inside and that the first tick sits on the 64-sample grid of the drift control, so the coarse
// re-basing happens before the loop and a tick is pole recurrences -> coefficients -> the DSP with no branch.  The
// arithmetic of every tick is renderGeneralF32T's, operation for operation: a stream may change between the two (and the
// hold loop) at any chunk boundary without changing an output bit.  ticks is a multiple of kGroupTicks (any number of
// kCoarseTicks cells); Philox noise only (canFadeF32T refuses every other mode); even `samplesGenerated` follows from the
// grid condition.
// ---------------------------------------------------------------------------------------------------
template <int ROLE, class Out, class Xchg, class FM, class GS>
KLATT_HD void renderFadeF32T(FM &fm, GS &gs, const StreamDesc &desc, int sampleRate, uint32_t ticks, Out &out, const NoiseConfig &noise,
                             Xchg &xc) {
	using T = RoleTraits<ROLE>;
	const double srD = (double)sampleRate, srInv = 1.0 / (double)sampleRate;
	const uint32_t rel = fm.qHead - 1u - desc.qBase;
	const FadePlanF32 *plan = desc.plans + (rel < desc.qCount ? rel : 0u);  // (idle lanes run a dummy stream with an empty queue)
	uint32_t counter = fm.counter;
	DspState S;
	loadDspState<ROLE>(S, gs);
	F2 u[kNumPairs], v[kNumPairs], wr[kNumPairs], wi[kNumPairs];
	F2 dir0[kNumDirectPairs], dstep[kNumDirectPairs];
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { half(u, r) = -gs.zre[r]; half(v, r) = -gs.zim[r]; half(wr, r) = plan->wre[r]; half(wi, r) = plan->wim[r]; }
#pragma unroll
	for (int i = 0; i < kNumDirect; ++i)
		if (roleUsesDirectPair<ROLE>(i / 2)) {
			half(dir0, i) = roleUsesDirect<ROLE>(i) ? plan->dir0[i] : 0.0f;
			half(dstep, i) = roleUsesDirect<ROLE>(i) ? plan->dirStep[i] : 0.0f;
		}
	float kf = (float)counter;
	const int64_t vibIncStep = plan->vibIncStep;
	const double depthStep = plan->depthStep;
	const bool n0Inv = gs.n0Inv != 0;
	uint64_t gen = gs.samplesGenerated;
	const uint64_t streamId = desc.streamId;
	// A chunk is a sequence of CELLS of kCoarseTicks ticks (the last one may be shorter), each starting on the drift-control
	// grid: the poles of a cell's first tick come from the coarse recurrence when the previous grid point of this fade was
	// recorded, from the per-tick one otherwise; either way they become the new record.
	uint32_t coarseAt = gs.coarseAt;
#pragma unroll 1
	for (uint32_t c0 = 0; c0 < ticks; c0 += (uint32_t)kCoarseTicks) {
		const uint32_t cellTicks = ticks - c0 < (uint32_t)kCoarseTicks ? ticks - c0 : (uint32_t)kCoarseTicks;
		{
			if (counter + 1u - coarseAt == (uint32_t)kCoarseTicks) {
#pragma unroll
				for (int r = T::R0; r < T::R1; ++r) {
					float zr = gs.zc[r], zi = gs.zc[kNumResonators + r], Wr = plan->Wre[r], Wi = plan->Wim[r];
					float tr = fmaf(-zr, Wr, Wr);
					tr = fmaf(zi, Wi, tr);
					float ti = fmaf(-zr, Wi, Wi);
					ti = fmaf(-zi, Wr, ti);
					half(u, r) = -(zr + tr);
					half(v, r) = -(zi + ti);
				}
			} else {
				stepPoles<ROLE>(u, v, wr, wi);
			}
#pragma unroll
			for (int r = T::R0; r < T::R1; ++r) { gs.zc[r] = -half(u, r); gs.zc[kNumResonators + r] = -half(v, r); }
		}
		coarseAt = counter + 1u;
		for (uint32_t t = 0; t < cellTicks; t += kGroupTicks) {
			if (T::hasC && !T::hasP) xc.sync();  // the parallel side has finished this group
#pragma unroll 1
			for (int k = 0; k < kGroupTicks; k += 2) {
				Philox4 blk;
				if (T::hasP) blk = noiseBlock(noise.seed, streamId, (gen + k) >> 1);
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					const bool oscHere = T::hasO && !T::hasC;
					OscChain osc;
					counter++;
					kf += 1.0f;
					if (T::hasO) { S.vibInc += vibIncStep; S.depth += depthStep; }
					if (t + k + h != 0) stepPoles<ROLE>(u, v, wr, wi);
					if (oscHere) { osc.seg1(S); osc.seg2(); }
					CoefF32 C;
					{
						F2 dir[kNumDirectPairs];
						const F2 kf2 = f2s(kf);
#pragma unroll
						for (int q = 0; q < kNumDirectPairs; ++q)
							if (roleUsesDirectPair<ROLE>(q)) dir[q] = fma2(kf2, dstep[q], dir0[q]);
						if (oscHere) osc.seg3(S);
						buildCoef<ROLE>(C, u, v, dir, n0Inv);
					}
					if (oscHere) osc.seg4(srD, srInv);
					uint32_t wA = 0;
					float par = 0.0f, voice = 0.0f;
					if (T::hasP) {
						wA = blk.w[2 * h];
						if (oscHere) osc.seg5(S);
						par = parallelSide(S, C, blk.w[2 * h + 1]);
						if (oscHere) voice = osc.seg6();
						if (!T::hasC) xc.put(t + k + h, wA, par, voice);
					}
					if (T::hasC) {
						if (!T::hasP) xc.get(t + k + h, wA, par, voice);
						if (T::hasO) voice = oscillatorSide(S, C, srD, srInv);
						out.push(cascadeSide(S, C, wA, par, voice));
					}
				}
			}
			gen += kGroupTicks;
			if (T::hasP && !T::hasC) xc.sync();  // hand the group over
		}
	}
	storeDspState<ROLE>(gs, S);
#pragma unroll
	for (int r = T::R0; r < T::R1; ++r) { gs.zre[r] = -half(u, r); gs.zim[r] = -half(v, r); }
#pragma unroll
	for (int i = 0; i < kNumDirect; ++i)
		if (roleUsesDirect<ROLE>(i) && (T::hasC || i != dPreFormantGain)) gs.dir[i] = fmaf(kf, half(dstep, i), half(dir0, i));
	if (T::hasC) {
		fm.counter = counter;
		gs.samplesGenerated = gen;
		gs.coarseAt = coarseAt;
		gs.callPos += ticks;
	}
}

}  // namespace klatt
