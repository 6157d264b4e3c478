// klatt_tick_core: the FP32 tick of the two time-parallel renderers, stated once.  Kernel (b) (klatt_long.cu) and the
// low-latency pull path (klatt_pull_core.cuh) both render a tick as a closed form of (request plan, sampleCounter c); this
// header holds what a tick computes from that: the request laws, the pole walk, the source and one tick of a resonator
// stage.  Each caller keeps its own storage (kernel (b) caches the plan fields of the request in force in registers, the
// pull path reads its PullSeg) and passes plain values, so the next change to the reference law is made here only.
// KLATT_HD: tests/hostsim runs the same arithmetic on the host.
#pragma once
#include "klatt_common.h"
#include "klatt_f32_core.cuh"

namespace klatt {

// ---------------------------------------------------------------------------------------------------------------
// The request laws at counter c (reference src/frame.cpp:41-80): c == 0 is the pop tick, rendered with the values in
// force before it (`stale`: the predecessor's final values, or what the host frame manager left after a purge); the fade
// 0 < c < F (src/frame.cpp:49-52); the landed values from c == F on.
// ---------------------------------------------------------------------------------------------------------------
KLATT_HD float dirLaw(uint32_t c, uint32_t F, float stale, float d0, float ds, float dF) {
	return c == 0 ? stale : (c < F ? fmaf((float)c, ds, d0) : dF);
}

// the vibrato depth 0.06 * vibratoPitchOffset, in double (klatt_common.h FadePlanF32)
KLATT_HD double depthLaw(uint32_t c, uint32_t F, double stale, double d0, double ds, double dF) {
	return c == 0 ? stale : (c < F ? fma((double)(float)c, ds, d0) : dF);
}

// vibrato: the per-tick phase increment on tick c, and the sum of the increments of ticks [0, c)
KLATT_HD int64_t vibIncLaw(uint32_t c, uint32_t F, int64_t stale, int64_t v0, int64_t vs, int64_t vF) {
	return c == 0 ? stale : (c < F ? v0 + (int64_t)c * vs : vF);
}
KLATT_HD uint64_t vibBeforeLaw(uint32_t c, uint32_t F, int64_t stale, int64_t v0, int64_t vs, int64_t vF) {
	if (c == 0) return 0;
	uint64_t sum = (uint64_t)stale;
	const uint64_t kmax = (c - 1 < F - 1) ? c - 1 : F - 1;  // fade ticks 1 .. kmax are behind us
	sum += kmax * (uint64_t)v0 + (uint64_t)vs * (kmax * (kmax + 1) / 2);
	if (c > F) sum += (uint64_t)(c - F) * (uint64_t)vF;
	return sum;
}

// the anti-resonator is inverted (cfN0 != 0, reference src/speechWaveGenerator.cpp:120)
KLATT_HD bool n0InvLaw(uint32_t c, uint32_t F, uint32_t stale, uint32_t fade, uint32_t fin) {
	return (c == 0 ? stale : (c < F ? fade : fin)) != 0;
}

// cur.voicePitch: stale on the pop tick, the fade old+(new-old)*ratio (src/utils.h:20-23), the landing value on the landing
// and the swap tick, then the hold glide.  The reference adds voicePitchInc once per tick (src/frame.cpp:77), and a sum of
// roundings is not a product: glideExact (klatt_f32_core.cuh) reproduces the c - F - 1 additions bit for bit.
KLATT_HD double pitchLanding(double o, double n) { return (n != n) ? o : o + ((n - o) * 1.0); }
KLATT_HD double pitchLaw(uint32_t c, uint32_t F, double stale, double o, double n, double inc) {
	if (c == 0) return stale;
	if (c < F) return (n != n) ? o : o + ((n - o) * ((double)c / (double)F));
	const double landing = pitchLanding(o, n);
	if (c <= F + 1) return landing;
	return glideExact(landing, inc, (uint64_t)(c - F - 1));
}

// The pitch law walked tick by tick: `walk` holds the value the walk rendered last.  A hold tick that directly follows it
// adds voicePitchInc as the reference does (src/frame.cpp:77); every other tick -- the first one after a seek included --
// takes the closed form, which glideExact makes agree with the additions bit for bit.
KLATT_HD double pitchTick(double &walk, bool follows, uint32_t c, uint32_t F, double stale, double o, double n, double inc) {
	walk = (c > F + 1 && follows) ? walk + inc : pitchLaw(c, F, stale, o, n, inc);
	return walk;
}

// ---------------------------------------------------------------------------------------------------------------
// zeta = 1 - pole of one section along a request: planFade's start value and per-tick ratio w during the fade, re-based on
// the closed form of the pole every kCoarseTicks ticks (drift control), constant after the landing.  The closed form is
// the caller's `exact(k, zr, zi)` (zeta on fade tick k): the two paths evaluate it differently and each keeps its bits.
// ---------------------------------------------------------------------------------------------------------------
struct PoleWalk {
	float zr, zi, wr, wi;
	// state as it is AFTER the tick before c; (staleRe, staleIm): zeta in force on the pop tick
	template <class Exact>
	KLATT_HD void seek(const FadePlanF32 &p, uint32_t c, uint32_t F, int r, float staleRe, float staleIm, Exact exact) {
		wr = wi = 0.0f;
		if (c <= 1) {
			zr = staleRe; zi = staleIm;
		} else if (c <= F) {  // ticks 1 .. c-1 of the fade are behind us
			exact(c - 1, zr, zi);
			wr = p.wre[r]; wi = p.wim[r];
		} else {
			zr = p.zFre[r]; zi = p.zFim[r];
		}
	}
	// the update of tick c: afterwards (zr, zi) is what the tick renders with.  The pop tick (c == 0) leaves the state alone.
	template <class Exact>
	KLATT_HD void tick(const FadePlanF32 &p, uint32_t c, uint32_t F, int r, Exact exact) {
		if (c == 0 || c > F) return;  // after the landing: constant
		if (c == F) {
			zr = p.zFre[r]; zi = p.zFim[r]; wr = wi = 0.0f;
			return;
		}
		if (c == 1) {
			zr = p.z0re[r]; zi = p.z0im[r]; wr = p.wre[r]; wi = p.wim[r];
		}
		if ((c & (uint32_t)(kCoarseTicks - 1)) == 0) {
			exact(c, zr, zi);  // drift control: back onto the closed form
			return;
		}
		step();
	}
	// a plain interior fade tick (1 < c < F, not a multiple of kCoarseTicks): zeta <- zeta + (1 - zeta) w
	KLATT_HD void step() {
		float tr = fmaf(-zr, wr, wr);
		tr = fmaf(zi, wi, tr);
		float ti = fmaf(-zr, wi, wi);
		ti = fmaf(-zi, wr, ti);
		zr += tr;
		zi += ti;
	}
	KLATT_HD void coef(float &a, float &rho) const {
		a = fmaf(zr, zr, zi * zi);
		rho = fmaf(2.0f, zr, -a);
	}
};

// ---------------------------------------------------------------------------------------------------------------
// source (reference src/speechWaveGenerator.cpp:32-88, :204-206)
// ---------------------------------------------------------------------------------------------------------------
// one step of a noise colouring filter (:40) on the draw in word w (the 23 bits used are w >> 9, an exact integer)
KLATT_HD float colourNoise(float last, uint32_t w) { return fmaf(0.75f, last, bitsToFloat(0x4B000000u | (w >> 9)) - 8388608.0f); }

// What a tick adds to the glottal phase, in cycles: the vibrato phase steps by vibInc, then (pitch * (1 + depth * sine)) /
// sampleRate with the vibrato sine in FP32 and the rest in FP64, the division correctly rounded (:72-74, :55).
KLATT_HD double glottalInc(uint64_t &vibPos, int64_t vibInc, double pitch, double depth, double srD, double srInv) {
	vibPos += (uint64_t)vibInc;
	const float vph = (float)(int32_t)(uint32_t)(vibPos >> 32) * 2.3283064365386963e-10f;
	return divideBySampleRate(pitch * fma((double)sinTurns(vph), depth, 1.0), srD, srInv);
}

// The two excitation signals of a tick from its sawtooth value, its noise words and its direct parameters: cascade input ci
// (:204, :148) and parallel input pin (:206, :171).  aspLast / fricLast are the colouring filters' memories.
KLATT_HD void excitation(float voice, uint32_t wA, uint32_t wF, float vta, float goq, float va, float aa, float fa, float pfg,
                         float &aspLast, float &fricLast, float &ci, float &pin) {
	aspLast = colourNoise(aspLast, wA);
	const float asp = aspLast * (0.2f * kDrawScale);
	float turb = asp * vta;
	if (voice < goq) turb *= 0.01f;
	const float v = (fmaf(voice, 2.0f, -1.0f) + turb) * va;
	const float src = fmaf(asp, aa, v);
	const float halfGain = pfg * 0.5f;
	ci = src * halfGain;
	fricLast = colourNoise(fricLast, wF);
	pin = fricLast * (((0.3f * kDrawScale) * fa) * halfGain);
}

// ---------------------------------------------------------------------------------------------------------------
// resonator stages (reference src/speechWaveGenerator.cpp:112-182, :207-208), in the order they run:
//   kStageParallel: frication input -> sections 8..13 -> parallel output (:170-180)
//   kStageNasal   : cascade input -> rN0 (FIR) -> rNP (section 1) -> caNP mix (:148-150)
//   kStageCascade : one section r6 .. r2 (:151-155)
//   kStageLast    : like kStageCascade for r1, then (x + par) * outputGain * 4000, clamp, truncate (:207-208)
// ---------------------------------------------------------------------------------------------------------------
enum Stage : int { kStageParallel = 0, kStageNasal = 1, kStageCascade = 2, kStageLast = 3 };
template <int STAGE> struct StageTraits {
	static constexpr int NR = STAGE == kStageParallel ? 6 : 1;  // scanned sections
};

// the coefficients of one tick of a stage
template <int STAGE> struct StageCoefs {
	static constexpr int NR = StageTraits<STAGE>::NR;
	float a[NR], rho[NR], mix[NR];  // sections; mix: pa1..6 (parallel stage)
	float extra;                    // parallelBypass, caNP or outputGain
	float a0, rho0, rcp0;           // rN0 (nasal stage): a, rho and 1/a when inverted
	bool inv;
};

// The state of one stage along a chunk: delta-form section memories (y, d), the FIR inputs of rN0, and in pass 1 the affine
// map P of the chunk (each section is linear in its state for a given input).  PASS 1 runs from zero state and accumulates
// P; PASS 2 runs from the scanned start state and produces the stage's output.
template <int STAGE, int PASS> struct StageTick {
	static constexpr int NR = StageTraits<STAGE>::NR;
	float y[NR], d[NR];
	float p00[NR], p01[NR], p10[NR], p11[NR];
	float in1, in2;  // rN0: the last two inputs
	KLATT_HD void start() {
		for (int k = 0; k < NR; ++k) { y[k] = 0.0f; d[k] = 0.0f; p00[k] = 1.0f; p01[k] = 0.0f; p10[k] = 0.0f; p11[k] = 1.0f; }
		in1 = 0.0f; in2 = 0.0f;
	}
	// one tick on input x (par: the parallel output, read by the last stage); returns the stage's output (pass 2; for the last
	// stage the int16 value as a float)
	KLATT_HD float operator()(float x, float par, const StageCoefs<STAGE> &k) {
		const float xin = x;
		if (STAGE == kStageNasal) {  // rN0 on inputs: src/speechWaveGenerator.cpp:129-135 with anti == true
			const float dprev = in1 - in2;
			const float dx = x - in1;
			const float dx1 = fmaf(-k.rho0, dprev, dprev);
			x = k.inv ? fmaf(dx - dx1, k.rcp0, in1) : fmaf(k.a0, dx, dx1 + in1);
			in2 = in1;
			in1 = xin;
		}
		float acc = 0.0f;
		for (int s = 0; s < NR; ++s) {
			const float a = k.a[s], rho = k.rho[s];
			float w = fmaf(-rho, d[s], d[s]);
			w = fmaf(-a, y[s], w);
			const float dn = fmaf(a, x, w);
			d[s] = dn;
			y[s] += dn;
			if (PASS == 1) {  // P <- A P with A = [[1-a, 1-rho], [-a, 1-rho]] acting on (y, d)
				const float g = 1.0f - rho;
				const float n10 = fmaf(-a, p00[s], g * p10[s]), n11 = fmaf(-a, p01[s], g * p11[s]);
				p00[s] += n10; p01[s] += n11;
				p10[s] = n10; p11[s] = n11;
			}
			if (STAGE == kStageParallel) acc = fmaf(y[s] - x, k.mix[s], acc);
		}
		if (PASS == 1) return 0.0f;
		if (STAGE == kStageParallel) return fmaf(x - acc, k.extra, acc);
		if (STAGE == kStageNasal) return fmaf(y[0] - xin, k.extra, xin);
		if (STAGE == kStageCascade) return y[0];
		float s = (y[0] + par) * (k.extra * 4000.0f);
		s = fminf(s, 32000.0f);
		s = fmaxf(s, -32000.0f);
		return (float)(int)s;  // the int16 value, exactly representable
	}
	KLATT_HD Affine map(int s) const { return Affine{p00[s], p01[s], p10[s], p11[s], y[s], d[s]}; }
};

}  // namespace klatt
