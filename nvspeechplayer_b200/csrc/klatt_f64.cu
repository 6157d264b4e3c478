// klatt_batch_f64: the bit-exact parity kernel.  One stream per thread, the reference's arithmetic in the
// reference's evaluation order, in double.  THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false so that no
// multiply-add is contracted (the reference build is x86-64 SSE2: no FMA), which leaves libdevice's
// exp/cos/sin (<= 1-2 ulp from glibc's) as the only arithmetic difference from the compiled reference.
//
// What is restated (paths relative to the reference checkout):
//   frame manager tick            src/frame.cpp:41-80      -> frameTick()
//   purge prologue                src/frame.cpp:103-112    -> applyPurge()
//   NaN-keeping lerp              src/utils.h:20-23        -> fadeValue()
//   coloured noise                src/speechWaveGenerator.cpp:39-42
//   phase accumulators            src/speechWaveGenerator.cpp:54-58
//   voice source                  src/speechWaveGenerator.cpp:72-86
//   resonator coefficients / step src/speechWaveGenerator.cpp:112-135
//   cascade / parallel banks      src/speechWaveGenerator.cpp:147-158 / :170-180
//   mix, gain, clamp, int16       src/speechWaveGenerator.cpp:204-208
//
// Layout: the three 47-double frames of the frame manager (old/new/cur) and the 42 resonator coefficients
// live in shared memory, [slot][thread] so every access is bank-conflict free; resonator histories, phases
// and noise state live in registers; the frame queue is read from HBM only on pop ticks.
#include <cuda_runtime.h>
#include <math_constants.h>
#include "klatt_common.h"
#include "philox.cuh"
#include "out_writer.cuh"
#include "launch.h"

namespace klatt {

constexpr int kF64Block = 64;
constexpr int kF64SmemDoubles = (3 * kNumParams + 3 * kNumResonators);  // per thread

namespace {

struct SmemF64 {
	double *base;  // points at this thread's column
	__device__ __forceinline__ double &oldF(int i) { return base[(i)*kF64Block]; }
	__device__ __forceinline__ double &newF(int i) { return base[(kNumParams + i) * kF64Block]; }
	__device__ __forceinline__ double &cur(int i) { return base[(2 * kNumParams + i) * kF64Block]; }
	__device__ __forceinline__ double &ca(int r) { return base[(3 * kNumParams + r) * kF64Block]; }
	__device__ __forceinline__ double &cb(int r) { return base[(3 * kNumParams + kNumResonators + r) * kF64Block]; }
	__device__ __forceinline__ double &cc(int r) { return base[(3 * kNumParams + 2 * kNumResonators + r) * kF64Block]; }
};

// src/utils.h:20-23
__device__ __forceinline__ double fadeValue(double oldVal, double newVal, double ratio) {
	if (isnan(newVal)) return oldVal;
	return oldVal + ((newVal - oldVal) * ratio);
}

// src/speechWaveGenerator.cpp:112-127 (the change-detection cache is replaced by the caller's dirty flag:
// the coefficients are a pure function of frequency, bandwidth, sampleRate and anti)
__device__ __forceinline__ void setCoefficients(SmemF64 &sm, int r, double srD, double frequency, double bandwidth, bool anti) {
	const double PI = 3.14159265358979323846;
	const double PITWO = PI * 2;
	double rad = exp(-PI / srD * bandwidth);
	double c = -(rad * rad);
	double b = rad * cos(PITWO / srD * -frequency) * 2.0;
	double a = 1.0 - b - c;
	if (anti && frequency != 0) {
		a = 1.0 / a;
		c *= -a;
		b *= -a;
	}
	sm.ca(r) = a; sm.cb(r) = b; sm.cc(r) = c;
}

__device__ __noinline__ void recomputeAllCoefficients(SmemF64 sm, double srD) {
	for (int r = 0; r < kNumResonators; ++r)
		setCoefficients(sm, r, srD, sm.cur(resFreqParam(r)), sm.cur(resBwParam(r)), r == kResN0);
}

}  // namespace

__global__ void __launch_bounds__(kF64Block)
klatt_batch_f64_kernel(const StreamDesc *__restrict__ descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                       int16_t *__restrict__ out, size_t rowStride, uint32_t *__restrict__ samplesWritten,
                       StreamResult *__restrict__ results, NoiseConfig noise) {
	extern __shared__ double smemRaw[];
	const uint32_t s = blockIdx.x * kF64Block + threadIdx.x;
	if (s >= numStreams) return;
	SmemF64 sm;
	sm.base = smemRaw + threadIdx.x;

	const StreamDesc desc = descs[s];
	StreamState *st = desc.state;
	FrameMgrState &fm = st->fm;
	GenStateF64 &gs = st->gen.f64;

	// ---- load the stream ----------------------------------------------------------------------
	for (int i = 0; i < kNumParams; ++i) {
		sm.oldF(i) = fm.oldFrame[i];
		sm.newF(i) = fm.newFrame[i];
		sm.cur(i) = fm.curFrame[i];
	}
	uint32_t counter = fm.counter, qHead = fm.qHead;
	uint32_t oldM = fm.oldM, newM = fm.newM, newF = fm.newF;
	int32_t lastUserIndex = fm.lastUserIndex;
	bool hasNew = fm.hasNew, curIsNull = fm.curIsNull, oldIsNull = fm.oldIsNull, newIsNull = fm.newIsNull;
	double oldInc = fm.oldInc, newInc = fm.newInc;

	// purge prologue, src/frame.cpp:103-112 (the dropped requests were already removed on the host)
	if (fm.purgePending) {
		fm.purgePending = 0;
		counter = oldM;
		if (hasNew) {
			oldIsNull = newIsNull;
			for (int i = 0; i < kNumParams; ++i) sm.oldF(i) = sm.cur(i);
			hasNew = false;
		}
	}

	double pitchPos = gs.pitchPos, vibratoPos = gs.vibratoPos, aspLast = gs.aspLast, fricLast = gs.fricLast;
	double p1[kNumResonators], p2[kNumResonators];
#pragma unroll
	for (int r = 0; r < kNumResonators; ++r) { p1[r] = gs.p1[r]; p2[r] = gs.p2[r]; }
	uint64_t gen = gs.samplesGenerated;

	const double srD = (double)sampleRate;  // every "/sampleRate" of the reference divides by the converted int
	bool coefDirty = true;                  // Resonator::setOnce==false / (f,bw) changed
	Philox4 blk;
	uint64_t blkIndex = ~0ull;

	OutWriter ow;
	{
		int16_t *row = out + (size_t)s * rowStride;
		ow.init(row, ((reinterpret_cast<uintptr_t>(row) & 15u) == 0));
	}

	uint32_t produced = 0;
	for (; produced < sampleCount; ++produced) {
		// ================= frame manager tick, src/frame.cpp:41-80 =================
		counter++;
		if (hasNew) {
			if (counter > newF) {  // :44-47
				for (int i = 0; i < kNumParams; ++i) sm.oldF(i) = sm.newF(i);
				oldM = newM; oldInc = newInc; oldIsNull = newIsNull;
				hasNew = false;
			} else {  // :49-52
				double ratio = (double)counter / (double)newF;
				for (int i = 0; i < kNumParams; ++i) sm.cur(i) = fadeValue(sm.oldF(i), sm.newF(i), ratio);
				coefDirty = true;
			}
		} else if (counter > oldM) {  // :54
			uint32_t rel = qHead - desc.qBase;
			if (rel < desc.qCount) {  // :55-72
				curIsNull = false;
				newM = desc.minDur[rel];
				uint32_t fd = desc.fadeDur[rel];
				newF = fd > 1u ? fd : 1u;  // src/speechPlayer.cpp:36
				newIsNull = desc.isNull ? (desc.isNull[rel] != 0) : false;
				int32_t ux = desc.userIndex ? desc.userIndex[rel] : -1;
				qHead++;
				hasNew = true;
				if (newIsNull) {  // :59-63
					for (int i = 0; i < kNumParams; ++i) sm.newF(i) = sm.oldF(i);
					sm.newF(kPreFormantGain) = 0;
					sm.newF(kVoicePitch) = sm.cur(kVoicePitch);
					newInc = 0;
				} else {
					const double *fr = desc.frames + (size_t)rel * kNumParams;
					for (int i = 0; i < kNumParams; ++i) sm.newF(i) = fr[i];
					newInc = (fr[kEndVoicePitch] - fr[kVoicePitch]) / (double)newM;  // src/frame.cpp:98
					if (oldIsNull) {  // :64-67
						for (int i = 0; i < kNumParams; ++i) sm.oldF(i) = sm.newF(i);
						sm.oldF(kPreFormantGain) = 0;
					}
				}
				if (ux != -1) lastUserIndex = ux;  // :69
				counter = 0;                       // :70
				sm.newF(kVoicePitch) += (newInc * (double)newF);  // :71
			} else {
				curIsNull = true;  // :73-75
			}
		} else {  // :76-79
			double vp = sm.cur(kVoicePitch) + oldInc;
			sm.cur(kVoicePitch) = vp;
			sm.oldF(kVoicePitch) = vp;
		}
		if (curIsNull) break;  // src/speechWaveGenerator.cpp:210

		if (coefDirty) {
			recomputeAllCoefficients(sm, srD);
			coefDirty = false;
		}

		// ================= noise draws =================
		int drawA, drawF;
		if (noise.mode == kNoisePhilox) {
			uint64_t b = gen >> 1;
			if (b != blkIndex) { blk = noiseBlock(noise.seed, desc.streamId, b); blkIndex = b; }
			bool odd = (gen & 1ull) != 0;
			drawA = (int)((odd ? blk.w[2] : blk.w[0]) >> 1);
			drawF = (int)((odd ? blk.w[3] : blk.w[1]) >> 1);
		} else {
			uint64_t d0 = 2 * gen - desc.replayBase;
			drawA = (d0 < desc.replayLen) ? desc.replay[d0] : 0;
			drawF = (d0 + 1 < desc.replayLen) ? desc.replay[d0 + 1] : 0;
		}
		gen++;

		// ================= voice source, src/speechWaveGenerator.cpp:72-86 =================
		const double PITWO = 3.14159265358979323846 * 2;
		double vibCycle = fmod((sm.cur(kVibratoSpeed) / srD) + vibratoPos, 1.0);  // :55
		vibratoPos = vibCycle;
		double vibrato = (sin(vibCycle * PITWO) * 0.06 * sm.cur(kVibratoPitchOffset)) + 1;  // :73
		double voice = fmod(((sm.cur(kVoicePitch) * vibrato) / srD) + pitchPos, 1.0);      // :74,:55
		pitchPos = voice;
		aspLast = ((double)drawA / 2147483647.0) + 0.75 * aspLast;  // :40
		double aspiration = aspLast * 0.2;                          // :75
		double turbulence = aspiration * sm.cur(kVoiceTurbulenceAmplitude);
		bool glottisOpen = voice >= sm.cur(kGlottalOpenQuotient);
		if (!glottisOpen) turbulence *= 0.01;
		voice = (voice * 2) - 1;
		voice += turbulence;
		voice *= sm.cur(kVoiceAmplitude);
		aspiration *= sm.cur(kAspirationAmplitude);
		double source = aspiration + voice;

		const double preGain = sm.cur(kPreFormantGain);
		// ================= cascade, src/speechWaveGenerator.cpp:147-158 =================
		double input = (source * preGain) / 2.0;
		double n0Out;
		{  // rN0, anti-resonator: history holds INPUTS (:133)
			n0Out = sm.ca(kResN0) * input + sm.cb(kResN0) * p1[kResN0] + sm.cc(kResN0) * p2[kResN0];
			p2[kResN0] = p1[kResN0];
			p1[kResN0] = input;
		}
		double npOut = sm.ca(kResNP) * n0Out + sm.cb(kResNP) * p1[kResNP] + sm.cc(kResNP) * p2[kResNP];
		p2[kResNP] = p1[kResNP];
		p1[kResNP] = npOut;
		double cascade = fadeValue(input, npOut, sm.cur(kCaNP));  // :150
#pragma unroll
		for (int r = kResCascade; r < kResParallel; ++r) {  // r6 .. r1
			double o = sm.ca(r) * cascade + sm.cb(r) * p1[r] + sm.cc(r) * p2[r];
			p2[r] = p1[r];
			p1[r] = o;
			cascade = o;
		}
		// ================= frication + parallel bank, :205-206, :170-180 =================
		fricLast = ((double)drawF / 2147483647.0) + 0.75 * fricLast;
		double fric = fricLast * 0.3 * sm.cur(kFricationAmplitude);
		double pin = (fric * preGain) / 2.0;
		double parallel = 0;
#pragma unroll
		for (int k = 0; k < 6; ++k) {
			const int r = kResParallel + k;
			double o = sm.ca(r) * pin + sm.cb(r) * p1[r] + sm.cc(r) * p2[r];
			p2[r] = p1[r];
			p1[r] = o;
			parallel += (o - pin) * sm.cur(kPa1 + k);
		}
		parallel = fadeValue(parallel, pin, sm.cur(kParallelBypass));
		// ================= mix, clamp (Win32 macro semantics: NaN -> +32000), truncate, :207-208 =================
		double v = (cascade + parallel) * sm.cur(kOutputGain);
		double scaled = v * 4000;
		double lo = (scaled < 32000.0) ? scaled : 32000.0;
		double cl = (lo > -32000.0) ? lo : -32000.0;
		ow.push(__double2int_rz(cl));
	}
	ow.flush();
	// a drained stream leaves the rest of its row silent (the reference leaves it untouched; callers only look
	// at the returned prefix)
	for (uint32_t i = produced; i < sampleCount; ++i) ow.row[i] = 0;

	// ---- store the stream back -------------------------------------------------------------------
	for (int i = 0; i < kNumParams; ++i) {
		fm.oldFrame[i] = sm.oldF(i);
		fm.newFrame[i] = sm.newF(i);
		fm.curFrame[i] = sm.cur(i);
	}
	fm.counter = counter; fm.qHead = qHead; fm.oldM = oldM; fm.newM = newM; fm.newF = newF;
	fm.lastUserIndex = lastUserIndex;
	fm.hasNew = hasNew; fm.curIsNull = curIsNull; fm.oldIsNull = oldIsNull; fm.newIsNull = newIsNull;
	fm.oldInc = oldInc; fm.newInc = newInc;
	gs.pitchPos = pitchPos; gs.vibratoPos = vibratoPos; gs.aspLast = aspLast; gs.fricLast = fricLast;
#pragma unroll
	for (int r = 0; r < kNumResonators; ++r) { gs.p1[r] = p1[r]; gs.p2[r] = p2[r]; }
	gs.samplesGenerated = gen;
	if (samplesWritten) samplesWritten[s] = produced;
	if (results) {
		StreamResult res;
		res.written = produced; res.lastUserIndex = lastUserIndex; res.qHead = qHead; res.pad = 0;
		results[s] = res;
	}
}

cudaError_t launchKlattF64(const StreamDesc *descs, uint32_t numStreams, int sampleRate, uint32_t sampleCount,
                           int16_t *out, size_t rowStride, uint32_t *samplesWritten, StreamResult *results,
                           NoiseConfig noise, cudaStream_t stream) {
	const size_t smem = (size_t)kF64SmemDoubles * kF64Block * sizeof(double);
	// per-context attribute; cheap enough to set on every launch (one process may drive several devices)
	cudaError_t e = cudaFuncSetAttribute(klatt_batch_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (e != cudaSuccess) return e;
	if (numStreams == 0 || sampleCount == 0) return cudaSuccess;
	dim3 grid((numStreams + kF64Block - 1) / kF64Block);
	klatt_batch_f64_kernel<<<grid, kF64Block, smem, stream>>>(descs, numStreams, sampleRate, sampleCount, out, rowStride,
	                                                          samplesWritten, results, noise);
	return cudaGetLastError();
}

}  // namespace klatt
