// TEST INFRASTRUCTURE ONLY.  Compiles the FP32 production arithmetic (nvspeechplayer_b200/csrc/klatt_f32_core.cuh,
// the bodies of the CUDA kernels) for the HOST so that its numerics against the reference can be studied and
// regression-tested in the CPU-only container.  Nothing here is linked into libspeechPlayer.so; the product has
// no CPU path.  Differences from the device build: glibc libm instead of libdevice (<= 1-2 ulp), IEEE division
// instead of MUFU.RCP in fastRcp().
//
// hostsim_render_f32 mirrors how the engine drives the kernels:
//   mode 0  one general-kernel pass per `chunk` ticks, plans made inline at the pop tick (per-handle API)
//   mode 1  plans precomputed for the whole queue (klatt_plan_kernel), then ROUNDS: a stream with at least holdTicks
//           pure hold ticks ahead runs renderHoldF32(holdTicks), otherwise renderGeneralF32(genTicks)
// Both render entries take Philox noise keyed (seed, streamId), or, given `replay`, the caller's draws (draw 2g / 2g+1 of
// generated sample g, 0 past replayLen) as a batch under SPEECHPLAYER_NOISE_REPLAY feeds them.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../nvspeechplayer_b200/csrc/klatt_f32_core.cuh"

using namespace klatt;

namespace {
struct ArrayOut {
	int16_t *p;
	uint32_t n;
	void push(int s) { p[n++] = (int16_t)s; }
};
}  // namespace

extern "C" int hostsim_render_f32(int sampleRate, const double *frames, const uint32_t *minDur, const uint32_t *fadeDur,
                                  const int32_t *userIndex, const uint8_t *isNull, uint32_t nFrames, uint64_t seed,
                                  uint64_t streamId, uint32_t maxSamples, int16_t *out, uint32_t chunk, int32_t *lastIndexOut,
                                  int mode, uint32_t holdTicks, uint32_t genTicks, uint32_t *holdTicksUsedOut, const int32_t *replay,
                                  uint64_t replayLen) {
	StreamState *st = (StreamState *)calloc(1, sizeof(StreamState));
	st->fm.lastUserIndex = -1;
	st->fm.curIsNull = 1;
	st->fm.oldIsNull = 1;
	StreamDesc d;
	memset(&d, 0, sizeof d);
	d.state = st; d.frames = frames; d.minDur = minDur; d.fadeDur = fadeDur; d.userIndex = userIndex; d.isNull = isNull;
	d.qCount = nFrames; d.qBase = 0; d.streamId = streamId;
	d.replay = replay; d.replayLen = replay ? replayLen : 0; d.replayBase = 0;
	std::vector<FadePlanF32> plans;
	if (mode == 1) {
		plans.resize(nFrames);
		int prevReal = -1;
		for (uint32_t j = 0; j < nFrames; ++j) {
			bool prevNull = (j == 0) || (isNull && isNull[j - 1]);
			bool curNull = isNull && isNull[j];
			double o[kNumParams], n[kNumParams];
			plannedFrames(prevReal >= 0 ? frames + (size_t)prevReal * kNumParams : nullptr, prevNull,
			              frames + (size_t)j * kNumParams, curNull, o, n);
			uint32_t F = fadeDur[j] > 1u ? fadeDur[j] : 1u;
			planFade(o, n, F, sampleRate, plans[j]);
			if (!curNull) prevReal = (int)j;
		}
		d.plans = plans.data();
	}
	NoiseConfig nc;
	nc.mode = replay ? kNoiseReplay : kNoisePhilox; nc.seed = seed;
	uint32_t total = 0, holdUsed = 0;
	int32_t lui = -1;
	uint32_t qh = 0;
	if (chunk == 0) chunk = maxSamples;
	while (total < maxSamples) {
		uint32_t left = maxSamples - total;
		if (mode == 1 && holdTicks && left >= holdTicks && canHoldF32(*st, holdTicks)) {
			ArrayOut ao{out + total, 0};
			XchgSelf xc;
			renderHoldF32<kRoleBoth>(d, sampleRate, holdTicks, ao, nc, xc);
			total += holdTicks;
			holdUsed += holdTicks;
			lui = st->fm.lastUserIndex;
			continue;
		}
		uint32_t step = (mode == 1 && genTicks) ? genTicks : chunk;
		uint32_t want = left < step ? left : step;
		ArrayOut ao{out + total, 0};
		XchgSelf xc;
		uint32_t got = renderGeneralF32<kRoleBoth>(d, sampleRate, want, want, ao, nc, xc, &lui, &qh);
		total += got;
		if (got < want) break;
	}
	if (lastIndexOut) *lastIndexOut = lui;
	if (holdTicksUsedOut) *holdTicksUsedOut = holdUsed;
	free(st);
	return (int)total;
}

// mode "cells" of the block scheduler (klatt_f32_block.cu): the stream lives in the compact StreamStateLite and is handed, cell
// by cell, to the hold loop (holdTicks pure hold ticks ahead), the fade loop (64 interior fade ticks ahead, on the 64-sample
// grid) or the general loop (everything else; it re-aligns a stream to the grid).  Must render the same bits as mode 0 / 1.
extern "C" int hostsim_render_f32_cells(int sampleRate, const double *frames, const uint32_t *minDur, const uint32_t *fadeDur,
                                        const int32_t *userIndex, const uint8_t *isNull, uint32_t nFrames, uint64_t seed,
                                        uint64_t streamId, uint32_t maxSamples, int16_t *out, uint32_t holdTicks, uint32_t fadeTicks,
                                        uint32_t *ticksByClass /* [3]: hold, fade, general */, int32_t *lastIndexOut, uint32_t fadeMax,
                                        const int32_t *replay, uint64_t replayLen) {
	StreamStateLite *st = (StreamStateLite *)calloc(1, sizeof(StreamStateLite));
	st->fm.lastUserIndex = -1;
	st->fm.curIsNull = 1;
	st->fm.oldIsNull = 1;
	StreamDesc d;
	memset(&d, 0, sizeof d);
	d.state = nullptr; d.frames = frames; d.minDur = minDur; d.fadeDur = fadeDur; d.userIndex = userIndex; d.isNull = isNull;
	d.qCount = nFrames; d.qBase = 0; d.streamId = streamId;
	d.replay = replay; d.replayLen = replay ? replayLen : 0; d.replayBase = 0;
	std::vector<FadePlanF32> plans(nFrames);
	int prevReal = -1;
	for (uint32_t j = 0; j < nFrames; ++j) {
		bool prevNull = (j == 0) || (isNull && isNull[j - 1]);
		bool curNull = isNull && isNull[j];
		double o[kNumParams], n[kNumParams];
		plannedFrames(prevReal >= 0 ? frames + (size_t)prevReal * kNumParams : nullptr, prevNull, frames + (size_t)j * kNumParams, curNull, o, n);
		uint32_t F = fadeDur[j] > 1u ? fadeDur[j] : 1u;
		planFade(o, n, F, sampleRate, plans[j]);
		if (!curNull) prevReal = (int)j;
	}
	d.plans = plans.data();
	NoiseConfig nc;
	nc.mode = replay ? kNoiseReplay : kNoisePhilox; nc.seed = seed;
	uint32_t total = 0;
	uint32_t used[3] = {0, 0, 0};
	int32_t lui = -1;
	uint32_t qh = 0;
	while (total < maxSamples) {
		const uint32_t left = maxSamples - total;
		ArrayOut ao{out + total, 0};
		XchgSelf xc;
		if (left >= holdTicks && canHoldF32T(st->fm, st->f32, holdTicks)) {
			renderHoldF32T<kRoleBoth>(st->fm, st->f32, d, sampleRate, holdTicks, ao, nc, xc);
			total += holdTicks; used[0] += holdTicks;
			lui = st->fm.lastUserIndex;
			continue;
		}
		if (left >= fadeTicks && canFadeF32T(st->fm, st->f32, fadeTicks, nc)) {
			// (the ring scheduler stretches a fade chunk to the interior fade ticks its streams have left, in whole cells)
			uint32_t ticks = fadeTicks;
			if (fadeMax > fadeTicks) {
				uint32_t can = st->fm.newF - 1u - st->fm.counter;
				if (can > left) can = left;
				if (can > fadeMax) can = fadeMax;
				can &= ~63u;
				if (can > ticks) ticks = can;
			}
			renderFadeF32T<kRoleBoth>(st->fm, st->f32, d, sampleRate, ticks, ao, nc, xc);
			total += ticks; used[1] += ticks;
			continue;
		}
		uint32_t want = (uint32_t)kCoarseTicks - (uint32_t)(st->f32.samplesGenerated & (uint64_t)(kCoarseTicks - 1));
		if (want > left) want = left;
		const uint32_t got = renderGeneralF32T<kRoleBoth>(st->fm, st->f32, d, sampleRate, want, want, ao, nc, xc, &lui, &qh);
		total += got; used[2] += got;
		if (got < want) break;
	}
	if (ticksByClass) { ticksByClass[0] = used[0]; ticksByClass[1] = used[1]; ticksByClass[2] = used[2]; }
	if (lastIndexOut) *lastIndexOut = lui;
	free(st);
	return (int)total;
}

// ---------------------------------------------------------------------------------------------------------------
// Low-latency pull path (nvspeechplayer_b200/csrc/klatt_pull_core.cuh + pull_manager.h): the host frame manager is
// the product's own; the kernel is emulated "thread by thread" -- the same per-thread passes in the same order, the
// block scans replaced by plain loops over the 512 chunks.
// ---------------------------------------------------------------------------------------------------------------
#include "../../nvspeechplayer_b200/csrc/pull_manager.h"
#include "../../nvspeechplayer_b200/csrc/klatt_long_phase.cuh"
#include <algorithm>

namespace {
struct HostPullPlayer {
	PullManager mgr;
	PullState state;
	int sampleRate;
	uint64_t seed, streamId;
	int phaseMode = 0;
	HostPullPlayer(int sr, uint64_t sd, uint64_t sid) : mgr(sr), sampleRate(sr), seed(sd), streamId(sid) { memset(&state, 0, sizeof state); }
};

// exclusive prefixes of `maps` (one per chunk) seeded with (y0, d0): what blockExclusive() computes on the device
void hostScan(const std::vector<PullAffine> &maps, int stride, int k, float y0, float d0, std::vector<PullStart> &out) {
	std::vector<PullAffineD> own(kPullThreads), pre(kPullThreads);
	for (int ch = 0; ch < kPullThreads; ++ch) own[ch] = pullToD(maps[(size_t)ch * stride + k]);
	pullBlockExclusiveModel(own.data(), pullSeed(y0, d0), pre.data());
	for (int ch = 0; ch < kPullThreads; ++ch) {
		out[(size_t)ch * stride + k].y = (float)pre[ch].zy;
		out[(size_t)ch * stride + k].d = (float)pre[ch].zd;
	}
}

template <int STAGE> void hostStage(const PullCtx &X, int res) {
	constexpr int NR = PullStageTraits<STAGE>::NR;
	std::vector<PullAffine> maps((size_t)kPullThreads * NR);
	std::vector<PullStart> st((size_t)kPullThreads * NR);
	std::vector<float> fir((size_t)kPullThreads * 2, 0.0f);
	std::vector<PullPole> poles((size_t)kPullThreads * (NR + 1));
	for (int ch = 0; ch < kPullThreads; ++ch)
		pullStage<STAGE, 1>(X, ch, res, &maps[(size_t)ch * NR], nullptr, &fir[(size_t)ch * 2], &poles[(size_t)ch * (NR + 1)]);
	for (int k = 0; k < NR; ++k) {
		const int r = STAGE == kPullParallel ? kResParallel + k : res;
		hostScan(maps, NR, k, X.state->y[r], X.state->d[r], st);
	}
	for (int ch = 0; ch < kPullThreads; ++ch)
		pullStage<STAGE, 2>(X, ch, res, nullptr, &st[(size_t)ch * NR], &fir[(size_t)ch * 2], &poles[(size_t)ch * (NR + 1)]);
}

unsigned long long g_runsLaunches = 0, g_runsSpecials = 0;

void hostPullRender(PullCtx X) {
	X.L = pullTicksPerThread(X.n);
	std::vector<float> sig((size_t)2 * X.L * kPullThreads, 0.0f);
	X.sigA = sig.data();
	X.sigB = sig.data() + (size_t)X.L * kPullThreads;
	std::vector<double> inc((size_t)X.L * kPullThreads, 0.0);
	X.inc = inc.data();
	std::vector<int64_t> runI((size_t)X.L * kPullThreads, 0);
	std::vector<uint16_t> runMeta(X.n + 8, 0);
	std::vector<PullPhaseRec> rec(kPullMaxSpecial);
	X.runI = runI.data(); X.runMeta = runMeta.data(); X.rec = rec.data();
	{
		std::vector<PullSourceSums> sums(kPullThreads);
		for (int ch = 0; ch < kPullThreads; ++ch) pullSourcePass1(X, ch, sums[ch]);
		std::vector<PullAffineD> own(kPullThreads), pre(kPullThreads);
		for (int ch = 0; ch < kPullThreads; ++ch) own[ch] = PullAffineD{sums[ch].decay, 0, 0, sums[ch].decay, sums[ch].zAsp, sums[ch].zFric};
		pullBlockExclusiveModel(own.data(), pullSeed(X.state->aspLast, X.state->fricLast), pre.data());
		std::vector<float> a0(kPullThreads), f0(kPullThreads);
		for (int ch = 0; ch < kPullThreads; ++ch) { a0[ch] = (float)pre[ch].zy; f0[ch] = (float)pre[ch].zd; }
		bool runsDone = false;
		if (X.phaseMode) {  // the run decomposition, scans as plain loops (integer arithmetic: the order does not matter)
			const double pos0 = X.state->pitchPos;
			uint64_t fixed = 0;
			const bool okStart = pullRunsStart(pos0, fixed);
			std::vector<PullRunSum> mine(kPullThreads), before(kPullThreads);
			for (int ch = 0; ch < kPullThreads; ++ch) {
				pullRunsClassify(X, ch, fixed, mine[ch]);
				fixed += sums[ch].phaseFixed;
			}
			if (!okStart) mine[0].specials += kPullMaxSpecial + 1;
			PullRunSum acc{0, 0u, 0u};
			for (int ch = 0; ch < kPullThreads; ++ch) { before[ch] = acc; acc = pullRunCombine(acc, mine[ch]); }
			if (acc.specials <= kPullMaxSpecial) {
				std::vector<double> incCopy;
				if (getenv("HOSTSIM_CHECK_RUNS")) incCopy.assign(X.inc, X.inc + (size_t)X.L * kPullThreads);
				for (int ch = 0; ch < kPullThreads; ++ch) pullRunsOffsets(X, ch, before[ch]);
				pullRunsSerial(X, acc.specials, pos0);
				for (int ch = 0; ch < kPullThreads; ++ch) pullRunsFinish(X, ch, before[ch].specials, pos0);
				if (!incCopy.empty()) {  // debug: the plain recurrence on a copy, first mismatch reported
					double pos = pos0;
					for (uint32_t t = 0; t < X.n; ++t) {
						const uint32_t at = pullIdx(X, t);
						const double x = incCopy[at];
						pos = fracRef(x + pos);
						if (memcmp(&pos, &X.inc[at], 8) != 0) {
							fprintf(stderr, "[runs mismatch] n=%u t=%u inc=%.17g want=%.17g got=%.17g meta=%04x prevmeta=%04x pos0=%.17g specials=%u\n",
							        X.n, t, x, pos, X.inc[at], X.runMeta[t], t ? X.runMeta[t - 1] : 0, pos0, acc.specials);
							break;
						}
					}
				}
				runsDone = true;
				g_runsLaunches++;
				g_runsSpecials += acc.specials;
			}
		}
		if (!runsDone) pullPhaseSerial(X);
		for (int ch = 0; ch < kPullThreads; ++ch) pullSourcePass2(X, ch, a0[ch], f0[ch]);
	}
	hostStage<kPullParallel>(X, 0);
	hostStage<kPullNasal>(X, kResNP);
	for (int r = kResCascade; r < kResParallel - 1; ++r) hostStage<kPullCascade>(X, r);
	hostStage<kPullLast>(X, kResParallel - 1);
	X.state->generated += X.n;
}
}  // namespace

extern "C" void *hostsim_pull_create(int sampleRate, uint64_t seed, uint64_t streamId) {
	return new HostPullPlayer(sampleRate, seed, streamId);
}
extern "C" void hostsim_pull_phase_mode(void *h, int mode) { ((HostPullPlayer *)h)->phaseMode = mode; }
extern "C" void hostsim_pull_runs_stats(unsigned long long *launches, unsigned long long *specials) {
	*launches = g_runsLaunches; *specials = g_runsSpecials;
}
extern "C" void hostsim_pull_destroy(void *h) { delete (HostPullPlayer *)h; }
extern "C" void hostsim_pull_queue(void *h, const double *frame, uint32_t minDur, uint32_t fadeDur, int32_t userIndex, int purge) {
	((HostPullPlayer *)h)->mgr.queueFrame(frame, minDur, fadeDur, userIndex, purge != 0);
}
extern "C" int hostsim_pull_last_index(void *h) { return ((HostPullPlayer *)h)->mgr.lastIndex(); }
// maxTicks / maxSegs: per-"launch" limits (0: the product's)
extern "C" int hostsim_pull_synthesize(void *h, uint32_t n, int16_t *out, uint32_t maxTicks, uint32_t maxSegs) {
	HostPullPlayer *p = (HostPullPlayer *)h;
	if (maxTicks == 0 || maxTicks > kPullMaxTicks) maxTicks = kPullMaxTicks;
	if (maxSegs == 0 || maxSegs > kPullMaxSegs) maxSegs = kPullMaxSegs;
	uint32_t total = 0;
	std::vector<PullSeg> segs;
	while (total < n) {
		const uint32_t want = (n - total) < maxTicks ? (n - total) : maxTicks;
		segs.clear();
		bool drained = false;
		const uint32_t got = p->mgr.advance(want, 0, maxSegs, segs, drained);
		if (got) {
			PullCtx X;
			memset(&X, 0, sizeof X);
			X.segs = segs.data(); X.nSeg = (uint32_t)segs.size(); X.n = got; X.sampleRate = p->sampleRate;
			X.state = &p->state; X.noiseMode = kNoisePhilox; X.seed = p->seed; X.streamId = p->streamId;
			X.pcm = out + total;
			X.phaseMode = p->phaseMode;
			hostPullRender(X);
		}
		total += got;
		if (drained) break;
	}
	return (int)total;
}

// The two renditions of the glottal-phase recurrence on a caller-supplied increment sequence (n <= 8192 ticks):
// out[0..n) = phase after every tick.  mode 0: the plain loop, mode 1: the run decomposition.  Returns the number of
// special ticks the serial thread visited (mode 1), n (mode 0), or -1 when mode 1 handed the pull back to the plain loop.
extern "C" int hostsim_phase(const double *incs, uint32_t n, double pos0, int mode, double *out, double *carry) {
	PullState st;
	memset(&st, 0, sizeof st);
	st.pitchPos = pos0;
	PullCtx X;
	memset(&X, 0, sizeof X);
	X.n = n; X.L = pullTicksPerThread(n); X.state = &st; X.phaseMode = mode;
	std::vector<double> inc((size_t)X.L * kPullThreads, 0.0);
	std::vector<int64_t> runI((size_t)X.L * kPullThreads, 0);
	std::vector<uint16_t> runMeta(n + 8, 0);
	std::vector<PullPhaseRec> rec(kPullMaxSpecial);
	X.inc = inc.data(); X.runI = runI.data(); X.runMeta = runMeta.data(); X.rec = rec.data();
	for (uint32_t t = 0; t < n; ++t) inc[pullIdx(X, t)] = incs[t];
	int visited = (int)n;
	bool done = false;
	if (mode == 1) {
		uint64_t fixed = 0;
		const bool okStart = pullRunsStart(pos0, fixed);
		std::vector<PullRunSum> mine(kPullThreads), before(kPullThreads);
		for (int ch = 0; ch < kPullThreads; ++ch) {
			pullRunsClassify(X, ch, fixed, mine[ch]);
			uint32_t t0, t1;
			pullChunkRange(X, ch, t0, t1);
			for (uint32_t t = t0; t < t1; ++t) fixed += (uint64_t)cyclesToFixed(incs[t]);
		}
		if (!okStart) mine[0].specials += kPullMaxSpecial + 1;
		PullRunSum acc{0, 0u, 0u};
		for (int ch = 0; ch < kPullThreads; ++ch) { before[ch] = acc; acc = pullRunCombine(acc, mine[ch]); }
		if (acc.specials <= kPullMaxSpecial) {
			for (int ch = 0; ch < kPullThreads; ++ch) pullRunsOffsets(X, ch, before[ch]);
			pullRunsSerial(X, acc.specials, pos0);
			for (int ch = 0; ch < kPullThreads; ++ch) pullRunsFinish(X, ch, before[ch].specials, pos0);
			visited = (int)acc.specials;
			done = true;
		} else {
			visited = -1;
		}
	}
	if (!done) pullPhaseSerial(X);
	for (uint32_t t = 0; t < n; ++t) out[t] = inc[pullIdx(X, t)];
	*carry = st.pitchPos;
	return visited;
}

// n-fold FP64 accumulation in closed form per binade (klatt_f32_core.cuh glideExact) -- compared with the plain loop by
// tests/test_long_phase_cpu.py
extern "C" double hostsim_glide(double p, double inc, uint64_t n) { return glideExact(p, inc, n); }

// The exact parallel phase of the long-utterance path (klatt_long_phase.cuh) on a caller-supplied increment sequence, chunk
// by chunk in the kernels' order: fixed-point prefix -> speculative runs -> scan of the offset maps -> true runs + check.
// out[t] = phase after tick t.  Returns 1 when every run ended on the next run's start (the device's condition for keeping
// the result), 0 when the check failed or a chunk could not be anchored (the device then takes the serial fallback).
namespace {
struct ArraySrc {
	const double *q;
	uint64_t t;
	void tick(double &quot, uint64_t &fi) { quot = q[t]; fi = (uint64_t)cyclesToFixed(quot); ++t; }
};
}
extern "C" int hostsim_long_phase(const double *quot, uint64_t n, uint32_t L, double *out, uint64_t *anchoredOut) {
	const uint64_t numChunks = (n + L - 1) / L;
	std::vector<uint64_t> startPhase(numChunks);
	uint64_t phi = 0;
	for (uint64_t c = 0; c < numChunks; ++c) {
		startPhase[c] = phi;
		for (uint64_t t = c * L; t < std::min<uint64_t>((c + 1) * L, n); ++t) phi += (uint64_t)cyclesToFixed(quot[t]);
	}
	std::vector<PhaseChunk> chunks(numChunks);
	bool ok = true;
	uint64_t anchored = 0;
	for (uint64_t c = 0; c < numChunks; ++c) {
		ArraySrc src{quot, c * L};
		ok = phaseSpeculateChunk(src, c, L, n, startPhase[c], 16ull * L, chunks[c]) && ok;
		anchored += chunks[c].anchor != kNoAnchor;
	}
	if (anchoredOut) *anchoredOut = anchored;
	std::vector<double> startP(numChunks, 0.0);
	PhaseMap pre = phaseMapIdentity();
	for (uint64_t c = 0; c < numChunks; ++c) {
		if (chunks[c].anchor != kNoAnchor) startP[c] = phaseFromOffset(chunks[c].s0, phaseMapApply(pre, 0));
		pre = phaseMapCompose(chunks[c].map, pre);
	}
	for (uint64_t c = 0; c < numChunks; ++c) {
		if (chunks[c].anchor == kNoAnchor) continue;
		double pos = startP[c];
		for (uint64_t t = chunks[c].anchor; t < chunks[c].next; ++t) { pos = phaseStep(pos, quot[t]); out[t] = pos; }
		if (chunks[c].next < n) {
			const uint64_t nx = chunks[c].next / L;
			if (nx >= numChunks || chunks[nx].anchor != chunks[c].next || startP[nx] != pos) ok = false;
		}
	}
	return ok ? 1 : 0;
}


// ---- the helper threads of the batched pull (nvspeechplayer_b200/csrc/host_pool.h): every index exactly once, any n / grain ----
#include "../../nvspeechplayer_b200/csrc/host_pool.h"
extern "C" int hostsim_host_pool(unsigned reps, unsigned maxN, unsigned *helpersOut) {
	klatt::HostPool &pool = klatt::HostPool::get();
	if (helpersOut) *helpersOut = (unsigned)pool.helpers();
	for (unsigned rep = 0; rep < reps; ++rep) {
		const size_t n = 1 + rep % maxN, grain = 1 + (rep * 7u) % 40u;
		std::vector<int> hits(n, 0);
		std::atomic<long long> sum{0};
		pool.parallelFor(n, grain, [&](size_t i) { hits[i] += 1; sum.fetch_add((long long)i); });
		for (size_t i = 0; i < n; ++i)
			if (hits[i] != 1) return -(int)rep - 1;
		if (sum.load() != (long long)n * (long long)(n - 1) / 2) return -(int)rep - 1;
	}
	return 0;
}


// ---- voicePitch of the pull path on ticks c0 .. c0+n-1 of one request, as a chunk's PullOsc walks them (seek, then tick by
// tick): must be the reference's fade formula followed by its repeated addition (src/frame.cpp:49-52, :77), bit for bit ----
extern "C" void hostsim_pull_pitch_walk(double pitchOld, double pitchNew, double pitchInc, uint32_t F, uint32_t c0, uint32_t n, double *out) {
	PullSeg seg;
	memset(&seg, 0, sizeof seg);
	seg.F = F; seg.pitchOld = pitchOld; seg.pitchNew = pitchNew; seg.pitchInc = pitchInc; seg.pitchStale = pitchOld;
	PullOsc w;
	memset(&w, 0, sizeof w);
	w.glideSeg = 0xffffffffu;
	w.cur.s = 0;
	for (uint32_t i = 0; i < n; ++i) {
		w.cur.c = c0 + i;
		out[i] = w.pitch(seg);
	}
}

// the vibrato sine of every FP32 path (klatt_f32_core.cuh sinTurns) and the depth that multiplies it
extern "C" void hostsim_sin_turns(const float *t, uint32_t n, float *out) {
	for (uint32_t i = 0; i < n; ++i) out[i] = sinTurns(t[i]);
}
extern "C" double hostsim_vibrato_depth(double vibratoPitchOffset) { return vibratoDepth(vibratoPitchOffset); }
