// Host side of the low-latency pull path (klatt_pull_core.cuh): the reference's frame manager
// (src/frame.cpp:30-127) run at REQUEST granularity.  The reference enters updateCurrentFrame() once per sample; all it
// does between two events (pop, swap, drain) is a linear interpolation or an arithmetic progression of the tick counter,
// so the manager here jumps from event to event in FP64 and describes the ticks in between in closed form: a pull of n
// samples becomes a handful of PullSeg records, and the device renders the ticks.
//
//   pop    src/frame.cpp:54-72   NULL-frame rewrites, userIndex, voicePitch += inc * F
//   fade   src/frame.cpp:48-52   ticks 1..F of a request (src/utils.h:20-23: a NaN target keeps the old value)
//   swap   src/frame.cpp:44-47   tick F+1: old = new, curFrame untouched
//   hold   src/frame.cpp:76-78   ticks F+2..M: curFrame.voicePitch += inc, written back into the old request
//   drain  src/frame.cpp:73-75   nothing queued when the hold runs out: no sample, the caller gets a short count
//   purge  src/frame.cpp:103-112 queue dropped, a fade in progress frozen into the old request, next tick pops
//
// Header-only and host-only; included by api_player.cu and by the host build of the kernel arithmetic under tests/hostsim.
#pragma once
#include <stdint.h>
#include <string.h>
#include <deque>
#include <vector>
#include "klatt_pull_core.cuh"

namespace klatt {

struct PullRequest {  // reference frameRequest_t, src/frame.cpp:21-28
	uint32_t M = 0, F = 1;
	bool isNull = true;
	double frame[kNumParams] = {};
	double inc = 0.0;
	int32_t userIndex = -1;
};

class PullManager {
public:
	explicit PullManager(int sampleRate_) : sampleRate(sampleRate_) {
		memset(cur, 0, sizeof cur);
		memset(&info, 0, sizeof info);
		info.F = 1;
	}

	// reference FrameManagerImpl::queueFrame, src/frame.cpp:90-115 (fadeDuration already >= 1: src/speechPlayer.cpp:36)
	void queueFrame(const double *frame, uint32_t minNumSamples, uint32_t numFadeSamples, int32_t userIndex, bool purgeQueue) {
		PullRequest r;
		r.M = minNumSamples;
		r.F = numFadeSamples > 1u ? numFadeSamples : 1u;
		if (frame) {
			r.isNull = false;
			memcpy(r.frame, frame, sizeof r.frame);
			r.inc = (frame[kEndVoicePitch] - frame[kVoicePitch]) / (double)r.M;
		} else {
			r.isNull = true;
		}
		r.userIndex = userIndex;
		if (purgeQueue) {
			queue.clear();
			syncToCounter();
			counter = old.M;
			if (hasNew) {
				old.isNull = nw.isNull;
				memcpy(old.frame, cur, sizeof cur);
				hasNew = false;
			}
			inRequest = false;  // whatever happens next is a pop (or a drain): no request's closed form applies any more
		}
		queue.push_back(r);
	}

	int32_t lastIndex() const { return lastUserIndex; }
	size_t pending() const { return queue.size(); }

	// Describe the next samples of the stream, at most n ticks and at most maxSegs segments, appended to `segs` with
	// tickStart counted from tickBase.  Returns the number of ticks described; `drained` tells a short count caused by an
	// empty queue (reference: synthesize returns less than it was asked for) from one caused by the segment limit.
	uint32_t advance(uint32_t n, uint32_t tickBase, uint32_t maxSegs, std::vector<PullSeg> &segs, bool &drained) {
		drained = false;
		uint32_t written = 0;
		const size_t segs0 = segs.size();
		while (written < n) {
			if (hasNew) {  // ticks counter+1 .. F (fade) and F+1 (swap)
				const uint32_t run = umin(n - written, nw.F + 1 - counter);
				if (!emit(segs, segs0, maxSegs, tickBase + written, counter + 1, run)) break;
				counter += run;
				written += run;
				if (counter == nw.F + 1) {  // src/frame.cpp:44-47
					old = nw;
					hasNew = false;
				}
			} else if (!inRequest || counter >= old.M) {  // src/frame.cpp:53: sampleCounter > minNumSamples on the next tick
				if (queue.empty()) {
					curIsNull = true;
					drained = true;
					break;
				}
				if (segs.size() - segs0 >= maxSegs) break;
				pop();
				emit(segs, segs0, maxSegs + 1, tickBase + written, 0, 1);
				written += 1;
			} else {  // hold ticks counter+1 .. M
				const uint32_t run = umin(n - written, old.M - counter);
				if (!emit(segs, segs0, maxSegs, tickBase + written, counter + 1, run)) break;
				counter += run;
				written += run;
			}
		}
		generated += written;
		return written;
	}

	uint64_t samplesGenerated() const { return generated; }

private:
	static uint32_t umin(uint32_t a, uint32_t b) { return a < b ? a : b; }
	static double lerp(double o, double nv, double ratio) { return (nv != nv) ? o : o + ((nv - o) * ratio); }  // src/utils.h:20-23

	// Bring curFrame (and the pitch written back into the old request, src/frame.cpp:77-78) to what the reference holds
	// after the last generated tick.  Only pops and purges look at them, so they are evaluated lazily (the hold glide as the
	// reference's repeated addition, seeked with glideExact).
	void syncToCounter() {
		if (!inRequest) return;
		const uint32_t c = counter, F = info.F;
		vibPos = info.vibPosAtPop + pullVibBefore(info, c + 1);
		if (c == 0) return;  // pop tick: curFrame untouched
		const uint32_t k = c < F ? c : F;
		const double ratio = (double)k / (double)F;
		for (int i = 0; i < kNumParams; ++i) cur[i] = lerp(reqOld[i], reqNew[i], ratio);
		if (c >= F + 2) {  // the hold glide: c - F - 1 additions of the increment, with the reference's roundings (glideExact)
			cur[kVoicePitch] = glideExact(cur[kVoicePitch], info.pitchInc, (uint64_t)(c - F - 1));
			old.frame[kVoicePitch] = cur[kVoicePitch];
		}
	}

	// src/frame.cpp:54-72
	void pop() {
		syncToCounter();
		curIsNull = false;
		nw = queue.front();
		queue.pop_front();
		if (nw.isNull) {
			memcpy(nw.frame, old.frame, sizeof nw.frame);
			nw.frame[kPreFormantGain] = 0;
			nw.frame[kVoicePitch] = cur[kVoicePitch];
			nw.inc = 0;
		} else if (old.isNull) {
			memcpy(old.frame, nw.frame, sizeof old.frame);
			old.frame[kPreFormantGain] = 0;
		}
		if (nw.userIndex != -1) lastUserIndex = nw.userIndex;
		counter = 0;
		nw.frame[kVoicePitch] += nw.inc * (double)nw.F;
		hasNew = true;
		inRequest = true;
		++popCount;
		// everything the ticks of this request need, in closed form of the counter
		memcpy(reqOld, old.frame, sizeof reqOld);
		memcpy(reqNew, nw.frame, sizeof reqNew);
		memset(&info, 0, sizeof info);
		planFade(reqOld, reqNew, nw.F, sampleRate, info.plan);
		const double srInv = 1.0 / (double)sampleRate;
		for (int r = 0; r < kNumResonators; ++r) {
			double f0 = reqOld[resFreqParam(r)], f1 = reqNew[resFreqParam(r)];
			double b0 = reqOld[resBwParam(r)], b1 = reqNew[resBwParam(r)];
			if (f1 != f1) f1 = f0;
			if (b1 != b1) b1 = b0;
			info.fb[r][0] = f0; info.fb[r][1] = f1; info.fb[r][2] = b0; info.fb[r][3] = b1;
			poleTerms(cur[resFreqParam(r)], cur[resBwParam(r)], srInv, info.zStaleRe[r], info.zStaleIm[r]);
		}
		for (int i = 0; i < kNumDirect; ++i) info.dirStale[i] = (float)cur[directParam(i)];
		info.n0InvStale = cur[kCfN0] != 0;
		info.vibIncStale = vibratoIncrement(cur[kVibratoSpeed], srInv);
		info.depthStale = vibratoDepth(cur[kVibratoPitchOffset]);
		info.vibPosAtPop = vibPos;
		info.pitchStale = cur[kVoicePitch];
		info.pitchOld = reqOld[kVoicePitch];
		info.pitchNew = reqNew[kVoicePitch];
		info.pitchInc = nw.inc;
		info.F = nw.F;
	}

	// append ticks [c0, c0+count) of the request in progress; one request is one segment of a pull
	bool emit(std::vector<PullSeg> &segs, size_t segs0, uint32_t maxSegs, uint32_t tickStart, uint32_t c0, uint32_t count) {
		if (count == 0) return true;
		if (segs.size() > segs0) {
			PullSeg &last = segs.back();
			if (lastSegSerial == popCount && last.c0 + last.count == c0 && last.tickStart + last.count == tickStart) {
				last.count += count;
				return true;
			}
		}
		if (segs.size() - segs0 >= maxSegs) return false;
		PullSeg s = info;
		s.c0 = c0;
		s.tickStart = tickStart;
		s.count = count;
		segs.push_back(s);
		lastSegSerial = popCount;
		return true;
	}

	int sampleRate;
	std::deque<PullRequest> queue;   // frameRequestQueue
	PullRequest old, nw;             // oldFrameRequest (initially NULL, M = 0: src/frame.cpp:86-87), newFrameRequest
	bool hasNew = false;
	bool inRequest = false;          // `counter` counts inside the request described by `info`
	double cur[kNumParams];          // curFrame
	bool curIsNull = true;
	uint32_t counter = 0;            // sampleCounter
	int32_t lastUserIndex = -1;
	uint64_t vibPos = 0;             // vibrato phase after the last generated tick
	uint64_t generated = 0;
	uint64_t popCount = 0, lastSegSerial = ~0ull;  // requests are numbered by their pops: one request, one segment per pull
	double reqOld[kNumParams] = {}, reqNew[kNumParams] = {};  // the frames the request in progress fades between
	PullSeg info;                    // its segment template
};

}  // namespace klatt
