// Host-side helper threads (plain C++, no CUDA): see HostPool below.  Used by api_player.cu for the batched pull; tests/hostsim
// builds it on the CPU (tests/test_host_pool_cpu.py).
#pragma once
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include <unistd.h>

namespace klatt {

// A few helper threads for the per-player HOST work of a batched pull (frame-manager walk, segment staging, PCM copies):
// 148 players x 8192 samples cost ~0.9 ms of serial bookkeeping around a 0.2 ms launch.  parallelFor hands out index blocks
// from an atomic cursor; the calling thread takes part and returns when every helper has checked in.  NVSP_HOST_THREADS=0
// turns the helpers off.
class HostPool {
public:
	static HostPool &get() {
		static HostPool pool;
		return pool;
	}
	size_t helpers() const { return workers.size(); }
	void parallelFor(size_t n, size_t grain, const std::function<void(size_t)> &fn) {
		if (workers.empty() || n <= grain || getpid() != owner) {  // (a forked child has the pool object but not its threads)
			for (size_t i = 0; i < n; ++i) fn(i);
			return;
		}
		std::lock_guard<std::mutex> one(callMu);  // one job at a time
		{
			std::lock_guard<std::mutex> lk(mu);
			job = &fn; total = n; step = grain; next.store(0); pending = workers.size(); ++epoch;
		}
		cv.notify_all();
		run(fn, n, grain);
		std::unique_lock<std::mutex> lk(mu);
		cvDone.wait(lk, [&] { return pending == 0; });
		job = nullptr;
	}
	~HostPool() {
		{
			std::lock_guard<std::mutex> lk(mu);
			stop = true;
		}
		cv.notify_all();
		for (std::thread &t : workers) {
			if (getpid() == owner) t.join();
			else t.detach();
		}
	}

private:
	HostPool() {
		unsigned want = std::thread::hardware_concurrency();
		want = want > 1 ? std::min(want - 1, 7u) : 0;
		if (const char *e = getenv("NVSP_HOST_THREADS")) want = (unsigned)std::min(std::max(atoi(e), 0), 64);
		for (unsigned i = 0; i < want; ++i) workers.emplace_back([this] { loop(); });
	}
	void run(const std::function<void(size_t)> &fn, size_t n, size_t grain) {
		for (;;) {
			const size_t a = next.fetch_add(grain);
			if (a >= n) return;
			const size_t b = std::min(a + grain, n);
			for (size_t i = a; i < b; ++i) fn(i);
		}
	}
	void loop() {
		uint64_t seen = 0;
		std::unique_lock<std::mutex> lk(mu);
		for (;;) {
			cv.wait(lk, [&] { return stop || epoch != seen; });
			if (stop) return;
			seen = epoch;
			const std::function<void(size_t)> *fn = job;
			const size_t n = total, grain = step;
			lk.unlock();
			run(*fn, n, grain);
			lk.lock();
			if (--pending == 0) cvDone.notify_one();
		}
	}
	std::vector<std::thread> workers;
	const pid_t owner = getpid();
	std::mutex mu, callMu;
	std::condition_variable cv, cvDone;
	const std::function<void(size_t)> *job = nullptr;
	size_t total = 0, step = 1, pending = 0;
	std::atomic<size_t> next{0};
	uint64_t epoch = 0;
	bool stop = false;
};

}  // namespace klatt
