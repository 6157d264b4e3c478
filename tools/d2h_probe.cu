// Host-gather probe (VERDICT r1 item 5): how fast can N GPUs of one box copy device memory into pinned host memory
// AT THE SAME TIME, with no kernels running?  The batch path's end-to-end number is this copy (28.9 GB of int16 per
// GPU per step of config 3), so its ceiling at N GPUs is what this program prints -- not a property of the engine.
//
//   shapes:  contig : one cudaMemcpyAsync of B bytes (device -> pinned host)
//            2d     : cudaMemcpy2DAsync of the engine's gather shape: `rows` rows of `width` bytes out of a device
//                     staging buffer (pitch = width) into a host buffer of pitch `hostPitch` (host.cu renderToHost:
//                     65 536 rows, 2 s slices of a 10 s row -> width 88 200 B, host pitch 441 000 B)
//            2dtight: the same rows into a host buffer of pitch == width (what a [chunk][stream]-blocked host layout
//                     would see)
//   modes:   one host thread + one stream per GPU, all released by a barrier; each repeats `reps` copies; the
//            aggregate is total bytes / (last finish - first start) by the host clock, per-GPU rates by CUDA events.
//
// build: nvcc -O2 -o tools/d2h_probe tools/d2h_probe.cu      run: tools/d2h_probe [gpus] [MiB per copy] [reps]
#include <cuda_runtime.h>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); exit(2); } } while (0)

static double nowS() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Barrier {
	std::atomic<int> count{0}, gen{0};
	int n;
	explicit Barrier(int n_) : n(n_) {}
	void wait() {
		int g = gen.load();
		if (count.fetch_add(1) + 1 == n) { count.store(0); gen.fetch_add(1); }
		else while (gen.load() == g) std::this_thread::yield();
	}
};

int main(int argc, char **argv) {
	int have = 0;
	CK(cudaGetDeviceCount(&have));
	int gpus = argc > 1 ? atoi(argv[1]) : have;
	if (gpus > have) gpus = have;
	const size_t mib = argc > 2 ? (size_t)atoll(argv[2]) : 1024;
	const int reps = argc > 3 ? atoi(argv[3]) : 6;
	const size_t width = 88200, hostPitch = 441000;
	const size_t rows = (mib << 20) / width, bytes = rows * width;
	printf("{\"probe\": \"d2h\", \"gpus\": %d, \"bytes_per_copy\": %zu, \"rows\": %zu, \"width\": %zu, \"host_pitch\": %zu, \"reps\": %d, \"results\": [\n",
	       gpus, bytes, rows, width, hostPitch, reps);
	const char *shapes[3] = {"contig", "2d", "2dtight"};
	for (int shape = 0; shape < 3; ++shape) {
		std::vector<double> rate(gpus, 0.0), t0(gpus, 0.0), t1(gpus, 0.0);
		Barrier bar(gpus);
		std::vector<std::thread> th;
		for (int g = 0; g < gpus; ++g)
			th.emplace_back([&, g] {
				CK(cudaSetDevice(g));
				void *d = nullptr, *h = nullptr;
				const size_t hostBytes = shape == 1 ? rows * hostPitch : bytes;
				CK(cudaMalloc(&d, bytes));
				CK(cudaMemset(d, 1, bytes));
				CK(cudaMallocHost(&h, hostBytes));
				cudaStream_t s;
				CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
				cudaEvent_t e0, e1;
				CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
				auto copy = [&] {
					if (shape == 0) CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s));
					else CK(cudaMemcpy2DAsync(h, shape == 1 ? hostPitch : width, d, width, width, rows, cudaMemcpyDeviceToHost, s));
				};
				copy();  // warm-up: page-lock mappings, first touch
				CK(cudaStreamSynchronize(s));
				bar.wait();
				t0[g] = nowS();
				CK(cudaEventRecord(e0, s));
				for (int r = 0; r < reps; ++r) copy();
				CK(cudaEventRecord(e1, s));
				CK(cudaStreamSynchronize(s));
				t1[g] = nowS();
				float ms = 0;
				CK(cudaEventElapsedTime(&ms, e0, e1));
				rate[g] = (double)bytes * reps / (ms * 1e-3) / 1e9;
				bar.wait();
				CK(cudaFreeHost(h)); CK(cudaFree(d));
				CK(cudaStreamDestroy(s));
			});
		for (auto &t : th) t.join();
		double first = t0[0], last = t1[0], lo = rate[0], hi = rate[0];
		for (int g = 0; g < gpus; ++g) {
			if (t0[g] < first) first = t0[g];
			if (t1[g] > last) last = t1[g];
			if (rate[g] < lo) lo = rate[g];
			if (rate[g] > hi) hi = rate[g];
		}
		printf("  {\"shape\": \"%s\", \"aggregate_GBps\": %.2f, \"per_gpu_min_GBps\": %.2f, \"per_gpu_max_GBps\": %.2f}%s\n", shapes[shape],
		       (double)bytes * reps * gpus / (last - first) / 1e9, lo, hi, shape < 2 ? "," : "");
	}
	printf("]}\n");
	return 0;
}
