// libbeng core: version / launch accounting, the host thread fan-out and the synthetic action-tape kernel.
#include <thread>
#include <vector>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {

std::atomic<uint64_t> g_launch_count{0};

bool for_each_chunk(int64_t n, int32_t n_threads, const std::function<bool(int64_t, int64_t)> &chunk) {
    if (n <= 0) return true;
    const int64_t nt = n_threads < 1 ? 1 : (n_threads < n ? n_threads : n);
    std::vector<char> ok((size_t)nt, 1);
    std::vector<std::thread> workers;
    for (int64_t t = 1; t < nt; ++t) {
        const int64_t b = n * t / nt, e = n * (t + 1) / nt;
        auto job = [=, &ok, &chunk] { ok[t] = chunk(b, e); };
        try {
            workers.emplace_back(job);
        } catch (...) {
            job();
        }
    }
    ok[0] = chunk(0, n / nt);
    for (std::thread &w : workers) w.join();
    for (const char o : ok)
        if (!o) return false;
    return true;
}

int device_sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            return 148;
    }
    return cached;
}

// One thread per env; each thread walks its n_cols draws so Philox blocks are reused.
__global__ void __launch_bounds__(256) fill_random_actions_kernel(long long *__restrict__ actions, long long n_envs,
                                                                  int n_cols, int n_choices, uint32_t step_index,
                                                                  uint64_t env_id_base, uint64_t seed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_envs) return;
    EnvStream rng(seed, env_id_base + (uint64_t)i, BENG_STREAM_ACTION, step_index * (uint32_t)n_cols);
    for (int c = 0; c < n_cols; ++c) actions[i * n_cols + c] = rng.randint(0, n_choices - 1);
}

}  // namespace beng

extern "C" {

int beng_version(void) { return BENG_VERSION; }

int beng_compiled_arch(void) {
#ifdef BENG_ARCH
    return BENG_ARCH;
#else
    return 0;
#endif
}

uint64_t beng_launch_count(void) { return beng::g_launch_count.load(std::memory_order_relaxed); }

int beng_fill_random_actions(int64_t *actions_dev, int64_t n_envs, int32_t n_cols, int32_t n_choices,
                             uint32_t step_index, uint64_t env_id_base, uint64_t seed, void *stream) {
    if (!actions_dev || n_envs < 0 || n_cols < 1 || n_choices < 1) return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    const int threads = 256;
    const unsigned blocks = (unsigned)((n_envs + threads - 1) / threads);
    beng::fill_random_actions_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(
        (long long *)actions_dev, (long long)n_envs, n_cols, n_choices, step_index, env_id_base, seed);
    return beng::finish_launch();
}

}  // extern "C"
