// Shared host/device helpers of libbeng: launch accounting, error mapping, PTX wrappers for the
// bulk asynchronous copy engine (TMA, non-tensor form) used to drain observation tiles.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdlib>
#include <functional>

#include "../../include/beng.h"

namespace beng {

extern std::atomic<uint64_t> g_launch_count;

inline int finish_launch() {
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaGetLastError();
}

int device_sm_count();

// ---- bulk async copy (cp.async.bulk, SASS UBLKCP) shared -> global -------------------------
// One thread issues a contiguous copy of `bytes` (multiple of 16, both addresses 16-B aligned)
// from this CTA's shared memory to global memory; completion is tracked per issuing thread in
// bulk async-groups.
__device__ __forceinline__ void bulk_store_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// Wait until at most N of this thread's bulk groups still have to READ their shared-memory source.
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// Wait until at most N of this thread's bulk groups are incomplete (writes performed).
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// Make generic-proxy writes to shared memory visible to the async proxy (the copy engine).
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// A step kernel depends on the previous step's state writes.  Launched with programmatic stream serialization, its
// CTAs may become resident while the previous grid drains; everything before pdl_wait() (index math, shared-memory
// setup) overlaps that tail, and pdl_wait() returns once the previous grid has completed and flushed its memory.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- launch-uniform state that the launch advances itself -------------------------------------------------------------
// A value every CTA of a step needs and every step changes (crypto's window head, snake's done-counter parity), kept in
// device memory instead of in the kernel arguments: the launch then has the same arguments every step, so a launch
// captured in a CUDA graph is the right program on every replay.  Call once per launch, after pdl_wait(), from every
// thread of every CTA of a 1-D grid (it contains a __syncthreads()).  Returns *word as it was when the launch started;
// the last CTA to arrive on *arrivals writes next(value) to *word and rewinds *arrivals to 0 (it must be 0 when the
// launch starts).  Every CTA arrives only after it holds the value, so no CTA can read the advanced one; the next launch
// reads *word after its own pdl_wait(), i.e. after this grid has completed and flushed its memory -- with PDL, without
// it, and across a programmatic edge of a graph alike.
template <typename Next>
__device__ __forceinline__ uint32_t grid_uniform_advance(uint32_t *word, uint32_t *arrivals, Next next) {
    __shared__ uint32_t s_value;
    if (threadIdx.x == 0) s_value = __ldcg(word);
    __syncthreads();
    const uint32_t v = s_value;
    if (threadIdx.x == 0) {
        __threadfence();  // this CTA's read of *word is ordered before its arrival
        if (atomicAdd(arrivals, 1u) == gridDim.x - 1) {
            __threadfence();  // ... and every other CTA's read before the write below
            *word = next(v);
            *arrivals = 0;
        }
    }
    return v;
}

// Launch `kern<<<grid, block, smem, stream>>>(args...)` with the PDL attribute (BENG_NO_PDL=1 disables it) and count
// the attempt in g_launch_count.
template <typename Kern, typename... Args>
inline cudaError_t launch_pdl(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, const Args &...args) {
    static const bool use_pdl = getenv("BENG_NO_PDL") == nullptr;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = use_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return e;
}

// Device -> host copy of `bytes` on `stream` for an optional output: a null `dst` is skipped.
inline cudaError_t d2h(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
    return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream) : cudaSuccess;
}

// Host fan-out of the *_apply_obs_delta functions: runs chunk(begin, end) over [0, n) split into nt = clamp(n_threads,
// 1, n) contiguous chunks [n * t / nt, n * (t + 1) / nt), one thread each, the calling thread taking chunk 0, and joins
// them all.  A chunk whose thread cannot be started runs on the calling thread instead (this never throws).  True
// when every chunk returned true.
bool for_each_chunk(int64_t n, int32_t n_threads, const std::function<bool(int64_t, int64_t)> &chunk);

// streaming (evict-first) 128-bit / 64-bit global loads for read-once inputs
__device__ __forceinline__ uint4 ld_stream_u4(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
// (coherent, not .nc: under programmatic dependent launch the producer of the action tensor may still be running when
// this grid becomes resident, and .nc data must be read-only for the whole lifetime of the grid)
__device__ __forceinline__ long long ld_stream_s64(const long long *p) {
    long long r;
    asm volatile("ld.global.L1::no_allocate.s64 %0, [%1];" : "=l"(r) : "l"(p));
    return r;
}
// ... and the same load with an L2 evict-first policy, for an input that no later launch reads again (a step's action
// tensor): its lines are the first the L2 gives up, so they do not push out lines the next launch would hit.
__device__ __forceinline__ long long ld_once_s64(const long long *p) {
    uint64_t policy;
    long long r;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.s64 %0, [%1], %2;" : "=l"(r) : "l"(p), "l"(policy));
    return r;
}

// Correctly rounded x / B (float64) for a compile-time integer B without the IEEE division subroutine (a ~60-instruction
// call on sm_100a): y = RN(1 / B), q = RN(x * y), r = x - B * q exactly (FMA), result RN(q + r * y) -- Markstein's
// final iteration, which returns the correctly rounded quotient when y is the correctly rounded reciprocal and q is
// within an ulp of x / B.  For finite x whose quotient neither overflows nor is subnormal (the callers divide sums of
// small integers).  tests/test_traffic_oracle.py restates the sequence in exact rational arithmetic against x / B.
template <int B>
__device__ __forceinline__ double div_const(double x) {
    constexpr double y = 1.0 / (double)B;
    const double q = x * y;
    const double r = fma(-(double)B, q, x);
    return fma(r, y, q);
}

// NumPy's pairwise summation order (np.sum / np.mean / np.var, n <= 128) over f(0..n-1), without materialising the
// array: the values are produced on demand so that the caller never holds all of them in registers.
template <typename F>
__device__ __forceinline__ double np_sum_fn(F f, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r += f(i);
        return r;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = f(j);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] += f(i + j);
    }
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += f(i);
    return res;
}

}  // namespace beng
