// Running normalization of observations and rewards (Stable-Baselines3 VecNormalize semantics) for the batched envs.
//
// One training step is two launches:
//   moments  every CTA sums a contiguous range of rows, per column, as float64 (x - x_row0) and (x - x_row0)^2, plus
//            the same two sums of the updated discounted returns (shifted by env 0's); the CTA's partials go to the
//            workspace.  The last CTA to arrive on the workspace counter adds all partials up in CTA order (so the
//            statistics are bit-identical run to run and do not depend on which CTA finished last), turns them into the
//            batch mean and variance and merges them into obs_rms / ret_rms with Chan's update.
//   apply    normalizes the observations and rewards with the updated statistics, writes the updated returns and zeroes
//            the returns of finished envs.
// With BENG_NORM_UPDATE clear only the apply pass runs.  Shifting by the batch's first row, which every CTA can read,
// keeps the cross-CTA combine to plain additions and the batch variance float64-accurate for columns with a large
// offset (a plain sum of squares loses every digit of 1e6 + 1e-3 * noise).
//
// Launch shape: one thread per (column, row group); a CTA holds R row groups of W = min(dim, 1024) columns, R chosen
// so that R * W is at least 512 threads (for dim = 261: 2 x 261 in a 544-thread CTA), and walks its rows R at a time.
// Columns past 1024 are handled in chunks of 1024.  The grid depends on (n, dim) only -- never on the device -- so the
// order of every float64 sum, and with it the statistics, is the same on every GPU.
#include "beng_common.cuh"

namespace beng {
namespace {

constexpr int NORM_MAX_CTAS = 296;          // two CTAs per SM of a 148-SM B200
constexpr long long NORM_ELEMS_PER_CTA = 32768;  // fewer, fuller CTAs below this much work each
constexpr int NORM_UNROLL = 8;              // independent loads in flight per thread
constexpr size_t NORM_WS_HEADER = 16;       // uint32 arrival counter, padded

struct Shape {
    int W, R, T, chunks, ctas;
};

Shape shape_of(int64_t n, int32_t dim) {
    Shape s;
    s.W = dim < 1024 ? dim : 1024;
    s.R = (512 + s.W - 1) / s.W;
    if (s.R * s.W > 1024) s.R = 1024 / s.W;
    if (s.R < 1) s.R = 1;
    s.T = (s.R * s.W + 31) / 32 * 32;
    s.chunks = (dim + s.W - 1) / s.W;
    long long g = ((long long)n * dim + NORM_ELEMS_PER_CTA - 1) / NORM_ELEMS_PER_CTA;
    if (g > NORM_MAX_CTAS) g = NORM_MAX_CTAS;
    if (g > n) g = n;
    s.ctas = g < 1 ? 1 : (int)g;
    return s;
}

struct KArgs {
    beng_normalize_params p;
    beng_normalize_io io;
    long long n;
    int dim, W, R, chunks;
    bool obs, reward, update;
};

__device__ __forceinline__ long long row_begin(long long n, int b, int g) { return n * b / g; }

// Correctly rounded a / s from s and y = RN(1 / s): Markstein's final iteration (see div_const in beng_common.cuh).
__device__ __forceinline__ double div_by(double a, double s, double y) {
    const double q = a * y;
    const double r = fma(-s, q, a);
    return fma(r, y, q);
}

__device__ __forceinline__ double clip(double x, double c) { return fmin(fmax(x, -c), c); }

__device__ __forceinline__ double discounted(const KArgs &a, long long e) {
    return __ldcg(a.io.returns + e) * a.p.gamma + (double)__ldcg(a.io.reward + e);
}

// Deterministic CTA-wide sum of (x, y) in a fixed order; the result is valid in thread 0.  `red` holds 2 * 32 doubles.
__device__ __forceinline__ double2 block_sum2(double x, double y, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x += __shfl_down_sync(0xFFFFFFFFu, x, o);
        y += __shfl_down_sync(0xFFFFFFFFu, y, o);
    }
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0) red[2 * w] = x, red[2 * w + 1] = y;
    __syncthreads();
    double2 r = make_double2(0.0, 0.0);
    if (threadIdx.x == 0)
        for (int i = 0; i < nw; ++i) r.x += red[2 * i], r.y += red[2 * i + 1];
    return r;
}

// Chan's merge of a batch (shifted sums s1, s2 over n rows, shift x0) into the running record (mean, var, count),
// in the operation order of SB3's RunningMeanStd.update_from_moments.
__device__ __forceinline__ void merge(double *mean, double *var, double count, double n, double x0, double s1,
                                      double s2) {
    const double m1 = s1 / n;
    const double b_mean = x0 + m1;
    const double b_var = fmax(s2 / n - m1 * m1, 0.0);
    const double delta = b_mean - *mean;
    const double tot = count + n;
    const double new_mean = *mean + delta * n / tot;
    const double m2 = *var * count + b_var * n + delta * delta * count * n / tot;
    *mean = new_mean;
    *var = m2 / tot;
}

// 56 registers (no spills): two CTAs of up to 576 threads fit an SM, so the 296-CTA grid is one wave on a B200.
__global__ void __maxnreg__(56) normalize_moments_kernel(const KArgs a) {
    extern __shared__ double2 sm[];  // [blockDim.x]
    __shared__ double red[64];
    __shared__ bool s_last;
    pdl_launch_dependents();
    pdl_wait();
    const int t = threadIdx.x, T = blockDim.x, b = blockIdx.x, G = gridDim.x;
    const long long r0 = row_begin(a.n, b, G), r1 = row_begin(a.n, b + 1, G);
    const int dim = a.dim, W = a.W, R = a.R;
    double2 *ws = reinterpret_cast<double2 *>(static_cast<char *>(a.io.workspace) + NORM_WS_HEADER);
    double2 *part = ws + (size_t)b * (dim + 1);

    if (a.obs) {
        const int rg = t / W, cl = t % W;
        for (int j = 0; j < a.chunks; ++j) {
            const int c = j * W + cl;
            double s1 = 0.0, s2 = 0.0;
            if (rg < R && c < dim) {
                const double x0 = (double)__ldcg(a.io.obs + c);
                const float *p = a.io.obs + (r0 + rg) * dim + c;
                const long long step = (long long)R * dim;
                long long r = r0 + rg;
                for (; r + (long long)(NORM_UNROLL - 1) * R < r1; r += (long long)NORM_UNROLL * R) {
                    float v[NORM_UNROLL];
#pragma unroll
                    for (int k = 0; k < NORM_UNROLL; ++k) v[k] = __ldcg(p + k * step);
#pragma unroll
                    for (int k = 0; k < NORM_UNROLL; ++k) {
                        const double d = (double)v[k] - x0;
                        s1 += d;
                        s2 = fma(d, d, s2);
                    }
                    p += NORM_UNROLL * step;
                }
                for (; r < r1; r += R, p += step) {
                    const double d = (double)__ldcg(p) - x0;
                    s1 += d;
                    s2 = fma(d, d, s2);
                }
            }
            sm[t] = make_double2(s1, s2);
            __syncthreads();
            if (rg == 0 && c < dim) {
                for (int g = 1; g < R; ++g) {
                    const double2 o = sm[g * W + cl];
                    s1 += o.x;
                    s2 += o.y;
                }
                part[c] = make_double2(s1, s2);
            }
            __syncthreads();
        }
    }
    if (a.reward) {
        const double y0 = discounted(a, 0);
        double s1 = 0.0, s2 = 0.0;
        for (long long e = r0 + t; e < r1; e += T) {
            const double d = discounted(a, e) - y0;
            s1 += d;
            s2 = fma(d, d, s2);
        }
        const double2 s = block_sum2(s1, s2, red);
        if (t == 0) part[dim] = s;
    }

    // arrival: the last CTA combines
    __threadfence();  // this thread's partials are visible device-wide before the CTA arrives
    __syncthreads();
    if (t == 0) {
        unsigned *arrivals = static_cast<unsigned *>(a.io.workspace);
        s_last = atomicAdd(arrivals, 1u) == (unsigned)G - 1;
        if (s_last) *arrivals = 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();

    // columns 0..dim-1 are the observation features, column dim the returns; P CTA subsets per column in parallel
    const int cols = dim + 1;
    const int P = T / cols > 1 ? T / cols : 1;
    const int Q = T / P;
    const double nd = (double)a.n;
    const double obs_count = a.obs ? a.io.obs_rms[2 * dim] : 0.0;
    for (int base = 0; base < cols; base += Q) {
        const int pp = t / Q, c = base + t % Q;
        const bool live = pp < P && c < cols && (c < dim ? a.obs : a.reward);
        double2 acc = make_double2(0.0, 0.0);
        if (live) {
            int g = pp;
            for (; g + 3 * P < G; g += 4 * P) {
                double2 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = __ldcg(ws + (size_t)(g + k * P) * cols + c);
#pragma unroll
                for (int k = 0; k < 4; ++k) acc.x += v[k].x, acc.y += v[k].y;
            }
            for (; g < G; g += P) {
                const double2 v = __ldcg(ws + (size_t)g * cols + c);
                acc.x += v.x, acc.y += v.y;
            }
        }
        sm[t] = acc;
        __syncthreads();
        if (live && pp == 0) {
            for (int q = 1; q < P; ++q) {
                const double2 o = sm[q * Q + (t % Q)];
                acc.x += o.x, acc.y += o.y;
            }
            if (c < dim)
                merge(a.io.obs_rms + c, a.io.obs_rms + dim + c, obs_count, nd, (double)__ldcg(a.io.obs + c), acc.x,
                      acc.y);
            else
                merge(a.io.ret_rms, a.io.ret_rms + 1, a.io.ret_rms[2], nd, discounted(a, 0), acc.x, acc.y);
        }
        __syncthreads();
    }
    if (t == 0) {
        if (a.obs) a.io.obs_rms[2 * dim] = obs_count + nd;
        if (a.reward) a.io.ret_rms[2] = a.io.ret_rms[2] + nd;
    }
}

__global__ void __launch_bounds__(1024) normalize_apply_kernel(const KArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const int t = threadIdx.x, T = blockDim.x, b = blockIdx.x, G = gridDim.x;
    const long long r0 = row_begin(a.n, b, G), r1 = row_begin(a.n, b + 1, G);
    const int dim = a.dim, W = a.W, R = a.R;

    if (a.obs && a.io.obs_out) {
        const int rg = t / W, cl = t % W;
        const double clip_obs = a.p.clip_obs;
        for (int j = 0; j < a.chunks; ++j) {
            const int c = j * W + cl;
            if (rg >= R || c >= dim) continue;
            const double mean = __ldcg(a.io.obs_rms + c);
            const double s = sqrt(__ldcg(a.io.obs_rms + dim + c) + a.p.epsilon);
            const double y = 1.0 / s;
            const long long off = (r0 + rg) * dim + c, step = (long long)R * dim;
            const float *p = a.io.obs + off;
            float *o = a.io.obs_out + off;
            long long r = r0 + rg;
            for (; r + (long long)(NORM_UNROLL - 1) * R < r1; r += (long long)NORM_UNROLL * R) {
                float v[NORM_UNROLL];
#pragma unroll
                for (int k = 0; k < NORM_UNROLL; ++k) v[k] = __ldcg(p + k * step);
#pragma unroll
                for (int k = 0; k < NORM_UNROLL; ++k)
                    __stcs(o + k * step, (float)clip(div_by((double)v[k] - mean, s, y), clip_obs));
                p += NORM_UNROLL * step;
                o += NORM_UNROLL * step;
            }
            for (; r < r1; r += R, p += step, o += step)
                __stcs(o, (float)clip(div_by((double)__ldcg(p) - mean, s, y), clip_obs));
        }
    }
    if (a.reward) {
        const double s = sqrt(__ldcg(a.io.ret_rms + 1) + a.p.epsilon);
        const double y = 1.0 / s;
        for (long long e = r0 + t; e < r1; e += T) {
            const bool done = (a.io.terminated && a.io.terminated[e]) || (a.io.truncated && a.io.truncated[e]);
            if (a.update)
                a.io.returns[e] = done ? 0.0 : discounted(a, e);
            else if (done)
                a.io.returns[e] = 0.0;
            if (a.io.reward_out)
                a.io.reward_out[e] = (float)clip(div_by((double)__ldcg(a.io.reward + e), s, y), a.p.clip_reward);
        }
    }
}

int check(const beng_normalize_params *p, const beng_normalize_io *io, int64_t n, int32_t dim) {
    if (!p || !io || n < 0 || dim < 1) return BENG_ERR_BAD_ARG;
    if (p->flags & ~(uint32_t)(BENG_NORM_OBS | BENG_NORM_REWARD | BENG_NORM_UPDATE)) return BENG_ERR_BAD_ARG;
    if (!(p->clip_obs >= 0.0) || !(p->clip_reward >= 0.0) || !(p->epsilon >= 0.0) || !(p->gamma >= 0.0))
        return BENG_ERR_BAD_ARG;  // (also rejects NaN)
    auto bad = [](const void *ptr, uintptr_t align, bool required) {
        return ptr ? ((uintptr_t)ptr & (align - 1)) != 0 : required;
    };
    const bool obs = p->flags & BENG_NORM_OBS, rew = p->flags & BENG_NORM_REWARD;
    const bool update = (p->flags & BENG_NORM_UPDATE) && (obs || rew);
    if (obs && (bad(io->obs, 4, true) || bad(io->obs_rms, 8, true) || bad(io->obs_out, 4, false))) return BENG_ERR_BAD_ARG;
    if (rew && (bad(io->reward, 4, true) || bad(io->returns, 8, true) || bad(io->ret_rms, 8, true) ||
                bad(io->reward_out, 4, false)))
        return BENG_ERR_BAD_ARG;
    if (update && bad(io->workspace, 16, true)) return BENG_ERR_BAD_ARG;
    return 0;
}

}  // namespace
}  // namespace beng

extern "C" {

size_t beng_normalize_workspace_bytes(int64_t n_envs, int32_t dim) {
    if (n_envs < 0 || dim < 1) return 0;
    const beng::Shape s = beng::shape_of(n_envs, dim);
    return beng::NORM_WS_HEADER + (size_t)s.ctas * ((size_t)dim + 1) * 2 * sizeof(double);
}

int beng_normalize(const beng_normalize_params *p, const beng_normalize_io *io, int64_t n_envs, int32_t dim,
                   void *stream) {
    if (int rc = beng::check(p, io, n_envs, dim)) return rc;
    const bool obs = p->flags & BENG_NORM_OBS, rew = p->flags & BENG_NORM_REWARD;
    const bool update = (p->flags & BENG_NORM_UPDATE) && (obs || rew);
    if (n_envs == 0 || !(obs || rew)) return 0;
    const beng::Shape s = beng::shape_of(n_envs, dim);
    const beng::KArgs a{*p, *io, (long long)n_envs, dim, s.W, s.R, s.chunks, obs, rew, update};
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)s.T * sizeof(double2);
    if (update)
        if (int rc = (int)beng::launch_pdl(beng::normalize_moments_kernel, dim3(s.ctas), dim3(s.T), smem, st, a))
            return rc;
    if (rew || io->obs_out)
        return (int)beng::launch_pdl(beng::normalize_apply_kernel, dim3(s.ctas), dim3(s.T), 0, st, a);
    return 0;
}

}  // extern "C"
