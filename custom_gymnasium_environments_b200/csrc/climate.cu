// Batched SmartClimateEnv for sm_100a (SURVEY.md section 8f rank 3): HVAC/lighting step in ONE kernel.
//
// Reference behaviour (paths relative to the reference root, directory smartclimate_rl-main/smartclimate/):
//   env.py:48-60 _init_state, :62-70 reset, :72-82 _get_obs, :84-117 step
//   utils.py:5-13 get_outside_temp, :15-22 update_occupancy, :24-28 room_temp_dynamics, :30-50 calculate_reward
//
// One thread per env over [field][env] float64 / int32 arrays; float64 arithmetic in the reference's order (Python
// floats); the 9-float observation tile of a CTA (256 x 36 B, contiguous in global memory) is composed in shared
// memory and drained with one bulk asynchronous copy.  RNG draws in the reference's order: normal(base, 5) then
// choice(4 values, p) as an inverse-CDF lookup (numpy Generator.choice's own rule; the cdf tables are the float64
// values numpy computes, see oracle/c/climate_oracle.c).  HBM-bound on paper (~160 B per env-step).
#include <cstdint>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {
namespace {

constexpr int KOBS = BENG_CLIMATE_OBS_DIM;
constexpr uint32_t KFLAG_NEEDS_RESET = 1u;

struct KArgs {
    beng_climate_params p;
    beng_climate_state st;
    beng_climate_io io;
    const float *ac_temp;
    const int8_t *lights;
    const uint8_t *mask;
    long long n;
    int first_call;
};

__device__ __forceinline__ double kclip(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }

// get_outside_temp, utils.py:5-13
__device__ __forceinline__ double outside_base(double tod) {
    return (0 <= tod && tod < 8) ? 25.0 : ((8 <= tod && tod < 16) ? 45.0 : 35.0);
}
__device__ __forceinline__ double outside_temp(double tod, EnvStream &rng) { return rng.normal(outside_base(tod), 5.0); }

// One env's state and action words as loaded (requested together, before anything is inspected).
struct KIn {
    double room, outside, ac, total, energy;
    uint32_t w0, ctr;
    int step, comfort_time;
    float act_ac;
    uint32_t lw;  // four int8 light flags
};

template <bool IS_RESET>
__device__ __forceinline__ KIn load_env(const KArgs &a, long long env) {
    const long long n = a.n;
    KIn in;
    in.act_ac = 0.0f;
    in.lw = 0;
    if constexpr (!IS_RESET) {
        in.act_ac = a.ac_temp[env];
        in.lw = *reinterpret_cast<const uint32_t *>(a.lights + 4 * env);
    }
    in.room = a.st.f64[env]; in.outside = a.st.f64[n + env]; in.ac = a.st.f64[2 * n + env];
    in.total = a.st.f64[3 * n + env]; in.energy = a.st.f64[4 * n + env];
    in.w0 = (uint32_t)a.st.i32[env];
    in.step = a.st.i32[n + env]; in.comfort_time = a.st.i32[2 * n + env];
    in.ctr = (uint32_t)a.st.i32[3 * n + env];
    return in;
}

// reset / step of one env (env.py:62-70, :84-117), its state and result stores, and its observation row
template <bool IS_RESET>
__device__ __forceinline__ void step_env(const KArgs &a, long long env, const KIn &in, float *row, bool &ended,
                                         double &st_ret, double &st_len) {
    const long long n = a.n;
    const float act_ac = in.act_ac;
    const uint32_t lw = in.lw;
    double room = in.room, outside = in.outside, ac = in.ac, total = in.total, energy = in.energy;
    const uint32_t w0 = in.w0;
    int people = w0 & 0xFF, lights = (w0 >> 8) & 0xF;
    uint32_t flags = w0 >> 16;
    int step = in.step, comfort_time = in.comfort_time;
    uint32_t ctr = in.ctr;
    bool selected = true;
    if constexpr (IS_RESET) {
        if (a.mask) selected = a.mask[env] != 0;
        if (selected && a.first_call) ctr = 0;
    }
    EnvStream rng(a.p.seed, a.p.env_id_base + (uint64_t)env, BENG_STREAM_ENV, ctr);
    double rew = 0.0, cf = 0.0, acp = 0.0, lp = 0.0;
    int term = 0, at_limit = 0;

    auto init_state = [&]() {  // env.py:48-60
        room = rng.uniform(22.0, 26.0);
        people = rng.randint(0, a.p.max_occupancy);  // integers(0, max_occupancy + 1)
        outside = outside_temp(0.0, rng);
        ac = 24.0;
        lights = 0;
        total = 0.0;
        comfort_time = 0;
        energy = 0.0;
        step = 0;
        flags = 0;
    };

    if constexpr (IS_RESET) {
        if (selected) init_state();
    } else {
        if (a.p.autoreset_mode == BENG_AUTORESET_NEXT_STEP && (flags & KFLAG_NEEDS_RESET)) {
            init_state();
        } else {
            ac = kclip((double)act_ac, 16.0, 32.0);  // env.py:85
            int lights_on = 0;
            lights = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int v = (int)(int8_t)((lw >> (8 * i)) & 0xFF);
                lights |= (v & 1) << i;  // MultiBinary(4): 0 / 1
                lights_on += v;
            }
            step = min(step + 1, 65535);
            const double tod = div_const<60>((double)(step % 1440));  // :91, (step % 1440) / 60 correctly rounded
            // the step's six draws (normal: four, choice: two) in one go
            uint32_t dr[6];
            rng.take(dr);
            outside = EnvStream::to_normal(outside_base(tod), 5.0, dr[0], dr[1], dr[2], dr[3]);  // get_outside_temp
            {   // update_occupancy, utils.py:15-22: rng.choice(values, p) == inverse-CDF lookup
                const bool day = (9 <= tod && tod < 18);
                const double u = EnvStream::to_random53(dr[4], dr[5]);
                const double c0 = day ? 0x1.999999999999ap-4 : 0x1.9999999999998p-3;
                const double c1 = day ? 0x1.999999999999ap-2 : 0x1.3333333333333p-1;
                const double c2 = day ? 0x1.999999999999ap-1 : 0x1.cccccccccccccp-1;
                const int idx = (c0 <= u) + (c1 <= u) + (c2 <= u);  // searchsorted(cdf, u, side='right')
                const int change = idx + (day ? -1 : -2);            // [-1,0,1,2] / [-2,-1,0,1]
                people = min(max(people + change, 0), a.p.max_occupancy);
            }
            // room_temp_dynamics, utils.py:24-28
            const double temp = room + 0.1 * (outside - room) + 0.2 * (ac - room) + (double)people * 1.0;
            room = kclip(temp, 10.0, 50.0);
            // calculate_reward, utils.py:30-50
            if (20 <= room && room <= 24) cf = 10;
            else if (18 <= room && room <= 26) cf = 5;
            else if (16 <= room && room <= 28) cf = 0;
            else cf = -15 * fabs(room - 22);
            acp = -0.5 * fabs(ac - outside);
            const int required = min(4, (people + 1) / 2);  // ceil(num_people / 2)
            lp = -1.0 * (double)max(0, lights_on - required);
            rew = cf + acp + lp;
            total += rew;
            if (20 <= room && room <= 24) comfort_time += 1;
            energy += fabs(ac - outside) + (double)lights_on;
            at_limit = step >= a.p.episode_minutes;
            term = at_limit;  // :107, reported as terminated
            if (term && a.p.autoreset_mode != BENG_AUTORESET_DISABLED) {
                ended = true;
                st_ret = total;
                st_len = (double)step;
                if (a.io.ep_return) a.io.ep_return[env] = total;
                if (a.io.ep_length) a.io.ep_length[env] = step;
                if (a.p.autoreset_mode == BENG_AUTORESET_SAME_STEP) init_state();
                else flags |= KFLAG_NEEDS_RESET;
            }
        }
    }

    // observation row, env.py:72-82
    row[0] = (float)room;
    row[1] = (float)people;
    row[2] = (float)div_const<60>((double)(step % 1440));
    row[3] = (float)outside;
    row[4] = (float)ac;
#pragma unroll
    for (int i = 0; i < 4; ++i) row[5 + i] = (float)((lights >> i) & 1);

    a.st.f64[env] = room;
    a.st.f64[n + env] = outside;
    a.st.f64[2 * n + env] = ac;
    a.st.f64[3 * n + env] = total;
    a.st.f64[4 * n + env] = energy;
    a.st.i32[env] = (int32_t)((uint32_t)people | ((uint32_t)lights << 8) | (flags << 16));
    a.st.i32[n + env] = step;
    a.st.i32[2 * n + env] = comfort_time;
    a.st.i32[3 * n + env] = (int32_t)rng.ctr;
    if constexpr (!IS_RESET) {
        a.io.reward[env] = (float)rew;
        a.io.terminated[env] = (uint8_t)term;
        if (a.io.truncated) a.io.truncated[env] = (uint8_t)(a.p.time_limit_truncation && at_limit);
        if (a.io.reward64) a.io.reward64[env] = rew;
        if (a.io.reward_terms) {
            a.io.reward_terms[env] = cf;
            a.io.reward_terms[n + env] = acp;
            a.io.reward_terms[2 * n + env] = lp;
        }
    }
}

constexpr int CLIMATE_T = 128;

// Reset kernel: one tile of CLIMATE_T envs per CTA.
__global__ void __launch_bounds__(CLIMATE_T, 8) climate_kernel(const KArgs a) {
    constexpr int T = CLIMATE_T;
    __shared__ __align__(128) float tile[T * KOBS];
    const int tid = threadIdx.x;
    const long long n = a.n;
    const long long first = (long long)blockIdx.x * T;
    const long long env = first + tid;
    pdl_launch_dependents();
    pdl_wait();

    bool ended = false;
    double st_ret = 0.0, st_len = 0.0;
    if (env < n) {
        const KIn in = load_env<true>(a, env);
        step_env<true>(a, env, in, tile + tid * KOBS, ended, st_ret, st_len);
    }

    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
        const long long n_here = min((long long)T, n - first);
        const uint32_t bytes = (uint32_t)(n_here * KOBS * sizeof(float));
        const uint32_t bulk = bytes & ~15u;
        if (bulk) bulk_store_s2g(a.io.obs + first * KOBS, tile, bulk);
        bulk_commit();
        for (uint32_t i = bulk / 4; i < bytes / 4; ++i) a.io.obs[first * KOBS + i] = tile[i];  // ragged last tile
    }
    if (tid == 0) bulk_wait_read<0>();
}

// Step kernel: a persistent CTA walks the tiles blockIdx.x, blockIdx.x + gridDim.x, ... and requests the NEXT
// tile's state and action words before it computes the current one, so that the memory round trip of a tile (40 % of
// the one-tile kernel's stall samples) runs under the float64 arithmetic of the previous one.  Three observation
// buffers: the bulk copy of tile k is only awaited before tile k+2 is drained, one CTA barrier per tile.
// 5 CTAs of 128 threads per SM (94 registers, no spills).  Same-box A/B at 1,048,576 envs, L2 flushed, us per step: the
// one-tile kernel 47.1; persistent (CTAs per SM x threads) 5 x 128 **41.1**, 10 x 64 41.2, 4 x 128 42.8, 3 x 192 43.3,
// 2 x 256 44.6; shapes that need a register cap below 94 spill and are slower than the one-tile kernel (6 x 128 at 80
// registers 53.8, 8 x 128 at 64 registers 58.4).
constexpr int CLIMATE_STEP_CTAS_PER_SM = 5;
__global__ void __launch_bounds__(CLIMATE_T, CLIMATE_STEP_CTAS_PER_SM) climate_step_persistent_kernel(const KArgs a) {
    constexpr int T = CLIMATE_T;
    __shared__ __align__(128) float tiles[3][T * KOBS];
    const int tid = threadIdx.x;
    const long long n = a.n;
    const long long n_tiles = (n + T - 1) / T;
    pdl_launch_dependents();
    pdl_wait();

    long long tile = blockIdx.x;
    KIn cur{};
    if (tile < n_tiles && tile * T + tid < n) cur = load_env<false>(a, tile * T + tid);
    int b = 0;
    for (; tile < n_tiles; tile += gridDim.x) {
        const long long first = tile * T, env = first + tid;
        const long long env_next = (tile + gridDim.x) * T + tid;
        KIn nxt{};
        if (env_next < n) nxt = load_env<false>(a, env_next);  // (past the last tile env_next >= n)
        float *buf = tiles[b];
        bool ended = false;
        double st_ret = 0.0, st_len = 0.0;
        if (env < n) step_env<false>(a, env, cur, buf + tid * KOBS, ended, st_ret, st_len);
        fence_proxy_async_smem();
        if (tid == 0) bulk_wait_read<1>();  // the buffer the NEXT tile writes (drained two tiles ago) is free
        __syncthreads();
        if (tid == 0) {
            const long long n_here = min((long long)T, n - first);
            const uint32_t bytes = (uint32_t)(n_here * KOBS * sizeof(float));
            const uint32_t bulk = bytes & ~15u;
            if (bulk) bulk_store_s2g(a.io.obs + first * KOBS, buf, bulk);
            bulk_commit();
            for (uint32_t i = bulk / 4; i < bytes / 4; ++i) a.io.obs[first * KOBS + i] = buf[i];  // ragged last tile
        }
        if (a.io.stats) {
            const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
            if (done_mask) {
                double r = st_ret, l = st_len;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
                    l += __shfl_xor_sync(0xFFFFFFFFu, l, o);
                }
                if ((tid & 31) == 0) {
                    atomicAdd(&a.io.stats[0], (double)__popc(done_mask));
                    atomicAdd(&a.io.stats[1], r);
                    atomicAdd(&a.io.stats[2], l);
                }
            }
        }
        cur = nxt;
        b = b == 2 ? 0 : b + 1;
    }
    if (tid == 0) bulk_wait_read<0>();
}

int launch_reset(const KArgs &a, cudaStream_t stream) {
    const unsigned grid = (unsigned)((a.n + CLIMATE_T - 1) / CLIMATE_T);
    return (int)launch_pdl(climate_kernel, dim3(grid), dim3(CLIMATE_T), 0, stream, a);
}

int launch_step(const KArgs &a, cudaStream_t stream) {
    const long long n_tiles = (a.n + CLIMATE_T - 1) / CLIMATE_T;
    const long long slots = (long long)device_sm_count() * CLIMATE_STEP_CTAS_PER_SM;
    const unsigned grid = (unsigned)(n_tiles < slots ? n_tiles : slots);
    return (int)launch_pdl(climate_step_persistent_kernel, dim3(grid), dim3(CLIMATE_T), 0, stream, a);
}

int check(const beng_climate_params *p, const beng_climate_state *st, const beng_climate_io *io, int64_t n) {
    if (!p || !st || !io || n < 0 || !st->f64 || !st->i32 || !io->obs) return BENG_ERR_BAD_ARG;
    if ((uintptr_t)io->obs & 15) return BENG_ERR_BAD_ARG;
    if (p->autoreset_mode < 0 || p->autoreset_mode > 2) return BENG_ERR_BAD_ARG;
    if (p->max_occupancy < 0 || p->max_occupancy > 255) return BENG_ERR_UNSUPPORTED;
    if (p->episode_minutes < 1 || p->episode_minutes > 65535) return BENG_ERR_UNSUPPORTED;
    return 0;
}

}  // namespace
}  // namespace beng

extern "C" {

int beng_climate_reset(const beng_climate_params *p, const beng_climate_state *st, const beng_climate_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (n_envs == 0) return 0;
    beng::KArgs a{*p, *st, *io, nullptr, nullptr, mask_dev, (long long)n_envs, first_call};
    return beng::launch_reset(a, (cudaStream_t)stream);
}

int beng_climate_step(const beng_climate_params *p, const beng_climate_state *st, const float *ac_temp_dev,
                      const int8_t *lights_dev, const beng_climate_io *io, int64_t n_envs, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (!ac_temp_dev || !lights_dev || !io->reward || !io->terminated) return BENG_ERR_BAD_ARG;
    if (((uintptr_t)lights_dev & 3) || ((uintptr_t)ac_temp_dev & 3)) return BENG_ERR_BAD_ARG;  // lights are read as one uint32 per env
    if (n_envs == 0) return 0;
    beng::KArgs a{*p, *st, *io, ac_temp_dev, lights_dev, nullptr, (long long)n_envs, 0};
    return beng::launch_step(a, (cudaStream_t)stream);
}

int beng_climate_step_host(const beng_climate_params *p, const beng_climate_state *st, float *ac_temp_dev,
                           int8_t *lights_dev, const beng_climate_io *io, int64_t n_envs, const float *ac_temp_host,
                           const int8_t *lights_host, float *obs_host, float *reward_host, uint8_t *terminated_host,
                           uint8_t *truncated_host, void *stream) {
    if (!ac_temp_host || !lights_host || !ac_temp_dev || !lights_dev) return BENG_ERR_BAD_ARG;
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (truncated_host && !io->truncated) return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)n_envs;
    cudaError_t e = cudaMemcpyAsync(ac_temp_dev, ac_temp_host, n * sizeof(float), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyAsync(lights_dev, lights_host, n * 4, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    if (int rc = beng_climate_step(p, st, ac_temp_dev, lights_dev, io, n_envs, stream)) return rc;
    if (int rc = beng::d2h(reward_host, io->reward, n * sizeof(float), s)) return rc;
    if (int rc = beng::d2h(terminated_host, io->terminated, n, s)) return rc;
    if (int rc = beng::d2h(truncated_host, io->truncated, n, s)) return rc;
    return beng::d2h(obs_host, io->obs, n * BENG_CLIMATE_OBS_DIM * sizeof(float), s);
}

}  // extern "C"
