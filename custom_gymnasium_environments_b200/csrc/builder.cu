// Batched WorldBuilderEnv for sm_100a (SURVEY.md section 8f rank 3): build + production + consumption + growth +
// "smart reward" + win/lose termination + auto-reset + observation in ONE kernel.
//
// Reference behaviour (paths relative to the reference root, directory world_builder_env/src/environment/):
//   world_builder_env.py:99-123 reset, :125-166 step, :186-217 _get_observation, :233-247 _check_termination
//   game_logic.py:33-57 reset, :59-123 execute_action, :125-156 _try_build, :158-203 costs/production/consumption/growth
//
// Integer dynamics, bit-exact.  One thread per env; the CTA's T x G*G grid bytes are contiguous in global memory: the
// tile is brought into shared memory with coalesced 128-bit loads, each thread works on its own row (the k-th empty
// cell in row-major order is what `np.random.randint(len(np.where(grid == 0)[0]))` selects, game_logic.py:131-138),
// and the tile is drained in place with one bulk asynchronous copy; the optional flattened observation
// (flatten_obs=True, :189-200) is composed in a second tile and drained the same way.
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {
namespace {

constexpr uint32_t BFLAG_NEEDS_RESET = 1u;
enum { FARM = 1, LUMBERYARD = 2, QUARRY = 3, HOUSE = 4 };

struct BArgs {
    beng_builder_params p;
    beng_builder_state st;
    beng_builder_io io;
    const long long *actions;
    const uint8_t *mask;
    long long n;
    int first_call;
    uint32_t *delta;  // DELTA step only: one BENG_BUILDER_DELTA record per env
};

// CELLS_T: G*G when it is known at compile time and a multiple of 4 (the default 10 x 10 board), 0 = any board.
// DELTA (step only): also store one change record per env to a.delta, describing how this step's grid row differs
// from the previous one.  It is assembled from the dynamics' registers (the cell and building of a successful build,
// the reset_env() call sites), never by reading the row back.
template <int T, bool IS_RESET, int CELLS_T, bool DELTA>
__global__ void __launch_bounds__(T) builder_kernel(const BArgs a) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ int s_stats[4];  // per-CTA: n_episodes, sum_return, sum_length, wins
    const int cells = CELLS_T ? CELLS_T : a.p.grid_size * a.p.grid_size, FD = cells + 6;
    uint8_t *tile = smem_raw;                                                     // [T][cells]
    float *flat = reinterpret_cast<float *>(smem_raw + (((size_t)T * cells + 15) & ~(size_t)15));  // [T][cells + 6]
    const int tid = threadIdx.x;
    const long long n = a.n;
    const long long first = (long long)blockIdx.x * T;
    const long long env = first + tid;
    const long long n_here = min((long long)T, n - first);
    const uint32_t tile_bytes = (uint32_t)(n_here * cells);
    if (tid < 4) s_stats[tid] = 0;
    pdl_launch_dependents();
    pdl_wait();

    // ---- per-env state words and the action are requested first, so that their memory round trip runs alongside
    // the tile's instead of after the barrier below
    int food = 0, wood = 0, stone = 0, pop = 0, cap = 0, steps = 0, ep_ret = 0;
    uint32_t counts = 0, w7 = 0, ctr = 0;
    long long act = 0;
    if (env < n) {
        const int32_t *w = a.st.words + env;
        food = w[0]; wood = w[n]; stone = w[2 * n]; pop = w[3 * n]; cap = w[4 * n];
        counts = (uint32_t)w[5 * n];
        steps = w[6 * n];
        w7 = (uint32_t)w[7 * n];
        ctr = (uint32_t)w[8 * n];
        ep_ret = w[9 * n];
        if constexpr (!IS_RESET) act = a.actions[env];
    }

    // ---- grid tile: global -> shared (coalesced 128-bit loads; byte tail for a ragged last tile)
    {
        const uint8_t *src = reinterpret_cast<const uint8_t *>(a.io.grid) + first * cells;
        const uint32_t vec = tile_bytes >> 4;
        for (uint32_t i = tid; i < vec; i += T)
            reinterpret_cast<uint4 *>(tile)[i] = reinterpret_cast<const uint4 *>(src)[i];
        for (uint32_t i = (vec << 4) + tid; i < tile_bytes; i += T) tile[i] = src[i];
    }
    __syncthreads();

    bool ended = false, won = false;
    int ep_ret_out = 0, ep_len_out = 0;
    if (env < n) {
        int32_t *w = a.st.words + env;
        int win_steps = w7 & 0xFFFF, reached = (w7 >> 16) & 1;
        uint32_t flags = w7 >> 24;
        uint8_t *row = tile + tid * cells;
        bool selected = true;
        if constexpr (IS_RESET) {
            if (a.mask) selected = a.mask[env] != 0;
            if (selected && a.first_call) ctr = 0;
        }
        EnvStream rng(a.p.seed, a.p.env_id_base + (uint64_t)env, BENG_STREAM_ENV, ctr);
        int rew = 0, term = 0;
        bool invalid = false;
        uint32_t rec = BENG_BUILDER_DELTA_NONE;  // DELTA: passes, failed builds, invalid actions change no cell

        // Rows start on 4-byte boundaries when G*G is a multiple of 4 (G even, e.g. the default 10): the three loops
        // over the row (clear, count empty cells, find the k-th empty cell) then run word-wise, 4 cells at a time.
        const bool wordwise = (cells & 3) == 0;
        uint32_t *row32 = reinterpret_cast<uint32_t *>(row);
        auto reset_env = [&]() {  // world_builder_env.py:99-123 + game_logic.py:33-57
            if (wordwise) { for (int i = 0; i < (cells >> 2); ++i) row32[i] = 0u; }
            else { for (int i = 0; i < cells; ++i) row[i] = 0; }
            food = 25; wood = 20; stone = 10; pop = 3; cap = 10;
            counts = 0; steps = 0; win_steps = 0; reached = 0; flags = 0; ep_ret = 0;
        };

        if constexpr (IS_RESET) {
            if (selected) reset_env();
        } else {
            if (a.p.autoreset_mode == BENG_AUTORESET_NEXT_STEP && (flags & BFLAG_NEEDS_RESET)) {
                reset_env();
                if constexpr (DELTA) rec = BENG_BUILDER_DELTA_CLEAR;
            } else if (act < 0 || act > 4) {
                invalid = true;  // the reference raises ValueError (:135-136); the env is left untouched
            } else {
                const int action = (int)act;
                steps += 1;
                // ---- GameLogic.execute_action, game_logic.py:59-123
                const int prev_pop = pop, prev_cap = cap;
                if (action != 0) {
                    bool ok = (action == FARM) ? wood >= 5 : (action == LUMBERYARD) ? stone >= 3
                            : (action == QUARRY) ? wood >= 5 : (wood >= 10 && stone >= 5);  // _can_afford_building
                    int n_empty = 0;
                    [[maybe_unused]] uint32_t emp[CELLS_T ? (CELLS_T / 4 + 7) / 8 : 1];  // bit c set <=> cell c is empty
                    if (ok) {
                        if constexpr (CELLS_T != 0) {
                            // Occupancy bitmap of the row, 4 cells per shared-memory word.  Cell values are 0..4, so
                            // adding 0x7F to every byte lane sets its top bit exactly when the cell is occupied (no
                            // carry between lanes); one multiply-high gathers the four top bits into a nibble.
                            // (The first version counted the empty cells in one pass over the row and searched the
                            // k-th in a second: 45 % of the kernel's instructions, issue slots 68 % busy.)
                            constexpr int NWORD = CELLS_T / 4, NMASK = (NWORD + 7) / 8;
                            uint32_t occ[NMASK];
#pragma unroll
                            for (int m = 0; m < NMASK; ++m) occ[m] = 0;
#pragma unroll
                            for (int i = 0; i < NWORD; ++i) {
                                const uint32_t top = (row32[i] + 0x7F7F7F7Fu) & 0x80808080u;  // bits 7, 15, 23, 31
                                const uint32_t nib = __umulhi(top, (1u << 25) | (1u << 18) | (1u << 11) | (1u << 4)) & 0xFu;
                                occ[i >> 3] |= nib << ((i & 7) * 4);
                            }
#pragma unroll
                            for (int m = 0; m < NMASK; ++m) {
                                const int bits = CELLS_T - 32 * m;  // cells covered by this word
                                emp[m] = ~occ[m] & (bits >= 32 ? 0xFFFFFFFFu : ((1u << (bits & 31)) - 1u));
                                n_empty += __popc(emp[m]);
                            }
                        } else if (wordwise) {  // __vcmpeq4: 0xFF in every byte lane that equals zero
                            for (int i = 0; i < (cells >> 2); ++i) n_empty += __popc(__vcmpeq4(row32[i], 0u)) >> 3;
                        } else {
                            for (int i = 0; i < cells; ++i) n_empty += (row[i] == 0);
                        }
                        ok = n_empty > 0;  // "No empty space", :133-134
                    }
                    if (ok) {
                        int idx = rng.randint(0, n_empty - 1);  // np.random.randint(n_empty), :137
                        int pos = 0;
                        if constexpr (CELLS_T != 0) {
                            constexpr int NMASK = (CELLS_T / 4 + 7) / 8;
                            uint32_t e = 0;
                            int cum = 0;
                            bool found = false;
#pragma unroll
                            for (int m = 0; m < NMASK; ++m) {  // the bitmap word that holds the idx-th empty cell
                                const int c = __popc(emp[m]);
                                if (!found && idx < cum + c) { e = emp[m]; pos = 32 * m; idx -= cum; found = true; }
                                cum += c;
                            }
                            int t = __popc(e & 0xFFFFu);  // the idx-th set bit of e (0-based), by halves
                            if (idx >= t) { idx -= t; pos += 16; e >>= 16; }
                            t = __popc(e & 0xFFu);
                            if (idx >= t) { idx -= t; pos += 8; e >>= 8; }
                            t = __popc(e & 0xFu);
                            if (idx >= t) { idx -= t; pos += 4; e >>= 4; }
                            t = __popc(e & 0x3u);
                            if (idx >= t) { idx -= t; pos += 2; e >>= 2; }
                            if (idx >= (int)(e & 1u)) pos += 1;
                        } else if (wordwise) {
                            for (int i = 0; i < (cells >> 2); ++i) {
                                const uint32_t m = __vcmpeq4(row32[i], 0u);
                                const int c = __popc(m) >> 3;
                                if (idx < c) {  // the idx-th empty byte lane of this word (row-major = little-endian lanes)
                                    uint32_t lanes = m & 0x01010101u;  // one bit per empty lane
                                    for (int k = 0; k < idx; ++k) lanes &= lanes - 1;  // drop the first idx empty lanes
                                    pos = i * 4 + ((__ffs(lanes) - 1) >> 3);
                                    break;
                                }
                                idx -= c;
                            }
                        } else {
                            for (int i = 0; i < cells; ++i) {
                                if (row[i] == 0 && idx-- == 0) { pos = i; break; }
                            }
                        }
                        if (action == FARM) wood -= 5;
                        else if (action == LUMBERYARD) stone -= 3;
                        else if (action == QUARRY) wood -= 5;
                        else { wood -= 10; stone -= 5; }
                        row[pos] = (uint8_t)action;
                        if constexpr (DELTA) rec = (uint32_t)pos | ((uint32_t)action << 8);
                        counts += 1u << (8 * (action - 1));
                        if (action == HOUSE) cap += 5;
                        rew += (action == FARM) ? 3 : (action == HOUSE) ? 4 : 2;
                        if (action == HOUSE && prev_pop >= prev_cap - 1) rew += 10;
                    } else {
                        rew -= 3;
                    }
                }
                food += 2 * (int)(counts & 0xFF);            // _process_production
                wood += 3 * (int)((counts >> 8) & 0xFF);
                stone += 2 * (int)((counts >> 16) & 0xFF);
                if (food < pop) pop = 0; else food -= pop;   // _process_consumption
                if (pop > 0 && food > 2 && pop < cap) { pop += 1; food -= 1; }  // _process_population_growth
                if (pop > prev_pop) rew += 5;
                if (pop < prev_pop) rew -= 50;
                if (food > pop * 2) rew += 1;
                if (food < pop) rew -= 2;
                if (food < max(2, pop)) rew -= 5;
                if (abs(wood - stone) < 5) rew += 1;
                if (action == FARM && food > pop * 3) rew -= 1;
                // ---- world_builder_env.py:144-157
                if (pop >= 20 && !reached) reached = 1;
                if (reached) win_steps = min(win_steps + 1, 65535);
                term = (pop <= 0) || (reached && win_steps >= 50);
                if (term) rew = (pop <= 0) ? -100 : ((win_steps >= 50) ? 100 : -50);
                ep_ret += rew;
                if (term && a.p.autoreset_mode != BENG_AUTORESET_DISABLED) {
                    ended = true;
                    won = pop > 0;
                    ep_ret_out = ep_ret;
                    ep_len_out = steps;
                    if (a.io.ep_return) a.io.ep_return[env] = ep_ret;
                    if (a.io.ep_length) a.io.ep_length[env] = steps;
                    if (a.p.autoreset_mode == BENG_AUTORESET_SAME_STEP) {
                        reset_env();
                        if constexpr (DELTA) rec = BENG_BUILDER_DELTA_CLEAR;  // also undoes this step's build
                    } else {
                        flags |= BFLAG_NEEDS_RESET;
                    }
                }
            }
            a.io.reward[env] = (float)rew;
            if constexpr (DELTA) a.delta[env] = rec;
            a.io.terminated[env] = (uint8_t)term;
            if (a.io.truncated) a.io.truncated[env] = 0;
            if (invalid && a.io.invalid_count) atomicAdd(a.io.invalid_count, 1);
        }

        w[0] = food; w[n] = wood; w[2 * n] = stone; w[3 * n] = pop; w[4 * n] = cap;
        w[5 * n] = (int32_t)counts;
        w[6 * n] = steps;
        w[7 * n] = (int32_t)((uint32_t)win_steps | ((uint32_t)reached << 16) | (flags << 24));
        w[8 * n] = (int32_t)rng.ctr;
        w[9 * n] = ep_ret;
        // observation, world_builder_env.py:186-217
        if (a.io.resources)
            reinterpret_cast<float4 *>(a.io.resources)[env] = make_float4((float)food, (float)wood, (float)stone, (float)pop);
        if (a.io.capacity) a.io.capacity[env] = (float)cap;
        if (a.io.win_steps) a.io.win_steps[env] = win_steps;
        if (a.io.flat_obs) {
            float *frow = flat + (size_t)tid * FD;
            for (int i = 0; i < cells; ++i) frow[i] = (float)row[i];
            frow[cells] = (float)food; frow[cells + 1] = (float)wood; frow[cells + 2] = (float)stone;
            frow[cells + 3] = (float)pop; frow[cells + 4] = (float)cap; frow[cells + 5] = (float)win_steps;
        }
    }

    if constexpr (!IS_RESET) {
        if (a.io.stats) {
            const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
            if (done_mask) {
                const int sr = __reduce_add_sync(0xFFFFFFFFu, ended ? ep_ret_out : 0);
                const int sl = __reduce_add_sync(0xFFFFFFFFu, ended ? ep_len_out : 0);
                const int sw = __reduce_add_sync(0xFFFFFFFFu, (ended && won) ? 1 : 0);
                if ((tid & 31) == 0) {
                    atomicAdd(&s_stats[0], __popc(done_mask));
                    atomicAdd(&s_stats[1], sr);
                    atomicAdd(&s_stats[2], sl);
                    atomicAdd(&s_stats[3], sw);
                }
            }
        }
    }

    // ---- drain: grid tile in place, flattened observation tile if requested
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
        const uint32_t bulk = tile_bytes & ~15u;
        int8_t *dst = a.io.grid + first * cells;
        if (bulk) bulk_store_s2g(dst, tile, bulk);
        for (uint32_t i = bulk; i < tile_bytes; ++i) dst[i] = (int8_t)tile[i];
        if (a.io.flat_obs) {
            const uint32_t fbytes = (uint32_t)(n_here * FD * sizeof(float)), fbulk = fbytes & ~15u;
            float *fdst = a.io.flat_obs + first * FD;
            if (fbulk) bulk_store_s2g(fdst, flat, fbulk);
            for (uint32_t i = fbulk / 4; i < fbytes / 4; ++i) fdst[i] = flat[i];
        }
        bulk_commit();
        bulk_wait_read<0>();
    }
    if constexpr (!IS_RESET) {
        if (a.io.stats && tid < 4 && s_stats[tid] != 0)
            atomicAdd((unsigned long long *)&a.io.stats[tid], (unsigned long long)(long long)s_stats[tid]);
    }
}

constexpr int BUILDER_T = 64;  // envs (= threads) per CTA; same-box sweep at 1M envs: 64 -> 75.6 us, 128 -> 76.8, 256 -> 82.7

template <bool IS_RESET, bool DELTA = false>
int launch(const BArgs &a, cudaStream_t stream) {
    const int cells = a.p.grid_size * a.p.grid_size;
    size_t smem = ((size_t)BUILDER_T * cells + 15) & ~(size_t)15;
    if (a.io.flat_obs) smem += (size_t)BUILDER_T * (cells + 6) * sizeof(float);
    auto kern = cells == 100 ? builder_kernel<BUILDER_T, IS_RESET, 100, DELTA>
                             : builder_kernel<BUILDER_T, IS_RESET, 0, DELTA>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    return (int)launch_pdl(kern, dim3((unsigned)((a.n + BUILDER_T - 1) / BUILDER_T)), dim3(BUILDER_T), smem, stream, a);
}

int check(const beng_builder_params *p, const beng_builder_state *st, const beng_builder_io *io, int64_t n) {
    if (!p || !st || !io || n < 0 || !st->words || !io->grid) return BENG_ERR_BAD_ARG;
    if (((uintptr_t)io->grid & 15) || (io->resources && ((uintptr_t)io->resources & 15)) ||
        (io->flat_obs && ((uintptr_t)io->flat_obs & 15)))
        return BENG_ERR_BAD_ARG;
    if (p->autoreset_mode < 0 || p->autoreset_mode > 2) return BENG_ERR_BAD_ARG;
    if (p->grid_size < 2 || p->grid_size > 15) return BENG_ERR_UNSUPPORTED;
    return 0;
}

// beng_builder_step without its public name: `delta` non-null selects the DELTA kernel.
int step(const beng_builder_params *p, const beng_builder_state *st, const int64_t *actions_dev,
         const beng_builder_io *io, int64_t n_envs, uint32_t *delta, cudaStream_t stream) {
    if (int rc = check(p, st, io, n_envs)) return rc;
    if (!actions_dev || !io->reward || !io->terminated) return BENG_ERR_BAD_ARG;
    if ((uintptr_t)actions_dev & 7) return BENG_ERR_BAD_ARG;  // 64-bit action loads (int64, or float32 pairs)
    if (n_envs == 0) return 0;
    BArgs a{*p, *st, *io, (const long long *)actions_dev, nullptr, (long long)n_envs, 0, delta};
    return delta ? launch<false, true>(a, stream) : launch<false>(a, stream);
}

// The body of beng_builder_step_host (delta_dev / delta_host null) and beng_builder_step_host_delta (grid_host null):
// H2D(actions) -> step kernel (the DELTA one when delta_dev is set) -> D2H of the change records, the results and the
// grid, each skipped when its host pointer is null.
int step_host(const beng_builder_params *p, const beng_builder_state *st, int64_t *actions_dev,
              const beng_builder_io *io, int64_t n_envs, const int64_t *actions_host, uint32_t *delta_dev,
              uint32_t *delta_host, int8_t *grid_host, float *resources_host, float *capacity_host,
              int32_t *win_steps_host, float *reward_host, uint8_t *terminated_host, cudaStream_t s) {
    if (!actions_host || !actions_dev) return BENG_ERR_BAD_ARG;
    if (int rc = check(p, st, io, n_envs)) return rc;
    if ((resources_host && !io->resources) || (capacity_host && !io->capacity) || (win_steps_host && !io->win_steps))
        return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    const size_t n = (size_t)n_envs, cells = (size_t)p->grid_size * p->grid_size;
    cudaError_t e = cudaMemcpyAsync(actions_dev, actions_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    if (int rc = step(p, st, actions_dev, io, n_envs, delta_dev, s)) return rc;
    if (int rc = d2h(delta_host, delta_dev, n * sizeof(uint32_t), s)) return rc;
    if (int rc = d2h(reward_host, io->reward, n * sizeof(float), s)) return rc;
    if (int rc = d2h(terminated_host, io->terminated, n, s)) return rc;
    if (int rc = d2h(resources_host, io->resources, n * 4 * sizeof(float), s)) return rc;
    if (int rc = d2h(capacity_host, io->capacity, n * sizeof(float), s)) return rc;
    if (int rc = d2h(win_steps_host, io->win_steps, n * sizeof(int32_t), s)) return rc;
    return d2h(grid_host, io->grid, n * cells, s);
}

// Applies the records of envs [begin, end); false on a malformed record (its row and the rest of the range are left
// as they are).
bool apply_delta_range(const uint32_t *delta, int8_t *grid, int64_t begin, int64_t end, uint32_t cells) {
    for (int64_t e = begin; e < end; ++e) {
        const uint32_t r = delta[e];
        if (r == BENG_BUILDER_DELTA_NONE) continue;
        const uint32_t cell = r & 0xFFu, value = (r >> 8) & 7u;
        if ((r & 0x7FFFF800u) || value > 4 || (value ? cell >= cells : cell != 0)) return false;
        int8_t *row = grid + e * cells;
        if (r & BENG_BUILDER_DELTA_CLEAR) memset(row, 0, cells);
        if (value) row[cell] = (int8_t)value;
    }
    return true;
}

}  // namespace
}  // namespace beng

extern "C" {

int beng_builder_reset(const beng_builder_params *p, const beng_builder_state *st, const beng_builder_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (n_envs == 0) return 0;
    beng::BArgs a{*p, *st, *io, nullptr, mask_dev, (long long)n_envs, first_call};
    return beng::launch<true>(a, (cudaStream_t)stream);
}

int beng_builder_step(const beng_builder_params *p, const beng_builder_state *st, const int64_t *actions_dev,
                      const beng_builder_io *io, int64_t n_envs, void *stream) {
    return beng::step(p, st, actions_dev, io, n_envs, nullptr, (cudaStream_t)stream);
}

int beng_builder_step_host(const beng_builder_params *p, const beng_builder_state *st, int64_t *actions_dev,
                           const beng_builder_io *io, int64_t n_envs, const int64_t *actions_host, int8_t *grid_host,
                           float *resources_host, float *capacity_host, int32_t *win_steps_host, float *reward_host,
                           uint8_t *terminated_host, void *stream) {
    return beng::step_host(p, st, actions_dev, io, n_envs, actions_host, nullptr, nullptr, grid_host, resources_host,
                           capacity_host, win_steps_host, reward_host, terminated_host, (cudaStream_t)stream);
}

int beng_builder_step_host_delta(const beng_builder_params *p, const beng_builder_state *st, int64_t *actions_dev,
                                 const beng_builder_io *io, int64_t n_envs, const int64_t *actions_host,
                                 uint32_t *delta_dev, uint32_t *delta_host, float *resources_host, float *capacity_host,
                                 int32_t *win_steps_host, float *reward_host, uint8_t *terminated_host, void *stream) {
    if (!delta_dev || !delta_host || ((uintptr_t)delta_dev & 3) || ((uintptr_t)delta_host & 3)) return BENG_ERR_BAD_ARG;
    return beng::step_host(p, st, actions_dev, io, n_envs, actions_host, delta_dev, delta_host, nullptr,
                           resources_host, capacity_host, win_steps_host, reward_host, terminated_host,
                           (cudaStream_t)stream);
}

int beng_builder_apply_obs_delta(const uint32_t *delta_host, int8_t *grid_host, int64_t n_envs, int32_t grid_size,
                                 int32_t n_threads) {
    if (n_envs < 0 || (n_envs > 0 && (!delta_host || !grid_host))) return BENG_ERR_BAD_ARG;
    if (grid_size < 2 || grid_size > 15) return BENG_ERR_UNSUPPORTED;
    const uint32_t cells = (uint32_t)(grid_size * grid_size);
    const bool ok = beng::for_each_chunk(n_envs, n_threads, [=](int64_t b, int64_t e) {
        return beng::apply_delta_range(delta_host, grid_host, b, e, cells);
    });
    return ok ? 0 : BENG_ERR_BAD_ARG;
}

}  // extern "C"
