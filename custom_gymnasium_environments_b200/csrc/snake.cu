// Batched SnakeEnvClassic for sm_100a: step + reward + termination + auto-reset + food RNG +
// observation encoding in ONE kernel.
//
// Reference behaviour (paths relative to the reference root):
//   SnakeEnvClassic.reset            snake_env_classic/snake_env.py:49-65
//   SnakeEnvClassic.step             snake_env_classic/snake_env.py:67-119
//   SnakeEnvClassic._place_food      snake_env_classic/snake_env.py:121-129
//   SnakeEnvClassic._get_observation snake_env_classic/snake_env.py:131-143
//
// Two step kernels with the same dynamics, results and state (DESIGN.md sections 3 and 6e):
//   * snake_kernel (beng_snake_reset, beng_snake_step, the host-buffer calls) composes every
//     observation row in full, into any buffer;
//   * snake_patch_kernel (beng_snake_step_inplace) expects io.obs to hold the previous observation
//     and writes only what changes -- the 32-byte sectors around at most two cells per env, the whole
//     row on a reset; the previous row doubles as the occupancy map (see the kernel).
//
// snake_kernel:
//   * one THREAD per env does the integer dynamics out of a 16-byte state record (one LDG.128 /
//     STG.128 per env, perfectly coalesced);
//   * one CTA owns a TILE of T consecutive envs; their T x G*G observation bytes are contiguous in
//     global memory, so the tile is composed in shared memory (zero fill, scatter body cells, food
//     last) and drained with ONE bulk asynchronous copy (cp.async.bulk shared->global, the TMA
//     engine, SASS UBLKCP) issued by a single thread -- no per-thread obs stores in this kernel;
//   * CTAs are persistent over tiles with one tile buffer each; several CTAs per SM keep the copy
//     engine draining one CTA's tile while the others compose theirs;
//   * the shared-memory tile doubles as the O(1) occupancy map for self-collision and for the
//     food rejection loop (the reference scans a Python list for both);
//   * finished episodes are counted with warp votes, accumulated per CTA in shared memory and
//     flushed with one set of global atomics per CTA; a warp-aggregated compaction emits the
//     list of finished envs.
//
// Both are HBM-bound: snake_kernel moves 450 algorithmic bytes per env-step, 400 of them the
// observation write; snake_patch_kernel about 150 (DESIGN.md sections 6e and 6f).  There is nothing
// GEMM-shaped here and no tensor-core path is wanted.
#include <climits>
#include <cstdint>
#include <cstring>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {
namespace {

constexpr uint32_t FLAG_NEEDS_RESET = 1u;  // NEXT_STEP auto-reset bookkeeping
constexpr int FOOD_NONE = 255;             // board full: no food on the grid (see place_food)

// ---- 16-byte state record ---------------------------------------------------------------------
// Byte 0 of v.y: bits 0-1 `dir`, bits 2-3 `last_move` (the direction of the last step that moved the head), bit 4
// `tail_known` (last_move is valid).  A length-2 body is the head and the cell the head last moved from, so with
// tail_known its tail is head - delta(last_move) and the ring is not needed (see tail_of).  Deaths and invalid actions
// do not move the head and leave both fields as they are; a reset clears them.
constexpr uint32_t DIR_MASK = 3u, LAST_MOVE_SHIFT = 2, TAIL_KNOWN_BIT = 1u << 4;

struct Core {
    int head_r, head_c, food_r, food_c;
    int dir, last_move;
    bool tail_known;
    uint32_t flags;
    int length, steps, ring_head;
    uint32_t ctr;
};

__device__ __forceinline__ Core unpack(const uint4 v) {
    Core s;
    s.head_r = v.x & 0xFF;
    s.head_c = (v.x >> 8) & 0xFF;
    s.food_r = (v.x >> 16) & 0xFF;
    s.food_c = (v.x >> 24) & 0xFF;
    s.dir = v.y & DIR_MASK;
    s.last_move = (v.y >> LAST_MOVE_SHIFT) & DIR_MASK;
    s.tail_known = (v.y & TAIL_KNOWN_BIT) != 0;
    s.flags = (v.y >> 8) & 0xFF;
    s.length = (v.y >> 16) & 0xFFFF;
    s.steps = v.z & 0xFFFF;
    s.ring_head = (v.z >> 16) & 0xFFFF;
    s.ctr = v.w;
    return s;
}

__device__ __forceinline__ uint4 pack(const Core &s) {
    uint4 v;
    v.x = (uint32_t)s.head_r | ((uint32_t)s.head_c << 8) | ((uint32_t)s.food_r << 16) | ((uint32_t)s.food_c << 24);
    v.y = (uint32_t)s.dir | ((uint32_t)s.last_move << LAST_MOVE_SHIFT) | (s.tail_known ? TAIL_KNOWN_BIT : 0u) |
          (s.flags << 8) | ((uint32_t)s.length << 16);
    v.z = (uint32_t)s.steps | ((uint32_t)s.ring_head << 16);
    v.w = s.ctr;
    return v;
}

struct Args {
    uint4 *core;
    uint16_t *ring;
    const long long *actions;  // step only
    const uint8_t *mask;       // reset only (nullable)
    beng_snake_io io;
    long long n_envs;
    uint64_t seed, env_id_base;
    int G, max_steps, mode, first_call, tl_trunc;
    uint32_t *delta;  // DELTA step only: one BENG_OBS_DELTA record per env
};

// _place_food (snake_env.py:121-129): draw (row, col) until the cell is not part of the snake.
// `occupied(cell)` tells whether a cell holds part of the body; the callers answer it from an
// observation row in which every body cell holds 1 and no food is marked (the food is written
// afterwards), so the membership test is one byte load.  The reference never returns when the board
// is full (length == G*G, unreachable at G = 20 within 1000 steps); there the engine and the oracle
// both leave the board without food instead of spinning.
template <typename Occupied>
__device__ __forceinline__ void place_food(Core &s, EnvStream &rng, int G, Occupied occupied) {
    if (s.length >= G * G) {
        s.food_r = s.food_c = FOOD_NONE;
        return;
    }
    for (;;) {
        const int r = rng.randint(0, G - 1);
        const int c = rng.randint(0, G - 1);
        if (!occupied(r * G + c)) {
            s.food_r = r;
            s.food_c = c;
            return;
        }
    }
}

// The finished-env counter of this launch is io.done_count + done_counter(io).  Called after pdl_wait(), from every
// thread (contains a __syncthreads()); block 0 zeroes the other counter for the next launch.  With
// io.done_count_next == io.done_count the pointer is the self-managed block {count0, count1, parity, arrivals} of beng.h:
// this launch counts into count[parity], zeroes count[parity ^ 1] and flips the parity; otherwise the offset is 0 and the
// caller's two counters are used as they are.  (An offset rather than a pointer: it costs the register-bound patch kernel
// one register across its body instead of two.)
__device__ __forceinline__ uint32_t done_counter(const beng_snake_io &io) {
    uint32_t *const count = io.done_count;
    uint32_t parity = 0, *next = io.done_count_next;
    if (count && next == count) {
        parity = grid_uniform_advance(count + 2, count + 3, [](uint32_t p) { return p ^ 1u; });
        next = count + (parity ^ 1u);
    } else {
        __syncthreads();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && next) *next = 0;
    return parity;
}

// Row tests for place_food: a byte of the row (shared or global memory; the kernels write these rows themselves, so
// the loads are plain coherent ones).
__device__ __forceinline__ auto body_in(const uint8_t *row) {
    return [row](int cell) { return row[cell] != 0; };
}

// The state record of reset (snake_env.py:49-65): a length-1 snake in the centre.  (The ring is not touched: it only
// holds bodies of length >= 3.)
__device__ __forceinline__ void reset_core(Core &s, int G) {
    const int center = G / 2;
    s.head_r = s.head_c = center;
    s.dir = 1;
    s.last_move = 0;
    s.tail_known = false;
    s.length = 1;
    s.steps = 0;
    s.ring_head = 0;
    s.flags = 0;
}

// reset (snake_env.py:49-65).  Expects `row` to be all zero.
__device__ __forceinline__ void reset_env(Core &s, EnvStream &rng, uint8_t *row, int G) {
    reset_core(s, G);
    row[s.head_r * G + s.head_c] = 1;
    place_food(s, rng, G, body_in(row));
}

// Index of the tail entry in the ring (valid for length >= 3, and for a length-2 snake whose tail is not known).
__device__ __forceinline__ int tail_index(const Core &s, int cells) {
    const int idx = s.ring_head - (s.length - 1);
    return idx < 0 ? idx + cells : idx;
}

// The tail cell of a length >= 2 snake.  The ring holds bodies of length >= 3 only: a length-2 body is the head and the
// cell it last moved from, head - delta(last_move), which the state record holds once the snake has moved (tail_known).
// A length-2 state without the bit (a record written before the bit existed, or built by hand) keeps its tail in the
// ring, at tail_index; its next move sets the bit.
__device__ __forceinline__ int tail_of(const Core &s, const uint16_t *ring, int cells, int G) {
    if (s.length == 2 && s.tail_known) {
        const int d = s.last_move;  // 0 up, 1 right, 2 down, 3 left
        return (s.head_r - (d == 2) + (d == 0)) * G + s.head_c - (d == 1) + (d == 3);
    }
    return ring[tail_index(s, cells)];
}

// Walk the body oldest -> newest, writing `mark` into the tile row.  Returns the tail cell and
// reports whether `probe` is one of the body cells (`new_head in self.snake`, snake_env.py:93).
// Only called for length >= 2.  `pre_tail` >= 0 is the tail cell fetched one tile ahead; the newest
// entry always equals the head held in the state record, so a length-2 snake needs no ring load here
// beyond its tail's (none when tail_of finds the tail in the state record).
__device__ __forceinline__ int scan_body(const Core &s, const uint16_t *ring, uint8_t *row, int cells, int G,
                                         uint8_t mark, int probe, bool &hit, int pre_tail = -1) {
    int idx = tail_index(s, cells);
    const int tail = (pre_tail >= 0) ? pre_tail : tail_of(s, ring, cells, G);
    row[tail] = mark;
    hit |= (tail == probe);
    for (int i = 1; i < s.length - 1; ++i) {
        if (++idx == cells) idx = 0;
        const int c = ring[idx];
        row[c] = mark;
        hit |= (c == probe);
    }
    const int head = s.head_r * G + s.head_c;
    row[head] = mark;
    hit |= (head == probe);
    return tail;
}

// Observation change records (include/beng.h, BENG_OBS_DELTA_*), built from the state record alone.
__device__ __forceinline__ uint32_t delta_pair(int cell, int value) { return (uint32_t)cell | ((uint32_t)value << 12); }
__device__ __forceinline__ uint32_t food_pair(const Core &s, int G) {
    return s.food_r == FOOD_NONE ? BENG_OBS_DELTA_UNUSED : delta_pair(s.food_r * G + s.food_c, 2);
}
// After reset_env: the row was cleared, then the head and the food were written.
__device__ __forceinline__ uint32_t reset_record(const Core &s, int G) {
    return BENG_OBS_DELTA_CLEAR | delta_pair(s.head_r * G + s.head_c, 1) | (food_pair(s, G) << 14);
}

// Per-env inputs of one tile, loaded one tile ahead of their use (software pipeline).
struct Loaded {
    uint4 raw;
    long long act;
    bool selected;
};

// Draw the current body into a zeroed row (no move).
__device__ __forceinline__ void draw_body(const Core &s, const uint16_t *ring, uint8_t *row, int cells, int G) {
    bool hit = false;
    if (s.length == 1) row[s.head_r * G + s.head_c] = 1;
    else if (s.length > 1) scan_body(s, ring, row, cells, G, 1, -1, hit);
}

template <bool IS_RESET>
__device__ __forceinline__ Loaded load_inputs(const Args &a, long long env) {
    Loaded l;
    l.raw = make_uint4(0, 0, 0, 0);
    l.act = 0;
    l.selected = true;
    if (env < a.n_envs) {
        l.raw = ld_stream_u4(a.core + env);
        if constexpr (!IS_RESET) l.act = ld_stream_s64(a.actions + env);
        else if (a.mask) l.selected = a.mask[env] != 0;
    }
    return l;
}

// Adds the episodes of one warp's finished envs (done_mask = ballot of `ended`) to the CTA's counters
// s_stats = {n_episodes, sum_return, sum_length, sum_score, max_score}.
__device__ __forceinline__ void add_warp_stats(int *s_stats, unsigned done_mask, bool ended, int ep_ret, int ep_len,
                                               int ep_score, int lane) {
    const int sr = __reduce_add_sync(0xFFFFFFFFu, ended ? ep_ret : 0);
    const int sl = __reduce_add_sync(0xFFFFFFFFu, ended ? ep_len : 0);
    const int ss = __reduce_add_sync(0xFFFFFFFFu, ended ? ep_score : 0);
    const int mx = __reduce_max_sync(0xFFFFFFFFu, ended ? ep_score : INT_MIN);
    if (lane == 0) {
        atomicAdd(&s_stats[0], __popc(done_mask));
        atomicAdd(&s_stats[1], sr);
        atomicAdd(&s_stats[2], sl);
        atomicAdd(&s_stats[3], ss);
        atomicMax(&s_stats[4], mx);
    }
}

// One set of global atomics per CTA for its counters (after a barrier that completes them).
__device__ __forceinline__ void flush_stats(int64_t *stats, const int *s_stats, int tid) {
    if (tid < 4) {
        if (s_stats[tid] != 0) atomicAdd((unsigned long long *)&stats[tid], (unsigned long long)(long long)s_stats[tid]);
    } else if (tid == 4) {
        if (s_stats[4] != INT_MIN) atomicMax((long long *)&stats[4], (long long)s_stats[4]);
    }
}

// OWNROW: every thread zero-fills its own env row with 16-byte stores (needs G*G % 16 == 0, and is
// bank-conflict free when G*G/16 is odd, e.g. G = 20: consecutive rows are 25 x 16 B apart so eight
// threads cover all 32 banks).  Otherwise the tile is zero-filled cooperatively + one more barrier.
// DELTA (step only): also store one change record per env to a.delta, describing how this step's
// observation row differs from the previous one.  It is assembled from the dynamics' registers (the
// cells a move, a meal or a reset wrote), never by reading the row back.
template <int T, bool IS_RESET, bool OWNROW, bool DELTA>
__global__ void __launch_bounds__(T) snake_kernel(const Args a) {
    extern __shared__ __align__(128) uint8_t buf[];  // the tile: T x G*G observation bytes
    __shared__ int s_stats[5];  // per-CTA, per-launch: n_episodes, sum_return, sum_length, sum_score, max_score

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int G = a.G;
    const int cells = G * G;
    const int tile_bytes = T * cells;  // multiple of 16 because T is
    const long long n_tiles = (a.n_envs + T - 1) / T;

    if (tid < 5) s_stats[tid] = (tid == 4) ? INT_MIN : 0;
    // PDL: let the next step's grid start becoming resident as this one drains, then wait for the PREVIOUS step's
    // grid to have completed and flushed before touching anything it wrote (state, counters).
    pdl_launch_dependents();
    pdl_wait();
    [[maybe_unused]] const uint32_t done_slot = done_counter(a.io);  // (a reset only zeroes the next counter)

    // deferred finished-env list entries of the previous tile (the global atomic's result is consumed one
    // iteration later so that its latency is off the critical path)
    unsigned pend_mask = 0, pend_base = 0;
    int pend_env = 0;

    Loaded cur = load_inputs<IS_RESET>(a, (long long)blockIdx.x * T + tid);
    // tail cell of this thread's env, fetched one tile ahead (-1: not fetched / not needed)
    int pre_tail = -1;
    if constexpr (!IS_RESET) {
        const long long env0 = (long long)blockIdx.x * T + tid;
        const Core c0 = unpack(cur.raw);
        if (env0 < a.n_envs && c0.length > 1) pre_tail = tail_of(c0, a.ring + env0 * cells, cells, G);
    }
    int it = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const long long env = tile * T + tid;
        const bool active = env < a.n_envs;

        // Prefetch the next tile's state + action into registers; consumed next iteration.
        const long long tile_next = tile + gridDim.x;
        Loaded nxt = cur;
        if (tile_next < n_tiles) nxt = load_inputs<IS_RESET>(a, tile_next * T + tid);

        if constexpr (!IS_RESET) {
            if (pend_mask) {  // warp-uniform
                const unsigned base = __shfl_sync(0xFFFFFFFFu, pend_base, 0);
                if (pend_mask & (1u << lane)) a.io.done_env[base + __popc(pend_mask & ((1u << lane) - 1u))] = pend_env;
                pend_mask = 0;
            }
        }

        // The bulk copy of the previous tile must have finished reading the buffer.
        if (it > 0) {
            if (tid == 0) bulk_wait_read<0>();
            __syncthreads();
        }
        uint8_t *row = buf + tid * cells;
        if constexpr (OWNROW) {
            uint4 *r16 = reinterpret_cast<uint4 *>(row);
            for (int i = 0; i < (cells >> 4); ++i) r16[i] = make_uint4(0, 0, 0, 0);
        } else {
            uint4 *buf16 = reinterpret_cast<uint4 *>(buf);
            for (int i = tid; i < (tile_bytes >> 4); i += T) buf16[i] = make_uint4(0, 0, 0, 0);
            __syncthreads();
        }

        // ---------------------------------------------------------------- per-env dynamics (smem + ring only)
        bool ended = false;
        int ep_ret = 0, ep_len = 0, ep_score = 0;
        float rew = 0.0f;
        int term = 0, trunc = 0;
        bool invalid = false;
        uint32_t rec = BENG_OBS_DELTA_NONE;  // DELTA: death and invalid actions change no cell
        Core s = unpack(cur.raw);
        if (active) {
            uint16_t *ring = a.ring + env * cells;
            if constexpr (IS_RESET) {
                if (cur.selected && a.first_call) s.ctr = 0;
            }
            EnvStream rng(a.seed, a.env_id_base + (uint64_t)env, BENG_STREAM_ENV, s.ctr);

            if constexpr (IS_RESET) {
                if (cur.selected) reset_env(s, rng, row, G);
                else draw_body(s, ring, row, cells, G);
            } else {
                const long long act = cur.act;
                if (a.mode == BENG_AUTORESET_NEXT_STEP && (s.flags & FLAG_NEEDS_RESET)) {
                    reset_env(s, rng, row, G);  // action ignored, reward 0, not terminated
                    if constexpr (DELTA) rec = reset_record(s, G);
                } else if (act < 0 || act > 3) {
                    // The reference raises ValueError (snake_env.py:69-70); here the env is left
                    // untouched and the event is counted for the host to raise on.
                    invalid = true;
                    draw_body(s, ring, row, cells, G);
                } else {
                    const int action = (int)act;
                    int d = action - s.dir;
                    if (d < 0) d = -d;
                    if (d != 2) s.dir = action;  // reversal guard, snake_env.py:73-74
                    // 0 up, 1 right, 2 down, 3 left in (row, col), snake_env.py:77-85
                    const int nr = s.head_r + (s.dir == 2) - (s.dir == 0);
                    const int nc = s.head_c + (s.dir == 1) - (s.dir == 3);
                    const bool wall = (unsigned)nr >= (unsigned)G || (unsigned)nc >= (unsigned)G;  // :88-90
                    const int new_cell = wall ? -1 : nr * G + nc;
                    const int head_cell = s.head_r * G + s.head_c;
                    const int food_cell = (s.food_r == FOOD_NONE) ? -2 : s.food_r * G + s.food_c;

                    // A wall death under SAME_STEP returns the reset observation: the old body is
                    // never drawn, so the row stays clean for reset_env below.
                    const bool draw = !(wall && a.mode == BENG_AUTORESET_SAME_STEP);
                    bool self_hit = false;
                    int tail_cell = head_cell;
                    if (draw) {
                        if (s.length == 1) row[head_cell] = 1;  // (a length-1 snake cannot hit itself)
                        else tail_cell = scan_body(s, ring, row, cells, G, 1, new_cell, self_hit, pre_tail);  // :93, tail included
                    }
                    const bool died = wall || self_hit;
                    if (died) {
                        rew = -10.0f;  // :90 / :94 -- nothing but `direction` was mutated
                        term = 1;
                    } else {
                        const bool eat = new_cell == food_cell;
                        // insert(0, new_head), :97.  The ring is only maintained for length >= 3: a length-1
                        // body IS the head held in the state record, and a length-2 body the head and the cell
                        // it came from (last_move, see tail_of).  That spares ~98 % of the env-steps a scattered
                        // 2-byte store (a partial-sector write costs a DRAM read-modify-write).  The meal that
                        // makes length 3 writes all three entries, tail first, where tail_index finds them.
                        if (s.length > 2 || (s.length == 2 && eat)) {
                            if (s.length == 2) {
                                ring[s.ring_head] = (uint16_t)tail_cell;
                                if (++s.ring_head == cells) s.ring_head = 0;
                                ring[s.ring_head] = (uint16_t)head_cell;
                            }
                            if (++s.ring_head == cells) s.ring_head = 0;
                            ring[s.ring_head] = (uint16_t)new_cell;
                        }
                        row[new_cell] = 1;
                        s.head_r = nr;
                        s.head_c = nc;
                        s.last_move = s.dir;
                        s.tail_known = true;
                        if (eat) {  // :101-104
                            s.length += 1;
                            rew = 10.0f;
                            place_food(s, rng, G, body_in(row));
                        } else {
                            row[tail_cell] = 0;  // pop(), :107
                        }
                        // (new_cell != tail_cell: moving into the tail is a self-hit, so the two pairs never collide)
                        if constexpr (DELTA)
                            rec = eat ? delta_pair(new_cell, 1) | (food_pair(s, G) << 14)
                                      : delta_pair(tail_cell, 0) | (delta_pair(new_cell, 1) << 14);
                        s.steps = min(s.steps + 1, 65535);     // :109
                        if (s.steps >= a.max_steps) {
                            term = 1;              // :112-114, reported as terminated
                            trunc = a.tl_trunc;    // gym.make's TimeLimit would add truncated=True here
                        }
                    }
                    if (term && a.mode != BENG_AUTORESET_DISABLED) {
                        ended = true;
                        ep_score = s.length - 1;
                        ep_ret = 10 * ep_score - (died ? 10 : 0);
                        ep_len = s.steps + (died ? 1 : 0);  // the death step does not bump `steps`
                        if (a.mode == BENG_AUTORESET_SAME_STEP) {
                            if (draw) {  // un-draw the body so the row is clean again
                                // Self-hit death: the body is unchanged.  Time limit: the body is the moved one
                                // (new head and last_move in the state record, everything older in the ring).
                                bool hit = false;
                                if (s.length == 1) row[s.head_r * G + s.head_c] = 0;
                                else scan_body(s, ring, row, cells, G, 0, -1, hit);
                            }
                            reset_env(s, rng, row, G);
                            if constexpr (DELTA) rec = reset_record(s, G);
                        } else {
                            s.flags |= FLAG_NEEDS_RESET;
                        }
                    }
                }
            }
            if (s.food_r != FOOD_NONE) row[s.food_r * G + s.food_c] = 2;  // food written last, :139-141
            s.ctr = rng.ctr;
        }

        // ---------------------------------------------------------------- drain the tile
        fence_proxy_async_smem();  // this thread's generic-proxy smem writes -> visible to the copy engine
        __syncthreads();
        if (tid == 0) {
            const long long first = tile * T;
            const long long n_here = min((long long)T, a.n_envs - first);
            const uint32_t bytes = (uint32_t)(n_here * cells);
            const uint32_t bulk = bytes & ~15u;
            if (bulk) bulk_store_s2g(a.io.obs + first * cells, buf, bulk);
            bulk_commit();
            for (uint32_t i = bulk; i < bytes; ++i) a.io.obs[first * cells + i] = (int8_t)buf[i];  // ragged last tile
        }

        // ---------------------------------------------------------------- per-env outputs (off the critical path)
        if (active) {
            a.core[env] = pack(s);
            if constexpr (!IS_RESET) {
                a.io.reward[env] = rew;
                if constexpr (DELTA) a.delta[env] = rec;
                a.io.terminated[env] = (uint8_t)term;
                if (a.io.truncated) a.io.truncated[env] = (uint8_t)trunc;  // raw class: never truncates, :119
                if (invalid && a.io.invalid_count) atomicAdd(a.io.invalid_count, 1);
            }
            if (a.io.score) a.io.score[env] = s.length - 1;
            if (a.io.snake_length) a.io.snake_length[env] = s.length;
            if (ended) {
                if (a.io.ep_return) a.io.ep_return[env] = (float)ep_ret;
                if (a.io.ep_length) a.io.ep_length[env] = ep_len;
                if (a.io.ep_score) a.io.ep_score[env] = ep_score;
            }
        }

        // ---------------------------------------------------------------- episode-done compaction + stats
        if constexpr (!IS_RESET) {
            const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
            if (done_mask) {
                if (a.io.done_env) {
                    // one global atomic per warp reserves the slots; the slots are written next iteration
                    if (lane == 0) pend_base = atomicAdd(a.io.done_count + done_slot, (unsigned)__popc(done_mask));
                    pend_mask = done_mask;
                    pend_env = (int)env;
                }
                if (a.io.stats) add_warp_stats(s_stats, done_mask, ended, ep_ret, ep_len, ep_score, lane);
            }
        }
        // Fetch the next tile's tail cell now (its state record, requested at the top of this iteration, has
        // arrived by now) so that a dependent ring load is not exposed at the start of the next tile.
        if constexpr (!IS_RESET) {
            pre_tail = -1;
            if (tile_next < n_tiles) {
                const long long env_n = tile_next * T + tid;
                const Core cn = unpack(nxt.raw);
                if (env_n < a.n_envs && cn.length > 1) pre_tail = tail_of(cn, a.ring + env_n * cells, cells, G);
            }
        }
        cur = nxt;
    }

    if constexpr (!IS_RESET) {
        if (pend_mask) {
            const unsigned base = __shfl_sync(0xFFFFFFFFu, pend_base, 0);
            if (pend_mask & (1u << lane)) a.io.done_env[base + __popc(pend_mask & ((1u << lane) - 1u))] = pend_env;
        }
    }
    if (tid == 0) bulk_wait_read<0>();  // the copy engine has read every tile before the CTA's shared memory retires
    if constexpr (!IS_RESET) {
        if (a.io.stats) {
            __syncthreads();
            flush_stats(a.io.stats, s_stats, tid);
        }
    }
}

// Zero an observation row with the widest stores its alignment allows: 16-byte stores throughout when G*G % 16 == 0
// (io->obs is 16-byte aligned, so every row then starts on a 16-byte boundary), byte stores around them otherwise.
__device__ __forceinline__ void clear_row(uint8_t *row, int cells) {
    uint8_t *p = row, *const end = row + cells;
    while (((uintptr_t)p & 15) && p < end) *p++ = 0;
    for (; p + 16 <= end; p += 16) *reinterpret_cast<uint4 *>(p) = make_uint4(0, 0, 0, 0);
    while (p < end) *p++ = 0;
}

// reset (snake_env.py:49-65) of an env whose observation row lives in global memory: the row is cleared, then the
// head and the food are written, as a BENG_OBS_DELTA_CLEAR record describes it.  The food test needs no memory read:
// the only body cell is the head.
__device__ __forceinline__ void reset_row(Core &s, EnvStream &rng, uint8_t *row, int G) {
    clear_row(row, G * G);
    reset_core(s, G);
    const int head = s.head_r * G + s.head_c;
    row[head] = 1;
    place_food(s, rng, G, [head](int cell) { return cell == head; });
    row[s.food_r * G + s.food_c] = 2;  // (a length-1 snake always leaves room for food)
}

// Adds value `v` at byte `o` of 16 bytes held as four words (nothing when o is outside 0..15).
__device__ __forceinline__ void put_byte(uint32_t (&w)[4], int o, uint32_t v) {
    const uint32_t q = (uint32_t)o >> 2, bits = v << ((o & 3) * 8);
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] |= q == (uint32_t)j ? bits : 0u;
}

// Writes the 32-byte sector of `row` that starts at cell `start` (32-byte aligned, inside the row): the body cells `head`
// and `body` hold 1, `food` holds 2, every other byte 0.  Two 16-byte stores from one thread, each built just before it
// is stored: one 256-bit store needs all eight words live at once, which costs the kernel spills at its 40 registers.
__device__ __forceinline__ void store_sector(uint8_t *row, int start, int head, int body, int food) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int s16 = start + 16 * half;
        uint32_t w[4] = {0, 0, 0, 0};
        put_byte(w, head - s16, 1);
        put_byte(w, body - s16, 1);
        put_byte(w, food - s16, 2);
        *reinterpret_cast<uint4 *>(row + s16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// The observation writes of a step that neither dies nor resets, of a snake whose whole row is known in registers: a
// length-1 snake (move or meal) and a length-2 snake that does not eat.  The row afterwards is all zeros but for the
// head (1), the food (2) and, unless a length-1 snake moved, the old head (1).  Each 32-byte sector holding a changed
// cell -- `clear` -> 0 and head -> 1 on a move (`clear` is the old head of a length-1 snake, the tail of a length-2
// one), head -> 1 and food -> 2 on a length-1 meal (`clear` < 0) -- is written whole, once, instead of with byte
// stores.  A partly written sector costs a DRAM read of the sector before the write (DESIGN.md section 6b); a whole one
// does not.  A sector that reaches into a neighbouring env's row keeps the byte store, since that env's thread may be
// writing its own part of the sector.  The sector bounds come from the row's address: io.obs is only 16-byte aligned
// and G*G need not be a multiple of 32.
__device__ __forceinline__ void patch_known_row(uint8_t *row, int cells, int old_head, int clear, int head, int food) {
    const int mis = (int)((uintptr_t)row & 31);  // the row starts `mis` bytes past a sector boundary
    const bool ate = clear < 0;
    const int body = clear != old_head ? old_head : -1;
    const int a = ate ? head : clear, b = ate ? food : head;  // the two changed cells, and their new values:
    const uint8_t va = ate ? 1 : 0, vb = ate ? 2 : 1;
    const int sa = ((a + mis) & ~31) - mis, sb = ((b + mis) & ~31) - mis;  // first cell of their sectors
    const bool whole_a = sa >= 0 && sa + 32 <= cells, whole_b = sb >= 0 && sb + 32 <= cells;
    if (whole_a) store_sector(row, sa, head, body, food);
    else row[a] = va;
    if (whole_b) {
        if (sb != sa) store_sector(row, sb, head, body, food);
    } else {
        row[b] = vb;
    }
}

// 1536 resident threads per SM (<= 40 registers, no spills): the kernel is bound by the latency of its dependent rounds
// of loads (state + action, then, for a snake of length >= 3, the row byte + tail entry), so resident threads are what
// it runs on.  Measured on B200 at 1M envs, G = 20: 61.5 us per step against 65.8 us at the 5 x 256 threads per SM that
// 46 registers give.  Measured shape of the whole-sector writes (DESIGN.md section 6f): two 16-byte stores per sector,
// 55.6 us per step.  One 256-bit store per sector compiles to 46 registers without spills; not timed.  At the same 1536
// threads per SM, fewer and larger CTAs are faster, since every CTA pays a fixed prologue and epilogue (the parity read,
// the arrival, barriers, the statistics flush): 2 CTAs of 768 threads, the fewest that keep 1536 (DESIGN.md section 6i).
constexpr int PATCH_THREADS = 768, PATCH_CTAS_PER_SM = 2;

// The step kernel of beng_snake_step_inplace: same dynamics, rewards, flags, state and statistics as snake_kernel, but
// io.obs must already hold the observation of the previous reset or step, and only the cells that change are written
// (move: old tail -> 0, new head -> 1; eat: new head -> 1, new food -> 2; death / invalid action: nothing; reset: clear,
// head -> 1, food -> 2 -- the order of the BENG_OBS_DELTA records).  One thread per env and no shared-memory tile:
//   * the previous observation is the occupancy map, so self-collision (`new_head in self.snake`, tail included,
//     snake_env.py:93) is the byte obs[new_cell] == 1 instead of a walk over the ring (for length 2, new_cell == tail);
//     the ring is read only for the tail cell a move of a length >= 3 snake clears (a length-2 tail comes from the
//     state record, tail_of), and written only where snake_kernel writes it, so a length <= 2 step loads nothing but
//     the state record and the action;
//   * the food rejection loop after a meal of a length >= 3 snake reads the same row, with the new head already
//     written over the old food; shorter snakes test their two or three body cells in registers;
//   * a step that does not reset of a length-1 snake (about 91 % of env-steps at G = 20 with random actions), or a
//     non-eating move of a length-2 snake (about 6 %), writes the 32-byte sectors holding its changed cells whole, with
//     two 16-byte stores each (patch_known_row), and byte stores only where a sector reaches into a neighbouring row;
//     longer snakes, length-2 meals, deaths and resets keep the stores above;
//   * with the self-managed counter block, the launch's parity reverses the order of the CTAs' env tiles every other
//     launch, so the envs a step writes last are the ones the next step reads and rewrites first, while their state
//     records and observation sectors may still be in L2 (DESIGN.md section 6h); callers with their own two counters
//     keep the ascending order;
//   * the action tensor is read once per step and loaded with an L2 evict-first policy.
// The row loads are plain coherent loads (no .nc / __ldg / __restrict__): this kernel writes those bytes itself.
__global__ void __launch_bounds__(PATCH_THREADS, PATCH_CTAS_PER_SM) snake_patch_kernel(const Args a) {
    __shared__ int s_stats[5];  // per-CTA: n_episodes, sum_return, sum_length, sum_score, max_score
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int G = a.G;
    const int cells = G * G;

    if (tid < 5) s_stats[tid] = (tid == 4) ? INT_MIN : 0;
    pdl_launch_dependents();
    pdl_wait();  // the previous step's state, observations and counters are complete from here on
    const uint32_t done_slot = done_counter(a.io);
    const unsigned tile = done_slot ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
    // (32-bit index math, n_envs < 2^32: a 64-bit product costs this register-bound kernel a spill)
    const long long env = tile * PATCH_THREADS + tid;
    const bool active = env < a.n_envs;

    bool ended = false;
    int ep_ret = 0, ep_len = 0, ep_score = 0;
    if (active) {
        const long long act = ld_once_s64(a.actions + env);
        Core s = unpack(ld_stream_u4(a.core + env));
        uint8_t *row = reinterpret_cast<uint8_t *>(a.io.obs) + env * cells;
        uint16_t *ring = a.ring + env * cells;
        EnvStream rng(a.seed, a.env_id_base + (uint64_t)env, BENG_STREAM_ENV, s.ctr);
        float rew = 0.0f;
        int term = 0, trunc = 0;
        // `invalid` is settled before any branch and used after them all, so that the action load is issued together
        // with the state load instead of being sunk into the move branch, one memory round trip later
        const bool needs_reset = a.mode == BENG_AUTORESET_NEXT_STEP && (s.flags & FLAG_NEEDS_RESET);
        const bool invalid = !needs_reset && (act < 0 || act > 3);  // the env is left untouched (see snake_kernel)
        bool reset = needs_reset;  // action ignored, reward 0, not terminated
        int known_old_head = -1;   // >= 0: the row is written by patch_known_row, with this old head ...
        int known_clear = -1;      // ... and this cell cleared (< 0: a length-1 meal)
        if (!needs_reset && !invalid) {
            const int action = (int)act;
            int d = action - s.dir;
            if (d < 0) d = -d;
            if (d != 2) s.dir = action;  // reversal guard, snake_env.py:73-74
            const int nr = s.head_r + (s.dir == 2) - (s.dir == 0);
            const int nc = s.head_c + (s.dir == 1) - (s.dir == 3);
            const bool wall = (unsigned)nr >= (unsigned)G || (unsigned)nc >= (unsigned)G;  // :88-90
            const int new_cell = nr * G + nc;
            const int head_cell = s.head_r * G + s.head_c;
            const int food_cell = (s.food_r == FOOD_NONE) ? -2 : s.food_r * G + s.food_c;

            bool self_hit = false;  // (a length-1 snake cannot hit itself)
            int tail_cell = head_cell;
            if (!wall && s.length > 1) {
                // length 2: the tail from the state record (a ring load only for a record without tail_known);
                // length >= 3: the ring entry and the row byte, both loads issued before either is used
                tail_cell = tail_of(s, ring, cells, G);
                // a length-2 body is the head, which the new head never is, and the tail: no row load
                self_hit = s.length == 2 ? new_cell == tail_cell : row[new_cell] == 1;
            }
            const bool died = wall || self_hit;
            if (died) {
                rew = -10.0f;  // :90 / :94 -- nothing but `direction` was mutated, the row is unchanged
                term = 1;
            } else {
                const bool eat = new_cell == food_cell;
                if (s.length > 2 || (s.length == 2 && eat)) {  // insert(0, new_head), :97 (the lazy ring of snake_kernel)
                    if (s.length == 2) {
                        ring[s.ring_head] = (uint16_t)tail_cell;
                        if (++s.ring_head == cells) s.ring_head = 0;
                        ring[s.ring_head] = (uint16_t)head_cell;
                    }
                    if (++s.ring_head == cells) s.ring_head = 0;
                    ring[s.ring_head] = (uint16_t)new_cell;
                }
                s.head_r = nr;
                s.head_c = nc;
                s.last_move = s.dir;
                s.tail_known = true;
                const bool len1 = s.length == 1;
                const bool known = len1 || (s.length == 2 && !eat);
                if (known) {
                    known_old_head = head_cell;
                    known_clear = eat ? -1 : tail_cell;  // (a length-1 snake's tail_cell is its old head)
                }
                if (eat) {  // :101-104
                    // The rejection loop of a length-1 or length-2 snake tests the body cells it holds in registers
                    // (new head, old head, tail; a length-1 snake's tail_cell is its old head); a longer one reads
                    // the row, with the new head marked over the old food.  A length-1 snake leaves its row to
                    // patch_known_row.
                    const bool short_body = s.length <= 2;
                    if (!len1) row[new_cell] = 1;
                    s.length += 1;
                    rew = 10.0f;
                    place_food(s, rng, G, [=](int cell) {
                        return short_body ? cell == new_cell || cell == head_cell || cell == tail_cell : row[cell] != 0;
                    });
                    if (!len1 && s.food_r != FOOD_NONE) row[s.food_r * G + s.food_c] = 2;
                } else if (!known) {
                    row[tail_cell] = 0;  // pop(), :107
                    row[new_cell] = 1;
                }
                s.steps = min(s.steps + 1, 65535);  // :109
                if (s.steps >= a.max_steps) {
                    term = 1;  // :112-114, reported as terminated
                    trunc = a.tl_trunc;
                }
            }
            if (term && a.mode != BENG_AUTORESET_DISABLED) {
                ended = true;
                ep_score = s.length - 1;
                ep_ret = 10 * ep_score - (died ? 10 : 0);
                ep_len = s.steps + (died ? 1 : 0);  // the death step does not bump `steps`
                if (a.mode == BENG_AUTORESET_SAME_STEP) reset = true;
                else s.flags |= FLAG_NEEDS_RESET;
            }
        }
        if (reset) {
            reset_row(s, rng, row, G);
            known_old_head = -1;  // (set here rather than tested below: then it is not live across reset_row)
        }
        s.ctr = rng.ctr;

        a.core[env] = pack(s);
        a.io.reward[env] = rew;
        a.io.terminated[env] = (uint8_t)term;
        if (a.io.truncated) a.io.truncated[env] = (uint8_t)trunc;
        if (invalid && a.io.invalid_count) atomicAdd(a.io.invalid_count, 1);
        if (a.io.score) a.io.score[env] = s.length - 1;
        if (a.io.snake_length) a.io.snake_length[env] = s.length;
        if (ended) {
            if (a.io.ep_return) a.io.ep_return[env] = (float)ep_ret;
            if (a.io.ep_length) a.io.ep_length[env] = ep_len;
            if (a.io.ep_score) a.io.ep_score[env] = ep_score;
        }
        if (known_old_head >= 0)
            patch_known_row(row, cells, known_old_head, known_clear, s.head_r * G + s.head_c, s.food_r * G + s.food_c);
    }

    // episode-done compaction + statistics (as snake_kernel, without its one-tile deferral)
    const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
    if (done_mask) {
        if (a.io.done_env) {
            unsigned base = 0;
            if (lane == 0) base = atomicAdd(a.io.done_count + done_slot, (unsigned)__popc(done_mask));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (ended) a.io.done_env[base + __popc(done_mask & ((1u << lane) - 1u))] = (int)env;
        }
        if (a.io.stats) add_warp_stats(s_stats, done_mask, ended, ep_ret, ep_len, ep_score, lane);
    }
    if (a.io.stats) {
        __syncthreads();
        flush_stats(a.io.stats, s_stats, tid);
    }
}

__global__ void __launch_bounds__(256) snake_export_kernel(const uint4 *__restrict__ core,
                                                           const uint16_t *__restrict__ ring, long long n_envs, int G,
                                                           int *head_r, int *head_c, int *food_r, int *food_c, int *dir,
                                                           int *steps, int *length, uint32_t *ctr, int *body) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_envs) return;
    const Core s = unpack(core[e]);
    if (head_r) head_r[e] = s.head_r;
    if (head_c) head_c[e] = s.head_c;
    if (food_r) food_r[e] = (s.food_r == FOOD_NONE) ? -1 : s.food_r;
    if (food_c) food_c[e] = (s.food_c == FOOD_NONE) ? -1 : s.food_c;
    if (dir) dir[e] = s.dir;
    if (steps) steps[e] = s.steps;
    if (length) length[e] = s.length;
    if (ctr) ctr[e] = s.ctr;
    if (body) {  // newest -> oldest; a length-1 body and a length-2 one with tail_known are in the state record
        const int cells = G * G;
        const int head = s.head_r * G + s.head_c;
        const bool in_core = s.length == 1 || (s.length == 2 && s.tail_known);
        int idx = s.ring_head;
        for (int i = 0; i < cells; ++i) {
            int c = -1;
            if (i < s.length) c = !in_core ? (int)ring[e * cells + idx] : i == 0 ? head : tail_of(s, ring, cells, G);
            body[e * cells + i] = c;
            if (--idx < 0) idx = cells - 1;
        }
    }
}

// ---- launch configuration ---------------------------------------------------------------------
struct Config {
    int tile;  // envs (= threads) per CTA tile
    int ctas_per_sm;
};

// Measured on B200 at 1M envs, G = 20 (profiles/snake_r1_sweep.txt): every single-stage shape that keeps
// >= 2 CTAs resident per SM reaches the same ~11.5 G env-steps/s (the kernel is DRAM-bound), two-stage shapes
// with fewer CTAs are ~15 % slower.  So: one tile buffer per CTA, as many CTAs per SM as shared memory
// allows, and the largest tile that still gives every SM >= 2 tiles of work.
Config pick_config(int G, long long n_envs) {
    const long long cells = (long long)G * G;
    const long long budget = 200 * 1024;  // of 227 KB: leaves room for static smem + 1 KB/CTA reservation
    Config c{256, 2};
    const long long sms = device_sm_count();
    while (c.tile > 32 && (c.tile * cells * 2 > budget || (n_envs + c.tile - 1) / c.tile < 2 * sms)) c.tile >>= 1;
    c.ctas_per_sm = (int)(budget / (c.tile * cells));
    if (c.ctas_per_sm < 1) c.ctas_per_sm = 1;
    if (c.ctas_per_sm > 8) c.ctas_per_sm = 8;
    return c;
}

template <int T, bool IS_RESET, bool OWNROW, bool DELTA>
int launch_one(const Args &a, const Config &c, cudaStream_t stream) {
    const size_t smem = (size_t)T * a.G * a.G;
    auto kern = snake_kernel<T, IS_RESET, OWNROW, DELTA>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const long long n_tiles = (a.n_envs + T - 1) / T;
    long long grid = (long long)device_sm_count() * c.ctas_per_sm;
    if (grid > n_tiles) grid = n_tiles;
    return (int)launch_pdl(kern, dim3((unsigned)grid), dim3(T), smem, stream, a);
}

template <bool IS_RESET, bool DELTA = false>
int launch(const Args &a, cudaStream_t stream) {
    const Config c = pick_config(a.G, a.n_envs);
    const int cells = a.G * a.G;
    const bool ownrow = (cells % 16 == 0) && ((cells / 16) % 2 == 1);
#define BENG_CASE(TT)                                                                       \
    case TT:                                                                                \
        return ownrow ? launch_one<TT, IS_RESET, true, DELTA>(a, c, stream)                \
                      : launch_one<TT, IS_RESET, false, DELTA>(a, c, stream);
    switch (c.tile) {
        BENG_CASE(256) BENG_CASE(128) BENG_CASE(64) BENG_CASE(32)
    }
#undef BENG_CASE
    return BENG_ERR_UNSUPPORTED;
}

int check_common(const beng_snake_params *p, const beng_snake_state *st, const beng_snake_io *io, int64_t n_envs) {
    if (!p || !st || !io || !st->core || !st->ring || !io->obs || n_envs < 0) return BENG_ERR_BAD_ARG;
    if (p->grid_size < 2 || p->grid_size > 64) return BENG_ERR_UNSUPPORTED;
    if (p->max_steps < 1 || p->max_steps > 65535) return BENG_ERR_UNSUPPORTED;
    if (p->autoreset_mode < 0 || p->autoreset_mode > 2) return BENG_ERR_BAD_ARG;
    if (((uintptr_t)st->core & 15) || ((uintptr_t)io->obs & 15)) return BENG_ERR_BAD_ARG;
    if (io->done_env && !io->done_count) return BENG_ERR_BAD_ARG;
    if (io->done_count && io->done_count_next == io->done_count && ((uintptr_t)io->done_count & 15))
        return BENG_ERR_BAD_ARG;  // the self-managed counter block (beng.h)
    return 0;
}

Args make_args(const beng_snake_params *p, const beng_snake_state *st, const beng_snake_io *io, int64_t n_envs) {
    Args a{};
    a.core = (uint4 *)st->core;
    a.ring = st->ring;
    a.io = *io;
    a.n_envs = n_envs;
    a.seed = p->seed;
    a.env_id_base = p->env_id_base;
    a.G = p->grid_size;
    a.max_steps = p->max_steps;
    a.mode = p->autoreset_mode;
    a.tl_trunc = p->time_limit_truncation;
    return a;
}

// beng_snake_step without its public name: `delta` non-null selects the DELTA kernel, `in_place` the patch kernel.
int step(const beng_snake_params *p, const beng_snake_state *st, const int64_t *actions_dev, const beng_snake_io *io,
         int64_t n_envs, uint32_t *delta, bool in_place, cudaStream_t stream) {
    if (int rc = check_common(p, st, io, n_envs)) return rc;
    if (!actions_dev || !io->reward || !io->terminated) return BENG_ERR_BAD_ARG;
    if ((uintptr_t)actions_dev & 7) return BENG_ERR_BAD_ARG;  // 64-bit action loads (int64, or float32 pairs)
    if (n_envs == 0) return 0;
    Args a = make_args(p, st, io, n_envs);
    a.actions = (const long long *)actions_dev;
    if (in_place) {
        if (n_envs > (int64_t)UINT32_MAX) return BENG_ERR_UNSUPPORTED;  // the patch kernel's 32-bit env index
        const long long blocks = (n_envs + PATCH_THREADS - 1) / PATCH_THREADS;
        return (int)launch_pdl(snake_patch_kernel, dim3((unsigned)blocks), dim3(PATCH_THREADS), 0, stream, a);
    }
    if (delta) {
        a.delta = delta;
        return launch<false, true>(a, stream);
    }
    return launch<false>(a, stream);
}

// The body of beng_snake_step_host (delta_dev / delta_host null) and beng_snake_step_host_delta (obs_host null):
// H2D(actions) -> step kernel (the DELTA one when delta_dev is set) -> D2H of the change records, the results and the
// observations, each skipped when its host pointer is null.
int step_host(const beng_snake_params *p, const beng_snake_state *st, int64_t *actions_dev, const beng_snake_io *io,
              int64_t n_envs, const int64_t *actions_host, uint32_t *delta_dev, uint32_t *delta_host, int8_t *obs_host,
              float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, int32_t *score_host,
              int32_t *snake_length_host, cudaStream_t s) {
    if (!actions_host || !actions_dev) return BENG_ERR_BAD_ARG;
    if (int rc = check_common(p, st, io, n_envs)) return rc;
    if ((truncated_host && !io->truncated) || (score_host && !io->score) || (snake_length_host && !io->snake_length))
        return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    const size_t n = (size_t)n_envs, cells = (size_t)p->grid_size * p->grid_size;
    cudaError_t e = cudaMemcpyAsync(actions_dev, actions_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    if (int rc = step(p, st, actions_dev, io, n_envs, delta_dev, false, s)) return rc;
    if (int rc = d2h(delta_host, delta_dev, n * sizeof(uint32_t), s)) return rc;
    if (int rc = d2h(reward_host, io->reward, n * sizeof(float), s)) return rc;
    if (int rc = d2h(terminated_host, io->terminated, n, s)) return rc;
    if (int rc = d2h(truncated_host, io->truncated, n, s)) return rc;
    if (int rc = d2h(score_host, io->score, n * sizeof(int32_t), s)) return rc;
    if (int rc = d2h(snake_length_host, io->snake_length, n * sizeof(int32_t), s)) return rc;
    return d2h(obs_host, io->obs, n * cells, s);
}

// Applies the records of envs [begin, end); false on a malformed record (the rest of the range is left as it is).
bool apply_delta_range(const uint32_t *delta, int8_t *obs, int64_t begin, int64_t end, int cells) {
    for (int64_t e = begin; e < end; ++e) {
        const uint32_t r = delta[e];
        if (r == BENG_OBS_DELTA_NONE) continue;
        if (r & 0x70000000u) return false;
        int8_t *row = obs + e * cells;
        if (r & BENG_OBS_DELTA_CLEAR) memset(row, 0, (size_t)cells);
        for (const uint32_t pr : {r & 0x3FFFu, (r >> 14) & 0x3FFFu}) {
            const uint32_t cell = pr & 0xFFFu, value = pr >> 12;
            if (value == 3) continue;
            if (cell >= (uint32_t)cells) return false;
            row[cell] = (int8_t)value;
        }
    }
    return true;
}

}  // namespace
}  // namespace beng

extern "C" {

int beng_snake_launch_config(int32_t grid_size, int64_t n_envs, int32_t *tile, int32_t *stages, int32_t *ctas_per_sm) {
    if (grid_size < 2 || grid_size > 64 || n_envs < 0) return BENG_ERR_BAD_ARG;
    const beng::Config c = beng::pick_config(grid_size, n_envs);
    if (tile) *tile = c.tile;
    if (stages) *stages = 1;
    if (ctas_per_sm) *ctas_per_sm = c.ctas_per_sm;
    return 0;
}

size_t beng_snake_core_bytes(int64_t n_envs) { return n_envs < 0 ? 0 : (size_t)n_envs * 16; }

size_t beng_snake_ring_bytes(int64_t n_envs, int32_t grid_size) {
    return (n_envs < 0 || grid_size < 1) ? 0 : (size_t)n_envs * (size_t)grid_size * grid_size * sizeof(uint16_t);
}

int beng_snake_reset(const beng_snake_params *p, const beng_snake_state *st, const beng_snake_io *io,
                     const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream) {
    if (int rc = beng::check_common(p, st, io, n_envs)) return rc;
    if (n_envs == 0) return 0;
    beng::Args a = beng::make_args(p, st, io, n_envs);
    a.mask = mask_dev;
    a.first_call = first_call;
    return beng::launch<true>(a, (cudaStream_t)stream);
}

int beng_snake_step(const beng_snake_params *p, const beng_snake_state *st, const int64_t *actions_dev,
                    const beng_snake_io *io, int64_t n_envs, void *stream) {
    return beng::step(p, st, actions_dev, io, n_envs, nullptr, false, (cudaStream_t)stream);
}

int beng_snake_step_inplace(const beng_snake_params *p, const beng_snake_state *st, const int64_t *actions_dev,
                            const beng_snake_io *io, int64_t n_envs, void *stream) {
    return beng::step(p, st, actions_dev, io, n_envs, nullptr, true, (cudaStream_t)stream);
}

int beng_snake_step_host(const beng_snake_params *p, const beng_snake_state *st, int64_t *actions_dev,
                         const beng_snake_io *io, int64_t n_envs, const int64_t *actions_host, int8_t *obs_host,
                         float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, int32_t *score_host,
                         int32_t *snake_length_host, void *stream) {
    return beng::step_host(p, st, actions_dev, io, n_envs, actions_host, nullptr, nullptr, obs_host, reward_host,
                           terminated_host, truncated_host, score_host, snake_length_host, (cudaStream_t)stream);
}

int beng_snake_step_host_delta(const beng_snake_params *p, const beng_snake_state *st, int64_t *actions_dev,
                               const beng_snake_io *io, int64_t n_envs, const int64_t *actions_host,
                               uint32_t *delta_dev, uint32_t *delta_host, float *reward_host, uint8_t *terminated_host,
                               uint8_t *truncated_host, int32_t *score_host, int32_t *snake_length_host, void *stream) {
    if (!delta_dev || !delta_host || ((uintptr_t)delta_dev & 3) || ((uintptr_t)delta_host & 3)) return BENG_ERR_BAD_ARG;
    return beng::step_host(p, st, actions_dev, io, n_envs, actions_host, delta_dev, delta_host, nullptr, reward_host,
                           terminated_host, truncated_host, score_host, snake_length_host, (cudaStream_t)stream);
}

int beng_snake_apply_obs_delta(const uint32_t *delta_host, int8_t *obs_host, int64_t n_envs, int32_t grid_size,
                               int32_t n_threads) {
    if (n_envs < 0 || (n_envs > 0 && (!delta_host || !obs_host))) return BENG_ERR_BAD_ARG;
    if (grid_size < 2 || grid_size > 64) return BENG_ERR_UNSUPPORTED;
    if (n_envs == 0) return 0;
    const int cells = grid_size * grid_size;
    const bool ok = beng::for_each_chunk(n_envs, n_threads, [=](int64_t b, int64_t e) {
        return beng::apply_delta_range(delta_host, obs_host, b, e, cells);
    });
    return ok ? 0 : BENG_ERR_BAD_ARG;
}

int beng_snake_export_state(const beng_snake_params *p, const beng_snake_state *st, int64_t n_envs, int32_t *head_r,
                            int32_t *head_c, int32_t *food_r, int32_t *food_c, int32_t *direction, int32_t *steps,
                            int32_t *length, uint32_t *rng_counter, int32_t *body_cells_dev, void *stream) {
    if (!p || !st || !st->core || !st->ring || n_envs < 0) return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    const unsigned blocks = (unsigned)((n_envs + 255) / 256);
    beng::snake_export_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
        (const uint4 *)st->core, st->ring, (long long)n_envs, p->grid_size, head_r, head_c, food_r, food_c, direction,
        steps, length, rng_counter, body_cells_dev);
    return beng::finish_launch();
}

}  // extern "C"
