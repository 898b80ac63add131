// Batched TrafficManagementEnv for sm_100a: light control + light timers + vehicle spawn/route + queue processing +
// reward + termination + auto-reset + the (14*NI+4)-feature observation in ONE kernel.
//
// Reference behaviour (paths relative to the reference root, directory traffic_management_env/):
//   config.py:6-35                      constants
//   utils.py:71-118   TrafficLight      update / _advance_phase / can_pass / set_phase
//   utils.py:121-171  Intersection      queues, process_vehicles
//   utils.py:174-248  routes            generate_vehicle_route, neighbours (N,S,W,E), direction
//   environment.py:141-166 reset, :168-203 step, :205-220 _apply_actions, :222-249 _spawn_vehicles,
//   :251-285 update/process/remove, :287-311 _calculate_reward, :313-363 _get_observation
//
// Vehicles never move in the reference (SURVEY.md section 0 fact 9): a vehicle waits in its start intersection's
// queue until the light lets the whole queue go, then either leaves `self.vehicles` (its random route ended where
// it started) or stays there forever.  A queue is therefore exactly (length, sum of waiting times, loop-back
// count) and the env needs one more integer, len(self.vehicles).  All dynamics are integer; reward and
// observation are float64 expressions of those integers in the reference's operation order (np.var = NumPy's
// pairwise sums), cast to float32 -- bit-exact against the reference.
//
// One warp per three intersections, one lane per env, over [field][env] arrays (coalesced); the four queues of an
// intersection are byte lanes of two state words; the 32 x obs_dim float observation tile is composed in shared
// memory and drained with one bulk asynchronous copy (cp.async.bulk, UBLKCP).  HBM-bound on paper (~1.2 KB per
// env-step) and in practice at 1M envs (0.94 of the measured copy bandwidth); at the BASELINE 65,536 envs the grid is
// two waves of a tile whose serial chain is loads -> lights -> spawn -> queues -> reward, see the kernel comment.
#include <cstdint>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {
namespace {

constexpr int MAXNI = BENG_TRAFFIC_MAX_INTERSECTIONS;
constexpr uint32_t TFLAG_NEEDS_RESET = 1u;
enum { NS_GREEN = 0, NS_YELLOW = 1, EW_GREEN = 2, EW_YELLOW = 3 };
enum { NORTH = 0, EAST = 1, SOUTH = 2, WEST = 3 };

struct TArgs {
    beng_traffic_params p;
    beng_traffic_state st;
    beng_traffic_io io;
    const long long *actions;
    const uint8_t *mask;
    long long n;
    int ni, first_call;
    uint32_t inv_cols;  // ceil(2^16 / grid_cols): (start * inv_cols) >> 16 == start / grid_cols for start < 25
};

// (float)((double)a / (double)b) for non-negative integers.  When both are exactly representable in binary32 the
// correctly rounded binary32 quotient is the same number (rounding a binary64 quotient of two binary32 values to
// binary32 is innocuous: 53 >= 2*24+2), so the common case is one IEEE float division instead of an FP64 one.
__device__ __forceinline__ float ratio_f32(long long a, long long b) {
    if (a < (1 << 24) && b < (1 << 24)) return __fdiv_rn((float)(int)a, (float)(int)b);
    return (float)((double)a / (double)b);
}

// The env warp's view of the env stream: the first SPEC_BLOCKS Philox blocks at/after the step's starting counter
// are computed BEFORE barrier 1 (while the intersection warps wait for their loads) and parked in shared memory, so
// the spawn logic between barriers 1 and 2 -- which every intersection warp waits for -- is table look-ups.  Draws
// beyond the table (many lights turning green in one step) fall back to computing their block.
constexpr int SPEC_BLOCKS = 3;

__device__ __noinline__ uint32_t philox_draw(uint32_t idx, uint64_t env, uint64_t seed) {
    const Philox4 p = philox_block(idx >> 2, stream_key(env, BENG_STREAM_ENV, seed));
    const uint32_t l = idx & 3u;
    return l == 0 ? p.v[0] : l == 1 ? p.v[1] : l == 2 ? p.v[2] : p.v[3];
}

struct CachedStream : Draws<CachedStream> {
    uint32_t ctr;
    uint32_t first;          // index of the first cached draw (a multiple of 4)
    const uint32_t *cache;   // [SPEC_BLOCKS * 4][32] in shared memory, already offset by the lane
    uint64_t env, seed;
    __device__ __forceinline__ uint32_t u32() {
        const uint32_t idx = ctr++, rel = idx - first;
        if (rel < SPEC_BLOCKS * 4) return cache[rel * 32];
        return philox_draw(idx, env, seed);
    }
};

// generate_vehicle_route (utils.py:174-193) + get_direction_between_intersections (:230-248) reduced to what the
// dynamics use: the first hop's direction and whether the walk ends on its start.
template <typename Stream>
__device__ __forceinline__ void spawn_route(const TArgs &a, Stream &rng, int &start, int &dir, int &loopback) {
    const int rows = a.p.grid_rows, cols = a.p.grid_cols;
    start = rng.randint(0, a.ni - 1);
    const int route_length = rng.randint(2, a.ni < 5 ? a.ni : 5);
    const int row0 = (int)(((uint32_t)start * a.inv_cols) >> 16), col0 = start - row0 * cols;  // start / cols, start % cols
    int row = row0, col = col0;
    dir = NORTH;
    for (int h = 1; h < route_length; ++h) {
        // neighbours in the reference's order N, S, W, E (utils.py:206), bounds of the FULL grid (ids up to rows*cols-1)
        uint32_t m = (uint32_t)(row > 0) | ((uint32_t)(row + 1 < rows) << 1) | ((uint32_t)(col > 0) << 2) |
                     ((uint32_t)(col + 1 < cols) << 3);
        const int pick = rng.randint(0, __popc(m) - 1);  // random.choice(neighbors)
        m = pick > 0 ? m & (m - 1) : m;                   // drop the `pick` lowest candidates
        m = pick > 1 ? m & (m - 1) : m;
        m = pick > 2 ? m & (m - 1) : m;
        const int c = __ffs((int)m) - 1;                  // 0 N, 1 S, 2 W, 3 E
        row += (c == 1) - (c == 0);
        col += (c == 3) - (c == 2);
        if (h == 1) dir = (0x1320 >> (c * 4)) & 3;        // -> Direction ids NORTH 0, EAST 1, SOUTH 2, WEST 3
    }
    loopback = row == row0 && col == col0;
}

// ---------------------------------------------------------------------------------------------------------------
// Per-intersection building blocks shared by the kernels below.  Written branch-free on the hot path: the profile of
// the first formulation showed ~500 warp-instructions per intersection, a third of them in divergent `if (cnt)` /
// `if (wipe)` regions executed with 2-4 live lanes, and another fifth in IEEE float divisions (the mean waiting time
// of every queue) that mostly took the slow path because the numerator was 0.
struct IxState {
    uint32_t l0, cnt4, lb4;  // light word; queue lengths / loop-back counts of the four directions, one byte each
    int passed, wait, qw[4];
};

__device__ __forceinline__ void load_ix(const TArgs &a, uint32_t i, uint32_t un, uint32_t e32, bool ok, IxState &s) {
    s.l0 = 0; s.cnt4 = 0; s.lb4 = 0; s.passed = 0; s.wait = 0;
#pragma unroll
    for (int d = 0; d < 4; ++d) s.qw[d] = 0;
    if (ok) {
        s.l0 = a.st.light[i * un + e32];
        s.passed = a.st.passed[i * un + e32];
        s.wait = a.st.waiting[i * un + e32];
        s.cnt4 = a.st.qmeta[(i * 2) * un + e32];
        s.lb4 = a.st.qmeta[(i * 2 + 1) * un + e32];
#pragma unroll
        for (int d = 0; d < 4; ++d) s.qw[d] = a.st.qwait[(i * 4 + d) * un + e32];
    }
}

// _apply_actions (:205-220) + TrafficLight.update (utils.py:79-97) of one light; returns whether the light turned green
// and therefore draws randint(5, 30) (the caller places that draw in the env's stream, in light-id order).
__device__ __forceinline__ bool light_update(uint32_t l0, long long act, bool step, int &ph, int &tm) {
    ph = (int)(l0 & 0xFF);
    tm = (int)(l0 >> 8);
    const bool to_ns = step && act == 1 && ph != NS_GREEN;  // set_phase: MIN_PHASE_DURATION
    const bool to_ew = step && act == 2 && ph != EW_GREEN;
    ph = to_ns ? (int)NS_GREEN : to_ew ? (int)EW_GREEN : ph;
    tm = (to_ns || to_ew) ? 5 : tm;
    tm -= step ? 1 : 0;
    const bool adv = step && tm <= 0;                        // _advance_phase
    ph = adv ? (ph + 1) & 3 : ph;
    const bool yellow = adv && (ph & 1);
    tm = yellow ? 3 : tm;                                    // YELLOW_DURATION
    return adv && !(ph & 1);
}

// 1 / cnt for the mean waiting time of a queue: (float)((double)qw * rcp[cnt]) equals the reference's
// float32(qw / cnt) wherever the quotient is below 2^24 (a float32 rounding breakpoint is at least 2^-33 away from
// qw / cnt in relative terms when cnt <= 255, the product is within 2^-52), and both are clamped to 100 above that.
// rcp[0] = 0: an empty queue reports 0.  The table is a compile-time constant (IEEE division in the host compiler),
// staged into shared memory by every CTA.
struct RcpTable {
    double v[256];
    constexpr RcpTable() : v{} {
        for (int i = 1; i < 256; ++i) v[i] = 1.0 / (double)i;
    }
};
__device__ const RcpTable g_rcp_table{};

__device__ __forceinline__ void fill_rcp_table(double *rcp, int tid, int nthreads) {
    for (int i = tid; i < 256; i += nthreads) rcp[i] = g_rcp_table.v[i];
}

struct IxOut {
    int pas, wt, qsum, left;
};

// _process_intersections (:271-281, utils.py:141-163), _remove_completed_vehicles (:283-285), the state write-back
// (only words that changed) and the per-intersection features of the observation (:313-363) for intersection i of one
// env.  `spq` = 4 * intersection + direction of the vehicle spawned this step (-1: none), `wipe`: the env is being
// reset (fresh TrafficLight, empty queues, zero counters) -- the totals returned are those BEFORE the wipe, which is
// what the reward of a same-step auto-reset is computed from.
__device__ __forceinline__ IxOut process_ix(const TArgs &a, int NI, int i, uint32_t un, uint32_t e32, const IxState &s,
                                            int ph, int tm, bool stepping, bool wipe, int spq, int sp_lb, float *row,
                                            const double *rcp) {
    // The four queues of an intersection are stepped together on their packed byte lanes (N, E, S, W = lanes 0..3;
    // a lane never exceeds 255 because len(self.vehicles) <= 255): `go` lanes empty into vehicles_passed, `wait`
    // lanes add their length to the waiting times; byte sums are one dot-product instruction (dp4a) each.
    const bool go_ns = stepping && ph == NS_GREEN, go_ew = stepping && ph == EW_GREEN;      // can_pass
    const uint32_t gm = go_ns ? 0x00FF00FFu : go_ew ? 0xFF00FF00u : 0u;
    const uint32_t wm = stepping ? ~gm : 0u;
    const uint32_t hit = (spq >> 2) == i ? 1u << ((spq & 3) * 8) : 0u;  // add_vehicle_to_queue, waiting_time 0
    uint32_t cnt4 = s.cnt4 + hit, lb4 = s.lb4 + (sp_lb ? hit : 0u);
    const uint32_t wait4 = cnt4 & wm;                                   // every queued vehicle waits one more step
    const int pas = s.passed + (int)__dp4a(cnt4 & gm, 0x01010101u, 0u);  // the whole queue proceeds ...
    const int left = (int)__dp4a(lb4 & gm, 0x01010101u, 0u);             // ... loop-back vehicles leave self.vehicles
    const int wt = s.wait + (int)__dp4a(wait4, 0x01010101u, 0u);
    cnt4 &= ~gm;
    lb4 &= ~gm;
    const int qsum = (int)__dp4a(cnt4, 0x01010101u, 0u);
    // (observation rows are 8-byte aligned and every feature group starts on an even float: pairs go out as float2)
    int qw_new[4];
    float qlen[4], qmean[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const bool go = (d & 1) ? go_ew : go_ns;
        const int cnt = (int)((cnt4 >> (8 * d)) & 0xFFu);
        const int qw = go ? 0 : s.qw[d] + (int)((wait4 >> (8 * d)) & 0xFFu);
        qw_new[d] = qw;
        if (qw != s.qw[d]) a.st.qwait[(uint32_t)(i * 4 + d) * un + e32] = qw;
        qlen[d] = (float)min(cnt, 20);                                    // MAX_QUEUE_LENGTH
        qmean[d] = fminf((float)((double)qw * rcp[cnt]), 100.0f);         // mean waiting time, <= 100
    }
    float2 *row2 = reinterpret_cast<float2 *>(row);
    row2[(NI * 4 + i * 4) / 2] = make_float2(qlen[0], qlen[1]);
    row2[(NI * 4 + i * 4) / 2 + 1] = make_float2(qlen[2], qlen[3]);
    row2[(NI * 8 + i * 4) / 2] = make_float2(qmean[0], qmean[1]);
    row2[(NI * 8 + i * 4) / 2 + 1] = make_float2(qmean[2], qmean[3]);
    if (cnt4 != s.cnt4) a.st.qmeta[(uint32_t)(i * 2) * un + e32] = cnt4;
    if (lb4 != s.lb4) a.st.qmeta[(uint32_t)(i * 2 + 1) * un + e32] = lb4;
    const uint32_t nl = (uint32_t)ph | ((uint32_t)tm << 8);
    if (nl != s.l0) a.st.light[(uint32_t)i * un + e32] = (uint16_t)nl;
    if (pas != s.passed) a.st.passed[(uint32_t)i * un + e32] = pas;
    if (wt != s.wait) a.st.waiting[(uint32_t)i * un + e32] = wt;
    row2[i * 2] = make_float2(ph == 0 ? 1.0f : 0.0f, ph == 1 ? 1.0f : 0.0f);
    row2[i * 2 + 1] = make_float2(ph == 2 ? 1.0f : 0.0f, ph == 3 ? 1.0f : 0.0f);
    row2[NI * 6 + i] = make_float2((float)pas, (float)min(wt, 1000));
    if (wipe) {  // rare (episode boundaries): zero whatever the step left non-zero, observation of a fresh env
        if (cnt4) a.st.qmeta[(uint32_t)(i * 2) * un + e32] = 0;
        if (lb4) a.st.qmeta[(uint32_t)(i * 2 + 1) * un + e32] = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            if (qw_new[d]) a.st.qwait[(uint32_t)(i * 4 + d) * un + e32] = 0;
            row[NI * 4 + i * 4 + d] = 0.0f;
            row[NI * 8 + i * 4 + d] = 0.0f;
        }
        if (nl != NS_GREEN) a.st.light[(uint32_t)i * un + e32] = NS_GREEN;
        if (pas) a.st.passed[(uint32_t)i * un + e32] = 0;
        if (wt) a.st.waiting[(uint32_t)i * un + e32] = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) row[i * 4 + q] = q == NS_GREEN ? 1.0f : 0.0f;
        row[NI * 12 + i * 2] = 0.0f;
        row[NI * 12 + i * 2 + 1] = 0.0f;
    }
    return IxOut{pas, wt, qsum, left};
}

// The three float32 ratios of the global metrics.  (float)((double)a / (double)b) for non-negative integers; a == 0
// short-cuts the IEEE division's slow path.
__device__ __forceinline__ float ratio0_f32(long long a, long long b) { return a == 0 ? 0.0f : ratio_f32(a, b); }

// _calculate_reward (:287-311): CUMULATIVE counters, float64, the reference's order of additions; q[i * stride] is the
// queue total of intersection i (np.var: population variance over NumPy's pairwise sums).
template <int NI_T>
__device__ __forceinline__ double step_reward(int tot_passed, int tot_wait, int tot_queue, const int32_t *q, int stride,
                                              int NI) {
    double rew = 0.0;
    rew += (double)tot_passed * 1.0;
    rew += (double)tot_wait * -0.1;
    rew += (double)tot_queue * -0.05;
    if (NI > 1) {
        const double sum = np_sum_fn([&](int i) { return (double)q[i * stride]; }, NI);
        const double mean = NI_T ? div_const<NI_T ? NI_T : 1>(sum) : sum / (double)NI;
        const double ssq = np_sum_fn([&](int i) { const double dq = (double)q[i * stride] - mean; return dq * dq; }, NI);
        const double var = NI_T ? div_const<NI_T ? NI_T : 1>(ssq) : ssq / (double)NI;
        rew += 0.5 / (1 + var);
    }
    return rew;
}

// ---------------------------------------------------------------------------------------------------------------
// Step / reset kernel: one WARP per IPW intersections, one lane per env.
//
// (The first version of this kernel ran one thread per env: ~2,500 dependent instructions per thread, 198 registers,
// ~8 resident warps per SM and 31 % of its stall samples on instruction-cache misses; DESIGN.md section 8.)  A CTA
// of NW+1 warps owns 32 envs: warp w < NW steps intersections w*IPW .. w*IPW+IPW-1 of those envs (their [field][env]
// rows are read with fully coalesced requests; IPW independent chains per thread), warp NW is the env warp (spawn,
// reward, termination, counters).  The two roles run different code between the same CTA-wide barriers; what
// crosses intersections goes through shared memory:
//   barrier 1: which lights need a randint draw (one ballot word per intersection) -> every light knows the index
//              of its own draw in the env's Philox stream (counter-based, so any thread can compute any draw)
//   barrier 2: the vehicle spawned this step (env warp, after the light draws in stream order)
//   barrier 3: per-intersection passed / waiting / queue totals -> reward (env warp), global metrics (warp 0)
//   barrier 4: observation tile complete -> one bulk asynchronous copy per CTA
// Every intersection warp waits for the env warp between barriers 1-2 and 3-4, so the env warp's code there is kept
// short: its Philox blocks are computed ahead of barrier 1 (CachedStream), the global metrics are warp 0's, the two
// float64 divisions by NI of the variance are FMA sequences instead of the division subroutine (div_const).
constexpr int WPI_E = 32;  // envs per CTA
// The default grid (9 intersections) runs 3 intersections per warp, 4-warp CTAs capped at 72 registers (7 CTAs per SM,
// the 2048 CTAs of 65,536 envs are 1.98 waves).  Same-box sweeps, us per step at 65,536 / 1,048,576 envs (L2 flushed),
// (intersections per warp, registers): before the queues were packed (1, 40) 30.4 / 256, (2, 48) 29.7 / 263,
// (2, 56) 28.3-29.0 / 225-253, (2, 64) 28.1-28.5 / 250-258, (3, 64) 30.7 / 255, (3, 72) 28.2 / 223, (3, 80) 30.3 / 233;
// with packed queues (2, 56) 28.2 / 220, (2, 64) 28.3 / 229, (3, 56) 28.9 / 230, (3, 64) 27.7 / 234,
// **(3, 72) 26.3-27.8 / 217**, (5, 80) 30.8 / 292, (5, 96) 31.7 / 285, (9, 128) 36.0 / 372.
constexpr int TRAFFIC_MAXREG = 72;

template <int NI_T, int IPW, bool IS_RESET>
__global__ void __maxnreg__(TRAFFIC_MAXREG) traffic_step_kernel(const TArgs a) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int NI = NI_T ? NI_T : a.ni;
    const int NW = (NI + IPW - 1) / IPW;  // intersection warps; warp NW is the env warp
    const int OD = NI * 14 + 4;
    double *s_rcp = reinterpret_cast<double *>(smem_raw);                      // [256]
    float *tile = reinterpret_cast<float *>(s_rcp + 256);                     // [32][OD]
    int32_t *s_part = reinterpret_cast<int32_t *>(tile + WPI_E * OD);         // [4][NI][32]
    int32_t *s_spawn = s_part + 4 * NI * WPI_E;                               // [32]
    uint32_t *s_phx = reinterpret_cast<uint32_t *>(s_spawn + WPI_E);          // [SPEC_BLOCKS*4][32]
    uint32_t *s_need = s_phx + SPEC_BLOCKS * 4 * WPI_E;                        // [NI]
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n = a.n;
    const long long first = (long long)blockIdx.x * WPI_E;
    const long long env = first + lane;
    const bool active = env < n;
    const uint32_t un = (uint32_t)n, e32 = (uint32_t)env;
    float *row = tile + lane * OD;
    auto cta_barrier = [&]() { asm volatile("bar.sync 1, %0;" ::"r"((NW + 1) * 32) : "memory"); };
    pdl_launch_dependents();
    pdl_wait();

    uint32_t m0 = 0, ctr = 0;
    bool selected = true;
    if (active) {
        m0 = a.st.misc[e32];
        ctr = a.st.misc[2u * un + e32];
        if (IS_RESET && a.mask) selected = a.mask[env] != 0;
    }
    int timestep = m0 & 0xFFFF;
    uint32_t flags = m0 >> 16;
    const bool do_reset =
        active && (IS_RESET ? selected : (a.p.autoreset_mode == BENG_AUTORESET_NEXT_STEP && (flags & TFLAG_NEEDS_RESET)));
    if (IS_RESET && selected && a.first_call) ctr = 0;
    const bool stepping = !IS_RESET && !do_reset && active;
    if (stepping) timestep = min(timestep + 1, 65535);                                  // :170
    const bool term = stepping && timestep >= a.p.max_timesteps;                        // :196, reported as terminated
    const bool ended = term && a.p.autoreset_mode != BENG_AUTORESET_DISABLED;
    const bool same_step = ended && a.p.autoreset_mode == BENG_AUTORESET_SAME_STEP;
    const bool wipe = do_reset || same_step;

    if (w < NW) {
        // ================= intersection warp: intersections w*IPW .. w*IPW+IPW-1 of 32 envs =================
        const int i0 = w * IPW;
        IxState s[IPW];
        long long act[IPW];
        int phase[IPW], timer[IPW];
#pragma unroll
        for (int k = 0; k < IPW; ++k) {
            const int i = i0 + k;
            load_ix(a, (uint32_t)i, un, e32, active && i < NI, s[k]);
            act[k] = 0;
            if constexpr (!IS_RESET)
                if (active && i < NI) act[k] = a.actions[e32 * (uint32_t)NI + (uint32_t)i];
        }
        // (after the state loads have been issued: the copy's own load -> store round trip then runs beside theirs
        // instead of ahead of them -- 12 % of the stall samples when it came first)
        fill_rcp_table(s_rcp, threadIdx.x, (NW + 1) * 32);
        int spawn = -1;
        if constexpr (!IS_RESET) {
            bool need[IPW];
#pragma unroll
            for (int k = 0; k < IPW; ++k) {
                const int i = i0 + k;
                need[k] = light_update(s[k].l0, act[k], stepping && i < NI, phase[k], timer[k]);
                const unsigned nb = __ballot_sync(0xFFFFFFFFu, need[k]);
                if (lane == 0 && i < NI) s_need[i] = nb;
            }
            cta_barrier();  // barrier 1
#pragma unroll
            for (int k = 0; k < IPW; ++k) {
                if (need[k]) {  // lights draw in id order: this one's draw follows those of the lower ids
                    uint32_t before = 0;
                    for (int j = 0; j < i0 + k; ++j) before += (s_need[j] >> lane) & 1u;
                    EnvStream rng(a.p.seed, a.p.env_id_base + (uint64_t)env, BENG_STREAM_ENV, ctr + before);
                    timer[k] = rng.randint(5, 30);
                }
            }
            cta_barrier();  // barrier 2
            spawn = s_spawn[lane];
        } else {
#pragma unroll
            for (int k = 0; k < IPW; ++k) { phase[k] = s[k].l0 & 0xFF; timer[k] = (int)(s[k].l0 >> 8); }
            cta_barrier();  // the reciprocal table is complete
        }
        const int spq = spawn >= 0 ? (spawn & 0xFF) * 4 + ((spawn >> 8) & 0xFF) : -1, sp_lb = (spawn >> 16) & 1;
#pragma unroll
        for (int k = 0; k < IPW; ++k) {
            const int i = i0 + k;
            if (i >= NI) break;
            const IxOut o = process_ix(a, NI, i, un, e32, s[k], phase[k], timer[k], stepping, wipe, spq, sp_lb, row, s_rcp);
            s_part[(0 * NI + i) * WPI_E + lane] = o.pas;
            s_part[(1 * NI + i) * WPI_E + lane] = o.wt;
            s_part[(2 * NI + i) * WPI_E + lane] = o.qsum;
            s_part[(3 * NI + i) * WPI_E + lane] = o.left;
        }
        cta_barrier();  // barrier 3
        if (w == 0 && active) {
            // global metrics (utils.py:251-267, environment.py:352-361), off the env warp's critical path
            int tot_passed = 0, tot_wait = 0, tot_queue = 0;
            if (!wipe) {
                for (int j = 0; j < NI; ++j) {
                    tot_passed += s_part[(0 * NI + j) * WPI_E + lane];
                    tot_wait += s_part[(1 * NI + j) * WPI_E + lane];
                    tot_queue += s_part[(2 * NI + j) * WPI_E + lane];
                }
            }
            row[NI * 14 + 1] = fminf(ratio0_f32(tot_wait, tot_passed > 1 ? tot_passed : 1), 100.0f);
            row[NI * 14 + 2] = fminf(ratio0_f32(tot_queue, NI), 50.0f);
            row[NI * 14 + 3] = ratio0_f32(tot_passed, NI);
        }
    } else {
        // ================= env warp: spawn, reward, termination, counters =================
        int listed = 0;
        double total_reward = 0.0;
        if (active) {
            listed = (int)a.st.misc[un + e32];
            total_reward = a.st.total_reward[env];
        }
        fill_rcp_table(s_rcp, threadIdx.x, (NW + 1) * 32);
        if constexpr (!IS_RESET) {
            const uint64_t env_id = a.p.env_id_base + (uint64_t)env;
            const uint32_t blk0 = ctr >> 2;
            if (stepping) {
#pragma unroll
                for (int b = 0; b < SPEC_BLOCKS; ++b) {
                    const Philox4 ph = philox_block(blk0 + b, stream_key(env_id, BENG_STREAM_ENV, a.p.seed));
#pragma unroll
                    for (int k = 0; k < 4; ++k) s_phx[(b * 4 + k) * WPI_E + lane] = ph.v[k];
                }
            }
            cta_barrier();  // barrier 1
            uint32_t draws = 0;
            for (int j = 0; j < NI; ++j) draws += (s_need[j] >> lane) & 1u;
            ctr += draws;
            int spawn = -1;
            // _spawn_vehicles (:222-249)
            if (stepping && listed < a.p.max_vehicles) {
                CachedStream rng{{}, ctr, blk0 << 2, s_phx + lane, env_id, a.p.seed};
                if (rng.random53() < a.p.spawn_rate) {
                    int sp_i, sp_d, sp_lb;
                    spawn_route(a, rng, sp_i, sp_d, sp_lb);
                    listed += 1;
                    spawn = sp_i | (sp_d << 8) | (sp_lb << 16);
                }
                ctr = rng.ctr;
            }
            s_spawn[lane] = spawn;
            cta_barrier();  // barrier 2
        } else {
            cta_barrier();  // the reciprocal table is complete
        }
        // While the intersection warps process the queues: everything of the env's outputs that does not depend on them.
        const int ep_len = timestep;
        if (active) {
            if (wipe) { timestep = 0; flags = 0; }
            else if (ended) flags |= TFLAG_NEEDS_RESET;
            a.st.misc[e32] = (uint32_t)timestep | (flags << 16);
            a.st.misc[2u * un + e32] = ctr;
            if (a.io.timestep) a.io.timestep[env] = timestep;
            if constexpr (!IS_RESET) {
                a.io.terminated[env] = (uint8_t)term;
                if (a.io.truncated) a.io.truncated[env] = (uint8_t)(a.p.time_limit_truncation && term);  // raw class: 0, :197
                if (ended && a.io.ep_length) a.io.ep_length[env] = ep_len;
            }
        }
        cta_barrier();  // barrier 3

        // ---- _calculate_reward (:287-311); the intersection warps wait for this at barrier 4
        double st_ret = 0.0, st_len = 0.0;
        if (active) {
            int tot_passed = 0, tot_wait = 0, tot_queue = 0, left = 0;
            for (int i = 0; i < NI; ++i) {
                tot_passed += s_part[(0 * NI + i) * WPI_E + lane];
                tot_wait += s_part[(1 * NI + i) * WPI_E + lane];
                tot_queue += s_part[(2 * NI + i) * WPI_E + lane];
                left += s_part[(3 * NI + i) * WPI_E + lane];
            }
            double rew = 0.0;
            if (do_reset) {
                total_reward = 0.0;
                listed = 0;
            } else if (!IS_RESET) {
                listed -= left;
                rew = step_reward<NI_T>(tot_passed, tot_wait, tot_queue, s_part + 2 * NI * WPI_E + lane, WPI_E, NI);
                total_reward += rew;
            }
            if (ended) {
                st_ret = total_reward;
                st_len = (double)ep_len;
                if (a.io.ep_return) a.io.ep_return[env] = total_reward;
                if (same_step) {  // reset() draws nothing and its observation is a constant
                    total_reward = 0.0;
                    listed = 0;
                }
            }
            row[NI * 14 + 0] = (float)listed;  // len(self.vehicles); the other three global metrics: warp 0
            a.st.misc[un + e32] = (uint32_t)listed;
            a.st.total_reward[env] = total_reward;
            if constexpr (!IS_RESET) {
                a.io.reward[env] = (float)rew;
                if (a.io.reward64) a.io.reward64[env] = rew;
            }
        }
        if constexpr (!IS_RESET) {
            if (a.io.stats) {
                const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
                if (done_mask) {
                    double r = st_ret, l = st_len;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
                        l += __shfl_xor_sync(0xFFFFFFFFu, l, o);
                    }
                    if (lane == 0) {
                        atomicAdd(&a.io.stats[0], (double)__popc(done_mask));
                        atomicAdd(&a.io.stats[1], r);
                        atomicAdd(&a.io.stats[2], l);
                    }
                }
            }
        }
    }

    fence_proxy_async_smem();
    cta_barrier();  // barrier 4: the observation tile is complete
    if (threadIdx.x == 0) {
        const long long n_here = min((long long)WPI_E, n - first);
        const uint32_t bytes = (uint32_t)(n_here * OD * sizeof(float));
        const uint32_t bulk = bytes & ~15u;
        if (bulk) bulk_store_s2g(a.io.obs + first * OD, tile, bulk);
        bulk_commit();
        for (uint32_t i = bulk / 4; i < bytes / 4; ++i) a.io.obs[first * OD + i] = tile[i];  // ragged last tile
        bulk_wait_read<0>();
    }
}

template <int NI_T, int IPW, bool IS_RESET>
int launch_shape(const TArgs &a, cudaStream_t stream) {
    const int od = a.ni * 14 + 4, nw = (a.ni + IPW - 1) / IPW;
    const size_t smem = 256 * sizeof(double) + (size_t)WPI_E * od * sizeof(float) +
                        (size_t)(4 * a.ni * WPI_E + WPI_E + SPEC_BLOCKS * 4 * WPI_E + a.ni) * sizeof(int32_t);
    const unsigned grid = (unsigned)((a.n + WPI_E - 1) / WPI_E);
    auto kern = traffic_step_kernel<NI_T, IPW, IS_RESET>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    return (int)launch_pdl(kern, dim3(grid), dim3((nw + 1) * 32), smem, stream, a);
}

// The default grid's 9 intersections get their own instantiation; any other count runs one intersection per warp.
template <bool IS_RESET>
int launch(const TArgs &a, cudaStream_t stream) {
    return a.ni == 9 ? launch_shape<9, 3, IS_RESET>(a, stream) : launch_shape<0, 1, IS_RESET>(a, stream);
}

int check(const beng_traffic_params *p, const beng_traffic_state *st, const beng_traffic_io *io, int64_t n) {
    if (!p || !st || !io || n < 0) return BENG_ERR_BAD_ARG;
    if (!st->light || !st->passed || !st->waiting || !st->qmeta || !st->qwait || !st->misc || !st->total_reward ||
        !io->obs)
        return BENG_ERR_BAD_ARG;
    if ((uintptr_t)io->obs & 15) return BENG_ERR_BAD_ARG;
    if (p->grid_rows < 1 || p->grid_cols < 1 || p->num_intersections < 1) return BENG_ERR_BAD_ARG;
    if (p->autoreset_mode < 0 || p->autoreset_mode > 2) return BENG_ERR_BAD_ARG;
    const long long cells = (long long)p->grid_rows * p->grid_cols;
    const long long ni = p->num_intersections < cells ? p->num_intersections : cells;
    if (ni > MAXNI || p->max_vehicles < 0 || p->max_vehicles > 255) return BENG_ERR_UNSUPPORTED;
    if (p->max_timesteps < 1 || p->max_timesteps > 65535) return BENG_ERR_UNSUPPORTED;
    if (cells < 2) return BENG_ERR_UNSUPPORTED;  // a 1x1 grid has no neighbours to route to
    if ((unsigned long long)n * (unsigned long long)ni * 4ull >= (1ull << 32)) return BENG_ERR_UNSUPPORTED;  // 32-bit offsets
    return 0;
}

TArgs make_args(const beng_traffic_params *p, const beng_traffic_state *st, const beng_traffic_io *io, int64_t n) {
    TArgs a{};
    a.p = *p;
    a.st = *st;
    a.io = *io;
    a.n = n;
    const int cells = p->grid_rows * p->grid_cols;
    a.ni = p->num_intersections < cells ? p->num_intersections : cells;
    a.inv_cols = (65536u + (uint32_t)p->grid_cols - 1u) / (uint32_t)p->grid_cols;
    return a;
}

}  // namespace
}  // namespace beng

extern "C" {

int beng_traffic_reset(const beng_traffic_params *p, const beng_traffic_state *st, const beng_traffic_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (n_envs == 0) return 0;
    beng::TArgs a = beng::make_args(p, st, io, n_envs);
    a.mask = mask_dev;
    a.first_call = first_call;
    return beng::launch<true>(a, (cudaStream_t)stream);
}

int beng_traffic_step(const beng_traffic_params *p, const beng_traffic_state *st, const int64_t *actions_dev,
                      const beng_traffic_io *io, int64_t n_envs, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (!actions_dev || !io->reward || !io->terminated) return BENG_ERR_BAD_ARG;
    if ((uintptr_t)actions_dev & 7) return BENG_ERR_BAD_ARG;  // 64-bit action loads (int64, or float32 pairs)
    if (n_envs == 0) return 0;
    beng::TArgs a = beng::make_args(p, st, io, n_envs);
    a.actions = (const long long *)actions_dev;
    return beng::launch<false>(a, (cudaStream_t)stream);
}

int beng_traffic_step_host(const beng_traffic_params *p, const beng_traffic_state *st, int64_t *actions_dev,
                           const beng_traffic_io *io, int64_t n_envs, const int64_t *actions_host, float *obs_host,
                           float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, void *stream) {
    if (!actions_host || !actions_dev) return BENG_ERR_BAD_ARG;
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (truncated_host && !io->truncated) return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    const beng::TArgs a = beng::make_args(p, st, io, n_envs);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)n_envs;
    cudaError_t e = cudaMemcpyAsync(actions_dev, actions_host, n * a.ni * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    if (int rc = beng_traffic_step(p, st, actions_dev, io, n_envs, stream)) return rc;
    if (int rc = beng::d2h(reward_host, io->reward, n * sizeof(float), s)) return rc;
    if (int rc = beng::d2h(terminated_host, io->terminated, n, s)) return rc;
    if (int rc = beng::d2h(truncated_host, io->truncated, n, s)) return rc;
    return beng::d2h(obs_host, io->obs, n * (a.ni * 14 + 4) * sizeof(float), s);
}

}  // extern "C"
