// Batched CryptoTradingEnv for sm_100a: trade execution + regime-switching price walk + new candle +
// termination + auto-reset + the 261-feature observation (OHLCV window, portfolio, RSI, MACD, Bollinger,
// psychology) in ONE kernel.
//
// Reference behaviour (paths relative to the reference root, file crypto_trading_env/crypto_trading_env.py):
//   TradingConfig :28-38                 TechnicalIndicators.{rsi,bollinger_bands,macd,_ema} :41-119
//   MarketSimulator.generate_next_price :132-164, _update_market_regime :166-186, volatility :188-198,
//                   trend :200-211, _update_market_psychology :213-221
//   CryptoTradingEnv.reset :301-340, step :342-398, _execute_action :400-447, _execute_buy :449-476,
//                   _execute_sell :478-503, _get_observation :505-561
//
// Design (DESIGN.md section 7; the kernel's own comment below has the details):
//   * state arrays are [slot/field][env] (env fastest), open/high/low/volume as one 16-byte record per (slot, env),
//     so every access of a warp is contiguous and 64/128-bit wide;
//   * the window is a ring over 50 slots with ONE head shared by all envs (params.window_head, or the device word
//     io.window_head_dev that the step advances itself): a step overwrites the oldest slot, a reset rewrites all 50
//     slots in rotation -- heads never diverge between envs, so the layout stays coalesced whatever the episode
//     boundaries are;
//   * money, prices and market state are float64 in the reference's operation order; the closes are kept in float64
//     (the MACD is a difference of two EMAs of ~5e4-magnitude prices: float32 closes would break the 1e-5
//     tolerance); open/high/low/volume only feed the observation and are stored and normalised in float32;
//   * the window is streamed ONCE per step: the threads that normalise it into the observation tile also accumulate
//     the MACD / signal-line dot products and the close range, and hand the last 20 closes to the RSI / Bollinger code;
//   * the 32 x 261 float observation tile is contiguous in global memory: composed in shared memory (row
//     stride 261 words = conflict-free) and drained with one bulk asynchronous copy (cp.async.bulk, UBLKCP).
//
// HBM-bound: ~2.4 KB per env-step (window read 1.4 KB + observation write 1.04 KB); no tensor-core work.
#include <cuda.h>

#include <cfloat>
#include <cstdint>

#include "beng_common.cuh"
#include "beng_rng.cuh"

namespace beng {
namespace {

constexpr int HIST = BENG_CRYPTO_HISTORY;
constexpr int OBS = BENG_CRYPTO_OBS_DIM;
constexpr uint32_t CFLAG_NEEDS_RESET = 1u;

enum { BULL_RUN = 0, BEAR_MARKET = 1, SIDEWAYS = 2, CRASH = 3, RECOVERY = 4 };

struct CArgs {
    beng_crypto_params p;
    beng_crypto_state st;
    beng_crypto_io io;
    const void *actions;
    const uint8_t *mask;
    long long n;
    long long pitch;  // row pitch (envs) of the close / ohlv windows: n rounded up to a multiple of 32
    int first_call;
};

struct Market {
    int regime;
    double trend, psych;
};

__device__ __forceinline__ double vol_mult(int r) {  // :190-196
    return r == BULL_RUN ? 1.2 : r == BEAR_MARKET ? 1.5 : r == SIDEWAYS ? 0.8 : r == CRASH ? 3.0 : 2.0;
}
__device__ __forceinline__ double base_trend(int r) {  // :202-208
    return r == BULL_RUN ? 0.001 : r == BEAR_MARKET ? -0.001 : r == SIDEWAYS ? 0.0 : r == CRASH ? -0.005 : 0.002;
}
__device__ __forceinline__ double clipd(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }

// _update_market_regime, :166-186, given its two draws: `pick` = random.choice of the two successors, `r` = the
// random() behind random.uniform(lo, hi) for the new trend strength
__device__ __forceinline__ void apply_regime(Market &m, int pick, double r) {
    int nr;
    switch (m.regime) {
        case BULL_RUN: nr = pick ? CRASH : SIDEWAYS; break;
        case BEAR_MARKET: nr = pick ? RECOVERY : SIDEWAYS; break;
        case SIDEWAYS: nr = pick ? BEAR_MARKET : BULL_RUN; break;
        case CRASH: nr = pick ? BEAR_MARKET : RECOVERY; break;
        default: nr = pick ? SIDEWAYS : BULL_RUN; break;
    }
    m.regime = nr;
    double lo, hi;
    if (nr == BULL_RUN || nr == RECOVERY) lo = 0.5, hi = 1.0;
    else if (nr == BEAR_MARKET || nr == CRASH) lo = -1.0, hi = -0.5;
    else lo = -0.2, hi = 0.2;
    m.trend = lo + (hi - lo) * r;  // == uniform(lo, hi) of the RNG contract
}
template <typename RNG>
__device__ __forceinline__ void update_regime(Market &m, RNG &rng) {
    const int pick = rng.randint(0, 1);
    const double r = rng.random53();
    apply_regime(m, pick, r);
}

// The state-dependent part of generate_next_price (:132-164) + _update_market_psychology (:213-221), given the
// standard-normal deviate z behind np.random.normal(0, volatility) and volume_factor; same operation order as
// next_price() below (normal(mu, sd) = mu + sd * z in the RNG contract).
__device__ __forceinline__ double price_update(const beng_crypto_params &p, Market &m, double cur, double z,
                                               double volume_factor) {
    const double volatility = p.volatility_base * vol_mult(m.regime);
    const double drift = (m.psych - 0.5) * p.market_psychology_factor;
    const double trend = base_trend(m.regime) * m.trend;
    const double eps = 0.0 + volatility * z;
    const double pct = (trend + drift + eps) * volume_factor;
    const double np_ = clipd(cur * (1.0 + pct), p.min_price, p.max_price);
    m.psych += pct * 10.0;
    m.psych = clipd(m.psych, 0.0, 1.0);
    m.psych += (0.5 - m.psych) * 0.01;
    return np_;
}

// generate_next_price, :132-164, and _update_market_psychology, :213-221
template <typename RNG>
__device__ __forceinline__ double next_price(const beng_crypto_params &p, Market &m, RNG &rng, double cur,
                                             double volume) {
    if (rng.random53() < 0.01) update_regime(m, rng);
    const double u1 = rng.random53(), u2 = rng.random53();  // np.random.normal(0, volatility): Box-Muller, RNG contract
    const double z = box_muller(u1, u2);
    return price_update(p, m, cur, z, 1.0 / (1.0 + volume * 0.1));
}

__device__ __forceinline__ void store_candle(double *close_arr, float4 *ohlv_arr, long long n, long long env, int slot,
                                             double open, double high, double low, double close, double volume) {
    close_arr[(long long)slot * n + env] = close;
    ohlv_arr[(long long)slot * n + env] = make_float4((float)open, (float)high, (float)low, (float)volume);
}

// reset, :301-340: 50 warm-up candles from 50000.0; the newest lands in slot `head`.  Market state carries over.
// Deliberately NOT inlined (it runs once per 1000 steps) and deliberately BY VALUE: taking the address of the
// caller's market / RNG state or of the kernel parameter block would force them into local memory for every
// thread on the hot path (measured: 135 us of a 300 us step).
struct WarmupResult {
    Market m;
    uint32_t ctr;
    double last;  // the newest close of the new window
};
__device__ __noinline__ WarmupResult warmup_window(double *close_arr, float4 *ohlv_arr, long long n, long long env,
                                                   int head, beng_crypto_params p, Market m, uint64_t gid,
                                                   uint32_t ctr) {
    EnvStream rng(p.seed, gid, BENG_STREAM_ENV, ctr);
    double price = 50000.0;
    int slot = head + 1 == HIST ? 0 : head + 1;  // oldest
    for (int k = 0; k < HIST; ++k) {
        const double volume = rng.uniform(0.5, 2.0);
        price = next_price(p, m, rng, price, volume);
        const double high = price * rng.uniform(1.0, 1.02);
        const double low = price * rng.uniform(0.98, 1.0);
        const double open = price * rng.uniform(0.99, 1.01);
        store_candle(close_arr, ohlv_arr, n, env, slot, open, high, low, price, volume);
        slot = slot + 1 == HIST ? 0 : slot + 1;
    }
    return WarmupResult{m, rng.ctr, price};
}

// The same reset done by a whole WARP for ONE env (sparse in-step auto-resets: an episode that ends on `value >= 10 x
// initial` or `value <= 0`).  Run by one lane, the 50-candle warm-up is a ~90 us serial chain, and the step kernel ends
// when its slowest CTA does: a handful of resets per step doubled the step time.  Here the lanes draw and transform the
// random numbers of all 50 candles in parallel (lane l: candles l and l+32) -- Philox, Box-Muller, volume factor -- and
// only the short state chain (regime -> volatility -> price -> psychology, ~12 dependent float64 operations per candle)
// stays serial; every lane runs it redundantly, so nothing has to be broadcast afterwards.
// Draw positions: a candle consumes 14 words (volume 2, regime check 2, normal 4, high 2, low 2, open 2) plus 3 when
// its regime check fires (choice 1, trend 2), so candle k starts at ctr + 14 k + 3 * (changes before k).  The lanes start
// from "no change anywhere", find the first candle whose check fires, shift everything behind it by 3 words, and
// repeat (one extra pass per regime change: 0.5 on average).
// `stage` is 100 doubles of warp-private shared memory, element d at stage[(d >> 4) * stage_stride + (d & 15)].
// All 32 lanes call this with identical arguments.  Bit-identical to warmup_window() (tests: sparse-reset rollouts).
// 20 consecutive words of an env's stream, starting at the Philox block that holds draw `c`: five blocks computed up
// front, no "is my block cached?" branch per draw (lanes of a warp sit at different alignments, so the lazy EnvStream
// evaluated Philox up to once per draw: ~30 times per candle instead of 5).
struct WordWindow : Draws<WordWindow> {
    uint32_t w[20];  // (indexed by a per-lane position: lives in local memory; this is the rare reset path)
    uint32_t pos;
    __device__ __forceinline__ WordWindow(uint64_t seed, uint64_t env, uint32_t c) : pos(c & 3u) {
#pragma unroll
        for (int b = 0; b < 5; ++b) {
            const Philox4 r = philox_block((c >> 2) + b, stream_key(env, BENG_STREAM_ENV, seed));
#pragma unroll
            for (int q = 0; q < 4; ++q) w[4 * b + q] = r.v[q];
        }
    }
    __device__ __forceinline__ uint32_t u32() { return w[pos++]; }
};

__device__ __noinline__ WarmupResult coop_warmup_window(double *close_arr, float4 *ohlv_arr, long long n, long long env,
                                                        int head, beng_crypto_params p, Market m, uint64_t gid,
                                                        uint32_t ctr, double *stage, int stage_stride) {
    const int lane = threadIdx.x & 31;
    auto at = [&](int d) -> double & { return stage[(d >> 4) * stage_stride + (d & 15)]; };
    double volume[2], z[2], vf[2], uh[2], ul[2], uo[2], rt[2] = {0.0, 0.0};
    int pick[2] = {0, 0};
    bool fires[2] = {false, false};
    unsigned long long fired = 0;  // candles whose regime check fires; bits <= resolved are final
    int resolved = -1, changes = 0;  // candles <= resolved sit at their final draw positions; `changes` fired among them
    for (;;) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int k = lane + 32 * h;
            if (k < HIST && k > resolved) {  // (first pass: every candle; later: the ones behind the new change)
                WordWindow r(p.seed, gid, ctr + 14u * (uint32_t)k + 3u * (uint32_t)changes);
                volume[h] = r.uniform(0.5, 2.0);
                fires[h] = r.random53() < 0.01;
                if (fires[h]) {
                    pick[h] = r.randint(0, 1);
                    rt[h] = r.random53();
                }
                const double u1 = r.random53(), u2 = r.random53();
                z[h] = box_muller(u1, u2);
                vf[h] = 1.0 / (1.0 + volume[h] * 0.1);
                uh[h] = r.uniform(1.0, 1.02);
                ul[h] = r.uniform(0.98, 1.0);
                uo[h] = r.uniform(0.99, 1.01);
            }
        }
        fired = (unsigned long long)__ballot_sync(0xFFFFFFFFu, fires[0]) |
                ((unsigned long long)__ballot_sync(0xFFFFFFFFu, lane + 32 < HIST && fires[1]) << 32);
        const unsigned long long done = resolved < 0 ? 0ull : ((2ull << resolved) - 1ull);  // bits <= resolved
        const unsigned long long behind = fired & ~done;
        if (!behind) break;  // nothing fires behind the resolved prefix: every candle is final
        resolved = __ffsll((long long)behind) - 1;  // the first one that does (its own draws were at the right place)
        ++changes;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        if (k < HIST) {
            at(k) = z[h];
            at(HIST + k) = vf[h];
        }
    }
    __syncwarp();
    // The serial state chain, run redundantly by every lane (nothing to broadcast, nothing to synchronise inside the
    // loop); a lane keeps the closes of its own two candles as they go by.
    double price = 50000.0, c0 = 0.0, c1 = 0.0;
#pragma unroll 1
    for (int k = 0; k < HIST; ++k) {
        if ((fired >> k) & 1ull) {  // warp-uniform
            const int src = k & 31;
            const int pk = __shfl_sync(0xFFFFFFFFu, k < 32 ? pick[0] : pick[1], src);
            const double r = __shfl_sync(0xFFFFFFFFu, k < 32 ? rt[0] : rt[1], src);
            apply_regime(m, pk, r);
        }
        price = price_update(p, m, price, at(k), at(HIST + k));
        if (k == lane) c0 = price;
        if (k == lane + 32) c1 = price;
    }
    const int oldest = head + 1 == HIST ? 0 : head + 1;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        if (k < HIST) {
            const double c = h ? c1 : c0;
            int slot = oldest + k;
            slot = slot >= HIST ? slot - HIST : slot;
            store_candle(close_arr, ohlv_arr, n, env, slot, c * uo[h], c * uh[h], c * ul[h], c, volume[h]);
        }
    }
    __syncwarp();  // (the stage may be reused, and the caller's lanes read these stores after their own __syncwarp)
    return WarmupResult{m, ctr + 14u * HIST + 3u * (uint32_t)changes, price};
}

// Streaming (evict-first) loads of the window.  Plain weak loads are enough for data written earlier in the SAME CTA:
// bar.sync orders the global-memory accesses of the participating threads, and no other CTA touches this env's window.
__device__ __forceinline__ double ld_win_f64(const double *p) { return __ldcs(p); }
__device__ __forceinline__ float4 ld_win_f32x4(const float4 *p) { return __ldcs(p); }

// _execute_buy, :449-476.  Returns 1 when the order executed.
template <typename RNG>
__device__ __forceinline__ int do_buy(const beng_crypto_params &p, RNG &rng, double &cash, double &holdings,
                                      double amount, double price) {
    if (amount <= 0 || cash < amount) return 0;
    const double slippage = price * p.slippage_rate * rng.uniform(0.5, 1.5);
    const double effective = price + slippage;
    const double fee = amount * p.trading_fee_rate;
    const double net = amount - fee;
    cash -= amount;
    holdings += net / effective;
    return 1;
}

// _execute_sell, :478-503.  Returns 2 when the order executed.
template <typename RNG>
__device__ __forceinline__ int do_sell(const beng_crypto_params &p, RNG &rng, double &cash, double &holdings,
                                       double crypto_amount, double price) {
    if (crypto_amount <= 0 || holdings < crypto_amount) return 0;
    const double slippage = price * p.slippage_rate * rng.uniform(0.5, 1.5);
    const double effective = price - slippage;
    const double received = crypto_amount * effective;
    const double fee = received * p.trading_fee_rate;
    holdings -= crypto_amount;
    cash += received - fee;
    return 2;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------------------------
// The step kernels.  Work unit: 32 consecutive envs (unit u = envs [32u, 32u+32)); units are strided over the grid
// (u(q) = blockIdx + gridDim * q), so every persistent CTA gets the same number +-1.
//
// Per unit there are two stages:
//   DYNAMICS (dynamics_phase, one warp, lane = env): ONLY what feeds back into the state -- trade, Philox draws,
//            Box-Muller price step, candle, termination, auto-reset -- in the reference's float64 operation order.
//   OBSERVATION (compose_unit + finish_unit, 16 warps): the unit's window is streamed ONCE.  Thread (e = lane, g = warp)
//            takes slots k = g, g+16, g+32, g+48 of env e, normalises them into the 32 x 261 float tile and accumulates
//            its share of the indicator work on the way:
//              * MACD line, signal line: an EMA seeded with prices[0] is a LINEAR function of the window, and so is the
//                reference's EMA-of-MACD-history (:94-100); both are dot products of the 50 closes with constant weight
//                vectors (c_macd, built at compile time by running the reference's recurrences on unit vectors).  The
//                weights sum to zero, so the products are taken with (close - newest close), which is exact (Sterbenz)
//                and keeps the partial sums small.  The 16 partials per env meet in shared memory.
//              * max/min of the closes for the MACD normalisation: float32 max/min of (close - newest close); the range
//                is only a divisor of an observation feature (relative error 1.2e-7 against the allowed 1e-5).
//              * the last 20 closes (Bollinger window; its last 15 give the RSI deltas) are dropped into shared memory.
//            After one barrier, warps 0..3 finish MACD / RSI / Bollinger / portfolio features for the 32 envs with short
//            tree-shaped float64 sums and fast float32 quotients (nothing in this loop may CALL: a call spills whatever
//            is live across it), then one thread drains the tile with a bulk asynchronous copy (UBLKCP).
// What keeps the reference's exact float64 operation order: everything that feeds back into the state (cash, holdings,
// price walk, psychology, reward).  What does not: the 11 indicator features, float32 outputs checked at rtol 1e-5 /
// atol 1e-6 (tests/test_crypto_gpu.py); their error against the oracle is ~1e-7, and tests/test_crypto_features_gpu.py
// bounds it feature by feature.  A window of 20 identical closes (a price pinned at a clip bound) takes the reference's
// own arithmetic for the Bollinger features, bit for bit (bollinger_constant).  The float32 shortcuts hold for prices
// in [2^-100, 2^100], the domain check() enforces on the price bounds.
//
// In the step, the window comes in through the TMA: a ring of two 38.4 KB shared-memory stages filled by
// cp.async.bulk.tensor (one [50 slots][32 envs] box of the close tensor and one of the open/high/low/volume tensor per
// unit, completion on an mbarrier), so the next unit's window is in flight whatever the threads are doing.  What a box
// fetched early cannot contain is handled explicitly: the newest candle (written by the dynamics after the box may have
// been read) comes from shared memory, and a unit in which some env reset in this call (its whole window was rewritten)
// is re-read with ordinary loads.
//
// Two kernels run these stages:
//   crypto5_kernel (the step)  warp-specialised, 768 threads, one CTA per SM: 16 OBSERVATION warps (64 registers after
//       setmaxnreg.dec) and 8 DYNAMICS warps (112 registers after setmaxnreg.inc) that run up to 16 units ahead; a
//       dynamics warp hands its unit over through a slot of a 16-deep shared-memory ring (mbarriers ready[]/freed[]).
//       The ~13,000-cycle dependency chain of a unit's dynamics therefore never sits on the observation path
//       (in the bulk-synchronous kernel it was 29 % of the step, profiles/crypto_step_r2_ncu_summary.txt).
//   crypto4_kernel (reset())  bulk-synchronous, 512 threads: rounds of 16 units, all warps run the dynamics of the
//       round, then the observation stage of its units one after the other.  Every window is rewritten in this
//       launch, so it reads them back with ordinary loads: nothing to prefetch through the TMA or to run ahead of.
//       (Run as the step kernel it measures ~8 % slower than crypto5_kernel, DESIGN.md section 7.)
constexpr int C3_SUB = 32;      // envs per unit
constexpr int C3_RNGW = 20;     // Philox words per env-step: <= 3 (block offset) + 2 (slippage) + 2 + 2 + 3 + 4 + 2 + 2
constexpr int C3_LAST = 20;     // closes kept for Bollinger / RSI
constexpr int C3_COOP_MAX = 8;  // resets per warp up to which each one is rebuilt by the whole warp
constexpr int C3_TILE_BYTES = C3_SUB * OBS * (int)sizeof(float);
static_assert(C3_TILE_BYTES % 128 == 0, "tile buffers stay 128-byte aligned");
constexpr int TMA_STAGES = 2;  // measured: 2 stages = 3 stages (133 vs 136 us); the third one buys nothing
constexpr int OBS_WARPS = 16, OBS_T = OBS_WARPS * 32, OBS_PER = (HIST + OBS_WARPS - 1) / OBS_WARPS;
constexpr int STAGE_O = HIST * C3_SUB * 16, STAGE_C = HIST * C3_SUB * 8;  // bytes per stage: 25600 + 12800

struct MacdWeights {
    double wm[HIST];  // MACD line   = sum_k wm[k] * close[k]   (k = 0 oldest)
    double wg[HIST];  // signal line = sum_k wg[k] * close[k]
};
// Runs TechnicalIndicators.macd (:79-106) / _ema (:108-119) symbolically: wf[k], ws[k] are the coefficients of close[k]
// in the fast / slow EMA after consuming closes 0..t, sg[k] those of the signal line.
constexpr MacdWeights make_macd_weights() {
    MacdWeights w{};
    const double mf = 2.0 / 13.0, ms = 2.0 / 27.0, mg = 2.0 / 10.0;
    double wf[HIST] = {}, ws[HIST] = {}, sg[HIST] = {};
    wf[0] = 1.0;
    ws[0] = 1.0;
    for (int t = 1; t < HIST; ++t) {
        for (int k = 0; k < t; ++k) {
            wf[k] = wf[k] * (1.0 - mf);
            ws[k] = ws[k] * (1.0 - ms);
        }
        wf[t] = mf;
        ws[t] = ms;
        if (t == 25) {
            for (int k = 0; k < HIST; ++k) sg[k] = wf[k] - ws[k];
        } else if (t > 25) {
            for (int k = 0; k < HIST; ++k) sg[k] = (wf[k] - ws[k]) * mg + sg[k] * (1.0 - mg);
        }
    }
    for (int k = 0; k < HIST; ++k) {
        w.wm[k] = wf[k] - ws[k];
        w.wg[k] = sg[k];
    }
    return w;
}
constexpr MacdWeights k_macd_weights = make_macd_weights();
__constant__ MacdWeights c_macd = k_macd_weights;

// One env's pre-computed Philox words in shared memory (word j of thread t at w[j * NT]).
template <int NT>
struct TableStream : Draws<TableStream<NT>> {
    const uint32_t *w;
    uint32_t pos, ctr;
    __device__ __forceinline__ uint32_t u32() {
        const uint32_t v = w[pos * NT];
        ++pos;
        ++ctr;
        return v;
    }
};

// The dynamics of one 32-env unit `u`, run by ONE warp (lane = env), one thread per env, in the reference's float64
// operation order: trade, Philox draws, Box-Muller price step, candle, termination, auto-reset.  Writes the state, the
// per-step outputs and this step's candle, rebuilds the windows of envs that reset, and hands (newest close, cash,
// holdings, psychology, newest open/high/low/volume) to `handover` for the observation stage.
// The step's Philox words are computed up front -- five blocks, no data-dependent branch -- and parked in shared memory
// (`tbl` = this thread's column of a [20][NT] table), so a draw is one LDS at a running index instead of a divergent
// "is my block cached?" branch per draw.  `coop_stage` (100 doubles, element d at (d >> 4) * coop_stride + (d & 15),
// warp-private, may alias the warp's table rows) is the scratch of coop_warmup_window.  Returns the warp's reset mask.
template <bool IS_RESET, int NT, typename Handover>
__device__ __forceinline__ unsigned dynamics_phase(const CArgs &a, long long u, bool unit_ok, int head, uint32_t *tbl,
                                                   double *coop_stage, int coop_stride, Handover handover) {
    const int lane = threadIdx.x & 31;
    const long long n = a.n, pitch = a.pitch;
    const long long env = u * C3_SUB + lane;
    const bool active = unit_ok && env < n;
    const uint64_t gid = a.p.env_id_base + (uint64_t)env;
    bool ended = false, need_reset = false;
    double st_ret = 0.0, st_len = 0.0, st_val = 0.0;
    double cash = 0.0, holdings = 0.0, ep_ret = 0.0, rew = 0.0, value = 0.0, price_out = 0.0, cur = 1.0;
    Market m{SIDEWAYS, 0.0, 0.5};
    int step = 0, term = 0, trade = 0;
    uint32_t flags = 0, ctr = 0;
    bool step_at_limit = false;
    float4 newest = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // open, high, low, volume of this step's candle
    // ---- (a) state in, one step of the dynamics, termination decision
    if (active) {
        // requested together with the state: the old price and the action head the dependency chain
        double price_pre = 0.0;
        long long act_pre = 0;
        float2 actf_pre = make_float2(0.0f, 0.0f);
        if constexpr (!IS_RESET) {
            price_pre = a.st.close[(long long)(head == 0 ? HIST - 1 : head - 1) * pitch + env];  // the newest candle
            if (a.p.action_type == 1) actf_pre = reinterpret_cast<const float2 *>(a.actions)[env];
            else act_pre = reinterpret_cast<const long long *>(a.actions)[env];
        }
        const uint32_t meta = a.st.meta[env];
        ctr = a.st.meta[n + env];
        cash = a.st.scal[env];
        holdings = a.st.scal[n + env];
        m.trend = a.st.scal[2 * n + env];
        m.psych = a.st.scal[3 * n + env];
        step = meta & 0xFFFF;
        m.regime = (meta >> 16) & 0xFF;
        flags = meta >> 24;
        ep_ret = a.st.ep_return[env];
        if constexpr (IS_RESET) {
            need_reset = a.mask ? a.mask[env] != 0 : true;
            if (need_reset && a.first_call) {  // constructor: MarketSimulator.__init__, :125-130
                m.regime = SIDEWAYS;
                m.trend = 0.0;
                m.psych = 0.5;
                ctr = 0;
            }
        } else if (a.p.autoreset_mode == BENG_AUTORESET_NEXT_STEP && (flags & CFLAG_NEEDS_RESET)) {
            need_reset = true;  // the ring head moved by one slot with this call: whole window at the new rotation
        } else {
            TableStream<NT> rng{{}, tbl, ctr & 3u, ctr};
            {
                const uint32_t blk0 = ctr >> 2;
#pragma unroll
                for (int b = 0; b < C3_RNGW / 4; ++b) {
                    const Philox4 r = philox_block(blk0 + b, stream_key(gid, BENG_STREAM_ENV, a.p.seed));
#pragma unroll
                    for (int q = 0; q < 4; ++q) tbl[(4 * b + q) * NT] = r.v[q];
                }
            }
            // _execute_action, :400-447
            const double price = price_pre;
            const double initial_value = cash + holdings * price;
            // Order side and size first, then ONE inlined copy of each execution routine, so that lanes of a
            // warp holding different actions do not walk through separate copies one after the other.
            int side = 0;  // 1 = buy `amount` of cash, 2 = sell `amount` of crypto
            double amount = 0.0;
            if (a.p.action_type == 1) {  // :408-422
                const float2 act = actf_pre;
                const double buy = clipd((double)act.x, 0.0, 1.0) * (cash * 0.1);
                const double sell = clipd((double)act.y, 0.0, 1.0) * (holdings * 0.1);
                if (buy > sell && buy > 0) side = 1, amount = buy;
                else if (sell > 0) side = 2, amount = sell;
            } else {  // :424-436; anything outside 1..4 is a hold: the reference does not validate
                const long long act = act_pre;
                if (act == 1 || act == 2) side = 1, amount = cash * (act == 1 ? 0.05 : 0.2);
                else if (act == 3 || act == 4) side = 2, amount = holdings * (act == 3 ? 0.05 : 0.2);
            }
            if (side == 1) trade = do_buy(a.p, rng, cash, holdings, amount, price);
            else if (side == 2) trade = do_sell(a.p, rng, cash, holdings, amount, price);
            const double final_value = cash + holdings * price;
            rew = final_value - initial_value;  // valued at the OLD price, :440-441
            if (!trade) rew -= 1.0;             // :444-445
            // next candle, :348-365
            const double volume = rng.uniform(0.5, 2.0);
            const double new_price = next_price(a.p, m, rng, price, volume);
            const double high = new_price * rng.uniform(1.0, 1.02);
            const double low = new_price * rng.uniform(0.98, 1.0);
            store_candle(a.st.close, reinterpret_cast<float4 *>(a.st.ohlv), pitch, env, head, price, high, low,
                         new_price, volume);
            newest = make_float4((float)price, (float)high, (float)low, (float)volume);
            ctr = rng.ctr;
            cur = new_price;
            value = cash + holdings * new_price;
            price_out = new_price;
            step = min(step + 1, 65535);
            step_at_limit = step >= a.p.max_steps;
            term = step_at_limit || (value <= 0) || (value >= a.p.initial_balance * 10);  // :382-386
            ep_ret += rew;
            if (term && a.p.autoreset_mode != BENG_AUTORESET_DISABLED) {
                ended = true;
                st_ret = ep_ret;
                st_len = (double)step;
                st_val = value;
                if (a.io.ep_return_out) a.io.ep_return_out[env] = ep_ret;
                if (a.io.ep_length) a.io.ep_length[env] = step;
                if (a.p.autoreset_mode == BENG_AUTORESET_SAME_STEP) need_reset = true;
                else flags |= CFLAG_NEEDS_RESET;
            }
        }
    }
    // ---- (b) state, hand-over to phase 2 and per-step outputs of every env that does not reset in this call
    // (done BEFORE the resets so that nothing of the hot path is live across their calls)
    auto put_state = [&]() {
        handover(cur, cash, holdings, m.psych, newest);
        a.st.scal[env] = cash;
        a.st.scal[n + env] = holdings;
        a.st.scal[2 * n + env] = m.trend;
        a.st.scal[3 * n + env] = m.psych;
        a.st.meta[env] = (uint32_t)step | ((uint32_t)m.regime << 16) | (flags << 24);
        a.st.meta[n + env] = ctr;
        a.st.ep_return[env] = ep_ret;
    };
    if (active) {
        if constexpr (IS_RESET) {
            if (!need_reset) cur = a.st.close[(long long)head * pitch + env];  // not selected: window unchanged
        } else {
            a.io.reward[env] = (float)rew;
            a.io.terminated[env] = (uint8_t)term;
            if (a.io.truncated)
                a.io.truncated[env] = (uint8_t)(a.p.time_limit_truncation && term && step_at_limit);
            if (a.io.reward64) a.io.reward64[env] = rew;
            if (a.io.trade_kind) a.io.trade_kind[env] = (uint8_t)trade;
            if (ended || !need_reset) {  // (a NEXT_STEP reset reports the fresh episode's values below)
                if (a.io.portfolio_value) a.io.portfolio_value[env] = value;
                if (a.io.current_price) a.io.current_price[env] = price_out;
            }
        }
        if (!need_reset) put_state();
    }
    if constexpr (!IS_RESET) {
        if (a.io.stats) {
            const unsigned done_mask = __ballot_sync(0xFFFFFFFFu, ended);
            if (done_mask) {  // rare: a handful of envs per step
                const double r = warp_sum(st_ret), l = warp_sum(st_len), v2 = warp_sum(st_val);
                if (lane == 0) {
                    atomicAdd(&a.io.stats[0], (double)__popc(done_mask));
                    atomicAdd(&a.io.stats[1], r);
                    atomicAdd(&a.io.stats[2], l);
                    atomicAdd(&a.io.stats[3], v2);
                }
            }
        }
    }
    // ---- (c) resets (:301-340).  A few per warp: the whole warp rebuilds each window together (see
    // coop_warmup_window); many (reset(), or a batch whose episodes all end on the same step): one lane per env.
    const unsigned reset_mask = __ballot_sync(0xFFFFFFFFu, need_reset);
    if (reset_mask) {
        WarmupResult wr{m, ctr, cur};
        float4 *ohlv4 = reinterpret_cast<float4 *>(a.st.ohlv);
        if (IS_RESET || __popc(reset_mask) > C3_COOP_MAX) {
            if (need_reset) wr = warmup_window(a.st.close, ohlv4, pitch, env, head, a.p, m, gid, ctr);
        } else {
            __syncwarp();  // every lane is done with its Philox words: their shared-memory rows become the stage
            for (unsigned rest = reset_mask; rest; rest &= rest - 1) {
                const int src = __ffs(rest) - 1;
                Market ms;
                ms.regime = __shfl_sync(0xFFFFFFFFu, m.regime, src);
                ms.trend = __shfl_sync(0xFFFFFFFFu, m.trend, src);
                ms.psych = __shfl_sync(0xFFFFFFFFu, m.psych, src);
                const uint32_t ctr_s = __shfl_sync(0xFFFFFFFFu, ctr, src);
                const long long env_s = u * C3_SUB + src;
                const WarmupResult w1 = coop_warmup_window(a.st.close, ohlv4, pitch, env_s, head, a.p, ms,
                                                           a.p.env_id_base + (uint64_t)env_s, ctr_s, coop_stage, coop_stride);
                if (lane == src) wr = w1;
            }
        }
        if (need_reset) {
            cash = a.p.initial_balance;
            holdings = 0.0;
            step = 0;
            flags = 0;
            ep_ret = 0.0;
            m = wr.m;
            ctr = wr.ctr;
            cur = wr.last;
            put_state();
            if constexpr (!IS_RESET) {
                if (!ended) {  // NEXT_STEP: this call only delivers the reset observation
                    if (a.io.portfolio_value) a.io.portfolio_value[env] = cash;
                    if (a.io.current_price) a.io.current_price[env] = cur;
                }
            }
        }
    }
    return reset_mask;
}

// ---- mbarrier / TMA wrappers ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MBAR_DONE;\n"
        "bra MBAR_WAIT;\n"
        "MBAR_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// Same wait for a warp that expects to wait LONG (a dynamics warp running ahead of the observation warps): back off
// between polls so that the spin does not take issue slots from the warps doing the work.
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
        __nanosleep(256);
    }
}
// One [rows][box_w] box of a 2-D tensor (tensor map in kernel-parameter space) -> shared memory, completion on `bar`.
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int x, int y, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"((unsigned long long)map), "r"(x), "r"(y), "r"(bar)
        : "memory");
}
// Barrier over the 512 observation threads only (id 1; id 0 is __syncthreads over the whole CTA).
__device__ __forceinline__ void obs_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(OBS_T) : "memory"); }

// ---- the observation stage ---------------------------------------------------------------------------------------
struct ObsSmem {
    const float *stage_o;   // [50][32] x float4 : this unit's open/high/low/volume box
    const double *stage_c;  // [50][32]          : this unit's close box
    double *pm, *pg;        // [16][32] MACD-line / signal-line partials
    float *mx, *mn;         // [16][32] max / min of (close - newest close)
    double *last;           // [20][32] the last 20 closes
};

// 1 / cur without the division subroutine: float32 reciprocal + one Newton step in float64 (error ~4e-15).  For
// cur inside the accepted price domain (check(): (float)cur is normal and below __fdividef's 2^126 limit).
__device__ __forceinline__ double recip_price(double cur) {
    const double r = (double)__fdividef(1.0f, (float)cur);
    return __fma_rn(r, __fma_rn(-cur, r, 1.0), r);
}

// Thread (e, g): slots k = g + 16 i of env `env` -> tile row `dst`, partial sums -> shared memory.
// DIRECT: read the window with ordinary loads (a reset rewrote it in this call, or there is no TMA stage at all); a
// separate instantiation, so that the common path carries none of its (predicated-off, but still issued) instructions.
template <bool DIRECT>
__device__ __forceinline__ void compose_unit(const CArgs &a, const ObsSmem &sm, int e, int g, long long env,
                                             const int (&slot_of)[OBS_PER], uint32_t pitch32, double cur, float4 newest,
                                             float *dst) {
    const double inv_d = recip_price(cur);
    const float inv_f = (float)inv_d;
    const float4 *so = reinterpret_cast<const float4 *>(sm.stage_o);
    const float4 *go = reinterpret_cast<const float4 *>(a.st.ohlv) + env;
    const double *gc = a.st.close + env;
    double pm = 0.0, pg = 0.0;
    float mx = 0.0f, mn = 0.0f;  // (the newest close itself contributes 0)
#pragma unroll
    for (int i = 0; i < OBS_PER; ++i) {
        const int k = g + OBS_WARPS * i;
        if (k < HIST) {
            float4 x;
            double c;
            if constexpr (DIRECT) {
                x = ld_win_f32x4(go + (uint32_t)slot_of[i] * pitch32);
                c = ld_win_f64(gc + (uint32_t)slot_of[i] * pitch32);
            } else if (k == HIST - 1) {  // this step's candle: the box may have been fetched before it existed
                x = newest;
                c = cur;
            } else {
                x = so[slot_of[i] * C3_SUB + e];
                c = sm.stage_c[slot_of[i] * C3_SUB + e];
            }
            dst[k * 5 + 0] = x.x * inv_f;  // price_data / current_price, :513-515
            dst[k * 5 + 1] = x.y * inv_f;
            dst[k * 5 + 2] = x.z * inv_f;
            dst[k * 5 + 3] = (float)(c * inv_d);
            dst[k * 5 + 4] = x.w * inv_f;
            const double d = c - cur;
            pm = __fma_rn(c_macd.wm[k], d, pm);
            pg = __fma_rn(c_macd.wg[k], d, pg);
            const float df = (float)d;
            mx = fmaxf(mx, df);
            mn = fminf(mn, df);
            if (k >= HIST - C3_LAST) sm.last[(k - (HIST - C3_LAST)) * C3_SUB + e] = c;
        }
    }
    sm.pm[g * C3_SUB + e] = pm;
    sm.pg[g * C3_SUB + e] = pg;
    sm.mx[g * C3_SUB + e] = mx;
    sm.mn[g * C3_SUB + e] = mn;
}

template <typename F>
__device__ __forceinline__ double tree_sum16(F v) {  // sum of v(0..15), depth 4
    const double a0 = v(0) + v(1), a1 = v(2) + v(3), a2 = v(4) + v(5), a3 = v(6) + v(7);
    const double a4 = v(8) + v(9), a5 = v(10) + v(11), a6 = v(12) + v(13), a7 = v(14) + v(15);
    return ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// x / y in float64 for a positive normal y without the IEEE division subroutine, whose slow-path CALL must not appear in
// finish_unit (see the kernel comment): the hardware's approximate reciprocal as a seed, two Newton steps, and
// Markstein's final correction, which rounds the quotient correctly unless the exact one lies within a tiny fraction
// of an ulp of a rounding boundary; the float32 features cast from it cannot tell.
__device__ __forceinline__ double div_rn_inline(double x, double y) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));
    r = __fma_rn(r, __fma_rn(-y, r, 1.0), r);
    r = __fma_rn(r, __fma_rn(-y, r, 1.0), r);
    const double q = x * r;
    return __fma_rn(__fma_rn(-y, q, x), r, q);
}

// Features 257..259 of a window of 20 identical closes c, as the reference computes them (:64-77, np.mean / np.std of
// 20 copies).  NumPy's pairwise sum of 20 copies is exact for some c (100.0, 30000.0) and not for most others (1000.1):
// then sma != c and std > 0.  t = c - sma is a few ulps of c, so t^2 and the 20-term sum of squares are exact, std is
// |t| exactly, upper and lower are sma +- 2|t| exactly, and the features reduce to 0.75 / 0.25 / 0.5 (t > 0 / t < 0 /
// t == 0), 4|t| / sma and t / sma (tests/test_crypto_features.py holds NumPy to this closed form).  Short on purpose:
// even when it never runs, a longer branch here costs the step ~4 % (same-box A/B on a B200).
__device__ __forceinline__ void bollinger_constant(double c, float *dst) {
    // np_sum_fn over 20 copies, written out: the eight partial sums 2c and their tree (16c) are exact, the four
    // remaining additions round
    double s = c * 16.0;
    s = s + c; s = s + c; s = s + c; s = s + c;
    const double sma = div_const<20>(s);
    const double t = c - sma;
    const double q = div_rn_inline(t, sma);
    dst[257] = t > 0.0 ? 0.75f : (t < 0.0 ? 0.25f : 0.5f);
    dst[258] = (float)(4.0 * fabs(q));
    dst[259] = (float)q;
}

// Warps 0..3 (lane e = env): the 11 features behind the window, features 250..260 of row `dst`.
__device__ __forceinline__ void finish_unit(const ObsSmem &sm, int e, int g, float4 port, float *dst) {
    if (g == 0) {  // MACD(12, 26, 9) normalised by the close range, :538-547
        const double pm = tree_sum16([&](int q) { return sm.pm[q * C3_SUB + e]; });
        const double pg = tree_sum16([&](int q) { return sm.pg[q * C3_SUB + e]; });
        float mx = 0.0f, mn = 0.0f;
#pragma unroll
        for (int q = 0; q < OBS_WARPS; ++q) {
            mx = fmaxf(mx, sm.mx[q * C3_SUB + e]);
            mn = fminf(mn, sm.mn[q * C3_SUB + e]);
        }
        const float range = mx - mn;
        float f0 = 0.0f, f1 = 0.0f, f2 = 0.0f;
        if (range > 0.0f) {
            f0 = __fdividef((float)pm, range);
            f1 = __fdividef((float)pg, range);
            f2 = __fdividef((float)(pm - pg), range);
        }
        dst[254] = f0;
        dst[255] = f1;
        dst[256] = f2;
    } else if (g == 1) {  // RSI(14) over the last 14 deltas, :45-61; rsi/100 = gain / (gain + loss)
        const double *wl = sm.last + 5 * C3_SUB + e;  // the last 15 closes
        auto delta = [&](int i) { return wl[(i + 1) * C3_SUB] - wl[i * C3_SUB]; };
        const double sg = np_sum_fn([&](int i) { const double d = delta(i); return d > 0 ? d : 0.0; }, 14);
        const double sl = np_sum_fn([&](int i) { const double d = delta(i); return d < 0 ? -d : 0.0; }, 14);
        dst[253] = (sl != 0) ? __fdividef((float)sg, (float)(sg + sl)) : 1.0f;
    } else if (g == 2) {  // Bollinger(20, 2 sigma, population std), :64-77 and :550-554
        // Mean and variance of the DIFFERENCES to the newest close (exact subtractions), so the sums are 4-deep trees
        // instead of NumPy's 8-deep pairwise chains.  div_const, not `/`: the division subroutine's slow-path CALL
        // would force every value live across it -- the prefetched window of the next unit -- into local memory.
        // The variance goes to float32 scaled by a power of two to the price's magnitude (var / 4^e, cur / 2^e in
        // [1, 2)), so the band holds for every price of the accepted domain, and sd is scaled back exactly.  A window of identical closes (a price pinned at a clip bound)
        // has var == 0 exactly; it takes the reference's arithmetic instead (bollinger_constant).
        const double *wl = sm.last + e;
        const double cur = wl[(C3_LAST - 1) * C3_SUB];
        auto dv = [&](int i) { return wl[i * C3_SUB] - cur; };
        const double s = tree_sum16(dv) + ((dv(16) + dv(17)) + (dv(18) + dv(19)));
        const double mean_d = div_const<20>(s);
        auto sq = [&](int i) { const double t = dv(i) - mean_d; return t * t; };
        const double var = div_const<20>(tree_sum16(sq) + ((sq(16) + sq(17)) + (sq(18) + sq(19))));
        if (var > 0.0) {
            // 2^-2e and 2^e for the binary exponent e of cur (cur / 2^e in [1, 2)), built from its bits: exact scalings
            const int ex = (__double2hiint(cur) >> 20) - 1023;
            const double down2 = __hiloint2double((1023 - 2 * ex) << 20, 0), up = __hiloint2double((1023 + ex) << 20, 0);
            const float var_f = (float)(var * down2);
            const double sd = (double)(var_f > 0.0f ? var_f * rsqrtf(var_f) : 0.0f) * up;  // float32 accuracy: it only scales features
            const double sma = cur + mean_d;
            const double upper = sma + (2 * sd), lower = sma - (2 * sd);
            const float width = (float)(upper - lower), mid = (float)sma;
            dst[257] = (upper > lower) ? __fdividef((float)(cur - lower), width) : 0.5f;
            dst[258] = (sma > 0) ? __fdividef(width, mid) : 0.0f;
            dst[259] = (sma > 0) ? __fdividef((float)-mean_d, mid) : 0.0f;  // (cur - sma) / sma
        } else {
            bollinger_constant(cur, dst);
        }
    } else if (g == 3) {  // portfolio features :519-527, psychology :559
        dst[250] = port.x;
        dst[251] = port.y;
        dst[252] = port.z;
        dst[260] = port.w;
    }
}

// One thread: hand the finished tile to the copy engine.
__device__ __forceinline__ void store_tile(const CArgs &a, const float *tile, long long sub_first) {
    const long long n_here = min((long long)C3_SUB, a.n - sub_first);
    const uint32_t bytes = (uint32_t)(n_here * OBS * sizeof(float));
    const uint32_t bulk = bytes & ~15u;
    if (bulk) bulk_store_s2g(a.io.obs + sub_first * OBS, tile, bulk);
    bulk_commit();
    for (uint32_t i = bulk / 4; i < bytes / 4; ++i) a.io.obs[sub_first * OBS + i] = tile[i];  // ragged tail
}

// ---- shared-memory layouts -----------------------------------------------------------------------------------------
// common prefix: two tiles, three TMA stages, the observation stage's scratch
constexpr size_t OFF_STAGE_O = 2 * (size_t)C3_TILE_BYTES;
constexpr size_t OFF_STAGE_C = OFF_STAGE_O + (size_t)TMA_STAGES * STAGE_O;
constexpr size_t OFF_PM = OFF_STAGE_C + (size_t)TMA_STAGES * STAGE_C;  // double [16][32]
constexpr size_t OFF_PG = OFF_PM + (size_t)OBS_T * 8;
constexpr size_t OFF_LAST = OFF_PG + (size_t)OBS_T * 8;                // double [20][32]
constexpr size_t OFF_MX = OFF_LAST + (size_t)C3_LAST * C3_SUB * 8;     // float [16][32]
constexpr size_t OFF_MN = OFF_MX + (size_t)OBS_T * 4;
constexpr size_t OFF_MBAR = OFF_MN + (size_t)OBS_T * 4;                // uint64 [3 full + 8 ready + 8 freed]
constexpr size_t OFF_COMMON_END = OFF_MBAR + 8 * 40;
static_assert(OFF_STAGE_O % 128 == 0 && OFF_STAGE_C % 128 == 0 && STAGE_O % 128 == 0 && STAGE_C % 128 == 0,
              "TMA destinations are 128-byte aligned");

__device__ __forceinline__ ObsSmem obs_smem(uint8_t *smem_raw, int stage) {
    ObsSmem sm;
    sm.stage_o = reinterpret_cast<const float *>(smem_raw + OFF_STAGE_O + (size_t)stage * STAGE_O);
    sm.stage_c = reinterpret_cast<const double *>(smem_raw + OFF_STAGE_C + (size_t)stage * STAGE_C);
    sm.pm = reinterpret_cast<double *>(smem_raw + OFF_PM);
    sm.pg = reinterpret_cast<double *>(smem_raw + OFF_PG);
    sm.last = reinterpret_cast<double *>(smem_raw + OFF_LAST);
    sm.mx = reinterpret_cast<float *>(smem_raw + OFF_MX);
    sm.mn = reinterpret_cast<float *>(smem_raw + OFF_MN);
    return sm;
}

// One thread: both boxes of the unit starting at env `env0` into stage `stage`.
__device__ __forceinline__ void issue_window_loads(uint8_t *smem_raw, int stage, int env0, const CUtensorMap *tm_close,
                                                   const CUtensorMap *tm_ohlv) {
    const uint32_t bar = smem_u32(smem_raw + OFF_MBAR) + 8u * stage;
    mbar_expect_tx(bar, STAGE_O + STAGE_C);
    tma_load_2d(smem_u32(smem_raw + OFF_STAGE_O + (size_t)stage * STAGE_O), tm_ohlv, env0 * 4, 0, bar);
    tma_load_2d(smem_u32(smem_raw + OFF_STAGE_C + (size_t)stage * STAGE_C), tm_close, env0, 0, bar);
}

// The window head of this launch, after pdl_wait(), from every thread (contains a __syncthreads()): the slot holding the
// newest candle before the call, from params.window_head or, when io.window_head_dev is set, from that device word.  A
// step (ADVANCE) moves the device word on by one slot for the next launch; the caller advances params.window_head.
template <bool ADVANCE>
__device__ __forceinline__ int window_head(const CArgs &a) {
    uint32_t *const dev = reinterpret_cast<uint32_t *>(a.io.window_head_dev);  // {head, arrivals}
    if (!dev) {
        __syncthreads();
        return a.p.window_head;
    }
    if constexpr (ADVANCE) return (int)grid_uniform_advance(dev, dev + 1, [](uint32_t h) { return h + 1 == HIST ? 0u : h + 1; });
    __syncthreads();
    return (int)__ldcg(dev);
}

// ---- crypto4: bulk-synchronous -------------------------------------------------------------------------------------
constexpr size_t C4_OFF_CUR = OFF_COMMON_END;                        // double [512]
constexpr size_t C4_OFF_NEWX = C4_OFF_CUR + (size_t)OBS_T * 8;       // float4 [512]
constexpr size_t C4_OFF_PORT = C4_OFF_NEWX + (size_t)OBS_T * 16;     // float4 [512]
constexpr size_t C4_SMEM_BYTES = C4_OFF_PORT + (size_t)OBS_T * 16;
static_assert(C4_SMEM_BYTES <= 227 * 1024, "one CTA per SM: everything has to fit in 227 KB");
static_assert((size_t)C3_RNGW * OBS_T * 4 <= 2 * (size_t)C3_TILE_BYTES, "the Philox table aliases the two tile buffers");

__global__ void __launch_bounds__(OBS_T, 1) crypto4_kernel(const CArgs a) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    float *tiles = reinterpret_cast<float *>(smem_raw);                        // [2][32][261]
    uint32_t *s_rng = reinterpret_cast<uint32_t *>(smem_raw);                  // [20][512], dynamics phase only
    double *s_cur = reinterpret_cast<double *>(smem_raw + C4_OFF_CUR);
    float4 *s_newx = reinterpret_cast<float4 *>(smem_raw + C4_OFF_NEWX);
    float4 *s_port = reinterpret_cast<float4 *>(smem_raw + C4_OFF_PORT);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long n = a.n;
    const long long n_units = (n + C3_SUB - 1) / C3_SUB;
    const uint32_t pitch32 = (uint32_t)a.pitch;
    const double inv_ib = 1.0 / a.p.initial_balance;  // (features divide by it; the product differs by <= 1 ulp of float64)
    // units of this CTA: u(q) = blockIdx.x + gridDim.x * q, q = 0 .. total-1
    const long long total = n_units > blockIdx.x ? (n_units - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto unit_of = [&](long long q) { return (long long)blockIdx.x + (long long)gridDim.x * q; };

    pdl_launch_dependents();  // the next step's grid may become resident as this one drains ...
    pdl_wait();               // ... and this one touches nothing before the previous step's grid has flushed
    const int head = window_head<false>(a);
    const int oldest = head + 1 == HIST ? 0 : head + 1;
    int slot_of[OBS_PER];  // ring slot of this thread's i-th candle (k = wid + 16 i, oldest first)
#pragma unroll
    for (int i = 0; i < OBS_PER; ++i) {
        const int slot = oldest + wid + OBS_WARPS * i;
        slot_of[i] = slot >= HIST ? slot - HIST : slot;
    }

#pragma unroll 1
    for (long long q0 = 0; q0 < total; q0 += OBS_WARPS) {
        // The Philox table of the dynamics phase lives in the tile buffers: the copy engine must have read them.
        if (tid == 0) bulk_wait_read<0>();
        __syncthreads();
        {
            const long long qw = q0 + wid;
            dynamics_phase<true, OBS_T>(
                a, unit_of(qw), qw < total, head, s_rng + tid, reinterpret_cast<double *>(s_rng + wid * C3_SUB), OBS_T / 2,
                [&](double cur, double cash, double holdings, double psych, float4 newest) {
                    const double hv = holdings * cur;  // portfolio features :519-527, psychology :559
                    s_cur[tid] = cur;
                    s_newx[tid] = newest;
                    s_port[tid] = make_float4((float)(cash * inv_ib), (float)(hv * inv_ib), (float)((cash + hv) * inv_ib),
                                              (float)psych);
                });
        }
        __syncthreads();  // orders this CTA's window writes (the new candle, a reset's whole window) before its reads below

#pragma unroll 1
        for (int sub = 0; sub < OBS_WARPS; ++sub) {
            const long long q = q0 + sub;
            if (q >= total) break;  // CTA-uniform
            const long long sub_first = unit_of(q) * C3_SUB;
            const long long env = sub_first + lane;
            const int le = sub * C3_SUB + lane;  // where the dynamics left this env's values
            float *tile = tiles + (q & 1) * (C3_SUB * OBS);
            float *dst = tile + lane * OBS;
            const ObsSmem sm = obs_smem(smem_raw, 0);
            if (env < n) compose_unit<true>(a, sm, lane, wid, env, slot_of, pitch32, s_cur[le], s_newx[le], dst);
            __syncthreads();  // partial sums and the last 20 closes are visible
            if (env < n && wid < 4) finish_unit(sm, lane, wid, s_port[le], dst);
            fence_proxy_async_smem();
            if (tid == 0) bulk_wait_read<0>();  // the copy issued one unit ago has read the other tile buffer
            __syncthreads();
            if (tid == 0) store_tile(a, tile, sub_first);
        }
    }
    if (tid == 0) bulk_wait_read<0>();  // shared memory must outlive the copy engine's reads
}

// ---- crypto5: warp-specialised -------------------------------------------------------------------------------------
constexpr int DYN_WARPS = 8, C5_T = OBS_T + DYN_WARPS * 32;      // 768 threads = 6 warpgroups (4 observation + 2 dynamics)
// setmaxnreg moves registers inside the CTA's OWN pool (what it was launched with: 768 threads x 80), it cannot draw on
// the rest of the register file: 512 * 64 + 256 * 112 = 61440 = 768 * 80.
// Measured: 64 / 112 is 3 us faster than 72 / 96.
constexpr int C5_LAUNCH_REGS = 80, C5_REGS_OBS = 64, C5_REGS_DYN = 112;
static_assert(OBS_T * C5_REGS_OBS + DYN_WARPS * 32 * C5_REGS_DYN <= C5_T * C5_LAUNCH_REGS, "setmaxnreg budget");
// Hand-over slots: unit q uses slot q % C5_RING (a multiple of DYN_WARPS).  Measured: 8 slots 133-144 us, 16 slots
// 126-133 us (the dynamics warps run further ahead).
constexpr int C5_RING = 16;
static_assert(C5_RING % DYN_WARPS == 0 && C5_RING <= 16, "each dynamics warp owns C5_RING / DYN_WARPS slots");
constexpr size_t C5_OFF_CUR = OFF_COMMON_END;                                 // double [ring][32]
constexpr size_t C5_OFF_NEWX = C5_OFF_CUR + (size_t)C5_RING * C3_SUB * 8;     // float4 [ring][32]
constexpr size_t C5_OFF_PORT = C5_OFF_NEWX + (size_t)C5_RING * C3_SUB * 16;   // float4 [ring][32]
constexpr size_t C5_OFF_URESET = C5_OFF_PORT + (size_t)C5_RING * C3_SUB * 16; // uint32 [ring]
constexpr size_t C5_OFF_RNG = C5_OFF_URESET + 128;                              // uint32 [8][20][32]
constexpr size_t C5_SMEM_BYTES = C5_OFF_RNG + (size_t)DYN_WARPS * C3_RNGW * C3_SUB * 4;
static_assert(C5_SMEM_BYTES <= 227 * 1024, "one CTA per SM: everything has to fit in 227 KB");

__global__ void __launch_bounds__(C5_T, 1) crypto5_kernel(const CArgs a, const __grid_constant__ CUtensorMap tm_close,
                                                          const __grid_constant__ CUtensorMap tm_ohlv) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    float *tiles = reinterpret_cast<float *>(smem_raw);  // [2][32][261]
    double *s_cur = reinterpret_cast<double *>(smem_raw + C5_OFF_CUR);
    float4 *s_newx = reinterpret_cast<float4 *>(smem_raw + C5_OFF_NEWX);
    float4 *s_port = reinterpret_cast<float4 *>(smem_raw + C5_OFF_PORT);
    uint32_t *s_ureset = reinterpret_cast<uint32_t *>(smem_raw + C5_OFF_URESET);
    const uint32_t mbar_full = smem_u32(smem_raw + OFF_MBAR);   // [3]  TMA stage filled
    const uint32_t mbar_ready = mbar_full + 8u * TMA_STAGES;    // [ring] slot filled by its dynamics warp
    const uint32_t mbar_freed = mbar_ready + 8u * C5_RING;      // [ring] slot consumed by the observation warps

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long n = a.n;
    const long long n_units = (n + C3_SUB - 1) / C3_SUB;
    const long long total = n_units > blockIdx.x ? (n_units - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto unit_of = [&](long long q) { return (long long)blockIdx.x + (long long)gridDim.x * q; };

    if (tid == 0) {
        for (int s = 0; s < TMA_STAGES + 2 * C5_RING; ++s) mbar_init(mbar_full + 8u * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async_smem();
    }
    pdl_launch_dependents();  // the next step's grid may become resident as this one drains ...
    pdl_wait();               // ... and this one touches nothing before the previous step's grid has flushed
    // (the only CTA-wide barrier is in here: the two roles part ways after it)
    const int newest = window_head<true>(a);
    const int head = newest + 1 == HIST ? 0 : newest + 1;  // the slot this step's candle goes to

    if (wid >= OBS_WARPS) {
        // =================================================================================== dynamics warps
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(C5_REGS_DYN));
        const int dw = wid - OBS_WARPS;  // this warp's ring slot
        const double inv_ib = 1.0 / a.p.initial_balance;
        uint32_t *table = reinterpret_cast<uint32_t *>(smem_raw + C5_OFF_RNG) + dw * (C3_RNGW * C3_SUB);  // [20][32]
#pragma unroll 1
        for (long long q = dw; q < total; q += DYN_WARPS) {
            const int rs = (int)(q % C5_RING);    // ring slot of this unit
            const int slot = rs * C3_SUB + lane;
            const long long use = q / C5_RING;    // how often this slot has been filled before
            if (use > 0) mbar_wait_backoff(mbar_freed + 8u * rs, (uint32_t)((use - 1) & 1));
            const unsigned resets = dynamics_phase<false, C3_SUB>(
                a, unit_of(q), true, head, table + lane, reinterpret_cast<double *>(table), C3_SUB / 2,
                [&](double cur, double cash, double holdings, double psych, float4 newest) {
                    const double hv = holdings * cur;  // portfolio features :519-527, psychology :559
                    s_cur[slot] = cur;
                    s_newx[slot] = newest;
                    s_port[slot] = make_float4((float)(cash * inv_ib), (float)(hv * inv_ib), (float)((cash + hv) * inv_ib),
                                               (float)psych);
                });
            if (lane == 0) s_ureset[rs] = resets;
            __syncwarp();  // every lane's shared- and global-memory writes are ordered before the release below
            if (lane == 0) mbar_arrive(mbar_ready + 8u * rs);
        }
    } else {
        // =================================================================================== observation warps
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(C5_REGS_OBS));
        const uint32_t pitch32 = (uint32_t)a.pitch;
        const int oldest = head + 1 == HIST ? 0 : head + 1;
        int slot_of[OBS_PER];  // ring slot of this thread's i-th candle (k = wid + 16 i, oldest first)
#pragma unroll
        for (int i = 0; i < OBS_PER; ++i) {
            const int slot = oldest + wid + OBS_WARPS * i;
            slot_of[i] = slot >= HIST ? slot - HIST : slot;
        }
        if (tid == 0) {
            for (long long q = 0; q < TMA_STAGES && q < total; ++q)
                issue_window_loads(smem_raw, (int)q, (int)(unit_of(q) * C3_SUB), &tm_close, &tm_ohlv);
        }
#pragma unroll 1
        for (long long q = 0; q < total; ++q) {
            const long long sub_first = unit_of(q) * C3_SUB;
            const long long env = sub_first + lane;
            const int dw = (int)(q % C5_RING);  // ring slot of this unit
            const int le = dw * C3_SUB + lane;
            const int stage = (int)(q % TMA_STAGES);
            float *tile = tiles + (q & 1) * (C3_SUB * OBS);
            float *dst = tile + lane * OBS;
            const ObsSmem sm = obs_smem(smem_raw, stage);
            mbar_wait(mbar_ready + 8u * dw, (uint32_t)((q / C5_RING) & 1));     // the unit's dynamics are done
            mbar_wait(mbar_full + 8u * stage, (uint32_t)((q / TMA_STAGES) & 1));  // its window box has landed
            const bool direct = s_ureset[dw] != 0;  // uniform over the 16 warps
            if (env < n) {
                if (direct) compose_unit<true>(a, sm, lane, wid, env, slot_of, pitch32, s_cur[le], s_newx[le], dst);
                else compose_unit<false>(a, sm, lane, wid, env, slot_of, pitch32, s_cur[le], s_newx[le], dst);
            }
            obs_bar_sync();  // the stage has been consumed; partial sums and the last 20 closes are visible
            if (tid == OBS_T - 1 && q + TMA_STAGES < total)  // refill the stage just freed
                issue_window_loads(smem_raw, stage, (int)(unit_of(q + TMA_STAGES) * C3_SUB), &tm_close, &tm_ohlv);
            if (env < n && wid < 4) finish_unit(sm, lane, wid, s_port[le], dst);
            fence_proxy_async_smem();
            if (tid == 0) bulk_wait_read<0>();  // the copy issued one unit ago has read the other tile buffer
            obs_bar_sync();
            if (tid == 0) store_tile(a, tile, sub_first);
            if (tid == 32) mbar_arrive(mbar_freed + 8u * dw);  // every read of the ring slot is behind the barrier above
        }
        if (tid == 0) bulk_wait_read<0>();  // shared memory must outlive the copy engine's reads
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (libbeng does not link libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}

// [50][pitch * elems_per_env] tensor of `type`, box = all 50 slots x one 32-env unit.
int make_window_map(CUtensorMap *map, void *base, long long pitch, CUtensorMapDataType type, int elem_bytes,
                    int elems_per_env) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return BENG_ERR_UNSUPPORTED;
    const cuuint64_t dims[2] = {(cuuint64_t)pitch * elems_per_env, (cuuint64_t)HIST};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch * elems_per_env * elem_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)(C3_SUB * elems_per_env), (cuuint32_t)HIST};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, type, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : BENG_ERR_BAD_ARG;
}

// One persistent CTA per SM (at most one per unit) of `threads` threads and `smem` bytes of dynamic shared memory.
template <typename Kern, typename... Extra>
int launch_persistent(Kern kern, int threads, size_t smem, const CArgs &a, cudaStream_t stream, const Extra &...extra) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const long long n_units = (a.n + C3_SUB - 1) / C3_SUB;
    long long grid = device_sm_count();
    if (grid > n_units) grid = n_units;
    return (int)launch_pdl(kern, dim3((unsigned)grid), dim3((unsigned)threads), smem, stream, a, extra...);
}

int launch_reset(const CArgs &a, cudaStream_t stream) {
    return launch_persistent(crypto4_kernel, OBS_T, C4_SMEM_BYTES, a, stream);
}

int launch_step(const CArgs &a, cudaStream_t stream) {
    CUtensorMap tm_close, tm_ohlv;
    if (int rc = make_window_map(&tm_close, a.st.close, a.pitch, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 8, 1)) return rc;
    if (int rc = make_window_map(&tm_ohlv, a.st.ohlv, a.pitch, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, 4)) return rc;
    return launch_persistent(crypto5_kernel, C5_T, C5_SMEM_BYTES, a, stream, tm_close, tm_ohlv);
}

int check(const beng_crypto_params *p, const beng_crypto_state *st, const beng_crypto_io *io, int64_t n) {
    if (!p || !st || !io || n < 0) return BENG_ERR_BAD_ARG;
    if (!st->scal || !st->meta || !st->ep_return || !st->close || !st->ohlv || !io->obs) return BENG_ERR_BAD_ARG;
    if (((uintptr_t)io->obs & 15) || ((uintptr_t)st->close & 7) || ((uintptr_t)st->ohlv & 15)) return BENG_ERR_BAD_ARG;
    if (io->window_head_dev ? ((uintptr_t)io->window_head_dev & 7) != 0 : (p->window_head < 0 || p->window_head >= HIST))
        return BENG_ERR_BAD_ARG;  // (a device head replaces params.window_head, which is then not read)
    if (p->autoreset_mode < 0 || p->autoreset_mode > 2 || p->action_type < 0 || p->action_type > 1) return BENG_ERR_BAD_ARG;
    if (p->max_steps < 1 || p->max_steps > 65535) return BENG_ERR_UNSUPPORTED;
    // Price domain (beng.h): every close lies in [min_price, max_price], so 1.02 x price, volume / price and the float32
    // reciprocal of the price stay normal floats well below __fdividef's 2^126 limit.  Rejects NaN and infinite
    // bounds, min_price <= 0 and min_price > max_price (the reference's np.clip would return max_price there).
    if (!(p->min_price >= 0x1p-100 && p->min_price <= p->max_price && p->max_price <= 0x1p100)) return BENG_ERR_UNSUPPORTED;
    if (n >= (1LL << 26)) return BENG_ERR_UNSUPPORTED;  // 32-bit element offsets in the window addressing (49 * n < 2^32)
    return 0;
}

}  // namespace
}  // namespace beng

extern "C" {

int64_t beng_crypto_window_pitch(int64_t n_envs) { return (n_envs + 31) & ~(int64_t)31; }

int beng_crypto_reset(const beng_crypto_params *p, const beng_crypto_state *st, const beng_crypto_io *io,
                      const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (n_envs == 0) return 0;
    beng::CArgs a{*p, *st, *io, nullptr, mask_dev, (long long)n_envs, beng_crypto_window_pitch(n_envs), first_call};
    return beng::launch_reset(a, (cudaStream_t)stream);
}

int beng_crypto_step(const beng_crypto_params *p, const beng_crypto_state *st, const void *actions_dev,
                     const beng_crypto_io *io, int64_t n_envs, void *stream) {
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (!actions_dev || !io->reward || !io->terminated) return BENG_ERR_BAD_ARG;
    if ((uintptr_t)actions_dev & 7) return BENG_ERR_BAD_ARG;  // 64-bit action loads (int64, or float32 pairs)
    if (n_envs == 0) return 0;
    beng::CArgs a{*p, *st, *io, actions_dev, nullptr, (long long)n_envs, beng_crypto_window_pitch(n_envs), 0};
    return beng::launch_step(a, (cudaStream_t)stream);
}

int beng_crypto_step_host(const beng_crypto_params *p, const beng_crypto_state *st, void *actions_dev,
                          const beng_crypto_io *io, int64_t n_envs, const void *actions_host, float *obs_host,
                          float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, void *stream) {
    if (!actions_host || !actions_dev) return BENG_ERR_BAD_ARG;
    if (int rc = beng::check(p, st, io, n_envs)) return rc;
    if (truncated_host && !io->truncated) return BENG_ERR_BAD_ARG;
    if (n_envs == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)n_envs;
    const size_t abytes = p->action_type == 1 ? n * 2 * sizeof(float) : n * sizeof(int64_t);
    cudaError_t e = cudaMemcpyAsync(actions_dev, actions_host, abytes, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return (int)e;
    if (int rc = beng_crypto_step(p, st, actions_dev, io, n_envs, stream)) return rc;
    if (int rc = beng::d2h(reward_host, io->reward, n * sizeof(float), s)) return rc;
    if (int rc = beng::d2h(terminated_host, io->terminated, n, s)) return rc;
    if (int rc = beng::d2h(truncated_host, io->truncated, n, s)) return rc;
    return beng::d2h(obs_host, io->obs, n * BENG_CRYPTO_OBS_DIM * sizeof(float), s);
}

}  // extern "C"
