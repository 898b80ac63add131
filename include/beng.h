/* beng.h -- C ABI of libbeng.so, the B200 (sm_100a) batched environment engine.
 *
 * This is the drop-in boundary for the step()/reset() hot path of the reference's Gymnasium
 * environments (SURVEY.md section 8b).  The reference is pure Python and has no FFI of its own;
 * the interface each entry point replaces is therefore a METHOD of the reference class, cited
 * per function below (paths relative to the reference root).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions (all entry points):
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - return int = cudaError_t (0 == success) or BENG_ERR_* (negative) for argument errors.
 *   - never allocate device memory, never synchronise, never throw: kernels are launched
 *     asynchronously on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - every `*_dev` / state / io pointer is a DEVICE pointer to caller-owned memory, 16-byte
 *     aligned, alive until the stream has drained.  The *_host entry points additionally take
 *     (pinned) HOST buffers and enqueue the H2D/D2H copies around the kernel on the same stream.
 *   - one host thread per GPU/process; env ids are GLOBAL (env_id_base + local index) so a given
 *     env has the same trajectory however the batch is sharded over GPUs.
 */
#ifndef BENG_H
#define BENG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BENG_VERSION 100 /* major*10000 + minor*100 + patch */

enum {
    BENG_ERR_BAD_ARG = -1,      /* NULL where a pointer is required, n_envs < 0, ... */
    BENG_ERR_UNSUPPORTED = -2,  /* e.g. grid_size outside [2, 64] */
};

/* Auto-reset modes of the batched classes (gymnasium.vector.AutoresetMode names).  The reference
 * has no auto-reset (SURVEY.md section 0 fact 4): DISABLED is exactly the reference class;
 * SAME_STEP is the reference's caller loop `if terminated: env.reset()` folded into the step. */
enum {
    BENG_AUTORESET_DISABLED = 0,
    BENG_AUTORESET_NEXT_STEP = 1,
    BENG_AUTORESET_SAME_STEP = 2,
};

/* RNG streams of the counter-based generator (Philox4x32-10, csrc/beng_rng.cuh). */
enum { BENG_STREAM_ENV = 0, BENG_STREAM_ACTION = 1 };

/* Library version (BENG_VERSION of the build). */
int beng_version(void);

/* SM architecture the library was compiled for (100 for sm_100a). */
int beng_compiled_arch(void);

/* Number of kernel launches this process has issued through the library since load
 * (bench.py reports it as `gpu_launches`). */
uint64_t beng_launch_count(void);

/* Synthetic uniform action tape on the device (bench / tests; stands in for a policy).
 *   actions_dev[i * n_cols + c] = randint(0, n_choices - 1) drawn from u32 number
 *   (step_index * n_cols + c) of stream BENG_STREAM_ACTION of env (env_id_base + i). */
int beng_fill_random_actions(int64_t *actions_dev, int64_t n_envs, int32_t n_cols, int32_t n_choices,
                             uint32_t step_index, uint64_t env_id_base, uint64_t seed, void *stream);

/* ------------------------------------------------------------------------------------------
 * snake_env_classic  (reference: snake_env_classic/snake_env.py, class SnakeEnvClassic)
 * ------------------------------------------------------------------------------------------ */

/* Constructor arguments of SnakeEnvClassic (snake_env.py:19-47) plus the batching parameters. */
typedef struct beng_snake_params {
    int32_t grid_size;      /* `grid_size` ctor kwarg, default 20 (snake_env.py:19); 2..64 */
    int32_t max_steps;      /* `self.max_steps = 1000` (snake_env.py:47); 1..65535 */
    int32_t autoreset_mode; /* BENG_AUTORESET_* */
    int32_t time_limit_truncation; /* 0: `truncated` is always 0, like the raw reference class (snake_env.py:119).
                                      1: ALSO set truncated on the step that reaches max_steps -- what gymnasium's
                                      TimeLimit wrapper adds when the env is built with gym.make
                                      (snake_env_classic/__init__.py:3-7, max_episode_steps=1000) */
    uint64_t seed;          /* key of the counter-based stream */
    uint64_t env_id_base;   /* global id of local env 0 */
} beng_snake_params;

/* Per-env state, structure-of-arrays in HBM.
 *   core : n_envs x 16 B record {u8 head_r, head_c, food_r, food_c; u8 direction; u8 flags;
 *          u16 length; u16 steps; u16 ring_head; u32 rng_counter}  -- one 128-bit load per env.
 *          (`score` is not stored: score == length - 1 always, snake_env.py:57,102 vs :97,107.)
 *          The direction byte: bits 0-1 the direction, bits 2-3 the direction of the last step
 *          that moved the head, bit 4 set when bits 2-3 are valid (every move or meal sets them,
 *          a reset clears them).
 *   ring : n_envs x (grid_size^2) u16 body cells (r * G + c); newest at ring_head, oldest
 *          (the tail) at ring_head - length + 1 (mod G^2).  Replaces the Python list
 *          `self.snake` (snake_env.py:54,97,107).  Only maintained from length 3 on: a length-1
 *          body is the head, a length-2 body with bit 4 set is the head and the cell one step
 *          against the last move; a length-2 record without bit 4 keeps its tail in the ring. */
typedef struct beng_snake_state {
    void *core;     /* uint4[n_envs] */
    uint16_t *ring; /* uint16_t[n_envs * grid_size * grid_size] */
} beng_snake_state;

/* Outputs of one batched step.  `obs`, `reward`, `terminated` are required; the rest may be NULL. */
typedef struct beng_snake_io {
    int8_t *obs;            /* [n_envs, G, G] 0 empty / 1 snake / 2 food  (_get_observation, snake_env.py:131-143) */
    float *reward;          /* [n_envs] -10 / 0 / +10                       (snake_env.py:90,94,100,103) */
    uint8_t *terminated;    /* [n_envs] death or steps >= max_steps        (snake_env.py:90,94,112-114) */
    uint8_t *truncated;     /* [n_envs] always 0                           (snake_env.py:119) */
    int32_t *score;         /* [n_envs] info["score"] after the step       (snake_env.py:117) */
    int32_t *snake_length;  /* [n_envs] info["snake_length"]               (snake_env.py:117) */
    /* written only for envs whose episode ended in this step (auto-reset modes): */
    float *ep_return;       /* [n_envs] 10 * score - 10 * died */
    int32_t *ep_length;     /* [n_envs] env steps in the episode (death step included) */
    int32_t *ep_score;      /* [n_envs] */
    /* warp-compacted list of the envs that finished this step (order unspecified): */
    uint32_t *done_count;   /* [1]  must be zero when the step starts (see done_count_next) */
    int32_t *done_env;      /* [n_envs] LOCAL env indices */
    uint32_t *done_count_next; /* [1] nullable; zeroed BY this launch so it can serve as `done_count` of the
                                  next step (ping-pong two counters: no memset launch between steps) */
    /* Self-managed counters: done_count_next == done_count (non-NULL) means that done_count points to
     * uint32_t[4] = {count0, count1, parity, arrivals}, 16-byte aligned, zero before the first call.  Every step and
     * reset launch then counts its finished envs into count[parity], zeroes count[parity ^ 1] and flips parity for
     * the next launch; `arrivals` is the launch's scratch counter and is 0 again when it ends.  The counter of the
     * last launch is count[parity ^ 1].  A step's arguments are then the same every call (a CUDA graph captures it
     * once and replays it), and no host state changes per step.  Every other combination is the contract above.
     * beng_snake_step_inplace also takes the parity as its sweep direction: on the self-managed block it visits the
     * env tiles in descending order every other launch (results are the same either way; only the order of
     * done_env, which is unspecified, differs), under the contract above always in ascending order. */
    /* running episode statistics, integer (exact, order independent):
     * {n_episodes, sum_return, sum_length, sum_score, max_score} */
    int64_t *stats;         /* [5] accumulated across steps; caller zeroes / all-reduces */
    int32_t *invalid_count; /* [1] number of out-of-space actions seen (reference raises ValueError,
                                   snake_env.py:69-70; here such an env is left untouched) */
} beng_snake_io;

/* Launch shape the observation-composing kernel of beng_snake_reset / beng_snake_step uses for (grid_size, n_envs) on
 * the current device: envs (= threads) per CTA tile, tile buffers per CTA, resident CTAs per SM.  Informational
 * (bench.py names the kernel with it).  beng_snake_step_inplace has no tile: one thread per env, 256 per CTA. */
int beng_snake_launch_config(int32_t grid_size, int64_t n_envs, int32_t *tile, int32_t *stages, int32_t *ctas_per_sm);

/* Bytes the caller must allocate. */
size_t beng_snake_core_bytes(int64_t n_envs);
size_t beng_snake_ring_bytes(int64_t n_envs, int32_t grid_size);

/* SnakeEnvClassic.reset (snake_env.py:49-65) for every env with mask[i] != 0 (mask NULL = all),
 * then the observation / info of EVERY env is written to io (io->obs required; reward etc. untouched).
 * `first_call` != 0 additionally zeroes rng_counter of the selected envs (constructor semantics). */
int beng_snake_reset(const beng_snake_params *p, const beng_snake_state *st, const beng_snake_io *io,
                     const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream);

/* SnakeEnvClassic.step (snake_env.py:67-119) + _place_food (:121-129) + _get_observation (:131-143)
 * + the auto-reset named in p->autoreset_mode, for all n_envs envs, in ONE kernel launch. */
int beng_snake_step(const beng_snake_params *p, const beng_snake_state *st, const int64_t *actions_dev,
                    const beng_snake_io *io, int64_t n_envs, void *stream);

/* The same step for a caller that keeps the observations in place.  Precondition: io->obs holds, byte for byte, the
 * observation that the last beng_snake_reset or step of these envs wrote (into any buffer); the function then writes
 * only the cells that change -- at most two per env, or the whole row on an auto-reset -- and reads io->obs as the
 * occupancy map of the bodies.  Results, state and statistics are those of beng_snake_step, and so is io->obs
 * afterwards.  Same arguments, checks and error codes as beng_snake_step; one kernel launch, none when n_envs == 0.
 * With any other io->obs content the observations, and the self-collision and food placement read from them, are
 * undefined. */
int beng_snake_step_inplace(const beng_snake_params *p, const beng_snake_state *st, const int64_t *actions_dev,
                            const beng_snake_io *io, int64_t n_envs, void *stream);

/* Same step with HOST action / result buffers (what a caller of the reference's numpy API holds):
 * enqueues H2D(actions) -> kernel -> D2H(obs, reward, terminated[, truncated, score, snake_length])
 * on `stream`.  Host pointers that are NULL are skipped (obs_host NULL keeps observations in HBM).
 * Does not synchronise; the caller waits on the stream before reading the host buffers. */
int beng_snake_step_host(const beng_snake_params *p, const beng_snake_state *st, int64_t *actions_dev,
                         const beng_snake_io *io, int64_t n_envs, const int64_t *actions_host, int8_t *obs_host,
                         float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, int32_t *score_host,
                         int32_t *snake_length_host, void *stream);

/* Observation change records of beng_snake_step_host_delta: one uint32_t per env and step, telling how the env's
 * observation row [G*G] differs from the one the previous step or reset wrote.
 *   pair    = cell | value << 12  (14 bits; cell = r * G + c < 4096; value 0 / 1 / 2 is written to the cell,
 *             value 3 marks an unused pair)
 *   record  = pair A (bits 0-13) | pair B << 14 (bits 14-27) | BENG_OBS_DELTA_CLEAR (bit 31); bits 28-30 are 0
 *   applied = clear the whole row if bit 31 is set, then write A, then B.
 * What the step kernel emits:
 *   move                        A = (old tail, 0), B = (new head, 1)
 *   eat                         A = (new head, 1), B = (new food, 2), or unused when the board is full
 *   death, invalid action       both unused (the row does not change)
 *   any auto-reset              CLEAR, A = (head, 1), B = (food, 2) */
#define BENG_OBS_DELTA_CLEAR 0x80000000u
#define BENG_OBS_DELTA_UNUSED 0x3000u                                       /* one unused pair */
#define BENG_OBS_DELTA_NONE (BENG_OBS_DELTA_UNUSED | (BENG_OBS_DELTA_UNUSED << 14)) /* no change */

/* beng_snake_step_host without the observation copy: enqueues H2D(actions) -> step kernel, which also writes one
 * change record per env to delta_dev -> D2H(records, reward, terminated[, truncated, score, snake_length]) on
 * `stream`.  io->obs on the device is written exactly as by beng_snake_step.  A caller that holds a host copy of
 * the observations from before this step brings it up to date with beng_snake_apply_obs_delta once the stream has
 * drained: 18 B per env cross the bus instead of G*G + 14.  delta_dev / delta_host (uint32_t[n_envs], device /
 * pinned host, 4-byte aligned) are required; NULL result host pointers are skipped.  Does not synchronise. */
int beng_snake_step_host_delta(const beng_snake_params *p, const beng_snake_state *st, int64_t *actions_dev,
                               const beng_snake_io *io, int64_t n_envs, const int64_t *actions_host,
                               uint32_t *delta_dev, uint32_t *delta_host, float *reward_host, uint8_t *terminated_host,
                               uint8_t *truncated_host, int32_t *score_host, int32_t *snake_length_host, void *stream);

/* Apply one step's change records (host memory, uint32_t[n_envs]) to a host copy of the observations
 * (int8_t[n_envs][G][G]).  Pure host code: touches no CUDA state and runs without a GPU.  The envs are split into
 * contiguous chunks over n_threads threads (<= 0 means one), all joined before it returns.  BENG_ERR_BAD_ARG for
 * NULL buffers, n_envs < 0 or a malformed record (set bits 28-30, or a cell >= G*G; obs_host is then partly
 * updated), BENG_ERR_UNSUPPORTED for grid_size outside [2, 64]. */
int beng_snake_apply_obs_delta(const uint32_t *delta_host, int8_t *obs_host, int64_t n_envs, int32_t grid_size,
                               int32_t n_threads);

/* Unpack the SoA state into plain int32 arrays (tests, checkpoints, debugging).  Any output may be NULL.
 * body_cells_dev, when given, is [n_envs, G*G] int32 filled head-first with r*G+c and -1 padding. */
int beng_snake_export_state(const beng_snake_params *p, const beng_snake_state *st, int64_t n_envs, int32_t *head_r,
                            int32_t *head_c, int32_t *food_r, int32_t *food_c, int32_t *direction, int32_t *steps,
                            int32_t *length, uint32_t *rng_counter, int32_t *body_cells_dev, void *stream);

/* ------------------------------------------------------------------------------------------
 * crypto_trading_env  (reference: crypto_trading_env/crypto_trading_env.py, class CryptoTradingEnv)
 * ------------------------------------------------------------------------------------------ */

#define BENG_CRYPTO_HISTORY 50  /* TradingConfig.history_length (crypto_trading_env.py:33); fixed */
#define BENG_CRYPTO_OBS_DIM 261 /* 50*5 + 3 + 8: what _get_observation really returns (:505-561); the declared
                                   space says 260 (:285-286) -- SURVEY.md section 0 fact 7 */

/* TradingConfig (crypto_trading_env.py:28-38) + episode limit (:298) + batching parameters. */
typedef struct beng_crypto_params {
    double initial_balance;          /* 10000.0 */
    double trading_fee_rate;         /* 0.001 */
    double slippage_rate;            /* 0.0005 */
    double min_price;                /* 100.0    price domain: 2^-100 <= min_price <= max_price <= 2^100, otherwise */
    double max_price;                /* 100000.0 reset / step return BENG_ERR_UNSUPPORTED (NaN bounds included) */
    double volatility_base;          /* 0.02 */
    double market_psychology_factor; /* 0.1 */
    int32_t max_steps;               /* 1000 (:298) */
    int32_t autoreset_mode;          /* BENG_AUTORESET_* */
    int32_t action_type;             /* 0 = Discrete(5) int64[n]; 1 = Box(-1,1,(2,)) float32[n][2]  (:288-296) */
    int32_t window_head;             /* slot (0..49) holding the NEWEST candle of every env before this call.
                                        A step writes the new candle to (window_head+1)%50 -- the caller then
                                        advances window_head by one; a reset leaves it unchanged.  Ignored when
                                        io->window_head_dev is set (the head then lives on the device). */
    int32_t time_limit_truncation;   /* 1: also set `truncated` when current_step reaches max_steps (gym.make's
                                        TimeLimit, crypto_trading_env.py:739-743); 0: never (raw class, :388) */
    int32_t reserved;
    uint64_t seed;
    uint64_t env_id_base;
} beng_crypto_params;

/* Per-env state, structure-of-arrays in HBM, env index fastest (coalesced for one thread per env).
 * All money/price arithmetic is float64 like the reference; open/high/low/volume are observation-only
 * features and are stored as float32. */
typedef struct beng_crypto_state {
    double *scal;      /* [4][n]  cash, holdings, trend_strength, market_psychology */
    uint32_t *meta;    /* [2][n]  {step | regime << 16 | flags << 24}, rng_counter */
    double *ep_return; /* [n]     running episode return */
    double *close;     /* [50][pitch] close prices, ring over slots (see window_head); pitch =
                          beng_crypto_window_pitch(n) = n rounded up to a multiple of 32, so that every 32-env unit of
                          every slot is one aligned box for the tensor-map (TMA) loads; 128-byte aligned */
    float *ohlv;       /* [50][pitch][4] open, high, low, volume: one 16-byte record per (slot, env); 128-byte aligned */
} beng_crypto_state;

typedef struct beng_crypto_io {
    float *obs;              /* [n][261]  _get_observation (:505-561) */
    float *reward;           /* [n]       (:440-445) cast to float32 */
    uint8_t *terminated;     /* [n]       step >= max_steps or value <= 0 or value >= 10 * initial (:382-386) */
    uint8_t *truncated;      /* [n]       always 0 (:388) */
    /* info dict (:390-398); all nullable */
    double *reward64;        /* [n] the float64 reward */
    double *portfolio_value; /* [n] */
    double *current_price;   /* [n] */
    uint8_t *trade_kind;     /* [n] 0 = no trade, 1 = buy, 2 = sell (info["trade_info"]["action"]) */
    /* written only for envs whose episode ended in this step (auto-reset modes); nullable */
    double *ep_return_out;   /* [n] */
    int32_t *ep_length;      /* [n] */
    double *stats;           /* [4] running {n_episodes, sum_return, sum_length, sum_final_value}; nullable */
    /* State that the launch itself advances, so that a step's arguments are the same every call (a CUDA graph
     * captures a step once and replays it):
     * NULL     : params.window_head is the head, as documented there (the caller advances it).
     * non-NULL : int32_t[2] = {head, arrivals}, 8-byte aligned, head 0..49 and arrivals 0 before the first call.
     *            params.window_head is then ignored (not validated).  beng_crypto_step reads the head and leaves it
     *            advanced by one slot (mod 50) for the next call; beng_crypto_reset reads it and leaves it as it is.
     *            `arrivals` is the launch's scratch counter and is 0 again when the launch ends. */
    int32_t *window_head_dev;
} beng_crypto_io;

/* Row pitch (in envs) of beng_crypto_state.close / .ohlv for a batch of n_envs. */
int64_t beng_crypto_window_pitch(int64_t n_envs);

/* CryptoTradingEnv.reset (:301-340) for envs with mask[i] != 0 (NULL = all): 50 warm-up candles from 50000.0,
 * cash/holdings/step reset, the MarketSimulator state is NOT reset (SURVEY.md fact 8).  first_call != 0 is the
 * constructor: market state = (SIDEWAYS, 0.0, 0.5) (:125-130) and rng_counter = 0 for the selected envs.
 * The observation of EVERY env is written to io->obs. */
int beng_crypto_reset(const beng_crypto_params *p, const beng_crypto_state *st, const beng_crypto_io *io,
                      const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream);

/* CryptoTradingEnv.step (:342-398) + _execute_action/_execute_buy/_execute_sell (:400-503) +
 * MarketSimulator.generate_next_price (:132-221) + _get_observation with all TechnicalIndicators (:41-119,
 * :505-561) + auto-reset, for all envs, in ONE kernel launch (persistent CTAs: per-env float64 dynamics, then the
 * window is streamed once and the indicators are accumulated on the way).  `actions_dev` is int64[n] or
 * float32[n][2] according to p->action_type.  n_envs must be below 2^26 (BENG_ERR_UNSUPPORTED otherwise). */
int beng_crypto_step(const beng_crypto_params *p, const beng_crypto_state *st, const void *actions_dev,
                     const beng_crypto_io *io, int64_t n_envs, void *stream);

/* Same step with HOST action / result buffers: H2D(actions) -> kernel -> D2H(obs, reward, terminated) on `stream`.
 * NULL host outputs are skipped.  Does not synchronise. */
int beng_crypto_step_host(const beng_crypto_params *p, const beng_crypto_state *st, void *actions_dev,
                          const beng_crypto_io *io, int64_t n_envs, const void *actions_host, float *obs_host,
                          float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, void *stream);

/* ------------------------------------------------------------------------------------------
 * traffic_management_env  (reference: traffic_management_env/{environment,utils,config}.py)
 * ------------------------------------------------------------------------------------------ */

#define BENG_TRAFFIC_MAX_INTERSECTIONS 25

/* Constructor arguments of TrafficManagementEnv (environment.py:61-66, defaults config.py:6-12) + config.py
 * MAX_TIMESTEPS + batching parameters.  The remaining config.py constants (phase durations 5/30/3, reward weights
 * 1.0/-0.1/-0.05/0.5, observation caps 20/100/1000/50) are compiled in. */
typedef struct beng_traffic_params {
    int32_t grid_rows, grid_cols; /* grid_size, default (5, 5) */
    int32_t num_intersections;    /* default 9; effective value = min(this, rows*cols) (environment.py:82); <= 25 */
    int32_t max_vehicles;         /* default 50; <= 255 */
    double spawn_rate;            /* default 0.3 */
    int32_t max_timesteps;        /* config.py:23 MAX_TIMESTEPS = 1000 */
    int32_t autoreset_mode;       /* BENG_AUTORESET_* */
    int32_t time_limit_truncation; /* 1: also set `truncated` at max_timesteps (gym.make's TimeLimit,
                                      traffic_management_env/__init__.py:7-17); 0: never (raw class, environment.py:197) */
    int32_t reserved;
    uint64_t seed;
    uint64_t env_id_base;
} beng_traffic_params;

/* Per-env state, [field][env] arrays (env index fastest).  Vehicles never move in the reference (SURVEY.md
 * section 0 fact 9), so a queue is fully described by (length, sum of waiting times, number of vehicles whose
 * route ends where it started) and the env by the length of `self.vehicles`. */
typedef struct beng_traffic_state {
    uint16_t *light;      /* [ni][n]    phase (low byte: 0 NS_GREEN 1 NS_YELLOW 2 EW_GREEN 3 EW_YELLOW) | timer << 8 */
    int32_t *passed;      /* [ni][n]    Intersection.vehicles_passed */
    int32_t *waiting;     /* [ni][n]    Intersection.total_waiting_time */
    uint32_t *qmeta;      /* [ni*2][n]  row 2i: queue lengths of intersection i, one byte per direction N, E, S, W (byte 0 = N);
                                        row 2i+1: loop-back vehicles (route ends where it started) per direction, same lanes */
    int32_t *qwait;       /* [ni*4][n]  sum of Vehicle.waiting_time over the queue */
    uint32_t *misc;       /* [3][n]     current_timestep | flags << 16 ; len(self.vehicles) ; rng_counter */
    double *total_reward; /* [n]        running episode return (info["total_reward"]) */
} beng_traffic_state;

typedef struct beng_traffic_io {
    float *obs;            /* [n][ni*14+4]  _get_observation (environment.py:313-363) */
    float *reward;         /* [n]           _calculate_reward (:287-311) cast to float32 */
    uint8_t *terminated;   /* [n]           current_timestep >= MAX_TIMESTEPS (:196) */
    uint8_t *truncated;    /* [n]           always 0 (:197) */
    double *reward64;      /* [n] nullable  the float64 reward */
    double *ep_return;     /* [n] nullable  written when an episode ends (auto-reset modes) */
    int32_t *ep_length;    /* [n] nullable */
    double *stats;         /* [3] nullable  running {n_episodes, sum_return, sum_length} */
    int32_t *timestep;     /* [n] nullable  info["timestep"] (environment.py:200): current_timestep after the call, 0 after a reset */
} beng_traffic_io;

/* TrafficManagementEnv.reset (environment.py:141-166) for envs with mask[i] != 0 (NULL = all); first_call != 0 also
 * rewinds the rng counter.  The observation of EVERY env is written to io->obs. */
int beng_traffic_reset(const beng_traffic_params *p, const beng_traffic_state *st, const beng_traffic_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream);

/* TrafficManagementEnv.step (environment.py:168-203): _apply_actions, every TrafficLight.update, _spawn_vehicles
 * (+ generate_vehicle_route), _process_intersections, _remove_completed_vehicles, _calculate_reward,
 * _get_observation and auto-reset, for all envs, in ONE kernel launch.  actions_dev: int64 [n][ni], values
 * 0 keep / 1 NS_GREEN / 2 EW_GREEN (anything else keeps, like the reference).  The kernels address the [field][env]
 * arrays with 32-bit element offsets: n_envs * ni * 4 must be below 2^32 (119 M envs on the default 9-intersection grid),
 * otherwise BENG_ERR_UNSUPPORTED. */
int beng_traffic_step(const beng_traffic_params *p, const beng_traffic_state *st, const int64_t *actions_dev,
                      const beng_traffic_io *io, int64_t n_envs, void *stream);

/* Same step with HOST action / result buffers; NULL host outputs are skipped; does not synchronise. */
int beng_traffic_step_host(const beng_traffic_params *p, const beng_traffic_state *st, int64_t *actions_dev,
                           const beng_traffic_io *io, int64_t n_envs, const int64_t *actions_host, float *obs_host,
                           float *reward_host, uint8_t *terminated_host, uint8_t *truncated_host, void *stream);

/* ------------------------------------------------------------------------------------------
 * smartclimate  (reference: smartclimate_rl-main/smartclimate/{env,utils}.py, class SmartClimateEnv)
 * SURVEY.md section 8(f) rank 3: the simplest float env on the same engine / boundary.
 * ------------------------------------------------------------------------------------------ */

#define BENG_CLIMATE_OBS_DIM 9

/* Constructor arguments (env.py:16-24) + batching parameters. */
typedef struct beng_climate_params {
    int32_t max_occupancy;         /* default 8 */
    int32_t episode_minutes;       /* default 1440; reported as `terminated` (env.py:107); <= 65535 */
    int32_t autoreset_mode;        /* BENG_AUTORESET_* */
    int32_t time_limit_truncation; /* 1: also set `truncated` at episode_minutes (gym.make's TimeLimit,
                                      smartclimate/__init__.py:6-10); 0: never (raw class, env.py:108) */
    uint64_t seed;
    uint64_t env_id_base;
} beng_climate_params;

/* Per-env state, [field][env] arrays (env index fastest).  float64 like the reference's Python floats. */
typedef struct beng_climate_state {
    double *f64;  /* [5][n] room_temp, outside_temp, ac_setting, total_reward, energy_usage */
    int32_t *i32; /* [4][n] num_people | lights << 8 | flags << 16 ; current_step ; comfort_time ; rng_counter */
} beng_climate_state;

typedef struct beng_climate_io {
    float *obs;           /* [n][9] room_temp, num_people, time_of_day, outside_temp, ac_setting, lights x4 (env.py:72-82) */
    float *reward;        /* [n]    calculate_reward (utils.py:30-50) cast to float32 */
    uint8_t *terminated;  /* [n]    current_step >= episode_minutes (env.py:107) */
    uint8_t *truncated;   /* [n]    always 0 (env.py:108) unless time_limit_truncation */
    double *reward64;     /* [n]    nullable */
    double *reward_terms; /* [3][n] nullable: info["comfort"], ["ac_penalty"], ["light_penalty"] (utils.py:46-50) */
    double *ep_return;    /* [n]    nullable, written when an episode ends (auto-reset modes) */
    int32_t *ep_length;   /* [n]    nullable */
    double *stats;        /* [3]    nullable running {n_episodes, sum_return, sum_length} */
} beng_climate_io;

/* SmartClimateEnv.reset / _init_state (env.py:48-70) for envs with mask[i] != 0 (NULL = all); first_call != 0 rewinds
 * the rng counter.  The observation of EVERY env is written to io->obs. */
int beng_climate_reset(const beng_climate_params *p, const beng_climate_state *st, const beng_climate_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream);

/* SmartClimateEnv.step (env.py:84-117) + utils.py:5-50 + auto-reset, ONE kernel launch.  The Dict action of the
 * reference is passed as two arrays: ac_temp_dev float32 [n] (action['ac_temp'][0]) and lights_dev int8 [n][4]. */
int beng_climate_step(const beng_climate_params *p, const beng_climate_state *st, const float *ac_temp_dev,
                      const int8_t *lights_dev, const beng_climate_io *io, int64_t n_envs, void *stream);

/* Same step with HOST action / result buffers; NULL host outputs are skipped; does not synchronise. */
int beng_climate_step_host(const beng_climate_params *p, const beng_climate_state *st, float *ac_temp_dev,
                           int8_t *lights_dev, const beng_climate_io *io, int64_t n_envs, const float *ac_temp_host,
                           const int8_t *lights_host, float *obs_host, float *reward_host, uint8_t *terminated_host,
                           uint8_t *truncated_host, void *stream);

/* ------------------------------------------------------------------------------------------
 * world_builder_env  (reference: world_builder_env/src/environment/{world_builder_env,game_logic}.py)
 * SURVEY.md section 8(f) rank 3: integer grid builder on the same engine / boundary.
 * ------------------------------------------------------------------------------------------ */

/* Constructor arguments (world_builder_env.py:38-44) + batching parameters.  The game constants (costs, production,
 * MAX_POPULATION 20, WIN_STEPS 50, initial resources) are compiled in (game_logic.py:13-57). */
typedef struct beng_builder_params {
    int32_t grid_size;      /* default 10; 2..15 */
    int32_t autoreset_mode; /* BENG_AUTORESET_* */
    uint64_t seed;
    uint64_t env_id_base;
} beng_builder_params;

/* Per-env scalar state, [word][env] int32 array (env index fastest):
 *   0 food  1 wood  2 stone  3 population  4 population_capacity
 *   5 building counts: farm | lumberyard << 8 | quarry << 16 | house << 24
 *   6 steps  7 win_steps | reached_win_population << 16 | flags << 24  8 rng_counter  9 running episode return
 * The grid itself lives in io->grid: it is both state and observation (one cell changes per successful build). */
typedef struct beng_builder_state {
    int32_t *words; /* [10][n] */
} beng_builder_state;

typedef struct beng_builder_io {
    int8_t *grid;            /* [n][G][G]  obs['grid'] AND the persistent grid state (0 empty, 1 farm, 2 lumberyard,
                                           3 quarry, 4 house); read and rewritten in place by every step */
    float *resources;        /* [n][4]     obs['resources'] = food, wood, stone, population (world_builder_env.py:205-210) */
    float *capacity;         /* [n][1]     obs['population_capacity'] */
    int32_t *win_steps;      /* [n][1]     obs['win_steps'] */
    float *flat_obs;         /* [n][G*G+6] nullable: the flatten_obs=True observation (:189-200) */
    float *reward;           /* [n]        execute_action's reward, or -100 / +100 on termination (:150-157) */
    uint8_t *terminated;     /* [n]        population <= 0, or 50 steps at population >= 20 (:233-247) */
    uint8_t *truncated;      /* [n]        always 0 (:148) */
    int32_t *ep_return;      /* [n] nullable, written when an episode ends (auto-reset modes) */
    int32_t *ep_length;      /* [n] nullable */
    int64_t *stats;          /* [4] nullable running {n_episodes, sum_return, sum_length, wins} (integer, exact) */
    int32_t *invalid_count;  /* [1] nullable: out-of-space actions seen (the reference raises ValueError, :135-136;
                                    such an env is left untouched) */
} beng_builder_io;

/* WorldBuilderEnv.reset (world_builder_env.py:99-123) for envs with mask[i] != 0 (NULL = all); first_call != 0 rewinds the
 * rng counter.  The observation of EVERY env is (re)written. */
int beng_builder_reset(const beng_builder_params *p, const beng_builder_state *st, const beng_builder_io *io,
                       const uint8_t *mask_dev, int64_t n_envs, int32_t first_call, void *stream);

/* WorldBuilderEnv.step (:125-166) + GameLogic.execute_action and helpers (game_logic.py:59-203) + auto-reset, ONE
 * kernel launch.  actions_dev: int64 [n], 0 pass / 1 farm / 2 lumberyard / 3 quarry / 4 house. */
int beng_builder_step(const beng_builder_params *p, const beng_builder_state *st, const int64_t *actions_dev,
                      const beng_builder_io *io, int64_t n_envs, void *stream);

/* Same step with HOST action / result buffers; NULL host outputs are skipped; does not synchronise. */
int beng_builder_step_host(const beng_builder_params *p, const beng_builder_state *st, int64_t *actions_dev,
                           const beng_builder_io *io, int64_t n_envs, const int64_t *actions_host, int8_t *grid_host,
                           float *resources_host, float *capacity_host, int32_t *win_steps_host, float *reward_host,
                           uint8_t *terminated_host, void *stream);

/* Grid change records of beng_builder_step_host_delta: one uint32_t per env and step, telling how the env's grid row
 * [G*G] differs from the one the previous step or reset wrote.  A step changes at most one cell.
 *   record  = cell (bits 0-7; cell = r * G + c < G*G <= 225) | value << 8 (bits 8-10; 0..4)
 *             | BENG_BUILDER_DELTA_CLEAR (bit 31); bits 11-30 are 0
 *   applied = clear the whole row if bit 31 is set, then, if value != 0, write value to the cell.
 *   A record is malformed when any of bits 11-30 is set, value > 4, value != 0 with cell >= G*G, or value == 0
 *   with cell != 0.
 * What the step kernel emits:
 *   successful build            cell | building << 8  (the k-th empty cell, building 1..4)
 *   pass, failed build (unaffordable or no empty cell), invalid action, end of episode without a reset
 *                               BENG_BUILDER_DELTA_NONE (the row does not change)
 *   any auto-reset              BENG_BUILDER_DELTA_CLEAR alone (a next-step reset at the start of the step, or a
 *                               same-step reset after the terminal step, which also undoes that step's build) */
#define BENG_BUILDER_DELTA_NONE 0x00000000u
#define BENG_BUILDER_DELTA_CLEAR 0x80000000u

/* beng_builder_step_host without the grid copy: enqueues H2D(actions) -> step kernel, which also writes one change
 * record per env to delta_dev -> D2H(records[, resources, capacity, win_steps], reward, terminated) on `stream`.
 * io->grid (and io->flat_obs when given) on the device is written exactly as by beng_builder_step.  A caller that
 * holds a host copy of the grids from before this step brings it up to date with beng_builder_apply_obs_delta once
 * the stream has drained: 33 B per env cross the bus instead of 129 B.  delta_dev / delta_host (uint32_t[n_envs],
 * device / pinned host, 4-byte aligned) are required; NULL result host pointers are skipped.  Does not synchronise. */
int beng_builder_step_host_delta(const beng_builder_params *p, const beng_builder_state *st, int64_t *actions_dev,
                                 const beng_builder_io *io, int64_t n_envs, const int64_t *actions_host,
                                 uint32_t *delta_dev, uint32_t *delta_host, float *resources_host, float *capacity_host,
                                 int32_t *win_steps_host, float *reward_host, uint8_t *terminated_host, void *stream);

/* Apply one step's change records (host memory, uint32_t[n_envs]) to a host copy of the grids (int8_t[n_envs][G][G]).
 * Pure host code: touches no CUDA state and runs without a GPU.  The envs are split into contiguous chunks over
 * n_threads threads (<= 0 means one), all joined before it returns.  Every record is checked before it is applied:
 * BENG_ERR_BAD_ARG for NULL buffers, n_envs < 0 or a malformed record (grid_host is then partly updated, the row of
 * the malformed record untouched), BENG_ERR_UNSUPPORTED for grid_size outside [2, 15]. */
int beng_builder_apply_obs_delta(const uint32_t *delta_host, int8_t *grid_host, int64_t n_envs, int32_t grid_size,
                                 int32_t n_threads);

/* ------------------------------------------------------------------------------------------
 * Running normalization of observations and rewards (Stable-Baselines3 VecNormalize semantics), for any env's
 * float32 [n][dim] observations and float32 [n] rewards.  INTEGRATION.md section "Normalizing observations and rewards"
 * states the semantics.
 * ------------------------------------------------------------------------------------------ */

#define BENG_NORM_OBS 1u    /* normalize io->obs into io->obs_out (skipped when obs_out is NULL) */
#define BENG_NORM_REWARD 2u /* normalize io->reward into io->reward_out (nullable) and zero io->returns where
                               terminated or truncated is set */
#define BENG_NORM_UPDATE 4u /* training: first update obs_rms with the batch (with BENG_NORM_OBS) and
                               returns = returns * gamma + reward, then ret_rms with the new returns (with BENG_NORM_REWARD) */

typedef struct beng_normalize_params {
    double clip_obs;    /* obs_out = clip((obs - mean) / sqrt(var + epsilon), -clip_obs, clip_obs) in float64, as float32 */
    double clip_reward; /* reward_out = clip(reward / sqrt(ret_var + epsilon), -clip_reward, clip_reward) */
    double epsilon;
    double gamma;
    uint32_t flags;     /* BENG_NORM_* */
    int32_t reserved;
} beng_normalize_params;

/* Running statistics records (float64, caller-owned, initialised to mean 0, var 1, count 1e-4):
 *   obs_rms : double[2 * dim + 1] = mean[dim], var[dim], count
 *   ret_rms : double[3]           = mean, var, count */
typedef struct beng_normalize_io {
    const float *obs;          /* [n][dim] row-major, 4-byte aligned (rows need not be 16-byte multiples) */
    const float *reward;       /* [n] */
    const uint8_t *terminated; /* [n] nullable (no env finished) */
    const uint8_t *truncated;  /* [n] nullable */
    double *returns;           /* [n] discounted running return of every env */
    double *obs_rms;
    double *ret_rms;
    void *workspace;           /* beng_normalize_workspace_bytes(n, dim) bytes, 16-byte aligned, zero before the first
                                  call; its arrival counter is 0 again when each call's launches end */
    float *obs_out;            /* [n][dim] nullable; must not overlap obs */
    float *reward_out;         /* [n] nullable */
} beng_normalize_io;

/* Workspace bytes beng_normalize needs for (n_envs, dim); 0 for n_envs < 0 or dim < 1. */
size_t beng_normalize_workspace_bytes(int64_t n_envs, int32_t dim);

/* One update / normalize of n_envs envs.  With BENG_NORM_UPDATE: two launches, a moments pass (every CTA sums its rows
 * shifted by row 0 in float64; the last CTA to arrive adds the partials in CTA order and merges the batch into obs_rms /
 * ret_rms with Chan's update) and an apply pass; without it only the apply pass.  None when n_envs == 0 or there is
 * nothing to write.  The statistics depend only on the inputs and (n_envs, dim): bit-identical run to run, on every
 * device and from a CUDA graph.  Pointers the flags need are checked (non-NULL, aligned: float / uint8 4 / 1 bytes,
 * double 8) before anything launches: BENG_ERR_BAD_ARG, also for n_envs < 0, dim < 1, unknown flags and negative or NaN
 * clip / epsilon / gamma.  obs and obs_rms are read only with BENG_NORM_OBS, dim is then the observation width;
 * reward / returns / ret_rms only with BENG_NORM_REWARD. */
int beng_normalize(const beng_normalize_params *p, const beng_normalize_io *io, int64_t n_envs, int32_t dim,
                   void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BENG_H */
