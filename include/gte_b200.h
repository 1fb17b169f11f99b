/*
 * gte_b200.h — C-ABI of libgte_b200.so: the B200 (sm_100a) batched drop-in for the per-step
 * simulation hot path of ten2net/Gym-Trading-Env.
 *
 * The reference has no FFI layer: the path sits behind the gymnasium Env API
 * (src/gym_trading_env/__init__.py:3-14 registers `TradingEnv` / `MultiDatasetTradingEnv`;
 * src/gym_trading_env/environments.py:163 `reset`, :233 `step`).  The entry points below are what a
 * binding for a batched version of exactly those calls needs; each one names the reference
 * function(s) it replaces.  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *  - plain C, POD structs, no torch types.  Every pointer inside the structs is a DEVICE pointer
 *    (e.g. torch.Tensor.data_ptr()) unless stated otherwise; the structs themselves live on the host.
 *  - the library never allocates, frees or retains device memory: it borrows the pointers for the
 *    duration of the call (the caller owns every buffer; outputs are overwritten in place).
 *  - calls only enqueue work on `stream` (a cudaStream_t passed as void*; NULL = default stream)
 *    and return without synchronising.
 *  - the library keeps a few process-wide caches (SM count, kernel attributes, side stream): make the calls
 *    from one host thread at a time.
 *  - return value: 0 = success, GTE_ERR_ARG (-1) = bad argument, GTE_ERR_CUDA (-2) = CUDA error;
 *    gte_last_error() returns a thread-local message for the last failing call.
 *  - all money math is IEEE fp64 round-to-nearest in the reference's exact operation order with
 *    no FMA contraction (utils/portfolio.py:7-46), so portfolio state and valuation are bit-exact.
 */
#ifndef GTE_B200_H
#define GTE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GTE_VERSION 203            /* 0.2.3 */
#define GTE_MAX_POSITIONS 64
#define GTE_MAX_DATASETS 64        /* least-used rotation keeps a 64-bit "used this round" mask per env */
#define GTE_N_METRICS 8
/* dynamic-feature ring: one block per tile of 32 consecutive envs (layout at GteState.dyn_ring) for any dynamic-feature
 * catalogue (GteParams.dyn_kinds): n_f32 blocks of W rows x 32 f32 values, one per f32 kind, then n_pos (0 or 1) blocks
 * of W rows x 32 u8 position indices. */
#define GTE_RING_TILE_ENVS 32
#define GTE_MAX_DYN 5
#define GTE_RING_TILE_BYTES_DYN(W, n_f32, n_pos) ((W) * (128 * (n_f32) + 32 * (n_pos)))
#define GTE_RING_BYTES_DYN(N, W, n_f32, n_pos) ((((int64_t)(N) + 31) / 32) * GTE_RING_TILE_BYTES_DYN(W, n_f32, n_pos))
#define GTE_RING_F32_OFFSET(W, k, s, e) ((k) * (W) * 128 + (s) * 128 + (((((e) >> 2) ^ ((s) & 7))) << 4) + (((e) & 3) << 2))
#define GTE_RING_POS_OFFSET_DYN(W, n_f32, s, e) ((n_f32) * (W) * 128 + (s) * 32 + (e))
/* The default pair (position, real_position): n_f32 = n_pos = 1, real_position in f32 block 0. */
#define GTE_RING_TILE_BYTES(W) GTE_RING_TILE_BYTES_DYN(W, 1, 1)
#define GTE_RING_BYTES(N, W) GTE_RING_BYTES_DYN(N, W, 1, 1)
#define GTE_RING_RP_OFFSET(s, e) GTE_RING_F32_OFFSET(0, 0, s, e)
#define GTE_RING_POS_OFFSET(W, s, e) GTE_RING_POS_OFFSET_DYN(W, 1, s, e)
#define GTE_STEP_THREADS 256       /* envs per tile of the step kernel */
#define GTE_MAX_PARTIAL_ROWS 4096  /* rows of GteStepOut.metric_partials (one per CTA; every grid is capped at this) */
/* Result block of gte_step_host — everything a host policy needs back from one iteration, in ONE piece of memory
 * (device copy and pinned host copy have the same layout):
 *   reward f64[N] | header (32 B) | ended u32[cap] | terminated u8[N] | truncated u8[N] | pad to 8
 *   header: error_flag i32 | sequence u32 | n_ended u32 | cap u32 | append counter u32 (device side) | 12 B pad
 *   ended[j] (j < min(n_ended, cap)): one entry per env whose episode ended in this iteration, in no particular order:
 *            bit 31 terminated, bit 30 truncated, bits 0..29 the env index.  Episode ends are rare (1 env in
 *            max_episode_duration per iteration), so `reward | header | ended` — the SPARSE prefix — carries the flags of
 *            a large batch in 8.1 instead of 10 bytes per env; the dense byte arrays are only needed when more than `cap`
 *            episodes ended at once.
 * The device copy must be zero-initialised before its first use (the append counter lives in it). */
#define GTE_HOST_RESULT_ENDED_CAP(N) ((((int64_t)(N) / 32 > 1024 ? (int64_t)(N) / 32 : 1024) + 3) / 4 * 4)
#define GTE_HOST_RESULT_ERROR_OFFSET(N) ((int64_t)(N) * 8)
#define GTE_HOST_RESULT_SEQ_OFFSET(N) (GTE_HOST_RESULT_ERROR_OFFSET(N) + 4)
#define GTE_HOST_RESULT_NENDED_OFFSET(N) (GTE_HOST_RESULT_ERROR_OFFSET(N) + 8)
#define GTE_HOST_RESULT_COUNTER_OFFSET(N) (GTE_HOST_RESULT_ERROR_OFFSET(N) + 16)
#define GTE_HOST_RESULT_ENDED_OFFSET(N) (GTE_HOST_RESULT_ERROR_OFFSET(N) + 32)
#define GTE_HOST_RESULT_SPARSE_BYTES(N) (GTE_HOST_RESULT_ENDED_OFFSET(N) + 4 * GTE_HOST_RESULT_ENDED_CAP(N))
#define GTE_HOST_RESULT_TERM_OFFSET(N) GTE_HOST_RESULT_SPARSE_BYTES(N)
#define GTE_HOST_RESULT_TRUNC_OFFSET(N) (GTE_HOST_RESULT_TERM_OFFSET(N) + (int64_t)(N))
#define GTE_HOST_RESULT_BYTES(N) ((GTE_HOST_RESULT_TRUNC_OFFSET(N) + (int64_t)(N) + 7) / 8 * 8)

#define GTE_OK 0
#define GTE_ERR_ARG (-1)
#define GTE_ERR_CUDA (-2)

/* metric slots: sums over the episodes that FINISHED in this call, except SUM_REWARD (all envs) */
enum GteMetric {
    GTE_M_EPISODES = 0,            /* number of finished episodes                                  */
    GTE_M_TERMINATED = 1,          /* ... that hit the valuation stop   (environments.py:246)       */
    GTE_M_TRUNCATED = 2,           /* ... that hit end-of-data / max duration (:248-251)            */
    GTE_M_SUM_PORTFOLIO_RETURN = 3,/* sum of valuation_end/initial - 1  (:282 "Portfolio Return")   */
    GTE_M_SUM_MARKET_RETURN = 4,   /* sum of close_end/close_start - 1  (:281 "Market Return")      */
    GTE_M_SUM_EPISODE_LENGTH = 5,  /* sum of episode lengths in steps                              */
    GTE_M_SUM_REWARD = 6,          /* sum of this iteration's rewards over all envs                */
    GTE_M_RESERVED = 7
};

/* Fused reward functors.  The reference takes an arbitrary Python `reward_function(history)`
 * (environments.py:50-51, :266); the catalogue covers the default and the variants its callers use:
 * luckymodel/envs/env.py:16-18 (log-return clipped to [-0.002, 0.005]), luckymodel/scripts/test_env.py:20-22
 * (100 x log-return), and the simple / positive-part return of env.py:19. */
enum GteRewardKind {
    GTE_REWARD_LOG_RETURN = 0,     /* f = log(v_t / v_{t-1})                 basic_reward_function, :17-18 */
    GTE_REWARD_SIMPLE_RETURN = 1   /* f = (v_t - v_{t-1}) / v_{t-1}                                         */
};

/* Dynamic-feature kinds (GteParams.dyn_kinds): the device catalogue standing in for the reference's
 * `dynamic_feature_functions` (environments.py:43-48, :153-154).  Each column is the fp64 value cast to float32;
 * in an episode's first row (the reset row, :191-192) position and real_position read the position, the others 0.
 * The STATEFUL kinds (6, 7) depend on the whole episode: they keep their running state in GteState.episode_acc
 * (row GTE_ACC_PEAK, shared with the max_drawdown metric, and row GTE_ACC_POSITION_AGE), so a configuration with
 * one of them needs episode_acc.  Their f32 ring blocks follow the others in kind-code order. */
enum GteDynKind {
    GTE_DYN_POSITION = 1,          /* history["position", -1]            (:20-21; u8 position index in the ring) */
    GTE_DYN_REAL_POSITION = 2,     /* history["real_position", -1]       (:23-24)                                */
    GTE_DYN_PORTFOLIO_RETURN = 3,  /* history["portfolio_valuation", -1] / history["portfolio_valuation", 0] - 1 */
    GTE_DYN_REWARD = 4,            /* history["reward", -1]: the step's reward (0 when terminated)               */
    GTE_DYN_EPISODE_PROGRESS = 5,  /* history["step", -1] / max_episode_duration                                 */
    GTE_DYN_CURRENT_DRAWDOWN = 6,  /* 1 - v[-1] / max(v), v = history["portfolio_valuation"] (stateful)          */
    GTE_DYN_POSITION_AGE = 7       /* History rows since the position last changed (by value), back to the reset
                                      row when it never did: a raw count, exact in f32 up to 2^24 (stateful)   */
};

/* Episode-metric kinds (GteParams.metric_kinds, bit 1 << kind): the device catalogue standing in for the reference's
 * TradingEnv.add_metric(name, function) (environments.py:274-294).  Each value is computed in the step kernel in fp64,
 * in the reference's operation order, over the episode's History (reset row included), and recorded at the episode's
 * end in GteStepOut.episode_record row 2 + kind. */
enum GteMetricKind {
    GTE_METRIC_POSITION_CHANGES = 0, /* np.sum(np.diff(history["position"]) != 0): rows whose position differs from the previous row */
    GTE_METRIC_EPISODE_LENGTH = 1,   /* len(history["position"]) = terminal step + 1                                               */
    GTE_METRIC_MAX_DRAWDOWN = 2,     /* max(1 - v / running max(v)), v = history["portfolio_valuation"]                             */
    GTE_METRIC_EPISODE_REWARD = 3,   /* sum(history["reward"]), Python's left-to-right sum                                          */
    GTE_METRIC_TIME_IN_MARKET = 4    /* mean(history["position"] != 0)                                                              */
};
#define GTE_N_METRIC_KINDS 5
#define GTE_METRIC_KINDS_ALL 0x1f
/* Rows of GteState.episode_acc (f64 [GTE_EPISODE_ACC_ROWS, N]): the running state of the current episode.  Counts are
 * stored as f64 (exact below 2^53).  Only the rows of configured kinds are read or written: row 5 only when the
 * position_age dynamic feature is configured, so a caller without that kind may allocate 5 rows ([5, N]). */
#define GTE_EPISODE_ACC_ROWS 6
enum GteEpisodeAccRow {
    GTE_ACC_PEAK = 0,                /* running max of the valuation (max_drawdown, current_drawdown) */
    GTE_ACC_DRAWDOWN = 1,            /* max drawdown so far (max_drawdown)                           */
    GTE_ACC_REWARD_SUM = 2,          /* sum of the rewards so far (episode_reward)                   */
    GTE_ACC_POSITION_CHANGES = 3,    /* rows whose position differs from the previous row            */
    GTE_ACC_IN_MARKET = 4,           /* rows whose position is not 0 (time_in_market)                */
    GTE_ACC_POSITION_AGE = 5         /* rows since the position last changed (position_age)          */
};
/* Rows of GteStepOut.episode_record (f64 [GTE_EPISODE_RECORD_ROWS, N]): row 0 the market return close[-1] / close[0] - 1,
 * row 1 the portfolio return valuation[-1] / valuation[0] - 1 (environments.py:281-282), row 2 + k metric kind k. */
#define GTE_EPISODE_RECORD_ROWS 7
/* the kinds that keep per-episode state in episode_acc (episode_length is the terminal step + 1) */
#define GTE_METRIC_KINDS_STATEFUL ((1 << GTE_METRIC_POSITION_CHANGES) | (1 << GTE_METRIC_MAX_DRAWDOWN) | \
                                   (1 << GTE_METRIC_EPISODE_REWARD) | (1 << GTE_METRIC_TIME_IN_MARKET))

/* GTE_E_PAST_END: an env stepped again after its episode reached the last row T-1 of its data (autoreset == 0, no reset
 * in between).  The step is an ordinary transition from row T-2 to row T-1, computed from the env's current portfolio:
 * the previous valuation is that portfolio valued at price[T-2] (portfolio_initial_value for an episode that started at
 * T-2), the trade happens at price[T-2], then interest, then the valuation at price[T-1]; it is reported as truncated,
 * counted in the batch metrics and folded into the episode accumulators like any truncation.  info idx / step and the
 * stored row ep_start + step stay at T-1 (episode_progress does not grow), so no reader leaves the data. */
enum GteErrorBit {
    GTE_E_ACTION_RANGE = 1, GTE_E_PAST_END = 2, GTE_E_PLAN_RANGE = 4, GTE_E_PLAN_EXHAUSTED = 8, GTE_E_NEGATIVE_ACTION = 16
};

/* observation-gather kernel variants (gte_gather_obs `variant`) */
enum GteObsVariant {
    GTE_OBS_AUTO = 0,              /* fastest variant the shape allows                              */
    GTE_OBS_GENERIC = 1,           /* scalar gather, any shape (windows=None, odd row sizes)        */
    GTE_OBS_VEC = 2,               /* 128-bit LDG/STG from the 16B-aligned window tables            */
    GTE_OBS_TMA = 3                /* cp.async.bulk global->smem->global, dynamic columns patched in smem */
};

/* Constructor parameters: TradingEnv.__init__ (environments.py:79-110) and
 * MultiDatasetTradingEnv.__init__ (:365-378). */
typedef struct GteParams {
    int32_t n_envs;                  /* envs owned by THIS process / GPU                               */
    int32_t n_positions;             /* len(positions)  (:98, action space Discrete(P) :112)           */
    int32_t windows;                 /* `windows` (:101); 0 = None                                     */
    int32_t n_static;                /* static "feature*" columns (:130)                               */
    int32_t n_dyn;                   /* dynamic feature columns, 0..GTE_MAX_DYN (see dyn_kinds)          */
    int32_t max_episode_duration;    /* (:94) -1 = 'max'                                               */
    int32_t n_datasets;              /* 1 for TradingEnv                                               */
    int32_t initial_position_idx;    /* index into positions, -1 = 'random' (:105, :167)               */
    int32_t episodes_between_switch; /* `episodes_between_dataset_switch` (:370)                       */
    int32_t plan_episodes;           /* E of reset_plan[N,E,3]; 0 = draw resets from Philox            */
    int32_t multi_dataset;           /* 1 = MultiDatasetTradingEnv.reset semantics (:393-400)          */
    int32_t reward_kind;             /* enum GteRewardKind: which fused reward functor (:50-51 `reward_function`) */
    int32_t n_limit_positions;       /* how many positions carry limit orders (0 = feature off, :217-231)          */
    int32_t action_bytes;            /* element width of the `actions` array: 1, 2, 4 or 8 (signed ints); 0 = 8.
                                        Discrete(P) fits int8 for every P <= GTE_MAX_POSITIONS: the narrow widths cut the
                                        host->device bytes of a host policy 8x and are widened in the step kernel's load */
    int32_t strict_actions;          /* 1: any negative action other than -1 sets error bit 4 (still treated as hold).
                                        The reference's positions[-k] would index from the END of the list (:234)        */
    int32_t dyn_kinds;               /* enum GteDynKind of dynamic column j in bits 4j..4j+3, each kind at most once.
                                        0 = the defaults: n_dyn == 0 none, n_dyn == 2 (position, real_position)
                                        (:20-24, :82), the same descriptor as the explicit 0x21.  episode_progress
                                        needs max_episode_duration > 0; current_drawdown and position_age need
                                        GteState.episode_acc (rows 0..5 with position_age, else rows 0..4)       */
    int64_t t_stride;                /* rows allocated per dataset in `price` / `features`             */
    int64_t env_id_offset;           /* global index of env 0 (multi-GPU sharding; keys the RNG)       */
    uint64_t seed;                   /* Philox key                                                     */
    double fee;                      /* `trading_fees` (:102)                                          */
    double rate;                     /* `borrow_interest_rate` (:103)                                  */
    double v0;                       /* `portfolio_initial_value` (:104)                               */
    double done_ratio;               /* terminated = valuation/v0 <= done_ratio; 0.7 in this fork (:246) */
    double reward_scale;             /* reward = clip(reward_scale * f(valuation, previous valuation),      */
    double reward_lo;                /*               reward_lo, reward_hi); defaults 1, -inf, +inf give   */
    double reward_hi;                /*               basic_reward_function bit for bit                    */
    double positions[GTE_MAX_POSITIONS]; /* `positions` (:98)                                          */
    int32_t metric_kinds;            /* episode metrics (add_metric, :274-294): bit 1 << k for enum GteMetricKind k.  Non-zero
                                        turns the per-episode record on (GteStepOut.episode_record, and GteState.episode_acc
                                        for the kinds in GTE_METRIC_KINDS_STATEFUL); 0 = off, the record is not written */
    int32_t pad_metric;              /* 0                                                              */
} GteParams;

/* Device-resident market data: what TradingEnv._set_df builds (environments.py:128-143). */
typedef struct GteData {
    const float* features;           /* f32 [n_datasets, t_stride, n_static]  (_obs_array static part, :141) */
    const double* price;             /* f64 [n_datasets, t_stride]            (_price_array, :143)            */
    const int32_t* lengths;          /* i32 [n_datasets]  len(df) of each dataset                              */
    const double* high;              /* f64 [n_datasets, t_stride] "high" column, or NULL (only limit orders read it, :221) */
    const double* low;               /* f64 [n_datasets, t_stride] "low" column, or NULL                                   */
    /* 16-byte-aligned window tables for the vector/TMA gather: copy c holds rows in the reference's
     * own [t, n_static+n_dyn] layout (dynamic columns zero) shifted so that a window starting at row
     * r0 with (r0*row_bytes) % 16 == 4*c starts on a 16-byte boundary.  NULL where unused. */
    const float* window_table[4];
    int64_t window_table_ds_stride;  /* bytes between datasets inside one copy (multiple of 16)               */
} GteData;

/* Per-env state, structure of arrays (the reference's Portfolio fields, utils/portfolio.py:2-6,
 * plus TradingEnv._position/_step/_idx as indices).  idx = ep_start + step. */
typedef struct GteState {
    double* asset;                   /* f64 [N]  signed: negative = borrowed asset (portfolio.py:53)    */
    double* fiat;                    /* f64 [N]  signed: negative = borrowed fiat  (portfolio.py:54)    */
    double* interest_asset;          /* f64 [N]                                                        */
    double* interest_fiat;           /* f64 [N]                                                        */
    int32_t* pos_idx;                /* i32 [N]  index of TradingEnv._position in positions            */
    int32_t* step;                   /* i32 [N]  TradingEnv._step                                      */
    int32_t* ep_start;               /* i32 [N]  _idx at reset (episode start row)                     */
    int32_t* dataset_idx;            /* i32 [N]  which dataset the env is on                           */
    /* Dynamic-feature ring, indexed by TIME: the row an env observed at lockstep iteration c (c = *ring_clock,
     * advanced by every gte_step / gte_step_obs call) lives in slot c % W, W = max(windows,1); a window reads slots
     * c-W+1 .. c, and its rows before ep_start read as zero (the env was reset less than W iterations ago).
     * Memory: one contiguous block per tile of 32 consecutive envs, so that the gather fetches a tile's whole ring
     * with one bulk copy while one iteration's stores are a full 128-byte line (+ a full 32-byte sector) per warp
     * and column.  Inside a block: for each configured f32 kind, in kind-code order (real_position, portfolio_return,
     * reward, episode_progress), W rows of 32 f32 values — f32 block k, env lane e of slot s at
     * GTE_RING_F32_OFFSET(W, k, s, e), 16-byte chunks XOR-swizzled by the slot so that column reads from shared memory
     * spread over the banks — then, when "position" is configured, W rows of 32 u8 position INDICES at
     * GTE_RING_POS_OFFSET_DYN(W, n_f32, s, e) (the feature is float32(positions[index]), :20-21).  The default pair is
     * GTE_RING_TILE_BYTES(W) per tile with real_position at GTE_RING_RP_OFFSET and the indices at GTE_RING_POS_OFFSET. */
    uint8_t* dyn_ring;               /* u8 [GTE_RING_BYTES_DYN(N, W, n_f32, n_pos)], 16-byte aligned; unused when n_dyn == 0 */
    uint64_t* ring_clock;            /* u64 [1]  lockstep iterations so far, advanced ON THE DEVICE              */
    int32_t* plan_cursor;            /* i32 [N]  next episode slot of reset_plan                       */
    uint64_t* ds_used;               /* u64 [N]  datasets used in the current rotation round (:383)    */
    int32_t* ds_episodes;            /* i32 [N]  _episodes_on_this_dataset (:381,394)                  */
    const int32_t* reset_plan;       /* i32 [N, E, 3] (start row, position idx, dataset idx) or NULL   */
    double* limit_price;             /* f64 [N, n_positions]: persistent limit order per target position
                                        (TradingEnv.add_limit_order :227-231), NaN = none; cleared at reset (:168) */
    const int32_t* limit_seq;        /* i32 [n_limit_positions]: position indices in the order the orders are tried
                                        (the reference iterates its dict in insertion order, :220)              */
    int32_t* error_flag;             /* i32 [1]  sticky bits, OR-ed by the kernels (enum GteErrorBit):
                                                 1 action >= n_positions (treated as hold); 2 an env was stepped past the
                                                 end of its data; 4 a reset_plan row out of range (clamped); 8 reset_plan
                                                 exhausted (wrapped around); 16 negative action other than -1 (strict_actions) */
    uint64_t* tick;                  /* u64 [1]  event counter keying the Philox draws; every gte_reset /
                                        gte_step / gte_step_obs call advances it by one ON THE DEVICE, so
                                        a captured CUDA graph of a step replays with fresh draws       */
    double* episode_acc;             /* f64 [GTE_EPISODE_ACC_ROWS, N] running state of the current episode (enum GteEpisodeAccRow),
                                        initialised from the reset row by every reset and by the auto-reset; needed when
                                        metric_kinds has a GTE_METRIC_KINDS_STATEFUL bit or dyn_kinds a stateful kind
                                        (6, 7), else may be NULL.  [5, N] suffices without position_age (row 5)     */
} GteState;

/* Outputs of one lockstep iteration.  reward / flags / valuation / real_position / info_* are the
 * values of the step just taken (terminal values where an episode ended); obs and GteState are
 * post-reset where the in-place auto-reset fired.  NULL pointers are skipped. */
typedef struct GteStepOut {
    double* reward;                  /* f64 [N]  log(valuation/previous valuation), 0 when terminated (:17-18,:263-267) */
    uint8_t* terminated;             /* u8  [N]                                                         */
    uint8_t* truncated;              /* u8  [N]                                                         */
    double* valuation;               /* f64 [N]  info["portfolio_valuation"] (:241)               or NULL */
    double* real_position;           /* f64 [N]  info["real_position"] (:259)                     or NULL */
    int32_t* info_idx;               /* i32 [N]  info["idx"]                                      or NULL */
    int32_t* info_step;              /* i32 [N]  info["step"]                                     or NULL */
    double* pre_reset_portfolio;     /* f64 [4, N] asset, fiat, interest_asset, interest_fiat before the auto-reset, or NULL */
    double* metric_partials;         /* f64 [GTE_MAX_PARTIAL_ROWS, GTE_N_METRICS] scratch (one row per CTA)   */
    double* metrics_step;            /* f64 [GTE_N_METRICS] this iteration's metrics                    */
    double* metrics_total;           /* f64 [GTE_N_METRICS] running totals (+= metrics_step)    or NULL */
    uint32_t* block_counter;         /* u32 [1]  zero-initialised scratch (self-resetting)              */
    int32_t* error_out;              /* i32 [1]  the last CTA of the launch stores *state->error_flag here, or NULL.
                                        May be mapped host memory: the flag then reaches the host with the results     */
    uint32_t* seq_out;               /* u32 [1]  or NULL: after every result of the launch is visible system-wide, the last
                                        CTA stores seq_value here — a host thread polling mapped memory sees the
                                        iteration complete without a driver call.  MUST be the upper half of an aligned
                                        8-byte word whose lower half is the error flag's destination (the layout of the
                                        host result block): the two are published with one 8-byte store, error_out itself
                                        is then not written                                                            */
    uint32_t seq_value;
    uint32_t ended_cap;              /* entries ended_list can hold                                                     */
    uint32_t* ended_list;            /* u32 [ended_cap] or NULL: every env whose episode ends in this launch appends
                                        (terminated << 31) | (truncated << 30) | env index (any order)                  */
    uint32_t* ended_counter;         /* u32 [1], device memory, zero before the first launch: the append cursor; the last
                                        CTA of the launch moves its value to ended_n_out and resets it                  */
    uint32_t* ended_n_out;           /* u32 [1]: how many episodes ended in this launch (may exceed ended_cap: the list
                                        then holds only the first ended_cap of them and the dense flags must be read)   */
    float* reward_f32;               /* f32 [N] or NULL: the reward ALSO rounded to float32 (numpy's cast) — the opt-in,
                                        LOSSY wire of a trainer that keeps float32 rewards anyway (stable-baselines3)   */
    double* episode_record;          /* f64 [GTE_EPISODE_RECORD_ROWS, N], required when metric_kinds != 0 (read only then): the
                                        metrics of each env's most recently FINISHED episode (row layout at
                                        GTE_EPISODE_RECORD_ROWS; rows 2 + k only for configured kinds k).  Written at
                                        an episode's end, from its terminal values, before the auto-reset; the columns of
                                        the other envs are left untouched.  gte_rollout does not replicate it per
                                        iteration: afterwards it holds the last episode each env finished.  With it, a
                                        gte_step_obs call never takes the fused launch (gte_step_obs_launches says so) */
} GteStepOut;

/* Host side of one lockstep iteration for a HOST policy (gte_step_host): actions come from pinned host memory,
 * reward / terminated / truncated / error flag land in ONE pinned host block, observations stay in HBM. */
enum GteHostIOMode {
    GTE_IO_AUTO = 0,                 /* MAPPED while N * (action_bytes + 10) <= 384 KiB (1 MiB with windows == 0), else COPY */
    GTE_IO_COPY = 1,                 /* copy engines: ONE cudaMemcpyAsync per direction, beside the gather  */
    GTE_IO_MAPPED = 2,               /* zero-copy: the step kernel reads the actions from, and writes its
                                        10 B/env of results straight into, the pinned (UVA-mapped) host memory:
                                        no copy to enqueue                                                 */
    GTE_IO_SERVER = 3                /* MAPPED without the launch: a resident kernel (launched by the first call, on a
                                        library-owned stream) waits for each call's request in mapped host memory and
                                        answers into the result block — no kernel launch, driver call or interrupt per
                                        step: the small-N latency floor.  Needs windows == 0 and a batch that is
                                        resident at once (n_envs <= 256 x SMs), else the call runs as MAPPED.  The kernel
                                        leaves when any other entry point of the library is called, on gte_serve_stop(),
                                        or after GTE_SERVER_IDLE_US (default 2000) without a request, and is launched
                                        again by the next call.  While it is resident the env state belongs to it: do
                                        not touch the state buffers from other streams.                      */
};
typedef struct GteHostIO {
    const void* actions;             /* HOST, pinned: [N] signed ints of params->action_bytes bytes each              */
    void* results;                   /* HOST, pinned: GTE_HOST_RESULT_BYTES(N) bytes, layout above                     */
    void* dev_actions;               /* DEVICE staging, N * action_bytes bytes (COPY mode)                             */
    void* dev_results;               /* DEVICE block of GTE_HOST_RESULT_BYTES(N) bytes, same layout (COPY mode)        */
    void* step_done_event;           /* cudaEvent_t recorded on `stream` right behind the step kernel, or NULL: lets the
                                        caller hang more work (the metric all-reduce) beside the gather                */
    void* obs_host;                  /* HOST, pinned, or NULL: the observation batch is ALSO delivered here (a host policy
                                        that reads observations: gymnasium / stable-baselines3 numpy semantics) — with
                                        windows == 0 in the MAPPED / SERVER modes the step kernel writes its one-row
                                        observations straight into it (the device `obs` is then left untouched), else
                                        one more device-to-host copy behind the gather; the call returns when it landed */
    int64_t obs_bytes;               /* size of the observation batch in bytes (N * W * F * 4)                          */
    void* reward_f32_host;           /* HOST, pinned, f32 [N], or NULL.  With dev_reward_f32 (copy engines only): the rewards
                                        cross PCIe rounded to float32 (4 instead of 8 bytes per env: LOSSY, opt-in) and the
                                        fp64 rewards stay on the device; the result block then only brings back its
                                        header + ended list (sparse_flags) or header + list + dense flags              */
    void* dev_reward_f32;            /* DEVICE, f32 [N], or NULL                                                          */
    int64_t reward_host_count;       /* copy engines only; 0 or N = all.  0 < count < N: this call's own device-to-host copy
                                        delivers only the FIRST count rewards (and the header / ended list / flags); rewards
                                        [count, N) stay in the device block for the caller to route to the host through a
                                        peer GPU's PCIe link (gte_relay_push) — the multi-GPU result relay              */
    int32_t mode;                    /* enum GteHostIOMode                                                             */
    int32_t sparse_flags;            /* copy engines only: bring back just the sparse prefix of the result block
                                        (GTE_HOST_RESULT_SPARSE_BYTES: reward | header | ended list) — the dense
                                        terminated / truncated bytes follow, inside the same call, only when more than
                                        `cap` episodes ended at once (header: n_ended > cap)                            */
} GteHostIO;

/* Lazily computed info columns (History's last row, environments.py:253-264 / utils/history.py). */
typedef struct GteInfo {
    int32_t* idx; int32_t* step; int32_t* position_index; int32_t* dataset_idx;   /* i32 [N] or NULL */
    double* position; double* real_position; double* portfolio_valuation;         /* f64 [N] or NULL */
    double* data_close;                                                            /* f64 [N] or NULL */
    double* distribution;            /* f64 [6, N]: asset, fiat, borrowed_asset, borrowed_fiat,
                                        interest_asset, interest_fiat (portfolio.py:49-57) or NULL  */
} GteInfo;

int gte_version(void);
const char* gte_last_error(void);
/* Hash of the CUDA sources the library was compiled from (set by the build line, -DGTE_BUILD_ID=...); bindings
 * compare it with the hash of the sources they ship to refuse a stale binary. */
const char* gte_build_id(void);

/* Replaces TradingEnv.reset (environments.py:163-199) [+ MultiDatasetTradingEnv.reset :393-400 and,
 * with first != 0, ONLY the dataset draw of MultiDatasetTradingEnv.__init__ :377-378] for every env
 * whose mask byte is non-zero (mask == NULL: all envs).  Episode start / initial position / dataset
 * come from state->reset_plan when params->plan_episodes > 0, else from Philox4x32-10 keyed by
 * (seed, *state->tick, global env id). */
int gte_reset(const GteParams* params, const GteData* data, const GteState* state,
              const uint8_t* mask, int first, void* stream);

/* Replaces TradingEnv.step (environments.py:233-272) for N envs: _take_action/_trade (:204-215) ->
 * Portfolio.trade_to_position (portfolio.py:18-43) -> index advance -> update_interest (:44-46) ->
 * valorisation (:7-13) -> done/truncated (:244-251) -> basic_reward_function (:17-18) -> episode
 * metrics (:279-283) -> in-place auto-reset when autoreset != 0.  actions: [N] signed ints of
 * params->action_bytes bytes (i64 by default), indices into positions; a negative action = hold (the reference's
 * position_index=None, :234). */
int gte_step(const GteParams* params, const GteData* data, const GteState* state,
             const void* actions, const GteStepOut* out, int autoreset, void* stream);

/* Replaces TradingEnv._get_obs (environments.py:152-160): obs f32 [N, F] (windows=None) or
 * [N, W, F], F = n_static + n_dyn; static columns gathered from the device-resident tables,
 * dynamic columns (in dyn_kinds order) from the dynamic-feature ring; window rows before the episode start are 0. */
int gte_gather_obs(const GteParams* params, const GteData* data, const GteState* state,
                   float* obs, int variant, void* stream);

/* One whole lockstep iteration — what a vector env's step() returns: gte_step + gte_gather_obs.
 * n_chunks: 0 = the library's choice: ONE fused launch (every CTA advances its own envs, then gathers their windows)
 * while the batch fits a single wave with <= 256 envs per CTA (~100k envs on a B200), metric_kinds == 0 and no stateful
 * dynamic feature is configured, else two plain launches;
 * 1 = always two plain launches (measured fastest for large batches, profiles/r01_tuning.md).  n_chunks > 1
 * is an opt-in experiment: the envs are cut into that many ranges and the step kernel of range c+1 runs beside the
 * gather of range c on a library-owned side stream (forked from and joined back into `stream` with events, so the
 * call is still stream-ordered and graph-capturable).  With windows == 0 the call is ONE launch: the step kernel
 * writes the one-row observation itself. */
int gte_step_obs(const GteParams* params, const GteData* data, const GteState* state,
                 const void* actions, const GteStepOut* out, float* obs, int autoreset,
                 int variant, int n_chunks, void* stream);

/* One lockstep iteration for a policy that lives on the HOST — what a gymnasium VectorEnv.step(numpy actions) does
 * (environments.py:233-272 for N envs) — as ONE blocking call: host actions in -> step kernel -> reward / flags / error
 * flag out -> gather enqueued.  Returns once io->results holds this iteration's values; the observation gather may
 * still be running on `stream` (the observations stay device-resident for the next policy forward pass) — unless
 * io->obs_host asks for the observations on the host too, in which case the call also waits for those.
 * out->reward / terminated / truncated / error_out are ignored: the call points them into the result block itself.
 * COPY mode: one H2D cudaMemcpyAsync (N * action_bytes) on a library-owned stream, the step kernel, ONE D2H
 * cudaMemcpyAsync (GTE_HOST_RESULT_BYTES(N)) on a second library-owned stream beside the gather.  MAPPED mode: no copy
 * at all (see GteHostIOMode).  *mode_used (may be NULL) receives the mode the call resolved to. */
int gte_step_host(const GteParams* params, const GteData* data, const GteState* state, const GteHostIO* io,
                  const GteStepOut* out, float* obs, int autoreset, int variant, int* mode_used, void* stream);

/* gte_step_host split in two (copy engines only; io->mode and io->obs_host are ignored / must be NULL): _begin enqueues
 * the action copy, the transition, the copy of the result block and the gather, and returns at once; _end waits until
 * io->results holds that iteration's values.  A caller that alternates TWO GteHostIO sets (results, dev_results and
 * dev_actions each their own; out->reward / terminated / truncated are again ignored) may call _begin for iteration
 * k+1 before _end for iteration k — what gymnasium 0.x / stable-baselines3 vector envs call step_async / step_wait:
 * the device-to-host copy of iteration k then runs under the action copy, transition and gather of iteration k+1.
 * A set's buffers are free for the next _begin once its _end has returned; at most 4 result blocks IN FLIGHT (begun, not
 * yet ended) per device. */
int gte_step_host_begin(const GteParams* params, const GteData* data, const GteState* state, const GteHostIO* io,
                        const GteStepOut* out, float* obs, int autoreset, int variant, void* stream);
int gte_step_host_end(const GteHostIO* io);

/* ---- result relay (multi-GPU host IO) --------------------------------------------------------------------------
 * On a box where the GPUs' device-to-host paths are unequal under load (measured on an 8 x B200 node: 12.9 GB/s for each
 * of four GPUs against 22.6 GB/s for each of the other four when all eight copy at once), a rank on a slow path ships the
 * tail of its result block over NVLink into a buffer on a peer GPU with a fast path; the PEER's copy engine then writes
 * it into the slow rank's result block, which lives in host memory both processes map (POSIX shared memory, registered
 * with gte_host_register in both).  No kernel and no host thread is involved in the data path: the sender's copy engine
 * writes data then a sequence word into the peer buffer (CUDA IPC mapping), the peer's stream waits for that word with a
 * stream memory operation (cuStreamWaitValue32), copies the data to the host and, behind it, the sequence word — which
 * the slow rank's host polls.  A rank may push to one peer and serve any number of peers.  Nothing in the reference
 * corresponds to this (it has no device): it exists to keep gte_step_host's bytes-per-second up at 8 GPUs.
 *
 * gte_relay_supported: 1 when the current device can wait on memory from a stream (needed by gte_relay_serve).
 * gte_relay_alloc:  cudaMalloc a relay buffer of `bytes` payload (+ a 256-byte header holding the sequence word), zeroed;
 *                   *dev_base receives the buffer, ipc_handle (64 bytes) what another process passes to gte_relay_open.
 * gte_relay_open:   map a peer process's relay buffer into this process (peer access enabled lazily).
 * gte_relay_release: undo gte_relay_alloc (opened == 0) or gte_relay_open (opened != 0).
 * gte_relay_push:   (sender) on a library-owned stream: wait for after_event (a cudaEvent_t recorded behind the step
 *                   kernel: GteHostIO.step_done_event), copy `bytes` from src_dev into the peer buffer's payload, then
 *                   publish `seq` in the peer buffer's header; done_event (a cudaEvent_t or NULL) is recorded behind both
 *                   — the caller orders the next writer of src_dev behind it.
 * gte_relay_serve:  (peer) on a library-owned stream per `lane` (0..7, one per rank served): wait until the header of
 *                   own_base holds a sequence number >= seq, copy `bytes` of payload to host_dst, then the 4-byte
 *                   sequence word to host_seq.  Both host addresses must be pinned for this process (gte_host_register).
 *                   Returns at once; the sender's host learns of completion by polling *host_seq == seq.
 * gte_relay_unblock: (peer) write `seq` into own_base's header from this side: releases a serve stream whose sender will
 *                   never deliver (set-up self-test failed) so that the buffer can be freed.
 * gte_host_register / gte_host_unregister: page-lock a host range (e.g. a shared-memory mapping) for DMA. */
#define GTE_RELAY_HEADER_BYTES 256
int gte_relay_supported(void);
int gte_relay_alloc(int64_t bytes, void** dev_base, void* ipc_handle);
int gte_relay_open(const void* ipc_handle, void** dev_base);
int gte_relay_release(void* dev_base, int opened);
int gte_relay_push(void* peer_base, const void* src_dev, int64_t bytes, uint32_t seq, void* after_event, void* done_event);
int gte_relay_serve(int lane, void* own_base, int64_t bytes, uint32_t seq, void* host_dst, void* host_seq);
int gte_relay_unblock(void* own_base, uint32_t seq);
int gte_host_register(void* ptr, int64_t bytes);
int gte_host_unregister(void* ptr);

/* Stop the resident server kernel of the current device (GTE_IO_SERVER), if one is running, and wait for it.  Every
 * other entry point does this implicitly before it enqueues anything. */
int gte_serve_stop(void);

/* n_steps lockstep iterations from a device-resident action stream, enqueued by ONE host call (the open-loop driver:
 * replay of recorded actions, random-policy baselines, back-tests; at small N an iteration then costs a kernel launch
 * instead of a trip through the host language).  actions: [n_steps, N] ints of params->action_bytes bytes.  Every non-NULL per-env array of `out`
 * (reward, terminated, truncated, valuation, real_position, info_idx, info_step, pre_reset_portfolio) holds n_steps
 * consecutive copies of its one-iteration shape, iteration k writing copy k; metrics_step ends up holding the last
 * iteration's metrics, metrics_total accumulates all of them.  keep_obs != 0: obs is f32 [n_steps, N, (W,) F] and
 * every iteration's observation is gathered; keep_obs == 0: obs is f32 [N, (W,) F] and only the LAST iteration's
 * observation is gathered (the dynamic-feature ring is kept up to date by the step kernel either way). */
int gte_rollout(const GteParams* params, const GteData* data, const GteState* state,
                const void* actions, int n_steps, const GteStepOut* out, float* obs, int keep_obs,
                int autoreset, int variant, void* stream);

/* History's last row as tensors (environments.py:253-264, portfolio.py:49-57), from current state. */
int gte_info(const GteParams* params, const GteData* data, const GteState* state,
             const GteInfo* info, void* stream);

/* sizeof() of the ABI structs as compiled: 0 GteParams, 1 GteData, 2 GteState, 3 GteStepOut, 4 GteInfo, 5 GteHostIO
 * (bindings assert their own layout against it). */
int gte_struct_size(int which);

/* Kernel launches one gte_step_obs call issues for this shape: 1 (windows == 0, or the fused form, never taken with
 * params->metric_kinds != 0 or a stateful dynamic feature), else 2 per env
 * range (host-only helper; asks the CUDA runtime for the gather kernel's occupancy, so it needs a device). */
int gte_step_obs_launches(const GteParams* params, const GteData* data, int variant, int n_chunks);

/* How many env ranges gte_step_obs uses for n_chunks = 0 (host-only helper). */
int gte_default_chunks(int n_envs);

/* Which gather variant GTE_OBS_AUTO resolves to for this shape (host-only helper). */
int gte_obs_variant_for(const GteParams* params, const GteData* data);

#ifdef __cplusplus
}
#endif
#endif /* GTE_B200_H */
