// gte_step_env.cuh — the transition of ONE env (TradingEnv.step, environments.py:233-272, line by line) and the
// deterministic metric reduction, used by the step kernel (gte_step.cu).
#pragma once

#include "gte_device.cuh"

namespace gte {

constexpr int kChunkFirst = 1, kChunkLast = 2, kChunkTotalOnly = 4;

struct StepThreadOut {       // what the gather phase of the fused kernel needs from the step phase
    int idx, ep_start, ds;   // post-reset row index, episode start, dataset
    float dyn_pos, dyn_rp;   // the dynamic features of row idx (position, real_position), as written to the ring
    float dyn_pr, dyn_rew, dyn_prog;   // portfolio_return, reward, episode_progress of row idx (read when configured)
    float dyn_dd, dyn_age;             // current_drawdown, position_age of row idx (ACC only, read when configured)
};

struct MetricAcc {           // per-thread accumulators (deterministic: fixed tile order per thread)
    double sum_pr = 0.0, sum_mr = 0.0, sum_rew = 0.0;
    int episodes = 0, terminated = 0, truncated = 0, sum_len = 0;
};

// The transition of ONE env (the reference's step(), line by line).
// action i of an array of 1-, 2-, 4- or 8-byte signed ints (GteParams.action_bytes; warp-uniform switch).  The array may
// be mapped HOST memory (gte_step_host, MAPPED mode): plain loads, each element read exactly once.
__device__ __forceinline__ int64_t load_action(const void* __restrict__ actions, int bytes, int64_t i) {
    switch (bytes) {
        case 1: return (int64_t) reinterpret_cast<const int8_t*>(actions)[i];
        case 2: return (int64_t) reinterpret_cast<const int16_t*>(actions)[i];
        case 4: return (int64_t) reinterpret_cast<const int32_t*>(actions)[i];
        default: return reinterpret_cast<const int64_t*>(actions)[i];
    }
}

// Per-launch constants derived on the host (gte_step.cu: make_step_consts).
struct StepConsts {
    double done_thr;      // largest double x with fl(x / v0) <= done_ratio (IEEE division is monotonic in x), or NaN:
                          // `valuation <= done_thr` is then bit-for-bit `valuation / v0 <= done_ratio` (:246) without the divide
    int action_bytes;     // 1, 2, 4 or 8
    int T0;               // len(df) of dataset 0, filled in ON THE DEVICE by the kernel prologue (lengths is device memory)
    DynLayout dyn;        // dynamic-column descriptor (read by the general-catalogue instantiations only)
};

__device__ __forceinline__ void store_env(const GteState& S, int64_t i, const EnvRegs& e) {
    S.asset[i] = e.pf.asset;
    S.fiat[i] = e.pf.fiat;
    S.interest_asset[i] = e.pf.ia;
    S.interest_fiat[i] = e.pf.ifi;
    S.pos_idx[i] = e.pos_idx;
    S.step[i] = e.step;
    S.ep_start[i] = e.ep_start;
}

// What one transition reads: the env's state, its action (already range-checked) and the two prices it trades /
// is valued at, split from the arithmetic.
struct EnvIn {
    EnvRegs e;
    int a;                // action: index into positions, or -1 = hold (out-of-range and negative actions included)
    int idx, T;           // row before advancing (clamped to T-2, e.step with it, when the caller stepped past the data),
                          // dataset length
};

// CG: load through L2 only — a kernel that stays resident across iterations (server kernel) must not find a line in
// its L1 that another kernel has rewritten since.
template <bool CG = false>
__device__ __forceinline__ EnvRegs load_env_regs(const GteParams& P, const GteState& S, int64_t i) {
    EnvRegs e;
    if (CG) {
        e.pf.asset = __ldcg(S.asset + i); e.pf.fiat = __ldcg(S.fiat + i);
        e.pf.ia = __ldcg(S.interest_asset + i); e.pf.ifi = __ldcg(S.interest_fiat + i);
        e.pos_idx = __ldcg(S.pos_idx + i); e.step = __ldcg(S.step + i); e.ep_start = __ldcg(S.ep_start + i);
        e.ds = (P.n_datasets > 1) ? __ldcg(S.dataset_idx + i) : 0;
        return e;
    }
    e.pf.asset = S.asset[i];
    e.pf.fiat = S.fiat[i];
    e.pf.ia = S.interest_asset[i];
    e.pf.ifi = S.interest_fiat[i];
    e.pos_idx = S.pos_idx[i];
    e.step = S.step[i];
    e.ep_start = S.ep_start[i];
    e.ds = (P.n_datasets > 1) ? S.dataset_idx[i] : 0;
    return e;
}

// state in registers + the raw action -> what the transition consumes (range checks, row index)
__device__ __forceinline__ EnvIn make_env_in(const GteParams& P, const GteData& D, const GteState& S, const StepConsts& K,
                                             const EnvRegs& e, int64_t a) {
    EnvIn in;
    in.e = e;
    if (a >= (int64_t)P.n_positions) atomicOr(S.error_flag, GTE_E_ACTION_RANGE);
    if (P.strict_actions && a < -1) atomicOr(S.error_flag, GTE_E_NEGATIVE_ACTION);
    in.a = (a < 0 || a >= (int64_t)P.n_positions) ? -1 : (int)a;           // :234 None = hold
    // one dataset: its length was read once per CTA (K.T0) instead of once per env behind the state loads
    in.T = (P.n_datasets > 1) ? D.lengths[in.e.ds] : K.T0;
    in.idx = in.e.ep_start + in.e.step;
    if (in.idx + 1 >= in.T) {        // stepping past the end of the data without a reset (caller bug)
        atomicOr(S.error_flag, GTE_E_PAST_END);
        in.idx = in.T - 2;
        // the step counter moves back with the row: the transition stores row T-1 again, so every reader that starts
        // from the stored state (gathers, info) stays inside the data
        in.e.step = in.idx - in.e.ep_start;
    }
    return in;
}

__device__ __forceinline__ EnvIn load_env(const GteParams& P, const GteData& D, const GteState& S,
                                          const void* __restrict__ actions, const StepConsts& K, int64_t i) {
    return make_env_in(P, D, S, K, load_env_regs(P, S, i), load_action(actions, K.action_bytes, i));
}

// price BEFORE advancing (:204-207) and the price the new row is valued at (:239)
__device__ __forceinline__ void load_prices(const GteParams& P, const GteData& D, const EnvIn& in, double& p0, double& p1) {
    const double* __restrict__ price = D.price + (int64_t)in.e.ds * P.t_stride;
    p0 = __ldg(price + in.idx);
    p1 = __ldg(price + in.idx + 1);
}

// Episode accumulators (ACC): the state of env i after this step's History row (position after the market trade and
// the limit orders, valuation, reward) has been folded in, in the reference's operation order.  Stored back every step.
// current / age: the values of the stateful dynamic features for this row (0 when their kind is not configured).
struct EpisodeAcc {
    double peak, drawdown, reward_sum, changes, in_market, current, age;
};
template <bool GEN>
__device__ __forceinline__ EpisodeAcc episode_acc_fold(const GteParams& P, const RingLayout<GEN>& R, const GteState& S,
                                                       int i, double pos_before, double pos_after, double val, double rew) {
    const int64_t N = P.n_envs;
    double* __restrict__ A = S.episode_acc;
    EpisodeAcc a = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const bool dd_metric = metric_on(P, GTE_METRIC_MAX_DRAWDOWN);
    if (dd_metric || dyn_on(R, GTE_DYN_CURRENT_DRAWDOWN)) {                  // one peak update for both consumers
        a.peak = __ldcg(A + GTE_ACC_PEAK * N + i);
        if (dd_metric) a.drawdown = __ldcg(A + GTE_ACC_DRAWDOWN * N + i);
        a.peak = (val > a.peak) ? val : a.peak;                              // np.maximum.accumulate(v) / np.max(v)
        const double d = dsub(1.0, ddiv(val, a.peak));                       // 1 - v / peak
        a.current = d;
        if (dd_metric) a.drawdown = (d > a.drawdown) ? d : a.drawdown;       // np.max
        A[GTE_ACC_PEAK * N + i] = a.peak;
        if (dd_metric) A[GTE_ACC_DRAWDOWN * N + i] = a.drawdown;
    }
    if (metric_on(P, GTE_METRIC_EPISODE_REWARD)) {                           // sum(): left to right
        a.reward_sum = dadd(__ldcg(A + GTE_ACC_REWARD_SUM * N + i), rew);
        A[GTE_ACC_REWARD_SUM * N + i] = a.reward_sum;
    }
    if (metric_on(P, GTE_METRIC_POSITION_CHANGES)) {                         // np.diff(position) != 0: History rows
        a.changes = __ldcg(A + GTE_ACC_POSITION_CHANGES * N + i) + ((pos_after != pos_before) ? 1.0 : 0.0);
        A[GTE_ACC_POSITION_CHANGES * N + i] = a.changes;
    }
    if (metric_on(P, GTE_METRIC_TIME_IN_MARKET)) {
        a.in_market = __ldcg(A + GTE_ACC_IN_MARKET * N + i) + ((pos_after != 0.0) ? 1.0 : 0.0);
        A[GTE_ACC_IN_MARKET * N + i] = a.in_market;
    }
    if (dyn_on(R, GTE_DYN_POSITION_AGE)) {                                   // rows since the position last changed
        a.age = (pos_after != pos_before) ? 0.0 : __ldcg(A + GTE_ACC_POSITION_AGE * N + i) + 1.0;
        A[GTE_ACC_POSITION_AGE * N + i] = a.age;
    }
    return a;
}

// The episode of env i ended with this step: its metrics into GteStepOut.episode_record (rows: include/gte_b200.h).
// Written only with metrics configured: with stateful dynamic features alone, episode_record may be NULL.
__device__ __forceinline__ void episode_record(const GteParams& P, const GteStepOut& O, int i, const EpisodeAcc& a,
                                               double market_return, double portfolio_return, int step) {
    const int64_t N = P.n_envs;
    double* __restrict__ R = O.episode_record;
    const double len = (double)step + 1.0;                                   // len(history): the reset row + step rows
    if (P.metric_kinds != 0) {
        R[i] = market_return;
        R[N + i] = portfolio_return;
    }
    if (metric_on(P, GTE_METRIC_POSITION_CHANGES)) R[(2 + GTE_METRIC_POSITION_CHANGES) * N + i] = a.changes;
    if (metric_on(P, GTE_METRIC_EPISODE_LENGTH)) R[(2 + GTE_METRIC_EPISODE_LENGTH) * N + i] = len;
    if (metric_on(P, GTE_METRIC_MAX_DRAWDOWN)) R[(2 + GTE_METRIC_MAX_DRAWDOWN) * N + i] = a.drawdown;
    if (metric_on(P, GTE_METRIC_EPISODE_REWARD)) R[(2 + GTE_METRIC_EPISODE_REWARD) * N + i] = a.reward_sum;
    if (metric_on(P, GTE_METRIC_TIME_IN_MARKET)) R[(2 + GTE_METRIC_TIME_IN_MARKET) * N + i] = ddiv(a.in_market, len);
}

// The arithmetic of one transition.  STORE_STATE = false: the caller keeps the env's state in registers across iterations
// (rollout / server kernels) and takes it back through e_out.  GEN: the general dynamic-feature catalogue (K.dyn).
// ACC: the episode accumulators run (acc_on: an episode metric or a stateful dynamic feature): every step folds its row
// into them before the ring store, which takes the stateful features' values from them; with metrics, an episode's end
// writes the record.
template <bool STORE_STATE = true, bool GEN = false, bool ACC = false>
__device__ __forceinline__ StepThreadOut step_env(const GteParams& P, const GteData& D, const GteState& S,
                                                  const StepConsts& K, const GteStepOut& O, uint64_t tick, int ring_slot,
                                                  int autoreset, int i, const EnvIn& in, const double p0, const double p1,
                                                  MetricAcc& acc, const double* __restrict__ pos_tab,
                                                  EnvRegs* e_out = nullptr) {
    EnvRegs e = in.e;
    const int a = in.a;
    const int T = in.T;
    int idx = in.idx;
    const double* __restrict__ price = D.price + (int64_t)e.ds * P.t_stride;
    // history["portfolio_valuation", -2]: the previous row's valuation.  The state on entry is exactly
    // the state that row was valued with, at the same price, so it is recomputed bit-identically
    // instead of being stored; the first row of an episode holds portfolio_initial_value (:194).
    const double val0 = valorisation(e.pf, p0);
    const double prev_val = (e.step == 0) ? P.v0 : val0;

    if (a >= 0) {                                                            // :234 (None = hold)
        const double target = pos_tab[a];
        if (target != pos_tab[e.pos_idx]) {                              // :213-215 value compare
            trade_to_position(e.pf, target, p0, P.fee, val0);                // :204-211
            e.pos_idx = a;
        }
    }
    idx += 1;                                                                // :235
    e.step += 1;                                                             // :236
    if (P.n_limit_positions > 0) {                                           // _take_action_order_limit (:217-223)
        const double hi = __ldg(D.high + (int64_t)e.ds * P.t_stride + idx);
        const double lo = __ldg(D.low + (int64_t)e.ds * P.t_stride + idx);
        for (int k = 0; k < P.n_limit_positions; ++k) {                      // dict insertion order (:220)
            const int pk = S.limit_seq[k];
            const double lim = S.limit_price[(int64_t)i * P.n_positions + pk];
            if (lim == lim && pos_tab[pk] != pos_tab[e.pos_idx] && lim <= hi && lim >= lo) {   // :221
                trade_to_position(e.pf, pos_tab[pk], lim, P.fee, valorisation(e.pf, lim));       // :222 price = limit
                e.pos_idx = pk;
            }
        }
    }
    update_interest(e.pf, P.rate);                                           // :240
    const double val = valorisation(e.pf, p1);                               // :241
    const bool done = (K.done_thr == K.done_thr) ? (val <= K.done_thr)       // :246 without the divide (StepConsts)
                                                 : (ddiv(val, P.v0) <= P.done_ratio);
    bool trunc = idx >= T - 1;                                               // :248
    if (P.max_episode_duration >= 0 && e.step >= P.max_episode_duration - 1) trunc = true;   // :250
    const double rp = real_position(e.pf, p1, val);                          // :259
    double rew = 0.0;                                                        // :263 (stays 0 when terminated)
    if (!done) {                                                             // :265-267 reward_function(history)
        double x = (P.reward_kind == GTE_REWARD_SIMPLE_RETURN) ? ddiv(dsub(val, prev_val), prev_val)
                                                               : log(ddiv(val, prev_val));      // :17-18
        x = dmul(P.reward_scale, x);                                         // 1 * x is exact
        x = (x < P.reward_lo) ? P.reward_lo : x;                             // np.clip = minimum(maximum(x, lo), hi)
        x = (x > P.reward_hi) ? P.reward_hi : x;
        rew = x;
    }

    O.reward[i] = rew;
    if (O.reward_f32 != nullptr) O.reward_f32[i] = (float)rew;              // round-to-nearest-even, as numpy casts
    O.terminated[i] = (uint8_t)done;
    O.truncated[i] = (uint8_t)trunc;
    if ((done || trunc) && O.ended_list != nullptr) {                        // the sparse form of the two flag arrays
        const unsigned slot = atomicAdd(O.ended_counter, 1u);
        if (slot < O.ended_cap) O.ended_list[slot] = (unsigned)i | (done ? 0x80000000u : 0u) | (trunc ? 0x40000000u : 0u);
    }
    if (O.valuation) O.valuation[i] = val;
    if (O.real_position) O.real_position[i] = rp;
    if (O.info_idx) O.info_idx[i] = idx;
    if (O.info_step) O.info_step[i] = e.step;
    if (O.pre_reset_portfolio) {
        const int64_t N = P.n_envs;
        O.pre_reset_portfolio[i] = e.pf.asset;
        O.pre_reset_portfolio[N + i] = e.pf.fiat;
        O.pre_reset_portfolio[2 * N + i] = e.pf.ia;
        O.pre_reset_portfolio[3 * N + i] = e.pf.ifi;
    }
    const RingLayout<GEN> R{K.dyn};
    float dyn_pos = (float)pos_tab[e.pos_idx], dyn_rp = (float)rp;        // fp64 -> fp32 as numpy casts (:154)
    float dyn_pr = 0.0f, dyn_rew = (float)rew, dyn_prog = 0.0f, dyn_dd = 0.0f, dyn_age = 0.0f;
    // each value only when its kind is configured (the transition is issue-bound on fp64 divides)
    if (R.kind_block(GTE_DYN_PORTFOLIO_RETURN) != kDynNone) dyn_pr = (float)dsub(ddiv(val, P.v0), 1.0);
    if (R.kind_block(GTE_DYN_EPISODE_PROGRESS) != kDynNone)
        dyn_prog = (float)ddiv((double)e.step, (double)P.max_episode_duration);
    // the episode accumulators: folded before the ring store, which takes the stateful features' values from them.
    // A stateful feature is never the default pair: GEN = false keeps the fold after the store, as the metrics-only
    // kernels have always had it (the order is worth a register in their allocation)
    EpisodeAcc ea;
    if (ACC && GEN) {
        ea = episode_acc_fold(P, R, S, i, pos_tab[in.e.pos_idx], pos_tab[e.pos_idx], val, rew);
        dyn_dd = (float)ea.current;
        dyn_age = (float)ea.age;
    }
    // _get_obs write-back (:153-154); an auto-reset below overwrites the same slot with the new episode's first row
    if (P.n_dyn > 0) {
        const DynRow row = {dyn_rp, dyn_pr, dyn_rew, dyn_prog, dyn_dd, dyn_age, e.pos_idx};
        ring_store<GEN, ACC>(P, K.dyn, S, i, ring_slot, row);
    }
    if (ACC && !GEN) ea = episode_acc_fold(P, R, S, i, pos_tab[in.e.pos_idx], pos_tab[e.pos_idx], val, rew);
    acc.sum_rew = dadd(acc.sum_rew, rew);
    if (done || trunc) {                                                     // :269-271 calculate_metrics
        acc.episodes += 1;
        acc.terminated += done ? 1 : 0;
        acc.truncated += trunc ? 1 : 0;
        acc.sum_len += e.step;
        const double pr = dsub(ddiv(val, P.v0), 1.0);                        // :282
        const double mr = dsub(ddiv(p1, __ldg(price + e.ep_start)), 1.0);    // :281
        acc.sum_pr = dadd(acc.sum_pr, pr);
        acc.sum_mr = dadd(acc.sum_mr, mr);
        if (ACC) episode_record(P, O, i, ea, mr, pr, e.step);               // terminal values, before the auto-reset
        if (autoreset) {
            reset_env<GEN, ACC>(P, D, S, i, tick, ring_slot, e, K.dyn);      // in-place auto-reset
            idx = e.ep_start;
            dyn_pos = dyn_rp = (float)pos_tab[e.pos_idx];                // first row: (position, position) :191-192
            dyn_pr = dyn_rew = dyn_prog = dyn_dd = dyn_age = 0.0f;
            if (P.n_datasets > 1) S.dataset_idx[i] = e.ds;
        }
    }
    if (STORE_STATE) store_env(S, i, e);
    if (e_out != nullptr) *e_out = e;
    StepThreadOut r;
    r.idx = idx; r.ep_start = e.ep_start; r.ds = e.ds;
    r.dyn_pos = dyn_pos; r.dyn_rp = dyn_rp;
    r.dyn_pr = dyn_pr; r.dyn_rew = dyn_rew; r.dyn_prog = dyn_prog;
    r.dyn_dd = dyn_dd; r.dyn_age = dyn_age;
    return r;
}

// load + transition of env i in one go (step kernel; fused step+gather kernel, which never runs with ACC)
template <bool GEN = false, bool ACC = false>
__device__ __forceinline__ StepThreadOut step_env_now(const GteParams& P, const GteData& D, const GteState& S,
                                                      const void* __restrict__ actions, const StepConsts& K,
                                                      const GteStepOut& O, uint64_t tick, int ring_slot, int autoreset,
                                                      int i, MetricAcc& acc, const double* __restrict__ pos_tab) {
    const EnvIn in = load_env(P, D, S, actions, K, i);
    double p0, p1;
    load_prices(P, D, in, p0, p1);
    return step_env<true, GEN, ACC>(P, D, S, K, O, tick, ring_slot, autoreset, i, in, p0, p1, acc, pos_tab);
}

// Dynamic column j of r: the value of the kind whose ring block column j reads.  GEN && ACC: the stateful kinds may be
// configured.
template <bool GEN, bool ACC = false>
__device__ __forceinline__ float dyn_value(const RingLayout<GEN>& R, const StepThreadOut& r, int j) {
    if (R.is_pos(j)) return r.dyn_pos;
    const uint32_t b = (uint32_t)R.f32_block(j);
    if (GEN && ACC && b == R.kind_block(GTE_DYN_CURRENT_DRAWDOWN)) return r.dyn_dd;
    if (GEN && ACC && b == R.kind_block(GTE_DYN_POSITION_AGE)) return r.dyn_age;
    return b == R.kind_block(GTE_DYN_REAL_POSITION) ? r.dyn_rp : b == R.kind_block(GTE_DYN_PORTFOLIO_RETURN) ? r.dyn_pr
         : b == R.kind_block(GTE_DYN_REWARD) ? r.dyn_rew : r.dyn_prog;
}

// The one-row observations (windows=None, environments.py:156-157) of the 32 consecutive envs of a warp; every lane of
// the warp must call it (valid = this lane's env exists and r holds its step's result).
//   coalesced = false: each lane writes its own row — 4-byte stores 4*F bytes apart; fine for device memory, where L2
//                      merges the partial sectors;
//   coalesced = true : the warp's rows are ONE contiguous block of 32*F floats: lane l writes elements l, l+32, ...,
//                      fetching (row, dataset, dynamic features) of the owning env by shuffle -> full 128-byte stores.
//                      For MAPPED HOST memory, where every partial-sector store is its own PCIe transaction
//                      (4096 envs: 60 us -> 27 us per host step).
// GEN: dynamic columns in P.dyn_kinds order (general catalogue), else the default pair (RingLayout).  ACC: as dyn_value.
template <bool GEN = false, bool ACC = false>
__device__ __forceinline__ void write_obs_rows(const GteParams& P, const GteData& D, const DynLayout& L,
                                               float* __restrict__ obs_rows, int64_t i, bool valid, const StepThreadOut& r,
                                               bool coalesced) {
    const RingLayout<GEN> R{L};
    const int F = P.n_static + P.n_dyn;
    if (!coalesced) {
        if (valid) {
            const float* __restrict__ f = D.features + ((int64_t)r.ds * P.t_stride + r.idx) * P.n_static;
            float* __restrict__ o = obs_rows + i * F;
            for (int c = 0; c < P.n_static; ++c) o[c] = __ldg(f + c);
            if (P.n_dyn > 0)
                for (int j = 0; j < R.n_cols(); ++j) o[P.n_static + j] = dyn_value<GEN, ACC>(R, r, j);
        }
        return;
    }
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    float* __restrict__ o = obs_rows + (i - lane) * F;           // row of lane 0's env
    for (int j = lane; j < 32 * F; j += 32) {                    // F trips for every lane
        const int e = j / F, c = j - e * F;
        const int idx = __shfl_sync(FULL, r.idx, e), ds = __shfl_sync(FULL, r.ds, e);
        StepThreadOut q;
        q.dyn_pos = __shfl_sync(FULL, r.dyn_pos, e);
        q.dyn_rp = __shfl_sync(FULL, r.dyn_rp, e);
        q.dyn_pr = __shfl_sync(FULL, r.dyn_pr, e);
        q.dyn_rew = __shfl_sync(FULL, r.dyn_rew, e);
        q.dyn_prog = __shfl_sync(FULL, r.dyn_prog, e);
        q.dyn_dd = (GEN && ACC) ? __shfl_sync(FULL, r.dyn_dd, e) : 0.0f;
        q.dyn_age = (GEN && ACC) ? __shfl_sync(FULL, r.dyn_age, e) : 0.0f;
        const bool ok = __shfl_sync(FULL, (int)valid, e) != 0;
        if (ok) o[j] = c < P.n_static ? __ldg(D.features + ((int64_t)ds * P.t_stride + idx) * P.n_static + c)
                                      : dyn_value<GEN, ACC>(R, q, c - P.n_static);
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = dadd(v, __shfl_down_sync(0xffffffffu, v, o));
    return v;
}

// CTA-level metric reduction -> metric_partials[blockIdx.x]; the last CTA to arrive folds all
// partial rows in a fixed order (deterministic) into metrics_step / metrics_total.  NT = threads of the CTA, all of
// which must call it (step kernel: 256; fused step+gather kernel: 192).
//   flags   kChunkFirst: overwrite metrics_step (else add to it) and advance the ring clock; kChunkLast: advance the
//           Philox tick; kChunkTotalOnly: only add to metrics_total (no metrics_step, no counters, nothing published);
//   phase   0 / 1: a kernel that reduces twice (rollout kernel: all iterations but the last, then the last) uses the two
//           halves of the ticket word and two sets of partial rows, so that CTAs already in the second reduction do not
//           disturb the first (needs 2 * gridDim.x <= GTE_MAX_PARTIAL_ROWS);
//   n_iter  how many lockstep iterations the launch covered (what the tick / ring clock advance by).
template <int NT>
static __device__ void reduce_metrics(const MetricAcc& acc, const GteStepOut& O, const GteState& S, int flags,
                                      int phase = 0, unsigned n_iter = 1u) {
    constexpr int NW = NT / 32, NG = NT / GTE_N_METRICS;
    __shared__ double s_part[NW][GTE_N_METRICS];
    __shared__ double s_fold[NG][GTE_N_METRICS];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* __restrict__ rows = O.metric_partials + (int64_t)phase * gridDim.x * GTE_N_METRICS;

    const double w_rew = warp_sum(acc.sum_rew);
    const int w_ep = __reduce_add_sync(0xffffffffu, acc.episodes);
    double w_pr = 0.0, w_mr = 0.0;
    int w_term = 0, w_trunc = 0, w_len = 0;
    if (w_ep > 0) {                                      // warp-uniform: episode ends are rare
        w_pr = warp_sum(acc.sum_pr);
        w_mr = warp_sum(acc.sum_mr);
        w_term = __reduce_add_sync(0xffffffffu, acc.terminated);
        w_trunc = __reduce_add_sync(0xffffffffu, acc.truncated);
        w_len = __reduce_add_sync(0xffffffffu, acc.sum_len);
    }
    __syncthreads();                                     // a second reduction of the same CTA: s_part is free again
    if (lane == 0) {
        s_part[warp][GTE_M_EPISODES] = (double)w_ep;
        s_part[warp][GTE_M_TERMINATED] = (double)w_term;
        s_part[warp][GTE_M_TRUNCATED] = (double)w_trunc;
        s_part[warp][GTE_M_SUM_PORTFOLIO_RETURN] = w_pr;
        s_part[warp][GTE_M_SUM_MARKET_RETURN] = w_mr;
        s_part[warp][GTE_M_SUM_EPISODE_LENGTH] = (double)w_len;
        s_part[warp][GTE_M_SUM_REWARD] = w_rew;
        s_part[warp][GTE_M_RESERVED] = 0.0;
    }
    __syncthreads();
    if (threadIdx.x < GTE_N_METRICS) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) t = dadd(t, s_part[w][threadIdx.x]);
        rows[(int64_t)blockIdx.x * GTE_N_METRICS + threadIdx.x] = t;
    }
    __syncthreads();
    const unsigned one = phase ? 0x10000u : 1u;
    if (threadIdx.x == 0) {
        // ONE cumulative fence per CTA, by the thread that takes the ticket: the barrier above put every write of the
        // CTA (results, partial row) before it.  System scope when the results went straight into mapped host memory.
        if (O.seq_out != nullptr) __threadfence_system(); else __threadfence();
        s_last = (((atomicAdd(O.block_counter, one) >> (16 * phase)) & 0xffffu) == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int m = threadIdx.x % GTE_N_METRICS, g = threadIdx.x / GTE_N_METRICS;   // NG groups x 8 metrics
    double t = 0.0;
    for (int b = g; b < (int)gridDim.x; b += NG)
        t = dadd(t, __ldcg(rows + (int64_t)b * GTE_N_METRICS + m));
    s_fold[g][m] = t;
    __syncthreads();
    if (threadIdx.x < GTE_N_METRICS) {
        double tot = 0.0;
        for (int k = 0; k < NG; ++k) tot = dadd(tot, s_fold[k][threadIdx.x]);
        // env chunks of one lockstep iteration run as consecutive launches: the first one overwrites
        // metrics_step, later ones add to it in launch order (deterministic)
        if (!(flags & kChunkTotalOnly))
            O.metrics_step[threadIdx.x] = (flags & kChunkFirst) ? tot : dadd(O.metrics_step[threadIdx.x], tot);
        if (O.metrics_total) O.metrics_total[threadIdx.x] = dadd(O.metrics_total[threadIdx.x], tot);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicSub(O.block_counter, one * gridDim.x);     // self-resetting for the next launch (this phase's half only)
        if (flags & kChunkTotalOnly) return;
        // every CTA of this launch has read the tick / ring clock by now.  The Philox event counter advances with
        // the LAST env range of an iteration; the ring clock with the FIRST one, so that the later ranges and
        // every gather of the iteration (all stream-ordered behind this launch) read the new value
        if (O.ended_list != nullptr) {                   // every CTA's appends came before its ticket
            *O.ended_n_out = __ldcg(O.ended_counter);
            *O.ended_counter = 0u;
        }
        if (flags & kChunkLast) *S.tick = *S.tick + (uint64_t)n_iter;
        if (flags & kChunkFirst) *S.ring_clock = *S.ring_clock + (uint64_t)n_iter;
        // every CTA OR-ed its error bits before it took its ticket: the flag is complete here (may be mapped host memory)
        const int err = (O.error_out != nullptr || O.seq_out != nullptr) ? __ldcg(S.error_flag) : 0;
        if (O.seq_out != nullptr) {
            // LAST, and in ONE 8-byte store with the error flag that sits right in front of it in the result block
            // (GTE_HOST_RESULT_ERROR_OFFSET / _SEQ_OFFSET): a host thread polling the sequence word may hand the next
            // iteration to a kernel that is still resident.  Every CTA fenced its results system-wide BEFORE its
            // ticket, and the tickets were all observed before this store is issued; the counters above only have to
            // be visible on the device.
            __threadfence();
            *reinterpret_cast<volatile unsigned long long*>(O.seq_out - 1) =
                ((unsigned long long)O.seq_value << 32) | (unsigned long long)(unsigned)err;
        } else if (O.error_out != nullptr) {
            *O.error_out = err;
        }
    }
}

}  // namespace gte
