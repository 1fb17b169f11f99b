// gte_device.cuh — device-side building blocks shared by the step / reset / info kernels.
//
// Money math = the reference's Portfolio (src/gym_trading_env/utils/portfolio.py) restated in IEEE
// fp64 with explicit round-to-nearest intrinsics (__dmul_rn/__dadd_rn/__ddiv_rn), which nvcc never
// contracts into FMA, in exactly the Python operation order — so asset/fiat/interest/valuation/
// real_position are bit-identical to the CPU reference.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gte_b200.h"

namespace gte {

constexpr int kStepThreads = GTE_STEP_THREADS;
constexpr int kMaxPartialRows = GTE_MAX_PARTIAL_ROWS;     // metric_partials rows the step kernel may use (grid cap)

// Programmatic dependent launch: wait until the preceding kernel of the stream has completed and its writes are visible
// (returns at once for a kernel that was not launched with the attribute).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

struct Portfolio {        // signed state of utils/portfolio.py:2-6
    double asset, fiat, ia, ifi;
};

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
// IEEE division.  The inline fast path of the fp64 divide hands a ZERO numerator to a ~250-instruction subroutine,
// and zero numerators are everyday values here (a flat position: asset = 0, target = 0), so one flat env per warp
// would send the whole warp there several times per step.  0 / b for a finite non-zero b is a zero whose sign is
// the XOR of the operand signs: answer that directly and divide 1 / b instead (result discarded) — bit-identical.
__device__ __forceinline__ double ddiv(double a, double b) {
    const bool zero_num = (a == 0.0) && (b != 0.0) && (fabs(b) <= 1.7976931348623157e308);   // false for NaN / inf / 0
    double num = zero_num ? 1.0 : a;
    asm("" : "+d"(num));      // opaque: otherwise the compiler divides the original (zero) numerator, whose quotient is dead
    const double q = __ddiv_rn(num, b);
    const double z = __longlong_as_double((__double_as_longlong(a) ^ __double_as_longlong(b)) & (long long)0x8000000000000000ull);
    return zero_num ? z : q;
}

// Portfolio.valorisation (portfolio.py:7-13): sum([asset*price, fiat, -ia*price, -if]) left to right.
__device__ __forceinline__ double valorisation(const Portfolio& s, double price) {
    double v = dmul(s.asset, price);
    v = dadd(v, s.fiat);
    v = dadd(v, dmul(-s.ia, price));
    v = dadd(v, -s.ifi);
    return v;
}

// Portfolio.real_position (portfolio.py:14-15), with the valuation already at hand.
__device__ __forceinline__ double real_position(const Portfolio& s, double price, double val) {
    return ddiv(dmul(dsub(s.asset, s.ia), price), val);
}

// Portfolio.trade_to_position (portfolio.py:18-43).  `val` = valorisation(s, price) on entry.
__device__ __forceinline__ void trade_to_position(Portfolio& s, double target, double price,
                                                  double fee, double val) {
    const double current = ddiv(dmul(s.asset, price), val);                  // :20 position(price)
    double r = 1.0;                                                          // :21
    if (target <= 0.0 && current < 0.0) {                                    // :22-23
        const double q = ddiv(target, current);
        r = (q < 1.0) ? q : 1.0;                                             // min(1, q): first arg on ties
    } else if (target >= 1.0 && current > 1.0) {                             // :24-25
        const double q = ddiv(dsub(target, 1.0), dsub(current, 1.0));
        r = (q < 1.0) ? q : 1.0;
    }
    if (r < 1.0) {                                                           // :26-30 repay interest
        const double k = dsub(1.0, r);
        s.asset = dsub(s.asset, dmul(k, s.ia));
        s.fiat = dsub(s.fiat, dmul(k, s.ifi));
        s.ia = dmul(r, s.ia);
        s.ifi = dmul(r, s.ifi);
        val = valorisation(s, price);                                        // :33 recomputed after repay
    }
    double trade = dsub(ddiv(dmul(target, val), price), s.asset);            // :33
    if (trade > 0.0) {                                                       // :34-38 buy
        trade = ddiv(trade, dadd(dsub(1.0, fee), dmul(fee, target)));
        s.asset = dadd(s.asset, dmul(trade, dsub(1.0, fee)));
        s.fiat = dadd(s.fiat, dmul(-trade, price));
    } else {                                                                 // :39-43 sell
        trade = ddiv(trade, dsub(1.0, dmul(fee, target)));
        s.asset = dadd(s.asset, trade);
        s.fiat = dadd(s.fiat, dmul(dmul(-trade, price), dsub(1.0, fee)));
    }
}

// Portfolio.update_interest (portfolio.py:44-46).  Python's max(0, -x) returns the FIRST argument on
// ties, so -0.0 never appears: written as a compare-select, not fmax.
__device__ __forceinline__ void update_interest(Portfolio& s, double rate) {
    const double na = -s.asset, nf = -s.fiat;
    s.ia = dmul((na > 0.0) ? na : 0.0, rate);
    s.ifi = dmul((nf > 0.0) ? nf : 0.0, rate);
}

// TargetPortfolio.__init__ (portfolio.py:59-66)
__device__ __forceinline__ Portfolio target_portfolio(double position, double value, double price) {
    Portfolio s;
    s.asset = ddiv(dmul(position, value), price);
    s.fiat = dmul(dsub(1.0, position), value);
    s.ia = 0.0;
    s.ifi = 0.0;
    return s;
}

// ---- Philox4x32-10 (Salmon et al., SC'11; Random123 known-answer vectors in tests/) -------------
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

__device__ __forceinline__ void philox_draw(uint64_t seed, uint64_t tick, uint64_t env_id, uint32_t r[4]) {
    r[0] = (uint32_t)tick; r[1] = (uint32_t)(tick >> 32);
    r[2] = (uint32_t)env_id; r[3] = (uint32_t)(env_id >> 32);
    philox4x32_10(r, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// MultiDatasetTradingEnv.next_dataset (environments.py:380-391): uniform among the least-used
// datasets == among those not yet used in the current round (use counts differ by at most one).
__device__ __forceinline__ int next_dataset(const GteParams& P, const GteState& S, int i, uint32_t u) {
    const uint64_t full = (P.n_datasets >= 64) ? ~0ull : ((1ull << P.n_datasets) - 1ull);
    uint64_t used = S.ds_used[i];
    if ((used & full) == full) used = 0;
    const int n_free = P.n_datasets - __popcll(used & full);
    int pick = (int)(((uint64_t)u * (uint64_t)n_free) >> 32);                // :385
    int ds = 0;
    for (int d = 0; d < P.n_datasets; ++d) {
        if (!((used >> d) & 1ull)) {
            if (pick == 0) { ds = d; break; }
            --pick;
        }
    }
    S.ds_used[i] = used | (1ull << ds);                                      // :388
    S.ds_episodes[i] = 0;                                                    // :381
    return ds;
}

// Dynamic-feature ring (time-indexed, one block per 32-env tile: include/gte_b200.h): the row env i observes at
// lockstep iteration c lives in slot c % W.  All envs write the same slot in one iteration: a warp stores one
// full 128-byte line per f32 column and one full 32-byte sector of position indices.
__device__ __forceinline__ int ring_slot_of(const GteParams& P, uint64_t clock) {
    const int W = P.windows > 0 ? P.windows : 1;
    return (int)(clock % (uint64_t)W);
}

// Dynamic-column descriptor, derived once on the host from (n_dyn, dyn_kinds) by dyn_layout(): drives the ring layout
// (include/gte_b200.h, GteState.dyn_ring) on both the step and the gather side.  `general` is false for no dynamic
// columns and for the default pair (position, real_position): those run the GEN = false instantiations, whose layout
// is known at compile time (RingLayout).
constexpr uint32_t kDynPosBlock = 0xF, kDynNone = 0xE;
struct DynLayout {
    uint32_t col_src;     // nibble j: the ring block column j reads: f32 block 0..4, or kDynPosBlock (u8 position indices)
    uint32_t kind_blk;    // nibble k (enum GteDynKind 1..7): the block of kind k, or kDynNone when it is not configured
    int n_f32, n_pos;     // f32 blocks, position-index blocks (0 or 1)
    int tile_bytes;       // GTE_RING_TILE_BYTES_DYN(W, n_f32, n_pos)
    bool general;
};

// The ring layout as the kernels see it, and the only code that branches on GEN to describe it.  GEN = false: the
// default pair, every answer a compile-time constant (column 0 reads the position-index block, column 1 f32 block 0;
// per-column answers fold by column index, which keeps the pair's registers where a decoded constant descriptor would
// not).  GEN = true: the general catalogue, answers read from L.  Kernels that may run without dynamic columns check
// n_dyn > 0 before they touch the ring.
template <bool GEN>
struct RingLayout {
    const DynLayout& L;
    __device__ __forceinline__ int n_cols() const { return GEN ? L.n_f32 + L.n_pos : 2; }
    __device__ __forceinline__ bool is_pos(int j) const { return GEN ? ((L.col_src >> (4 * j)) & 15u) == kDynPosBlock : j == 0; }
    __device__ __forceinline__ int f32_block(int j) const { return GEN ? (int)((L.col_src >> (4 * j)) & 15u) : 0; }
    // f32 block of kind k, kDynPosBlock for position, or kDynNone when the kind is not configured
    __device__ __forceinline__ uint32_t kind_block(int k) const {
        return GEN ? (L.kind_blk >> (4 * k)) & 15u
                   : (k == GTE_DYN_POSITION ? kDynPosBlock : k == GTE_DYN_REAL_POSITION ? 0u : kDynNone);
    }
    __device__ __forceinline__ int n_f32() const { return GEN ? L.n_f32 : 1; }
    __device__ __forceinline__ int n_pos() const { return GEN ? L.n_pos : 1; }
    __device__ __forceinline__ int tile_bytes(int W) const { return GEN ? L.tile_bytes : GTE_RING_TILE_BYTES_DYN(W, 1, 1); }
    // the ring block of the 32-env tile that holds env
    __device__ __forceinline__ const uint8_t* tile_of(const uint8_t* ring, int W, int64_t env) const {
        return ring + (env >> 5) * (int64_t)tile_bytes(W);
    }
};

// dyn_kinds with the legacy 0 spelled out (n_dyn == 2: the default pair, 0x21)
static inline uint32_t dyn_kinds_of(const GteParams& P) {
    return (P.dyn_kinds == 0 && P.n_dyn == 2) ? 0x21u : (uint32_t)P.dyn_kinds;
}

static inline DynLayout dyn_layout(const GteParams& P) {
    DynLayout L;
    const uint32_t kinds = dyn_kinds_of(P);
    const int W = P.windows > 0 ? P.windows : 1;
    L.n_pos = 0;
    for (int j = 0; j < P.n_dyn; ++j) L.n_pos += ((kinds >> (4 * j)) & 15u) == GTE_DYN_POSITION;
    L.n_f32 = P.n_dyn - L.n_pos;
    L.kind_blk = 0u;
    for (int k = 0; k < 8; ++k) L.kind_blk |= kDynNone << (4 * k);
    int blk = 0;
    for (int k = GTE_DYN_REAL_POSITION; k <= GTE_DYN_POSITION_AGE; ++k)         // f32 blocks in kind-code order
        for (int j = 0; j < P.n_dyn; ++j)
            if (((kinds >> (4 * j)) & 15u) == (uint32_t)k) L.kind_blk = (L.kind_blk & ~(15u << (4 * k))) | ((uint32_t)blk++ << (4 * k));
    if (L.n_pos) L.kind_blk = (L.kind_blk & ~(15u << (4 * GTE_DYN_POSITION))) | (kDynPosBlock << (4 * GTE_DYN_POSITION));
    L.col_src = 0u;
    for (int j = 0; j < P.n_dyn; ++j) L.col_src |= ((L.kind_blk >> (4 * ((kinds >> (4 * j)) & 15u))) & 15u) << (4 * j);
    L.tile_bytes = GTE_RING_TILE_BYTES_DYN(W, L.n_f32, L.n_pos);
    L.general = P.n_dyn > 0 && kinds != 0x21u;
    return L;
}

// One row of every dynamic column, fp64 values already cast to f32 as numpy casts (:154); the kinds that are not
// configured are ignored.
struct DynRow {
    float rp, pr, rew, prog;      // real_position, portfolio_return, reward, episode_progress
    float dd, age;                // current_drawdown, position_age (stateful: written by the ACC instantiations only)
    int pos_idx;                  // position: index into positions
};
// Writes row r of env i into ring slot `slot` (step and reset side); needs n_dyn > 0.  GEN && ACC: the stateful kinds
// may be configured (they need the episode accumulators and are never the default pair; otherwise their stores are
// not compiled).
template <bool GEN, bool ACC = false>
__device__ __forceinline__ void ring_store(const GteParams& P, const DynLayout& L, const GteState& S, int i, int slot,
                                           const DynRow& r) {
    const RingLayout<GEN> R{L};
    const int W = P.windows > 0 ? P.windows : 1;
    const int e = i & 31;
    uint8_t* tile = S.dyn_ring + (int64_t)(i >> 5) * R.tile_bytes(W);
    const float v[6] = {r.rp, r.pr, r.rew, r.prog, r.dd, r.age};
#pragma unroll
    for (int k = GTE_DYN_REAL_POSITION; k <= (GEN && ACC ? GTE_DYN_POSITION_AGE : GTE_DYN_EPISODE_PROGRESS); ++k) {
        const uint32_t b = R.kind_block(k);
        if (b < kDynNone) *reinterpret_cast<float*>(tile + GTE_RING_F32_OFFSET(W, (int)b, slot, e)) = v[k - GTE_DYN_REAL_POSITION];
    }
    if (R.n_pos()) tile[GTE_RING_POS_OFFSET_DYN(W, R.n_f32(), slot, e)] = (uint8_t)r.pos_idx;
}

// Dynamic column j of env lane e in ring slot s of a ring tile (the gathers' read).  CG: a global-memory tile read
// through L2 only, as the vec gather reads the ring.
template <bool GEN, bool CG = false>
__device__ __forceinline__ float ring_value(const GteParams& P, const RingLayout<GEN>& R, int W, const uint8_t* tile,
                                            int j, int s, int e) {
    if (R.is_pos(j)) {
        const uint8_t* p = tile + GTE_RING_POS_OFFSET_DYN(W, R.n_f32(), s, e);
        return (float)P.positions[CG ? __ldcg(p) : *p];           // fp64 -> fp32 as numpy casts (:154)
    }
    const float* p = reinterpret_cast<const float*>(tile + GTE_RING_F32_OFFSET(W, R.f32_block(j), s, e));
    return CG ? __ldcg(p) : *p;
}

struct EnvRegs {          // the per-env state a step keeps in registers
    Portfolio pf;
    int pos_idx, step, ep_start, ds;
};

// Episode metrics (GteParams.metric_kinds, TradingEnv.add_metric :274-294) and the stateful dynamic features: the
// running state of env i's episode in GteState.episode_acc, one f64 row per quantity (enum GteEpisodeAccRow).  Only the
// rows of configured kinds are touched; the peak row serves both max_drawdown and current_drawdown.
__device__ __forceinline__ bool metric_on(const GteParams& P, int kind) { return (P.metric_kinds >> kind) & 1; }
// the stateful dynamic feature of kind k is a column (compile-time false for GEN = false: never the default pair)
template <bool GEN>
__device__ __forceinline__ bool dyn_on(const RingLayout<GEN>& R, int k) { return R.kind_block(k) != kDynNone; }

// The reset row (:186-197): valuation v0, reward 0, the episode's first position.
template <bool GEN>
__device__ __forceinline__ void episode_acc_init(const GteParams& P, const RingLayout<GEN>& R, const GteState& S, int i,
                                                 double position) {
    const int64_t N = P.n_envs;
    double* __restrict__ A = S.episode_acc;
    if (metric_on(P, GTE_METRIC_MAX_DRAWDOWN) || dyn_on(R, GTE_DYN_CURRENT_DRAWDOWN)) A[GTE_ACC_PEAK * N + i] = P.v0;
    if (metric_on(P, GTE_METRIC_MAX_DRAWDOWN)) A[GTE_ACC_DRAWDOWN * N + i] = 0.0;        // 1 - v0 / v0
    if (metric_on(P, GTE_METRIC_EPISODE_REWARD)) A[GTE_ACC_REWARD_SUM * N + i] = 0.0;
    if (metric_on(P, GTE_METRIC_POSITION_CHANGES)) A[GTE_ACC_POSITION_CHANGES * N + i] = 0.0;
    if (metric_on(P, GTE_METRIC_TIME_IN_MARKET)) A[GTE_ACC_IN_MARKET * N + i] = (position != 0.0) ? 1.0 : 0.0;
    if (dyn_on(R, GTE_DYN_POSITION_AGE)) A[GTE_ACC_POSITION_AGE * N + i] = 0.0;
}

// TradingEnv.reset (environments.py:163-199) preceded by MultiDatasetTradingEnv.reset (:393-400).
// Rare path (once per episode): plan/rotation bookkeeping goes straight to global memory.
// GEN: the general dynamic-feature catalogue (L.general), else no dynamic columns or the default pair (RingLayout).
// ACC: the episode accumulators run (an episode metric or a stateful dynamic feature): they start from the reset row.
template <bool GEN = false, bool ACC = false>
__device__ __forceinline__ void reset_env(const GteParams& P, const GteData& D, const GteState& S,
                                       int i, uint64_t tick, int ring_slot, EnvRegs& e, const DynLayout& L) {
    uint32_t r[4];
    philox_draw(P.seed, tick, (uint64_t)(P.env_id_offset + i), r);
    const bool have_plan = P.plan_episodes > 0 && S.reset_plan != nullptr;
    int plan_start = 0, plan_pos = 0, plan_ds = 0;
    if (have_plan) {
        const int cur = S.plan_cursor[i];
        if (cur >= P.plan_episodes) atomicOr(S.error_flag, GTE_E_PLAN_EXHAUSTED);     // replays from the start
        const int32_t* pl = S.reset_plan + ((int64_t)i * P.plan_episodes + (cur % P.plan_episodes)) * 3;
        plan_start = pl[0]; plan_pos = pl[1]; plan_ds = pl[2];
        S.plan_cursor[i] = cur + 1;
        // a plan row must name a dataset, a position and a start row the reference could have drawn
        // (environments.py:167-177): clamp and flag instead of reading out of bounds
        bool bad = plan_pos < 0 || plan_pos >= P.n_positions || plan_ds < 0 || plan_ds >= P.n_datasets;
        plan_pos = min(max(plan_pos, 0), P.n_positions - 1);
        plan_ds = P.multi_dataset ? min(max(plan_ds, 0), P.n_datasets - 1) : e.ds;
        const int Tp = D.lengths[plan_ds], lo = P.windows > 0 ? P.windows - 1 : 0;
        if (plan_start < lo || plan_start > Tp - 2) { bad = true; plan_start = min(max(plan_start, lo), Tp - 2); }
        if (bad) atomicOr(S.error_flag, GTE_E_PLAN_RANGE);
    }
    if (P.multi_dataset) {                                                   // :394-398
        const int n = S.ds_episodes[i] + 1;
        if (n % P.episodes_between_switch == 0) {
            if (have_plan) S.ds_episodes[i] = 0;
            else e.ds = next_dataset(P, S, i, r[3]);
        } else {
            S.ds_episodes[i] = n;
        }
        // a plan records the dataset every episode ran on (incl. the one drawn in __init__, :378)
        if (have_plan) e.ds = plan_ds;
    }
    const int T = D.lengths[e.ds];
    e.step = 0;                                                              // :166
    if (have_plan) e.pos_idx = plan_pos;                                     // :167
    else if (P.initial_position_idx >= 0) e.pos_idx = P.initial_position_idx;
    else e.pos_idx = (int)(((uint64_t)r[2] * (uint64_t)P.n_positions) >> 32);
    int start = P.windows > 0 ? P.windows - 1 : 0;                           // :171-172
    if (have_plan) start = plan_start;
    else if (P.max_episode_duration >= 0) {                                  // :173-177 randint(low, high)
        const int64_t lo = start, hi = (int64_t)T - P.max_episode_duration - start;
        const uint64_t x = ((uint64_t)r[1] << 32) | r[0];
        start = (int)(lo + (int64_t)__umul64hi(x, (uint64_t)(hi - lo)));
    }
    e.ep_start = start;
    const double position = P.positions[e.pos_idx];
    const double price = D.price[(int64_t)e.ds * P.t_stride + start];
    e.pf = target_portfolio(position, P.v0, price);                          // :179-183
    for (int k = 0; k < P.n_limit_positions; ++k)                            // self._limit_orders = {} (:168)
        S.limit_price[(int64_t)i * P.n_positions + S.limit_seq[k]] = __longlong_as_double(0x7ff8000000000000ll);
    if (P.n_dyn > 0) {                        // first obs row (:191-192): position, real_position = position, else 0
        const DynRow r = {(float)position, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, e.pos_idx};
        ring_store<GEN, ACC>(P, L, S, i, ring_slot, r);
    }
    if (ACC) episode_acc_init(P, RingLayout<GEN>{L}, S, i, position);
}

}  // namespace gte
