// gte_step.cu — fused per-env transition kernel, reset kernel and info kernel (sm_100a).
//
// One thread per env, structure-of-arrays state in HBM (coalesced 8/4-byte accesses), 256-env tiles; a grid of at
// most one resident wave of CTAs, each walking through consecutive tiles.
// Replaces TradingEnv.step (environments.py:233-272) for N envs in lockstep; see
// include/gte_b200.h for the boundary and DESIGN.md for the data layout / roofline.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <immintrin.h>

#include "gte_step_env.cuh"
#include "gte_launch.h"

namespace gte {

// Each CTA owns `tiles_per_cta` CONSECUTIVE 256-env tiles: 1 while the grid fits on the GPU at once, more beyond that
// (see step_tiles_per_cta).  GEN: the general dynamic-feature catalogue (K0.dyn); every kernel below that writes the
// ring runs one code path, instantiated with GEN = false for no dynamic columns / the default pair, whose ring layout
// is then known at compile time (RingLayout).  ACC (here and in every kernel below): the episode accumulators run
// (acc_on: an episode metric or a stateful dynamic feature); the ACC = false instantiations are the kernels of a run
// without them.
template <int MIN_CTAS, bool GEN = false, bool ACC = false>
__global__ void __launch_bounds__(kStepThreads, MIN_CTAS)
step_kernel(const GteParams P, const GteData D, const GteState S, const void* __restrict__ actions, const StepConsts K0,
            const GteStepOut O, int autoreset, int tiles_per_cta, int env_begin, int env_end, int chunk_flags,
            float* __restrict__ obs_rows, int obs_on_host) {
    // the positions table in shared memory: a per-lane index into the kernel-parameter constant bank would be
    // replayed once per distinct address
    __shared__ double s_pos[GTE_MAX_POSITIONS];
    __shared__ int s_T0;
    if (threadIdx.x < GTE_MAX_POSITIONS) s_pos[threadIdx.x] = P.positions[threadIdx.x];
    if (threadIdx.x == 0) s_T0 = D.lengths[0];          // static data: may be read before the dependency wait
    __syncthreads();
    pdl_wait();                              // everything below reads what the previous kernel of the stream wrote
    StepConsts K = K0;
    K.T0 = s_T0;
    MetricAcc acc;
    const uint64_t tick = *S.tick;
    // the slot this iteration's row goes to: the first env range of an iteration still sees the old clock
    const int ring_slot = ring_slot_of(P, *S.ring_clock + ((chunk_flags & kChunkFirst) ? 1ull : 0ull));
    const int64_t base0 = (int64_t)env_begin + (int64_t)blockIdx.x * tiles_per_cta * kStepThreads;
    for (int t = 0; t < tiles_per_cta; ++t) {
        const int64_t i = base0 + (int64_t)t * kStepThreads + threadIdx.x;
        const bool valid = i < env_end;
        StepThreadOut r = {};
        if (valid) r = step_env_now<GEN, ACC>(P, D, S, actions, K, O, tick, ring_slot, autoreset, (int)i, acc, s_pos);
        // windows=None (environments.py:156-157): the observation is the single row idx, written by the step kernel
        // itself -> one launch per lockstep iteration at small N
        if (obs_rows != nullptr) write_obs_rows<GEN, ACC>(P, D, K.dyn, obs_rows, i, valid, r, obs_on_host != 0);
    }
    reduce_metrics<kStepThreads>(acc, O, S, chunk_flags);
}

// K lockstep iterations in ONE launch (open-loop action stream, batches that fit the GPU at once): one thread per env,
// the env's state stays in REGISTERS for all K iterations and nothing is exchanged between the CTAs on the way — the
// Philox tick and the ring slot of iteration k are tick0 + k / clock0 + 1 + k, and the episode metrics are folded once
// at the end (all iterations but the last into metrics_total, the last one into metrics_step as well).  An iteration
// then costs the transition's own dependency chain (~1.5 us) instead of a kernel launch (~8 us).
// Every per-env output array of O holds n_steps consecutive copies, iteration k writing copy k (gte_rollout).
// obs_rows (windows == 0 only): the one-row observations, every iteration (keep_obs) or the last one.
// The episode record is not replicated: it ends up holding the last episode each env finished.
template <bool GEN = false, bool ACC = false>
__global__ void __launch_bounds__(kStepThreads, 2)
rollout_kernel(const GteParams P, const GteData D, const GteState S, const void* __restrict__ actions, const StepConsts K0,
               const GteStepOut O, int autoreset, int n_steps, int keep_obs, float* __restrict__ obs_rows) {
    __shared__ double s_pos[GTE_MAX_POSITIONS];
    __shared__ int s_T0;
    if (threadIdx.x < GTE_MAX_POSITIONS) s_pos[threadIdx.x] = P.positions[threadIdx.x];
    if (threadIdx.x == 0) s_T0 = D.lengths[0];
    __syncthreads();
    pdl_wait();
    StepConsts K = K0;
    K.T0 = s_T0;
    const int64_t N = P.n_envs;
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    const bool valid = i < N;
    const int64_t ii = valid ? i : N - 1;                    // out-of-range threads shadow the last env and store nothing
    const uint64_t tick0 = __ldcg(S.tick), clock0 = __ldcg(S.ring_clock);
    const int ab = K.action_bytes, F = P.n_static + P.n_dyn;
    MetricAcc acc, acc_prev;
    EnvRegs e = load_env_regs(P, S, ii);
    int64_t a_next = load_action(actions, ab, ii);
    for (int k = 0; k < n_steps; ++k) {
        const int64_t a = a_next;
        if (k + 1 < n_steps) a_next = load_action(actions, ab, (int64_t)(k + 1) * N + ii);   // in flight during the transition
        if (k == n_steps - 1) { acc_prev = acc; acc = MetricAcc(); }
        if (valid) {
            const EnvIn in = make_env_in(P, D, S, K, e, a);
            double p0, p1;
            load_prices(P, D, in, p0, p1);
            GteStepOut o = O;
            o.reward += (int64_t)k * N; o.terminated += (int64_t)k * N; o.truncated += (int64_t)k * N;
            if (o.valuation) o.valuation += (int64_t)k * N;
            if (o.real_position) o.real_position += (int64_t)k * N;
            if (o.info_idx) o.info_idx += (int64_t)k * N;
            if (o.info_step) o.info_step += (int64_t)k * N;
            if (o.pre_reset_portfolio) o.pre_reset_portfolio += (int64_t)k * 4 * N;
            const StepThreadOut r = step_env<false, GEN, ACC>(P, D, S, K, o, tick0 + (uint64_t)k, ring_slot_of(P, clock0 + 1ull + (uint64_t)k),
                                                         autoreset, (int)i, in, p0, p1, acc, s_pos, &e);
            if (obs_rows != nullptr && (keep_obs || k == n_steps - 1))
                write_obs_rows<GEN, ACC>(P, D, K.dyn, obs_rows + (keep_obs ? (int64_t)k * N * F : 0), i, true, r, false);
        }
    }
    if (valid) store_env(S, i, e);
    reduce_metrics<kStepThreads>(acc_prev, O, S, kChunkTotalOnly, 0);
    reduce_metrics<kStepThreads>(acc, O, S, kChunkFirst | kChunkLast, 1, (unsigned)n_steps);
}

// ---- resident "env server" for a HOST policy at small N (gte_step_host, GTE_IO_SERVER) -----------------------------
// A synchronous host step costs launch -> run -> completion -> wake-up (~20 us on this box) however small the kernel.
// The server kernel is launched ONCE and stays resident: every iteration the host writes its actions into mapped pinned
// memory and writes a request word (ctl->req); CTA 0 polls that word over PCIe and hands the command to the other CTAs through a word in
// device memory; every thread advances its env (actions read from, results written straight into, mapped host memory)
// and the last CTA publishes the iteration's sequence number to the host, which polls it.  No launch, no driver call
// and no interrupt on the path.  The kernel leaves by itself when told to (req = kServeStop), or when no request arrived for
// idle_ns — so a cudaDeviceSynchronize() elsewhere in the process waits at most that long — and tells the host
// (ctl->alive = 0), which simply launches it again with the next request.
struct ServeCtl {                // pinned, mapped host memory, owned by the library (one per device)
    // host -> device, ONE 16-byte word pair the kernel fetches with a single PCIe read per poll:
    volatile unsigned long long req;      // (sequence number of the requested iteration << 8) | action_bytes; kServeStop = leave
    volatile unsigned long long actions;  // the request's action array (mapped host memory), written BEFORE req
    volatile uint32_t alive;              // host sets 1 before a launch, the kernel sets 0 on its way out
    uint32_t pad[11];
};
constexpr unsigned long long kServeStop = ~0ull;

// one 16-byte system-scope read of {req, actions}: the host writes `actions` first, so a snapshot that shows the new
// request also shows its action pointer
__device__ __forceinline__ void ld_ctl(const ServeCtl* c, unsigned long long& req, unsigned long long& actions) {
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(req), "=l"(actions) : "l"(c) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// an element of the host's action array: never through a cache that could hold last iteration's line
__device__ __forceinline__ int64_t load_action_volatile(const void* actions, int bytes, int64_t i) {
    switch (bytes) {
        case 1: return (int64_t) __ldcv(reinterpret_cast<const signed char*>(actions) + i);
        case 2: return (int64_t) __ldcv(reinterpret_cast<const short*>(actions) + i);
        case 4: return (int64_t) __ldcv(reinterpret_cast<const int*>(actions) + i);
        default: return (int64_t) __ldcv(reinterpret_cast<const long long*>(actions) + i);
    }
}

template <bool GEN = false, bool ACC = false>
__global__ void __launch_bounds__(kStepThreads, 2)
serve_kernel(const GteParams P, const GteData D, const GteState S, const StepConsts K0, const GteStepOut O, int autoreset,
             float* __restrict__ obs_rows, int obs_on_host, ServeCtl* ctl, unsigned long long* dctl, uint32_t first_seq,
             unsigned long long idle_ns) {
    __shared__ double s_pos[GTE_MAX_POSITIONS];
    __shared__ int s_T0;
    __shared__ unsigned long long s_cmd[2];
    if (threadIdx.x < GTE_MAX_POSITIONS) s_pos[threadIdx.x] = P.positions[threadIdx.x];
    if (threadIdx.x == 0) s_T0 = D.lengths[0];
    __syncthreads();
    StepConsts K = K0;
    K.T0 = s_T0;
    const int64_t i = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
    const bool valid = i < P.n_envs;
    for (uint32_t seq = first_seq;; ++seq) {
        // ---- wait for the host: CTA 0 watches the mapped control block, the others two words in device memory
        //      dctl[0] = (seq << 9) | (leave << 8) | action_bytes, dctl[1] = action pointer (written first)
        if (threadIdx.x == 0) {
            unsigned long long cmd, act;
            if (blockIdx.x == 0) {
                const unsigned long long t0 = global_timer_ns();
                for (;;) {
                    unsigned long long req;
                    ld_ctl(ctl, req, act);
                    if (req != kServeStop && (uint32_t)(req >> 8) == seq) { cmd = ((unsigned long long)seq << 9) | (req & 0xffull); break; }
                    if (req == kServeStop || global_timer_ns() - t0 > idle_ns) { cmd = ((unsigned long long)seq << 9) | 0x100ull; break; }
                }
                // no system-scope fence: the action array is read with volatile (system-scope) loads that are issued only
                // after this poll has RETURNED the new request (data dependency through dctl), and the host wrote the
                // actions before the request word — a fence here costs a PCIe round trip per step
                dctl[1] = act;
                st_release_gpu_u64(dctl, cmd);
            } else {
                for (;;) {
                    cmd = ld_acquire_gpu_u64(dctl);
                    if ((uint32_t)(cmd >> 9) == seq) break;
                }
                act = __ldcg(dctl + 1);
            }
            s_cmd[0] = cmd; s_cmd[1] = act;
        }
        __syncthreads();
        if (s_cmd[0] & 0x100ull) break;
        const int action_bytes = (int)(s_cmd[0] & 0xffull);
        const void* actions = reinterpret_cast<const void*>(s_cmd[1]);
        // ---- one lockstep iteration
        MetricAcc acc;
        const uint64_t tick = __ldcg(S.tick);
        const int ring_slot = ring_slot_of(P, __ldcg(S.ring_clock) + 1ull);
        StepThreadOut r = {};
        if (valid) {
            const int64_t a = load_action_volatile(actions, action_bytes, i);         // over PCIe, beside the state loads
            const EnvIn in = make_env_in(P, D, S, K, load_env_regs<true>(P, S, i), a);
            double p0, p1;
            load_prices(P, D, in, p0, p1);
            r = step_env<true, GEN, ACC>(P, D, S, K, O, tick, ring_slot, autoreset, (int)i, in, p0, p1, acc, s_pos);
        }
        if (obs_rows != nullptr) write_obs_rows<GEN, ACC>(P, D, K.dyn, obs_rows, i, valid, r, obs_on_host != 0);
        GteStepOut o = O;
        o.seq_value = seq;                               // what the last CTA publishes to the host when all is visible
        reduce_metrics<kStepThreads>(acc, o, S, kChunkFirst | kChunkLast);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        __threadfence_system();
        ctl->alive = 0u;
    }
}

// TradingEnv.reset for the masked envs (environments.py:163-199, :393-400); `first` also performs
// the dataset draw of MultiDatasetTradingEnv.__init__ (:377-378).
template <bool GEN = false, bool ACC = false>
__global__ void __launch_bounds__(kStepThreads)
reset_kernel(const GteParams P, const GteData D, const GteState S, const uint8_t* __restrict__ mask,
             int first, const DynLayout L) {
    const int i = blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= P.n_envs) return;
    const uint64_t tick = *S.tick;
    if (first) {
        S.ds_used[i] = 0;
        S.ds_episodes[i] = 0;
        S.plan_cursor[i] = 0;
        int ds = 0;
        if (P.multi_dataset && !(P.plan_episodes > 0 && S.reset_plan != nullptr)) {
            uint32_t r[4];
            philox_draw(P.seed, tick, (uint64_t)(P.env_id_offset + i), r);
            ds = next_dataset(P, S, i, r[3]);
        }
        S.dataset_idx[i] = ds;
        return;
    }
    if (mask != nullptr && mask[i] == 0) return;
    EnvRegs e;
    e.ds = S.dataset_idx[i];
    reset_env<GEN, ACC>(P, D, S, i, tick, ring_slot_of(P, *S.ring_clock), e, L);    // the row currently observed
    S.asset[i] = e.pf.asset;
    S.fiat[i] = e.pf.fiat;
    S.interest_asset[i] = e.pf.ia;
    S.interest_fiat[i] = e.pf.ifi;
    S.pos_idx[i] = e.pos_idx;
    S.step[i] = e.step;
    S.ep_start[i] = e.ep_start;
    S.dataset_idx[i] = e.ds;
}

__global__ void bump_tick_kernel(uint64_t* tick) { *tick = *tick + 1ull; }

// History's last row from the current state (environments.py:253-264, portfolio.py:49-57).
__global__ void __launch_bounds__(kStepThreads)
info_kernel(const GteParams P, const GteData D, const GteState S, const GteInfo I) {
    const int i = blockIdx.x * kStepThreads + threadIdx.x;
    if (i >= P.n_envs) return;
    Portfolio pf;
    pf.asset = S.asset[i]; pf.fiat = S.fiat[i]; pf.ia = S.interest_asset[i]; pf.ifi = S.interest_fiat[i];
    const int step = S.step[i], ep_start = S.ep_start[i], ds = S.dataset_idx[i], pidx = S.pos_idx[i];
    const int idx = ep_start + step;
    const double price = D.price[(int64_t)ds * P.t_stride + idx];
    const double position = P.positions[pidx];
    // the reset row holds portfolio_initial_value and real_position = position (:192-194)
    const double val = (step == 0) ? P.v0 : valorisation(pf, price);
    const double rp = (step == 0) ? position : real_position(pf, price, val);
    if (I.idx) I.idx[i] = idx;
    if (I.step) I.step[i] = step;
    if (I.position_index) I.position_index[i] = pidx;
    if (I.dataset_idx) I.dataset_idx[i] = ds;
    if (I.position) I.position[i] = position;
    if (I.real_position) I.real_position[i] = rp;
    if (I.portfolio_valuation) I.portfolio_valuation[i] = val;
    if (I.data_close) I.data_close[i] = price;
    if (I.distribution) {                                                    // portfolio.py:49-57
        const int64_t N = P.n_envs;
        const double na = -pf.asset, nf = -pf.fiat;
        I.distribution[i] = (pf.asset > 0.0) ? pf.asset : 0.0;
        I.distribution[N + i] = (pf.fiat > 0.0) ? pf.fiat : 0.0;
        I.distribution[2 * N + i] = (na > 0.0) ? na : 0.0;
        I.distribution[3 * N + i] = (nf > 0.0) ? nf : 0.0;
        I.distribution[4 * N + i] = pf.ia;
        I.distribution[5 * N + i] = pf.ifi;
    }
}

// ---- host launchers -------------------------------------------------------------------------------

// Largest double x with fl(x / v0) <= ratio.  Correctly rounded division is monotonic in x, so `valuation <= x` decides
// the reference's `valuation / initial <= ratio` (environments.py:246) bit for bit without dividing on the device.
// NaN when the search does not settle within a few ulps (denormal ratios): the kernel then divides.
static double done_threshold(double v0, double ratio) {
    if (!(v0 > 0.0) || !std::isfinite(v0) || !std::isfinite(ratio)) return NAN;
    volatile double x = ratio * v0;
    for (int k = 0; k < 64 && (double)(x / v0) <= ratio; ++k) x = std::nextafter((double)x, INFINITY);
    for (int k = 0; k < 128; ++k) {
        volatile double q = x / v0;
        if (q <= ratio) {
            volatile double up = std::nextafter((double)x, INFINITY);
            volatile double qu = up / v0;
            return (qu > ratio) ? (double)x : NAN;
        }
        x = std::nextafter((double)x, -INFINITY);
    }
    return NAN;
}

StepConsts make_step_consts(const GteParams& P) {
    static const bool no_thr = [] { const char* e = getenv("GTE_NO_DONE_THRESHOLD"); return e != nullptr && atoi(e) != 0; }();
    StepConsts K;
    K.done_thr = no_thr ? NAN : done_threshold(P.v0, P.done_ratio);
    K.action_bytes = P.action_bytes == 0 ? 8 : P.action_bytes;
    K.T0 = 0;                                // filled in on the device
    K.dyn = dyn_layout(P);
    return K;
}

bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("GTE_PDL"); return e == nullptr || atoi(e) != 0; }();
    return on;
}

static int g_num_sms = 0;
int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

// Consecutive 256-env tiles per CTA: the grid is capped at the CTAs that are resident at once (SMs x 3), so a large
// batch runs as ONE wave of CTAs that each walk through their tiles — the per-CTA set-up and the metric fold are paid
// once per CTA instead of once per tile or two (C5 shard: 0.112 -> 0.089 ms; GTE_STEP_MAX_CTAS overrides the cap).
static int step_tiles_per_cta(int n_envs) {
    static const int max_ctas = [] { const char* e = getenv("GTE_STEP_MAX_CTAS"); return e ? atoi(e) : 0; }();
    int64_t cap = max_ctas > 0 ? max_ctas : (int64_t)num_sms() * 3;
    if (cap > kMaxPartialRows) cap = kMaxPartialRows;
    const int64_t tiles = ((int64_t)n_envs + kStepThreads - 1) / kStepThreads;
    return (int)((tiles + cap - 1) / cap);
}

int step_grid(int n_envs) {
    const int64_t tiles = ((int64_t)n_envs + kStepThreads - 1) / kStepThreads;
    const int tpc = step_tiles_per_cta(n_envs);
    return (int)((tiles + tpc - 1) / tpc);
}

cudaError_t launch_step_range(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                              const GteStepOut& O, int autoreset, int env_begin, int env_end, int chunk_flags,
                              cudaStream_t stream, float* obs_rows, bool obs_on_host) {
    const StepConsts K = make_step_consts(P);
    const int n = env_end - env_begin;
    const int grid = step_grid(n), tpc = step_tiles_per_cta(n);
    // same shared-memory carve-out as the gather kernel, so CTAs of both can be resident on one SM
    static bool carveout_set[16] = {};                 // per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (!carveout_set[dev & 15]) {
        cudaFuncSetAttribute(step_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(step_kernel<3, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(step_kernel<3, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(step_kernel<3, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carveout_set[dev & 15] = true;
    }
    // ONE build: 3 CTAs per SM at 80 registers with no local-memory spills.  The 4-CTAs/SM build (64 registers, 18 STL /
    // 15 LDL) measures the same on the C5 shard (0.0925 vs 0.0930 ms): the kernel is bound by the issue rate of its
    // dependent fp64 chains, not by resident warps, loads or stores (profiles/r02_tuning.md has the diagnostic runs)
    auto kern = acc_on(P) ? (K.dyn.general ? step_kernel<3, true, true> : step_kernel<3, false, true>)
                                    : (K.dyn.general ? step_kernel<3, true> : step_kernel<3>);
    return launch_pdl(kern, dim3(grid), dim3(kStepThreads), 0, stream, P, D, S, actions, K, O, autoreset, tpc,
                      env_begin, env_end, chunk_flags, obs_rows, obs_on_host ? 1 : 0);
}

cudaError_t launch_step(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                        const GteStepOut& O, int autoreset, cudaStream_t stream) {
    return launch_step_range(P, D, S, actions, O, autoreset, 0, P.n_envs, kChunkFirst | kChunkLast, stream, nullptr);
}

cudaError_t launch_reset(const GteParams& P, const GteData& D, const GteState& S, const uint8_t* mask,
                         int first, cudaStream_t stream) {
    const int grid = (P.n_envs + kStepThreads - 1) / kStepThreads;
    const DynLayout L = dyn_layout(P);
    auto kern = acc_on(P) ? (L.general ? reset_kernel<true, true> : reset_kernel<false, true>)
                                    : (L.general ? reset_kernel<true> : reset_kernel<false>);
    kern<<<grid, kStepThreads, 0, stream>>>(P, D, S, mask, first, L);
    bump_tick_kernel<<<1, 1, 0, stream>>>(S.tick);
    return cudaGetLastError();
}

// ---- one lockstep iteration = step + gather; optionally env chunks pipelined over two streams -----
// (opt-in: the step kernel is latency-bound and the gather HBM-bound, but running the step of chunk c+1
// beside the gather of chunk c did not beat two plain launches on B200)
struct AuxStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork[16] = {};
    cudaEvent_t join = nullptr;
    int device = -1;
};
static AuxStream g_aux[16];

static cudaError_t aux_for_current_device(AuxStream** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    AuxStream& a = g_aux[dev & 15];
    if (a.stream == nullptr) {
        if ((e = cudaStreamCreateWithFlags(&a.stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
        for (auto& ev : a.fork)
            if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming)) != cudaSuccess) return e;
        a.device = dev;
    }
    *out = &a;
    return cudaSuccess;
}

int default_chunks(int n_envs) {
    // Measured on B200 (profiles/r01_tuning.md): running the step kernel of range c+1 beside the gather of
    // range c does not beat two plain launches — the gather already saturates HBM writes and the extra
    // launches add tails — so pipelining is opt-in (n_chunks > 1 or GTE_CHUNKS).
    static const int forced = [] { const char* e = getenv("GTE_CHUNKS"); return e ? atoi(e) : 0; }();
    (void)n_envs;
    if (forced > 0) return forced > 16 ? 16 : forced;
    return 1;
}

cudaError_t launch_step_obs(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                            const GteStepOut& O, float* obs, int autoreset, int variant, int n_chunks,
                            cudaStream_t stream) {
    const bool may_fuse = n_chunks <= 0;     // an explicit n_chunks (1 = two plain launches) is honoured as given
    if (n_chunks <= 0) n_chunks = default_chunks(P.n_envs);
    if (n_chunks > 16) n_chunks = 16;
    cudaError_t e;
    if (P.windows == 0)            // windows=None: the step kernel writes the one-row observation itself
        return launch_step_range(P, D, S, actions, O, autoreset, 0, P.n_envs, kChunkFirst | kChunkLast, stream, obs);
    if (n_chunks == 1) {
        bool fused = false;                  // small batches: transition + gather in ONE launch
        if (may_fuse && (e = launch_fused_step_obs(P, D, S, actions, make_step_consts(P), O, obs, autoreset, variant, stream, &fused)) != cudaSuccess || fused)
            return e;
        if ((e = launch_step(P, D, S, actions, O, autoreset, stream)) != cudaSuccess) return e;
        return launch_obs_range(P, D, S, obs, variant, 0, P.n_envs, stream);
    }
    AuxStream* aux = nullptr;
    if ((e = aux_for_current_device(&aux)) != cudaSuccess) return e;
    const int64_t per = (((int64_t)P.n_envs + n_chunks - 1) / n_chunks + kStepThreads - 1) / kStepThreads * kStepThreads;
    n_chunks = (int)(((int64_t)P.n_envs + per - 1) / per);         // drop empty tail chunks
    for (int c = 0; c < n_chunks; ++c) {
        const int b = (int)(c * per);
        const int en = (int)((c + 1) * per < P.n_envs ? (c + 1) * per : P.n_envs);
        const int flags = (c == 0 ? kChunkFirst : 0) | (c == n_chunks - 1 ? kChunkLast : 0);
        if ((e = launch_step_range(P, D, S, actions, O, autoreset, b, en, flags, stream, nullptr)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(aux->fork[c], stream)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(aux->stream, aux->fork[c], 0)) != cudaSuccess) return e;
        if ((e = launch_obs_range(P, D, S, obs, variant, b, en, aux->stream)) != cudaSuccess) return e;
    }
    if ((e = cudaEventRecord(aux->join, aux->stream)) != cudaSuccess) return e;
    return cudaStreamWaitEvent(stream, aux->join, 0);
}

// ---- n_steps iterations from one host call (open-loop action stream) ------------------------------
// Whether gte_rollout runs as ONE persistent launch (rollout_kernel): the batch must fit the GPU at once (every env owns
// a thread for the whole call) and windowed observations must not be wanted for every iteration.
bool rollout_is_persistent(const GteParams& P, int n_steps, int keep_obs) {
    static const bool enabled = [] { const char* e = getenv("GTE_ROLLOUT_PERSISTENT"); return e == nullptr || atoi(e) != 0; }();
    const int64_t grid = ((int64_t)P.n_envs + kStepThreads - 1) / kStepThreads;
    return enabled && n_steps >= 2 && grid <= (int64_t)num_sms() * 2 && 2 * grid <= kMaxPartialRows &&
           (P.windows == 0 || !keep_obs);
}

cudaError_t launch_rollout(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                           int n_steps, const GteStepOut& O, float* obs, int keep_obs, int autoreset, int variant,
                           cudaStream_t stream) {
    const int64_t N = P.n_envs;
    const int64_t obs_elems = N * (int64_t)(P.windows > 0 ? P.windows : 1) * (P.n_static + P.n_dyn);
    cudaError_t e;
    if (rollout_is_persistent(P, n_steps, keep_obs)) {
        const int grid = (int)((N + kStepThreads - 1) / kStepThreads);
        const StepConsts K = make_step_consts(P);
        auto kern = acc_on(P) ? (K.dyn.general ? rollout_kernel<true, true> : rollout_kernel<false, true>)
                                        : (K.dyn.general ? rollout_kernel<true> : rollout_kernel<false>);
        e = launch_pdl(kern, dim3(grid), dim3(kStepThreads), 0, stream,
                       P, D, S, actions, K, O, autoreset, n_steps, keep_obs, P.windows == 0 ? obs : (float*)nullptr);
        if (e != cudaSuccess || P.windows == 0) return e;
        return launch_obs_range(P, D, S, obs, variant, 0, P.n_envs, stream);     // the last iteration's windows
    }
    for (int k = 0; k < n_steps; ++k) {
        GteStepOut o = O;                                   // iteration k writes copy k of every per-env array
        o.reward += k * N; o.terminated += k * N; o.truncated += k * N;
        if (o.valuation) o.valuation += k * N;
        if (o.real_position) o.real_position += k * N;
        if (o.info_idx) o.info_idx += k * N;
        if (o.info_step) o.info_step += k * N;
        if (o.pre_reset_portfolio) o.pre_reset_portfolio += k * 4 * N;
        const bool want_obs = keep_obs || k == n_steps - 1;
        float* obs_k = obs + (keep_obs ? k * obs_elems : 0);
        const void* a = static_cast<const char*>(actions) + (int64_t)k * N * (P.action_bytes == 0 ? 8 : P.action_bytes);
        if (P.windows == 0) {                               // the step kernel writes the one-row observation itself
            e = launch_step_range(P, D, S, a, o, autoreset, 0, P.n_envs, kChunkFirst | kChunkLast, stream,
                                  want_obs ? obs_k : nullptr);
        } else {
            bool fused = false;
            if (want_obs) e = launch_fused_step_obs(P, D, S, a, make_step_consts(P), o, obs_k, autoreset, variant, stream, &fused);
            if (!fused) {
                e = launch_step(P, D, S, a, o, autoreset, stream);
                if (e == cudaSuccess && want_obs) e = launch_obs_range(P, D, S, obs_k, variant, 0, P.n_envs, stream);
            }
        }
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ---- one lockstep iteration for a HOST policy: actions from pinned host memory, results into one pinned block ----
struct HostIOStreams {
    cudaStream_t in = nullptr, out = nullptr;
    cudaEvent_t ev_in = nullptr, ev_step = nullptr;
    uint32_t seq = 0;                // MAPPED / SERVER mode: number of the last call (what its kernel writes into the block)
    // SERVER mode: the resident kernel's stream, its mapped control block, the device-side command word, and what the
    // running instance was launched for (a call with anything else quiesces it and launches a new one)
    cudaStream_t serve = nullptr;
    ServeCtl* ctl = nullptr;
    unsigned long long* dctl = nullptr;
    bool serving = false;
    GteParams sp; GteData sd; GteState ss; GteStepOut so; float* sobs = nullptr; int sauto = 0;
    // gte_step_host_begin / _end: completion events of the result copies in flight, keyed by the host result block
    struct Pending { const void* results = nullptr; cudaEvent_t ev = nullptr; cudaEvent_t ev_in = nullptr; cudaEvent_t ev_step = nullptr;
                     int64_t n = 0; bool sparse = false; bool open = false; } pending[4];     // open: begun, not yet ended
};
static HostIOStreams g_hio[16];

static cudaError_t hio_for_current_device(HostIOStreams** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    HostIOStreams& h = g_hio[dev & 15];
    if (h.in == nullptr) {
        if ((e = cudaStreamCreateWithFlags(&h.in, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaStreamCreateWithFlags(&h.out, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&h.ev_in, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&h.ev_step, cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    *out = &h;
    return cudaSuccess;
}

// Stop the resident server kernel of the current device, if any: every other entry point of the library calls this
// first, so the server never runs beside a kernel that touches the same env state.
cudaError_t serve_quiesce() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return cudaSuccess;
    HostIOStreams& h = g_hio[dev & 15];
    if (!h.serving) return cudaSuccess;
    h.ctl->req = kServeStop;
    const cudaError_t e = cudaStreamSynchronize(h.serve);
    h.ctl->req = 0ull;
    h.serving = false;
    return e;
}

static unsigned long long serve_idle_ns() {
    static const unsigned long long ns = [] { const char* e = getenv("GTE_SERVER_IDLE_US"); return (unsigned long long)(e ? atoll(e) : 2000) * 1000ull; }();
    return ns;
}

bool serve_supported(const GteParams& P) {
    // the whole batch must be resident at once (every env owns a thread for as long as the kernel lives), and the
    // observation must be the step kernel's own one-row write (windows == 0)
    const int64_t grid = ((int64_t)P.n_envs + kStepThreads - 1) / kStepThreads;
    return P.windows == 0 && grid <= (int64_t)num_sms() && grid <= kMaxPartialRows;
}

// out->reward / flags / error / (device block only) the sparse episode-end list -> a result block (include/gte_b200.h)
static void point_results(GteStepOut& o, char* blk, int64_t N, bool device_block) {
    o.reward = reinterpret_cast<double*>(blk);
    o.terminated = reinterpret_cast<uint8_t*>(blk + GTE_HOST_RESULT_TERM_OFFSET(N));
    o.truncated = reinterpret_cast<uint8_t*>(blk + GTE_HOST_RESULT_TRUNC_OFFSET(N));
    o.error_out = reinterpret_cast<int32_t*>(blk + GTE_HOST_RESULT_ERROR_OFFSET(N));
    o.ended_list = nullptr; o.ended_counter = nullptr; o.ended_n_out = nullptr; o.ended_cap = 0;
    if (device_block) {          // the append counter needs device atomics: mapped host blocks carry dense flags only
        o.ended_list = reinterpret_cast<uint32_t*>(blk + GTE_HOST_RESULT_ENDED_OFFSET(N));
        o.ended_counter = reinterpret_cast<uint32_t*>(blk + GTE_HOST_RESULT_COUNTER_OFFSET(N));
        o.ended_n_out = reinterpret_cast<uint32_t*>(blk + GTE_HOST_RESULT_NENDED_OFFSET(N));
        o.ended_cap = (uint32_t)GTE_HOST_RESULT_ENDED_CAP(N);
    }
}

// The device-to-host copies of one result block (copy engines).  Default: ONE copy of the block (its sparse prefix when
// the flags travel as a list).  float32 reward wire (opt-in, lossy): the fp64 rewards stay in the device block, the block
// copy starts behind them and the rounded rewards come back with a copy of their own.  reward_host_count (result relay,
// gte_relay_*): only that many leading rewards take this GPU's own link — the caller routes the rest through a peer.
static bool f32_wire(const GteHostIO& io) { return io.reward_f32_host != nullptr && io.dev_reward_f32 != nullptr; }
static cudaError_t copy_results_to_host(const GteHostIO& io, int64_t N, bool sparse, cudaStream_t s) {
    const size_t end = sparse ? (size_t)GTE_HOST_RESULT_SPARSE_BYTES(N) : (size_t)GTE_HOST_RESULT_BYTES(N);
    const size_t hdr = (size_t)GTE_HOST_RESULT_ERROR_OFFSET(N);
    const int64_t own = (io.reward_host_count > 0 && io.reward_host_count < N) ? io.reward_host_count : N;
    char* dst = static_cast<char*>(io.results);
    const char* src = static_cast<const char*>(io.dev_results);
    cudaError_t e;
    if (f32_wire(io)) {
        if ((e = cudaMemcpyAsync(io.reward_f32_host, io.dev_reward_f32, (size_t)own * 4, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
        return cudaMemcpyAsync(dst + hdr, src + hdr, end - hdr, cudaMemcpyDeviceToHost, s);
    }
    if (own == N) return cudaMemcpyAsync(dst, src, end, cudaMemcpyDeviceToHost, s);
    if ((e = cudaMemcpyAsync(dst, src, (size_t)own * 8, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    return cudaMemcpyAsync(dst + hdr, src + hdr, end - hdr, cudaMemcpyDeviceToHost, s);
}

// After the sparse prefix has landed: more episodes ended than the list holds -> fetch the dense flag bytes as well.
static cudaError_t fetch_dense_flags_if_needed(const GteHostIO& io, int64_t N, cudaStream_t copy_stream) {
    const uint32_t n_ended = *reinterpret_cast<volatile uint32_t*>(static_cast<char*>(io.results) + GTE_HOST_RESULT_NENDED_OFFSET(N));
    if (n_ended <= (uint32_t)GTE_HOST_RESULT_ENDED_CAP(N)) return cudaSuccess;
    const int64_t off = GTE_HOST_RESULT_TERM_OFFSET(N);
    cudaError_t e = cudaMemcpyAsync(static_cast<char*>(io.results) + off, static_cast<char*>(io.dev_results) + off, (size_t)(2 * N),
                                    cudaMemcpyDeviceToHost, copy_stream);
    return e != cudaSuccess ? e : cudaStreamSynchronize(copy_stream);
}

// The host polls mapped memory for a kernel's answer; whatever goes wrong on the device, it gives up after
// GTE_HOST_SPIN_TIMEOUT_S (default 20 s) instead of spinning for ever.
static double host_now_s() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
static bool spin_deadline_passed(double t_start) {
    static const double limit = [] { const char* e = getenv("GTE_HOST_SPIN_TIMEOUT_S"); return e ? atof(e) : 20.0; }();
    return host_now_s() - t_start > limit;
}

int host_io_mode(const GteParams& P, int mode) {
    if (mode == GTE_IO_SERVER) return serve_supported(P) ? GTE_IO_SERVER : GTE_IO_MAPPED;
    // measured on B200 (tools/host_path_probe.py, profiles/r02_tuning.md): with a gather behind the step kernel the
    // mapped writes delay it, so the copy engines win from ~40k envs on; without one mapped wins up to >= 64k envs
    static const long long forced_max = [] { const char* e = getenv("GTE_IO_MAPPED_MAX_BYTES"); return e ? atoll(e) : -1ll; }();
    if (mode == GTE_IO_COPY || mode == GTE_IO_MAPPED) return mode;
    const int ab = P.action_bytes == 0 ? 8 : P.action_bytes;
    const long long mapped_max = forced_max >= 0 ? forced_max : (P.windows > 0 ? 384ll << 10 : 1ll << 20);
    return (int64_t)P.n_envs * (ab + 10) <= mapped_max ? GTE_IO_MAPPED : GTE_IO_COPY;
}

cudaError_t launch_step_host(const GteParams& P, const GteData& D, const GteState& S, const GteHostIO& io,
                             const GteStepOut& O, float* obs, int autoreset, int variant, int* mode_used,
                             cudaStream_t stream) {
    const int64_t N = P.n_envs;
    const int ab = P.action_bytes == 0 ? 8 : P.action_bytes;
    const int mode = host_io_mode(P, io.mode);
    if (mode_used != nullptr) *mode_used = mode;
    HostIOStreams* h = nullptr;
    cudaError_t e;
    if ((e = hio_for_current_device(&h)) != cudaSuccess) return e;
    // the results of this iteration: one block, on the device (COPY) or straight in the mapped host memory (MAPPED)
    char* blk = static_cast<char*>(mode != GTE_IO_COPY ? io.results : io.dev_results);
    GteStepOut o = O;
    point_results(o, blk, N, mode == GTE_IO_COPY);
    const bool sparse = mode == GTE_IO_COPY && io.sparse_flags != 0;
    o.reward_f32 = (mode == GTE_IO_COPY && f32_wire(io)) ? static_cast<float*>(io.dev_reward_f32) : nullptr;
    volatile uint32_t* seq_word = reinterpret_cast<volatile uint32_t*>(static_cast<char*>(io.results) + GTE_HOST_RESULT_SEQ_OFFSET(N));
    uint32_t seq = 0;
    if (mode == GTE_IO_MAPPED || mode == GTE_IO_SERVER) {
        seq = ++h->seq ? h->seq : ++h->seq;                  // never 0
        *seq_word = 0;
        o.seq_out = const_cast<uint32_t*>(seq_word);
        o.seq_value = seq;
    } else {
        o.seq_out = nullptr;
    }
    if (mode == GTE_IO_SERVER) {
        // ---- resident server: (re)launch it if it is not running for exactly these buffers, then hand it the request
        if (h->serve == nullptr) {
            if ((e = cudaStreamCreateWithFlags(&h->serve, cudaStreamNonBlocking)) != cudaSuccess) return e;
            if ((e = cudaHostAlloc(reinterpret_cast<void**>(&h->ctl), sizeof(ServeCtl), cudaHostAllocMapped)) != cudaSuccess) return e;
            memset(h->ctl, 0, sizeof(ServeCtl));
            if ((e = cudaMalloc(reinterpret_cast<void**>(&h->dctl), 64)) != cudaSuccess) return e;
        }
        GteParams p0 = P;
        p0.action_bytes = 0;                                 // travels with every request, not with the launch
        if (io.obs_host != nullptr) obs = static_cast<float*>(io.obs_host);   // windows == 0: rows written straight to the host
        const bool same = h->serving && memcmp(&h->sp, &p0, sizeof(p0)) == 0 && memcmp(&h->sd, &D, sizeof(D)) == 0 &&
                          memcmp(&h->ss, &S, sizeof(S)) == 0 && h->so.metrics_step == O.metrics_step &&
                          h->so.reward == o.reward && h->so.episode_record == O.episode_record &&
                          h->sobs == obs && h->sauto == autoreset;
        if (h->serving && !same && (e = serve_quiesce()) != cudaSuccess) return e;
        auto launch = [&]() -> cudaError_t {
            cudaError_t le;
            // behind whatever the caller enqueued on its stream so far (reset, previous iterations ...)
            if ((le = cudaEventRecord(h->ev_step, stream)) != cudaSuccess) return le;
            if ((le = cudaStreamWaitEvent(h->serve, h->ev_step, 0)) != cudaSuccess) return le;
            if ((le = cudaMemsetAsync(h->dctl, 0, 64, h->serve)) != cudaSuccess) return le;
            h->ctl->alive = 1u;
            const int grid = (int)((N + kStepThreads - 1) / kStepThreads);
            const StepConsts K = make_step_consts(p0);
            auto kern = acc_on(p0) ? (K.dyn.general ? serve_kernel<true, true> : serve_kernel<false, true>)
                                             : (K.dyn.general ? serve_kernel<true> : serve_kernel<false>);
            kern<<<grid, kStepThreads, 0, h->serve>>>(p0, D, S, K, o, autoreset, obs, io.obs_host != nullptr ? 1 : 0, h->ctl,
                                                      h->dctl, seq, serve_idle_ns());
            if ((le = cudaGetLastError()) != cudaSuccess) return le;
            h->serving = true;
            h->sp = p0; h->sd = D; h->ss = S; h->so = O; h->so.reward = o.reward; h->sobs = obs; h->sauto = autoreset;
            return cudaSuccess;
        };
        if ((!h->serving || h->ctl->alive == 0u) && (e = launch()) != cudaSuccess) return e;
        const double t_start = host_now_s();
        h->ctl->actions = (unsigned long long)reinterpret_cast<uintptr_t>(io.actions);
        __atomic_thread_fence(__ATOMIC_RELEASE);             // the caller's action writes (and the pointer) before the request
        h->ctl->req = ((unsigned long long)seq << 8) | (unsigned long long)ab;
        for (uint32_t spins = 1; *seq_word != seq; ++spins) {
            _mm_pause();
            if (h->ctl->alive == 0u) {                       // it left (idle time-out) — possibly without seeing this request
                __atomic_thread_fence(__ATOMIC_ACQUIRE);
                if (*seq_word == seq) break;
                if ((e = cudaStreamSynchronize(h->serve)) != cudaSuccess) return e;
                if ((e = launch()) != cudaSuccess) return e;
            } else if ((spins & 0x3fffu) == 0) {
                if ((e = cudaStreamQuery(h->serve)) != cudaErrorNotReady && e != cudaSuccess) return e;   // a faulted kernel never answers
                if (spin_deadline_passed(t_start)) return cudaErrorLaunchTimeout;
            }
        }
        __atomic_thread_fence(__ATOMIC_ACQUIRE);
        return cudaSuccess;
    }
    if ((e = serve_quiesce()) != cudaSuccess) return e;
    const void* actions = io.actions;
    if (mode == GTE_IO_COPY) {
        // the previous call returned only after ITS step kernel's results had reached the host, so dev_actions is
        // free: the copy does not wait for `stream` and runs beside the previous iteration's gather
        if ((e = cudaMemcpyAsync(io.dev_actions, io.actions, (size_t)(N * ab), cudaMemcpyHostToDevice, h->in)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(h->ev_in, h->in)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(stream, h->ev_in, 0)) != cudaSuccess) return e;
        actions = io.dev_actions;
    }
    // windows=None: the step kernel writes the one-row observation itself — in the MAPPED mode straight into the host
    // copy when the caller wants the observations there
    const bool obs_mapped = P.windows == 0 && mode == GTE_IO_MAPPED && io.obs_host != nullptr;
    float* obs_rows = P.windows == 0 ? (obs_mapped ? static_cast<float*>(io.obs_host) : obs) : nullptr;
    if ((e = launch_step_range(P, D, S, actions, o, autoreset, 0, P.n_envs, kChunkFirst | kChunkLast, stream, obs_rows, obs_mapped)) != cudaSuccess) return e;
    if (io.step_done_event != nullptr &&
        (e = cudaEventRecord(static_cast<cudaEvent_t>(io.step_done_event), stream)) != cudaSuccess) return e;
    const bool obs_copy = io.obs_host != nullptr && !obs_mapped;     // one more D2H behind the gather, on `stream` itself
    if (mode == GTE_IO_COPY) {
        if ((e = cudaEventRecord(h->ev_step, stream)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(h->out, h->ev_step, 0)) != cudaSuccess) return e;
        if ((e = copy_results_to_host(io, N, sparse, h->out)) != cudaSuccess) return e;
        if (P.windows > 0 && (e = launch_obs_range(P, D, S, obs, variant, 0, P.n_envs, stream)) != cudaSuccess) return e;
        if (obs_copy) {
            if ((e = cudaMemcpyAsync(io.obs_host, obs, (size_t)io.obs_bytes, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
            if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
        }
        if ((e = cudaStreamSynchronize(h->out)) != cudaSuccess) return e;   // reward / flags / error flag are on the host; the gather runs on
        return sparse ? fetch_dense_flags_if_needed(io, N, h->out) : cudaSuccess;
    }
    // MAPPED: the kernel itself wrote the host block and, last, the call's sequence number: poll that word instead
    // of going through the driver (the lowest-latency completion signal there is)
    if (P.windows > 0 && (e = launch_obs_range(P, D, S, obs, variant, 0, P.n_envs, stream)) != cudaSuccess) return e;
    if (obs_copy) {
        if ((e = cudaMemcpyAsync(io.obs_host, obs, (size_t)io.obs_bytes, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
        return cudaStreamSynchronize(stream);               // everything of this iteration, observations included
    }
    const double t_start = host_now_s();
    for (uint32_t spins = 1; *seq_word != seq; ++spins) {
        _mm_pause();
        if ((spins & 0x3fffu) == 0) {                        // a faulted kernel never writes the word: ask the driver now and then
            e = cudaStreamQuery(stream);
            if (e != cudaErrorNotReady) return (e == cudaSuccess && *seq_word != seq) ? cudaErrorUnknown : e;
            if (spin_deadline_passed(t_start)) return cudaErrorLaunchTimeout;
        }
    }
    return cudaSuccess;
}

// ---- the same iteration split in two: begin() enqueues everything and returns, end() waits for the result block -----
// A caller that alternates TWO GteHostIO sets (host + device result block and action staging each) can call
// begin(k+1) before end(k): the device-to-host copy of iteration k then runs under the action copy, transition and
// gather of iteration k+1 (copy engines only; the blocks of a set are free again once its end() has returned).
cudaError_t launch_step_host_begin(const GteParams& P, const GteData& D, const GteState& S, const GteHostIO& io,
                                   const GteStepOut& O, float* obs, int autoreset, int variant, cudaStream_t stream) {
    const int64_t N = P.n_envs;
    const int ab = P.action_bytes == 0 ? 8 : P.action_bytes;
    HostIOStreams* h = nullptr;
    cudaError_t e;
    if ((e = hio_for_current_device(&h)) != cudaSuccess) return e;
    if ((e = serve_quiesce()) != cudaSuccess) return e;
    HostIOStreams::Pending* slot = nullptr;
    for (auto& p : h->pending) if (p.results == io.results) slot = &p;
    if (slot == nullptr) for (auto& p : h->pending) if (p.results == nullptr) { slot = &p; break; }
    if (slot == nullptr) for (auto& p : h->pending) if (!p.open) { slot = &p; break; }     // a block whose iteration has ended: its slot is free
    if (slot == nullptr) return cudaErrorInvalidValue;       // more than 4 result blocks in flight
    if (slot->ev == nullptr) {
        if ((e = cudaEventCreateWithFlags(&slot->ev, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&slot->ev_in, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&slot->ev_step, cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    slot->results = io.results;
    slot->open = true;
    slot->n = N;
    slot->sparse = io.sparse_flags != 0;
    GteStepOut o = O;
    point_results(o, static_cast<char*>(io.dev_results), N, true);
    o.seq_out = nullptr;
    o.reward_f32 = f32_wire(io) ? static_cast<float*>(io.dev_reward_f32) : nullptr;
    // this set's staging buffer is free: its previous iteration's end() has returned (the caller's contract)
    if ((e = cudaMemcpyAsync(io.dev_actions, io.actions, (size_t)(N * ab), cudaMemcpyHostToDevice, h->in)) != cudaSuccess) return e;
    if ((e = cudaEventRecord(slot->ev_in, h->in)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(stream, slot->ev_in, 0)) != cudaSuccess) return e;
    float* obs_rows = P.windows == 0 ? obs : nullptr;
    if ((e = launch_step_range(P, D, S, io.dev_actions, o, autoreset, 0, P.n_envs, kChunkFirst | kChunkLast, stream, obs_rows)) != cudaSuccess) return e;
    if (io.step_done_event != nullptr &&
        (e = cudaEventRecord(static_cast<cudaEvent_t>(io.step_done_event), stream)) != cudaSuccess) return e;
    if ((e = cudaEventRecord(slot->ev_step, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(h->out, slot->ev_step, 0)) != cudaSuccess) return e;
    if ((e = copy_results_to_host(io, N, slot->sparse, h->out)) != cudaSuccess) return e;
    if ((e = cudaEventRecord(slot->ev, h->out)) != cudaSuccess) return e;
    if (P.windows > 0 && (e = launch_obs_range(P, D, S, obs, variant, 0, P.n_envs, stream)) != cudaSuccess) return e;
    return cudaSuccess;
}

cudaError_t launch_step_host_end(const GteHostIO& io) {
    HostIOStreams* h = nullptr;
    cudaError_t e;
    if ((e = hio_for_current_device(&h)) != cudaSuccess) return e;
    for (auto& p : h->pending)
        if (p.results == io.results && p.ev != nullptr) {
            if ((e = cudaEventSynchronize(p.ev)) != cudaSuccess) return e;
            p.open = false;
            // (a later iteration's copy may be queued behind on the same stream: the rare dense fetch waits for it too)
            return p.sparse ? fetch_dense_flags_if_needed(io, p.n, h->out) : cudaSuccess;
        }
    return cudaErrorInvalidValue;                            // no begin() for this result block
}

cudaError_t launch_info(const GteParams& P, const GteData& D, const GteState& S, const GteInfo& I,
                        cudaStream_t stream) {
    const int grid = (P.n_envs + kStepThreads - 1) / kStepThreads;
    info_kernel<<<grid, kStepThreads, 0, stream>>>(P, D, S, I);
    return cudaGetLastError();
}

}  // namespace gte
