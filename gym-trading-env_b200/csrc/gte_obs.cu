// gte_obs.cu — observation-window gather kernels (sm_100a).  Replaces TradingEnv._get_obs
// (environments.py:152-160): obs[env] = rows idx-W+1..idx of [static features | dynamic features].
//
// Three variants (DESIGN.md §kernels):
//   generic : scalar gather, any shape (windows=None, odd row sizes); a power-of-two lane group per env.
//   vec     : one warp per env; 128-bit ld.global.nc from the 16-byte-aligned window table (rows in the
//             reference's own [t, F] layout, dynamic columns zero), dynamic columns patched in
//             registers from the per-env ring, 128-bit coalesced st.global.  No shared memory.
//   tma     : warp-specialised producer/consumer pipeline: cp.async.bulk (TMA, 1-D) pulls whole windows and
//             the dynamic-feature ring block of each 32-env tile global->shared, consumer warps patch the
//             dynamic columns in shared memory, cp.async.bulk pushes groups of finished windows shared->global.
//             The LSU only touches 12 bytes of per-env metadata.
#include <cstdlib>

#include "gte_tma.cuh"
#include "gte_step_env.cuh"
#include "gte_launch.h"

namespace gte {

// ------------------------------------------------------------------------------------------ generic
// GEN (every kernel below): dynamic columns of the general catalogue (sh.dyn), else none or the default pair, whose ring
// layout is known at compile time (RingLayout).
template <int G, bool GEN = false>
__global__ void __launch_bounds__(256)
obs_generic_kernel(const GteParams P, const GteData D, const GteState S, float* __restrict__ obs,
                   const ObsShape sh, const int env_begin, const int env_end) {
    const int groups_per_block = 256 / G;
    const int lane = threadIdx.x % G;
    const int64_t n_groups = (int64_t)gridDim.x * groups_per_block;
    const int per_env = sh.W * sh.F;
    const RingLayout<GEN> R{sh.dyn};
    const int s0 = sh.nd > 0 ? (int)((*S.ring_clock + 1ull) % (uint64_t)sh.W) : 0;    // ring slot of window row 0
    for (int64_t env = env_begin + (int64_t)blockIdx.x * groups_per_block + threadIdx.x / G; env < env_end;
         env += n_groups) {
        const int ep_start = S.ep_start[env];
        const int idx = ep_start + S.step[env];
        const int ds = S.dataset_idx[env];
        const int r0 = idx + 1 - sh.W;
        const float* __restrict__ feat = D.features + ((int64_t)ds * P.t_stride + r0) * sh.ns;
        float* __restrict__ out = obs + env * per_env;
        for (int e = lane; e < per_env; e += G) {
            const int w = e / sh.F, c = e - w * sh.F;
            float v;
            if (c < sh.ns) {
                v = __ldg(feat + (int64_t)w * sh.ns + c);
            } else {
                const int r = r0 + w;
                int slot = s0 + w;
                if (slot >= sh.W) slot -= sh.W;
                const int e32 = (int)(env & 31);
                const uint8_t* __restrict__ ring = R.tile_of(S.dyn_ring, sh.W, env);
                v = (r < ep_start) ? 0.0f : ring_value(P, R, sh.W, ring, c - sh.ns, slot, e32);
            }
            out[e] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ float4 ld_nc_v4(const void* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_cs_v4(void* p, const float4& v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ------------------------------------------------------------------------------------------ vec
template <bool PAIR, bool GEN = false>     // PAIR: the default pair and F even -> the dynamic pair is an aligned float2
__global__ void __launch_bounds__(256)
obs_vec_kernel(const GteParams P, const GteData D, const GteState S, float* __restrict__ obs,
               const ObsShape sh, const int env_begin, const int env_end) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const RingLayout<GEN> R{sh.dyn};
    const int s0 = sh.nd > 0 ? (int)((*S.ring_clock + 1ull) % (uint64_t)sh.W) : 0;    // ring slot of window row 0
    for (int64_t env = env_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); env < env_end;
         env += n_warps) {
        const int ep_start = S.ep_start[env];
        const int idx = ep_start + S.step[env];
        const int ds = S.dataset_idx[env];
        const int r0 = idx + 1 - sh.W;
        const char* __restrict__ src = window_src(D, sh, ds, r0);
        const uint8_t* __restrict__ ring = R.tile_of(S.dyn_ring, sh.W, env);
        const int e32 = (int)(env & 31);
        char* __restrict__ dst = reinterpret_cast<char*>(obs) + env * (int64_t)sh.win_bytes;
        for (int j = lane; j < sh.n_vec; j += 32) {
            float4 v = ld_nc_v4(src + 16 * j);
            if (sh.nd > 0) {
                float* pv = reinterpret_cast<float*>(&v);
#pragma unroll
                for (int k = 0; k < 4; k += (PAIR ? 2 : 1)) {
                    const uint32_t e = 4u * j + k;
                    const int w = (int)fast_div(e, sh.magicF);
                    const int c = (int)e - w * sh.F;
                    if (c >= sh.ns) {
                        const int r = r0 + w;
                        int slot = s0 + w;
                        if (slot >= sh.W) slot -= sh.W;
                        if (PAIR) {                      // c == sh.ns: columns 0 and 1 at once
                            const bool live = r >= ep_start;
                            pv[k] = live ? ring_value<GEN, true>(P, R, sh.W, ring, 0, slot, e32) : 0.0f;
                            pv[k + 1] = live ? ring_value<GEN, true>(P, R, sh.W, ring, 1, slot, e32) : 0.0f;
                        } else {
                            pv[k] = (r < ep_start) ? 0.0f : ring_value<GEN, true>(P, R, sh.W, ring, c - sh.ns, slot, e32);
                        }
                    }
                }
            }
            st_cs_v4(dst + 16 * j, v);
        }
    }
}

// ---- TMA gather: warp-specialised producer / consumer pipeline -----------------------------------------
// One CTA = 4 consumer warps + 1 producer warp + 1 store warp working on ONE pipeline over 32-env tiles (strided over the grid),
// each tile cut into groups of G consecutive envs:
//   producer warp : owns the metadata of the next tile (one env per lane, one coalesced load per array a whole
//                   tile ahead), turns it ONCE per env into the window address and the first live window row,
//                   waits for a free window stage (empty mbarrier), publishes the first live rows to shared
//                   memory and issues the group's G cp.async.bulk window copies from the L2-resident window
//                   table onto the stage's full mbarrier.  One tile ahead it issues the ONE cp.async.bulk of the
//                   tile's dynamic-feature ring block (HBM, contiguous: W x 160 bytes for the default pair — real_position
//                   rows whose 16-byte chunks are XOR-swizzled so the consumers' column reads spread over the banks,
//                   then position-index rows; GTE_RING_TILE_BYTES_DYN for the general catalogue);
//   consumer warps: wait on both full mbarriers, patch the dynamic columns smem->smem (128 threads = G envs x
//                   128/G slots per pass; rows before the episode start stay zero), fence.proxy.async, and each
//                   warp arrives on the stage's ready mbarrier (and, after the tile's last group, hands the ring
//                   block back) without ever meeting the other warps;
//   store warp    : one thread waits for a ready stage, issues the SINGLE bulk store of the G contiguous windows
//                   and, once the PREVIOUS group's store has finished reading shared memory, hands that window
//                   stage back to the producer — the store drain never blocks the consumers.
// Evidence for this shape is in profiles/r01_tuning.md (per-warp pipelines were bound by the instruction
// chain of too few resident warps; consumers of a unified pipeline mostly waited on the HBM ring loads).
constexpr int kCoopConsumerWarps = 4;
constexpr int kCoopThreads = (kCoopConsumerWarps + 2) * 32;       // + producer warp + store warp
constexpr int kTileEnvs = 32;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// WS window stages of G envs and RT ring-tile stages per CTA.  The ring tiles come from HBM (slow under a
// saturating write stream) and only need the tile index, the windows come from L2 and need the envs'
// metadata: ring tiles are requested a whole tile ahead, the big window buffers are only held for an L2
// round trip + patch + store drain.
// FUSED (single-wave grids only, gte_step_obs): the CTA first advances ITS OWN envs by one transition — every thread one
// env, the very step_env() of the step kernel — keeps each env's window address / first live row in shared memory,
// takes part in the metric fold, and then runs the gather pipeline below on those envs.  One launch per lockstep
// iteration and no grid-wide dependency between the transition and the gather: at 65 536 envs the two-launch form pays
// the step kernel's tail (metric fold, drain) plus the gather's ramp between two latency-bound kernels.
constexpr int kFusedMaxEnvs = 256;         // envs one CTA may own in the fused form (metadata kept in shared memory)
struct FusedStep {
    const void* actions;
    StepConsts K;
    GteStepOut O;
    int autoreset;
    unsigned int* sched;       // DYN only: {next tile to hand out (beyond the first gridDim.x), CTAs finished}, both 0 at launch
};

// DYN (large batches): tiles are CLAIMED, not assigned — tile 0 of a CTA is its block index, every further one comes from
// a global counter (one atomicAdd per tile, issued by the producer a whole tile before its answer is needed).  Measured
// (tools/store_path_probe.cu): a persistent grid that splits a 5.4 GB store stream EVENLY over the SMs writes 6.2 TB/s, the
// same stream handed out on demand 7.4-7.6 TB/s — the SMs do not all reach memory equally fast, and with a static split
// the launch lasts as long as the slowest of them.  The producer publishes each tile id through shared memory (ring of 4
// ids, riding on the release of the stage's full barrier); a tile id past the end stops consumers and store warp.
template <int WS, int RT, int G, int UNIT = kTileEnvs, bool FUSED = false, bool DYN = false, bool GEN = false>
__global__ void __launch_bounds__(kCoopThreads, FUSED ? 4 : 1)
obs_tma_coop_kernel(const GteParams P, const GteData D, const GteState S, float* __restrict__ obs,
                    const ObsShape sh, const int env_begin, const int env_end, const FusedStep FS) {
    static_assert(RT >= 2, "a ring tile is requested while the previous one is being consumed");
    static_assert(!DYN || (RT == 2 && !FUSED), "claimed tiles: the producer looks exactly one ring tile ahead; a fused CTA owns its envs");
    static_assert(UNIT % G == 0 && kTileEnvs % UNIT == 0, "a work unit is a whole number of groups inside one ring block");
    // work unit ("tile") = UNIT consecutive envs inside one 32-env ring block: 32 normally, 16 or 8 when the batch
    // is so small that whole blocks would leave CTAs idle or unevenly loaded (the block is then fetched once per unit)
    constexpr int unit_envs = UNIT;
    constexpr int GROUPS = UNIT / G;                             // groups per tile
    constexpr int NCONS = kCoopConsumerWarps * 32;
    constexpr int SPP = NCONS / G;                               // ring slots patched per pass
    constexpr int RING_AT = WS < GROUPS - 1 ? WS : GROUPS - 1;   // group at which the tile RT-1 ahead is requested:
                                                                 // by then the stage it reuses has been handed back
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_w[WS], ready_w[WS], empty_w[WS], full_r[RT], empty_r[RT];
    __shared__ int first_live[2][kTileEnvs];                     // per tile parity: first window row of the episode
    __shared__ unsigned long long f_src[FUSED ? kFusedMaxEnvs : 1];   // FUSED: window address / first live row of every
    __shared__ int f_live[FUSED ? kFusedMaxEnvs : 1];                 //        env this CTA owns, written by its step phase
    __shared__ double f_pos[FUSED ? GTE_MAX_POSITIONS : 1];
    __shared__ int f_T0;
    __shared__ int tile_id_s[4];                                 // DYN: id of tile k of this CTA at [k & 3]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool ring = sh.nd > 0;
    const uint32_t win_bytes = (uint32_t)sh.win_bytes;
    const uint32_t wstage_bytes = win_bytes * G;
    const RingLayout<GEN> R{sh.dyn};
    const uint32_t rstride = (uint32_t)R.tile_bytes(sh.W);
    auto ring_src = [&](int64_t env) -> const uint8_t* { return R.tile_of(S.dyn_ring, sh.W, env); };
    unsigned char* rbase = smem_raw;
    unsigned char* wbase = rbase + (ring ? (size_t)RT * rstride : 0);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < WS; ++s) {
            mbar_init(&full_w[s], 1); mbar_init(&ready_w[s], kCoopConsumerWarps); mbar_init(&empty_w[s], 1);
        }
#pragma unroll
        for (int s = 0; s < RT; ++s) { mbar_init(&full_r[s], 1); mbar_init(&empty_r[s], kCoopConsumerWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (FUSED && tid < GTE_MAX_POSITIONS) f_pos[tid] = P.positions[tid];
    if (FUSED && tid == 0) f_T0 = D.lengths[0];
    __syncthreads();
    pdl_wait();                              // state / ring / clock below were written by the kernel before us

    // tile k of this CTA = unit_envs consecutive envs, tiles strided over the grid; group gi of it = G envs
    auto tile_env0 = [&](int k) -> int64_t { return env_begin + ((int64_t)blockIdx.x + (int64_t)k * gridDim.x) * unit_envs; };
    auto env0_of = [&](int t) -> int64_t { return env_begin + (int64_t)t * unit_envs; };        // DYN: first env of tile id t
    // ring slot of window row 0 AFTER this iteration's transition.  Two launches: the step kernel has advanced the clock.
    // FUSED: the clock is advanced by the last CTA of THIS launch, after every CTA has read it here.
    int s0 = 0;
    if (FUSED) {
        const uint64_t tick = *S.tick, clock = *S.ring_clock;
        const int ring_slot = ring_slot_of(P, clock + 1ull);
        s0 = (int)((clock + 2ull) % (uint64_t)sh.W);
        MetricAcc acc;
        StepConsts K = FS.K;
        K.T0 = f_T0;
        for (int j = tid; j < kFusedMaxEnvs; j += kCoopThreads) {          // (the launcher guarantees the CTA owns <= 256 envs)
            const int64_t env = tile_env0(j / unit_envs) + (j % unit_envs);
            if (env < env_end) {
                const StepThreadOut r = step_env_now<GEN>(P, D, S, FS.actions, K, FS.O, tick, ring_slot, FS.autoreset, (int)env, acc, f_pos);
                f_live[j] = sh.W - 1 - (r.idx - r.ep_start);             // window row of ep_start (<= 0: the whole window is live)
                f_src[j] = (unsigned long long)window_src(D, sh, r.ds, r.idx + 1 - sh.W);
            }
        }
        // the ring entries just stored are read back below by the TMA unit (async proxy): order them across the proxies
        asm volatile("fence.proxy.async;" ::: "memory");
        reduce_metrics<kCoopThreads>(acc, FS.O, S, kChunkFirst | kChunkLast);   // ends with / contains CTA-wide barriers
        __syncthreads();
    } else if (sh.nd > 0) {
        s0 = (int)((*S.ring_clock + 1ull) % (uint64_t)sh.W);
    }
    auto group_env0 = [&](int k, int gi) -> int64_t { return tile_env0(k) + gi * G; };
    auto valid_from = [&](int64_t e0) -> int {                   // envs of the group starting at env e0 inside [.., env_end)
        const int64_t left = (int64_t)env_end - e0;
        return left >= G ? G : (left > 0 ? (int)left : 0);
    };
    auto group_valid = [&](int k, int gi) -> int { return valid_from(group_env0(k, gi)); };

    if (warp == kCoopConsumerWarps) {
        // ------------------------------------------------------------------ producer warp
        struct TilePre { unsigned long long src; int first_live; };
        auto load_tile = [&](int k) {
            TilePre p;
            p.src = 0ull; p.first_live = 0;
            const int64_t env = tile_env0(k) + lane;
            if (FUSED) {
                const int j = k * unit_envs + lane;
                if (lane < unit_envs && env < env_end && j < kFusedMaxEnvs) { p.src = f_src[j]; p.first_live = f_live[j]; }
            } else if (lane < unit_envs && env < env_end) {
                // per-env state is WRITTEN by the step kernel this grid may overlap with (programmatic dependent launch): never
                // through the non-coherent path (ld.global.nc is only defined for data that is read-only for the whole kernel)
                const int ep = __ldcg(S.ep_start + env), st = __ldcg(S.step + env), ds = __ldcg(S.dataset_idx + env);
                p.first_live = sh.W - 1 - st;                    // window row of ep_start (<= 0: the whole window is live)
                p.src = (unsigned long long)window_src(D, sh, ds, ep + st + 1 - sh.W);
            }
            return p;
        };
        auto issue_ring = [&](int k) {                           // lane 0; needs nothing but the tile index
            if (ring && tile_env0(k) < env_end) {
                const int stage = k % RT, use = k / RT;
                if (use > 0) mbar_wait(&empty_r[stage], (uint32_t)(use - 1) & 1u);
                mbar_expect_tx(&full_r[stage], rstride);
                bulk_g2s(rbase + (size_t)stage * rstride, ring_src(tile_env0(k)), rstride, &full_r[stage]);
            }
        };
        if (DYN) {
            auto load_tile_id = [&](int t) {
                TilePre p;
                p.src = 0ull; p.first_live = 0;
                const int64_t env = env0_of(t) + lane;
                if (lane < unit_envs && env < env_end) {
                    const int ep = __ldcg(S.ep_start + env), st = __ldcg(S.step + env), ds = __ldcg(S.dataset_idx + env);
                    p.first_live = sh.W - 1 - st;
                    p.src = (unsigned long long)window_src(D, sh, ds, ep + st + 1 - sh.W);
                }
                return p;
            };
            auto issue_ring_id = [&](int k, int t) {             // lane 0
                if (ring && env0_of(t) < env_end) {
                    const int stage = k % RT, use = k / RT;
                    if (use > 0) mbar_wait(&empty_r[stage], (uint32_t)(use - 1) & 1u);
                    mbar_expect_tx(&full_r[stage], rstride);
                    bulk_g2s(rbase + (size_t)stage * rstride, ring_src(env0_of(t)), rstride, &full_r[stage]);
                }
            };
            // lane 0 claims; the answer of a claim is only looked at one whole tile later (claim_use), so the round trip of
            // the atomic never stalls the pipeline
            auto claim = [&]() -> int { return lane == 0 ? (int)(gridDim.x + atomicAdd(FS.sched, 1u)) : 0; };
            auto claim_use = [&](int raw) -> int {
                asm volatile("" : "+r"(raw));                    // the value is waited for HERE, not where it was asked for
                return __shfl_sync(FULL, raw, 0);
            };
            int ta = (int)blockIdx.x;                            // T(0)
            int tb = claim_use(claim());                         // T(1): the one exposed round trip, once per CTA
            int tc_raw = claim();                                // T(2), in flight
            TilePre pc = load_tile_id(ta), pn = load_tile_id(tb);
            if (lane == 0) issue_ring_id(0, ta);
            int q = 0;
            for (int k = 0;; ++k) {
                const bool last = env0_of(ta) >= env_end;        // a tile id past the end: tell the others and stop
                for (int gi = 0; gi < GROUPS; ++gi, ++q) {
                    const int n_valid = last ? 0 : valid_from(env0_of(ta) + gi * G);
                    if (n_valid == 0 && !(last && gi == 0)) break;
                    if (!last && lane == 0 && gi == RING_AT) issue_ring_id(k + 1, tb);
                    __syncwarp();
                    const int stage = q % WS, use = q / WS;
                    if (use > 0) mbar_wait(&empty_w[stage], (uint32_t)(use - 1) & 1u);
                    if (gi == 0) {
                        first_live[k & 1][lane] = pc.first_live;
                        if (lane == 0) tile_id_s[k & 3] = last ? -1 : ta;
                        __syncwarp();
                    }
                    if (last) {                                  // completes the stage's phase without data (release: the -1)
                        if (lane == 0) mbar_arrive(&full_w[stage]);
                        break;
                    }
                    unsigned char* sbuf = wbase + (size_t)stage * wstage_bytes;
                    if (lane == 0) mbar_expect_tx(&full_w[stage], (uint32_t)n_valid * win_bytes);
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        const unsigned long long src = __shfl_sync(FULL, pc.src, gi * G + g);
                        if (lane == 0 && g < n_valid)
                            bulk_g2s(sbuf + (size_t)g * win_bytes, reinterpret_cast<const void*>(src), win_bytes, &full_w[stage]);
                    }
                }
                if (last) break;
                const int tc = claim_use(tc_raw);                // asked for one tile ago
                tc_raw = claim();
                pc = pn;
                pn = load_tile_id(tc);
                ta = tb; tb = tc;
            }
        } else {
        TilePre pc = load_tile(0), pn = load_tile(1);
        if (lane == 0)
            for (int k = 0; k < RT - 1; ++k) issue_ring(k);
        int q = 0;
        for (int k = 0; tile_env0(k) < env_end; ++k) {
            for (int gi = 0; gi < GROUPS; ++gi, ++q) {
                const int n_valid = group_valid(k, gi);
                if (n_valid == 0) break;
                if (lane == 0 && gi == RING_AT) issue_ring(k + RT - 1);
                __syncwarp();
                const int stage = q % WS, use = q / WS;
                if (use > 0) mbar_wait(&empty_w[stage], (uint32_t)(use - 1) & 1u);     // stage handed back
                if (gi == 0) {                                   // after the wait: tile k-2 is fully consumed
                    first_live[k & 1][lane] = pc.first_live;
                    __syncwarp();
                }
                unsigned char* sbuf = wbase + (size_t)stage * wstage_bytes;
                if (lane == 0) mbar_expect_tx(&full_w[stage], (uint32_t)n_valid * win_bytes);   // release: publishes first_live
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const unsigned long long src = __shfl_sync(FULL, pc.src, gi * G + g);
                    if (lane == 0 && g < n_valid)
                        bulk_g2s(sbuf + (size_t)g * win_bytes, reinterpret_cast<const void*>(src), win_bytes, &full_w[stage]);
                }
            }
            pc = pn;
            pn = load_tile(k + 2);
        }
        }
    } else if (warp == kCoopConsumerWarps + 1) {
        // ------------------------------------------------------------------ store warp (one thread)
        if (lane == 0) {
            int q = 0;
            int64_t e0 = 0;                                                  // DYN: first env of the current tile
            for (int k = 0; DYN || tile_env0(k) < env_end; ++k) {
                bool stop = false;
                for (int gi = 0; gi < GROUPS; ++gi, ++q) {
                    const int ws = q % WS;
                    if (DYN && gi == 0) {                                    // the tile id rides on the first group's barrier
                        mbar_wait(&ready_w[ws], (uint32_t)(q / WS) & 1u);
                        const int t = *reinterpret_cast<volatile int*>(&tile_id_s[k & 3]);
                        if (t < 0) { stop = true; break; }
                        e0 = env0_of(t);
                    }
                    const int n_valid = DYN ? valid_from(e0 + gi * G) : group_valid(k, gi);
                    if (n_valid == 0) break;
                    if (!(DYN && gi == 0))
                        mbar_wait(&ready_w[ws], (uint32_t)(q / WS) & 1u);    // every consumer warp has patched the group
                    bulk_s2g(reinterpret_cast<char*>(obs) + (DYN ? e0 + gi * G : group_env0(k, gi)) * (int64_t)win_bytes,
                             wbase + (size_t)ws * wstage_bytes, (uint32_t)n_valid * win_bytes);
                    bulk_commit();
                    if (q > 0) {
                        bulk_wait_read<1>();                     // the previous group's store has left smem
                        mbar_arrive(&empty_w[(q - 1) % WS]);
                    }
                }
                if (stop) break;
            }
            bulk_wait_read<0>();                                 // smem must outlive the last store's reads
        }
    } else {
        // ------------------------------------------------------------------ consumer warps
        // thread -> (env g of the group, slot t of the pass): the G lanes sharing a slot read one 16-byte chunk of
        // the swizzled real_position row, lanes of different slots hit different chunks (banks).  The warps never
        // meet: each one signals the store warp (and, after a tile's last group, the producer) on its own.
        const int g = tid % G, t = tid / G;
        int q = 0;
        int64_t e0 = 0;                                                      // DYN: first env of the current tile
        for (int k = 0; DYN || tile_env0(k) < env_end; ++k) {
            const int rs = k % RT;
            bool stop = false;
            for (int gi = 0; gi < GROUPS; ++gi, ++q) {
                const int ws = q % WS;
                if (DYN && gi == 0) {                                        // the tile id rides on the first group's barrier
                    mbar_wait(&full_w[ws], (uint32_t)(q / WS) & 1u);
                    const int tid_k = *reinterpret_cast<volatile int*>(&tile_id_s[k & 3]);
                    if (tid_k < 0) {                                         // no more tiles: pass the word on to the store warp
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&ready_w[ws]);
                        stop = true;
                        break;
                    }
                    e0 = env0_of(tid_k);
                }
                const int n_valid = DYN ? valid_from(e0 + gi * G) : group_valid(k, gi);
                if (n_valid == 0) break;
                unsigned char* sbuf = wbase + (size_t)ws * wstage_bytes;
                if (!(DYN && gi == 0))
                    mbar_wait(&full_w[ws], (uint32_t)(q / WS) & 1u);         // windows landed (acquire: first_live too)
                if (ring) {
                    mbar_wait(&full_r[rs], (uint32_t)(k / RT) & 1u);         // the tile's ring block landed
                    if (g < n_valid) {
                        const int live0 = first_live[k & 1][gi * G + g];
                        const int e = (int)((DYN ? e0 : tile_env0(k)) & 31) + gi * G + g;      // env lane within the 32-env ring block
                        float* fbuf = reinterpret_cast<float*>(sbuf + (size_t)g * win_bytes);
                        const unsigned char* rtile = rbase + (size_t)rs * rstride;
                        for (int s = t; s < sh.W; s += SPP) {
                            int w = s - s0;
                            if (w < 0) w += sh.W;
                            if (w >= live0) {                    // rows before the episode start stay zero
                                float* qd = fbuf + w * sh.F + sh.ns;
                                for (int j = 0; j < R.n_cols(); ++j) qd[j] = ring_value(P, R, sh.W, rtile, j, s, e);
                            }
                        }
                    }
                    fence_proxy_async();                         // generic-proxy smem writes -> visible to TMA
                }
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&ready_w[ws]);                   // release: this warp's share of the group is patched
                    if (ring && gi == GROUPS - 1) mbar_arrive(&empty_r[rs]);  // ... and its reads of the ring block are done
                }
            }
            if (stop) break;
        }
    }
    if (DYN) {
        // the last CTA to finish leaves both counters at zero for the next launch that is handed this slot
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            if (atomicAdd(FS.sched + 1, 1u) == gridDim.x - 1) {
                FS.sched[0] = 0u;
                FS.sched[1] = 0u;
                __threadfence();
            }
        }
    }
}

using ObsKernelFn = void (*)(const GteParams, const GteData, const GteState, float*, const ObsShape, int, int, const FusedStep);

struct TmaConfig { int wstages, rtiles, group; };

static size_t tma_smem_bytes(const ObsShape& sh, const TmaConfig& c) {
    const size_t ring = sh.nd > 0 ? (size_t)c.rtiles * sh.dyn.tile_bytes : 0;
    return (size_t)c.group * c.wstages * sh.win_bytes + ring;
}

// (window stages, ring-tile stages, envs per group) combinations compiled in: the default pipeline shape (3 window
// stages, 2 ring tiles, the groups tma_config() may pick) in every form — work units of 32, 16 and 8 envs, the fused
// step+gather form, the claimed-tiles form (large batches) — and, for no columns / the default pair, a few more
// shapes for tuning runs (GTE_TMA_STAGES / _RTILES / _GROUP).
template <bool GEN>
static ObsKernelFn tma_kernel_of(int key, int unit, bool fused, bool dyn) {
    if (dyn && !fused && unit == kTileEnvs) {
        switch (key) {
            case 30201: return obs_tma_coop_kernel<3, 2, 1, 32, false, true, GEN>;
            case 30202: return obs_tma_coop_kernel<3, 2, 2, 32, false, true, GEN>;
            case 30204: return obs_tma_coop_kernel<3, 2, 4, 32, false, true, GEN>;
        }
    }
    if (!dyn) {
        switch ((fused ? 1000000 : 0) + unit * 100000 + key) {
            case 3230201: return obs_tma_coop_kernel<3, 2, 1, 32, false, false, GEN>;
            case 3230202: return obs_tma_coop_kernel<3, 2, 2, 32, false, false, GEN>;
            case 3230204: return obs_tma_coop_kernel<3, 2, 4, 32, false, false, GEN>;
            case 1630201: return obs_tma_coop_kernel<3, 2, 1, 16, false, false, GEN>;
            case 1630202: return obs_tma_coop_kernel<3, 2, 2, 16, false, false, GEN>;
            case 1630204: return obs_tma_coop_kernel<3, 2, 4, 16, false, false, GEN>;
            case 830201: return obs_tma_coop_kernel<3, 2, 1, 8, false, false, GEN>;
            case 830202: return obs_tma_coop_kernel<3, 2, 2, 8, false, false, GEN>;
            case 830204: return obs_tma_coop_kernel<3, 2, 4, 8, false, false, GEN>;
            case 4230201: return obs_tma_coop_kernel<3, 2, 1, 32, true, false, GEN>;
            case 4230202: return obs_tma_coop_kernel<3, 2, 2, 32, true, false, GEN>;
            case 4230204: return obs_tma_coop_kernel<3, 2, 4, 32, true, false, GEN>;
            case 2630201: return obs_tma_coop_kernel<3, 2, 1, 16, true, false, GEN>;
            case 2630202: return obs_tma_coop_kernel<3, 2, 2, 16, true, false, GEN>;
            case 2630204: return obs_tma_coop_kernel<3, 2, 4, 16, true, false, GEN>;
            case 1830201: return obs_tma_coop_kernel<3, 2, 1, 8, true, false, GEN>;
            case 1830202: return obs_tma_coop_kernel<3, 2, 2, 8, true, false, GEN>;
            case 1830204: return obs_tma_coop_kernel<3, 2, 4, 8, true, false, GEN>;
        }
    }
    if constexpr (!GEN) {
        if (!fused && unit == kTileEnvs) {
            switch ((dyn ? 1000000 : 0) + key) {
                case 1030208: return obs_tma_coop_kernel<3, 2, 8, 32, false, true>;
                case 30208: return obs_tma_coop_kernel<3, 2, 8>;
                case 30304: return obs_tma_coop_kernel<3, 3, 4>;
                case 40204: return obs_tma_coop_kernel<4, 2, 4>;
                case 40304: return obs_tma_coop_kernel<4, 3, 4>;
                case 20204: return obs_tma_coop_kernel<2, 2, 4>;
                case 40202: return obs_tma_coop_kernel<4, 2, 2>;
                case 60202: return obs_tma_coop_kernel<6, 2, 2>;
                case 60302: return obs_tma_coop_kernel<6, 3, 2>;
                case 20208: return obs_tma_coop_kernel<2, 2, 8>;
            }
        }
    }
    return nullptr;
}

static ObsKernelFn tma_kernel(const TmaConfig& c, int unit = kTileEnvs, bool fused = false, bool dyn = false, bool gen = false) {
    const int key = c.wstages * 10000 + c.rtiles * 100 + c.group;
    return gen ? tma_kernel_of<true>(key, unit, fused, dyn) : tma_kernel_of<false>(key, unit, fused, dyn);
}

// Pipeline shape: 3 window stages of the largest group (4, 2, 1 envs) + 2 ring tiles that still leave two CTAs per
// SM; GTE_TMA_STAGES / GTE_TMA_RTILES / GTE_TMA_GROUP override it for tuning runs.
static TmaConfig tma_config(const ObsShape& sh) {
    static const int ws = [] { const char* e = getenv("GTE_TMA_STAGES"); return e ? atoi(e) : 0; }();
    static const int rt = [] { const char* e = getenv("GTE_TMA_RTILES"); return e ? atoi(e) : 0; }();
    static const int g = [] { const char* e = getenv("GTE_TMA_GROUP"); return e ? atoi(e) : 0; }();
    if (ws > 0 && rt > 0 && g > 0) {
        const TmaConfig c{ws, rt, g};
        if (tma_kernel(c, kTileEnvs, false, false, sh.dyn.general) != nullptr) return c;
    }
    TmaConfig c{3, 2, 4};
    if (sh.dyn.general) {
        // the general catalogue's ring stages grow with its f32 columns (W x 544 bytes per tile with all five): halving
        // the group no longer buys a CTA per SM, so take the group with the most windows in flight per SM
        int best = 0;
        for (int g = 4; g >= 1; g /= 2) {
            const TmaConfig t{3, 2, g};
            const size_t smem = tma_smem_bytes(sh, t);
            const int in_flight = (int)((227u * 1024u) / (smem + 2048u)) * g;
            if (smem <= 200 * 1024 && in_flight > best) { best = in_flight; c = t; }
        }
        return c;
    }
    while (c.group > 1 && tma_smem_bytes(sh, c) > 100 * 1024) c.group /= 2;
    return c;
}

// ------------------------------------------------------------------------------------------ launch
using GenericKernelFn = void (*)(const GteParams, const GteData, const GteState, float*, const ObsShape, int, int);

// the generic gather with G lanes per env
template <bool GEN>
static GenericKernelFn generic_kernel(int G) {
    switch (G) {
        case 32: return obs_generic_kernel<32, GEN>;
        case 16: return obs_generic_kernel<16, GEN>;
        case 8: return obs_generic_kernel<8, GEN>;
        case 4: return obs_generic_kernel<4, GEN>;
        case 2: return obs_generic_kernel<2, GEN>;
        default: return obs_generic_kernel<1, GEN>;
    }
}

bool obs_vec_supported(const GteParams& P, const GteData& D) {
    const ObsShape sh = make_shape(P);
    if (P.windows <= 0 || sh.win_bytes % 16 != 0) return false;
    if ((int64_t)sh.W * sh.F * (int64_t)sh.F >= (1ll << 31)) return false;     // fast_div range
    for (int r = 0; r < 4; ++r) {                       // every residue class a window start can have
        const int c = (int)((((int64_t)r * sh.row_bytes) >> 2) & 3);
        if (D.window_table[c] == nullptr) return false;
    }
    return D.window_table_ds_stride % 16 == 0;
}

bool obs_tma_supported(const GteParams& P, const GteData& D) {
    if (!obs_vec_supported(P, D)) return false;
    const ObsShape sh = make_shape(P);
    return tma_smem_bytes(sh, tma_config(sh)) <= 200 * 1024;
}

// Grid / work-unit choice of the TMA gather for n_envs envs (and the one-time per-device kernel attribute opt-ins).
struct TmaPlan {
    ObsKernelFn kern;
    int grid, unit, envs_per_cta;
    size_t smem;
    unsigned int* sched;       // claimed-tiles form: this launch's pair of counters, else nullptr
};

// Counters of the claimed-tiles form: 64 slots of {next tile, CTAs finished} per device, handed out round-robin (launches
// that overlap on different streams get different slots; the last CTA of a launch zeroes its slot again).  Allocated on
// first use — never inside a stream capture (the caller then falls back to the static split).
constexpr int kDynMinTilesPerCta = 8;
static unsigned int* dyn_sched_slot(cudaStream_t stream) {
    static unsigned int* pool[16] = {};
    static unsigned int next[16] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    unsigned int*& p = pool[dev & 15];
    if (p == nullptr) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return nullptr;
        if (cudaMalloc(reinterpret_cast<void**>(&p), 64 * 32) != cudaSuccess) { p = nullptr; (void)cudaGetLastError(); return nullptr; }
        if (cudaMemset(p, 0, 64 * 32) != cudaSuccess) { cudaFree(p); p = nullptr; (void)cudaGetLastError(); return nullptr; }
    }
    return p + 8 * (next[dev & 15]++ & 63u);
}

static cudaError_t plan_tma(const ObsShape& sh, int n_envs, bool fused, TmaPlan* out, cudaStream_t stream = nullptr) {
    const TmaConfig cfg = tma_config(sh);
    const size_t smem = tma_smem_bytes(sh, cfg);
    const bool gen = sh.dyn.general;
    ObsKernelFn probe = tma_kernel(cfg, kTileEnvs, fused, false, gen);
    if (probe == nullptr) return cudaErrorInvalidValue;
    int dev = 0;
    cudaGetDevice(&dev);
    // opt-in to > 48 KB dynamic smem once per kernel AND device (the attribute is per device), and how many CTAs of the
    // kernel an SM holds (registers, static + dynamic shared memory), asked of the runtime once
    struct Slot { ObsKernelFn kern; size_t smem_max, smem_asked; int per_sm; };
    static Slot slots[16][24] = {};
    auto configure = [&](ObsKernelFn k, int* per_sm) -> cudaError_t {
        Slot* sl = slots[dev & 15];
        int i = 0;
        while (i < 23 && sl[i].kern != nullptr && sl[i].kern != k) ++i;
        if (sl[i].kern != k) { sl[i].kern = k; sl[i].smem_max = 0; sl[i].smem_asked = (size_t)-1; }
        if (smem > sl[i].smem_max) {                        // the opt-in only ever has to grow
            cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            sl[i].smem_max = smem;
        }
        if (smem != sl[i].smem_asked) {                     // occupancy belongs to THIS launch's shared-memory size
            int n = 0;
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, kCoopThreads, smem);
            if (e != cudaSuccess) return e;
            sl[i].smem_asked = smem;
            sl[i].per_sm = n < 1 ? 1 : n;
        }
        *per_sm = sl[i].per_sm;
        return cudaSuccess;
    };
    int per_sm = 1;
    cudaError_t e = configure(probe, &per_sm);
    if (e != cudaSuccess) return e;
    // work unit = one 32-env tile, or half / a quarter of one when that spreads a small batch more evenly (the time
    // of the launch follows the units of the busiest CTA x the unit size); persistent grid of <= SMs x per_sm CTAs,
    // sized so that every CTA gets the same number of units (no straggler wave at mid-size N)
    const int64_t cap = (int64_t)num_sms() * per_sm;
    int unit = 32;
    int64_t best = -1;
    static const int forced_unit = [] { const char* e = getenv("GTE_TMA_UNIT"); return e ? atoi(e) : 0; }();   // tuning runs
    for (int u = 32; u >= 8 && u >= cfg.group; u /= 2) {
        if (forced_unit > 0 && tma_kernel(cfg, forced_unit, fused, false, gen) != nullptr) { unit = forced_unit; break; }
        if (tma_kernel(cfg, u, fused, false, gen) == nullptr) continue;
        const int64_t units = ((int64_t)n_envs + u - 1) / u;
        const int64_t per_cta = (units + cap - 1) / cap;
        if (u == 8 && per_cta > 1) break;                  // quarter tiles only while every CTA gets at most one
        // a smaller unit re-fetches the 32-env ring block once per unit (+5 % traffic per halving): it has to buy
        // more than that in balance (C4: 1792 -> 1776 envs on the busiest CTA is not worth it, C3: 128 -> 112 is)
        if (best < 0 || per_cta * u * 100 < best * 95) { best = per_cta * u; unit = u; }
    }
    const int64_t need = ((int64_t)n_envs + unit - 1) / unit;
    const int64_t waves = (need + cap - 1) / cap;
    out->grid = (int)((need + waves - 1) / waves);
    static const int tiles_per_cta = [] { const char* e = getenv("GTE_TMA_TILES_PER_CTA"); return e ? atoi(e) : 0; }();   // tuning runs
    if (tiles_per_cta > 0 && !fused && (need + tiles_per_cta - 1) / tiles_per_cta > out->grid)
        out->grid = (int)((need + tiles_per_cta - 1) / tiles_per_cta);
    out->unit = unit;
    out->envs_per_cta = (int)(((need + out->grid - 1) / out->grid) * unit);
    out->smem = smem;
    out->kern = tma_kernel(cfg, unit, fused, false, gen);
    out->sched = nullptr;
    // large batches: tiles are claimed from a counter instead of being split evenly over the CTAs (GTE_TMA_DYN=0: never,
    // 2: whenever the kernel exists, for tests of the small-batch corners)
    static const int dyn_mode = [] { const char* e = getenv("GTE_TMA_DYN"); return e ? atoi(e) : 1; }();
    ObsKernelFn dk = tma_kernel(cfg, unit, fused, true, gen);
    if (dyn_mode > 0 && dk != nullptr && tiles_per_cta <= 0 &&
        (dyn_mode >= 2 || (need + out->grid - 1) / out->grid >= kDynMinTilesPerCta)) {
        unsigned int* slot = dyn_sched_slot(stream);
        if (slot != nullptr) { out->kern = dk; out->sched = slot; }
    }
    int unused = 0;
    return out->kern == probe ? cudaSuccess : configure(out->kern, &unused);
}

// Whether gte_step_obs runs this shape as ONE fused launch: the batch must be small enough for every CTA of the
// single-wave grid to own at most kFusedMaxEnvs envs, and the episode accumulators must be off (acc_on: the fused kernel
// is not instantiated with them, it sits at its register cap).  *plan is filled when it does.
static cudaError_t fused_plan(const GteParams& P, const GteData& D, int variant, TmaPlan* plan, bool* eligible) {
    static const bool enabled = [] { const char* e = getenv("GTE_FUSED"); return e == nullptr || atoi(e) != 0; }();
    *eligible = false;
    if (!enabled || P.windows <= 0 || acc_on(P) || (variant != GTE_OBS_AUTO && variant != GTE_OBS_TMA) || !obs_tma_supported(P, D))
        return cudaSuccess;
    const ObsShape sh = make_shape(P);
    if (tma_kernel(tma_config(sh), kTileEnvs, true, false, sh.dyn.general) == nullptr) return cudaSuccess;
    // cheap pre-check before touching kernel attributes: even 8 CTAs per SM could not keep every CTA under the limit
    if ((int64_t)P.n_envs > (int64_t)num_sms() * 8 * kFusedMaxEnvs) return cudaSuccess;
    cudaError_t e = plan_tma(sh, P.n_envs, true, plan);
    if (e != cudaSuccess) return e;
    *eligible = plan->envs_per_cta <= kFusedMaxEnvs && plan->grid <= kMaxPartialRows;
    return cudaSuccess;
}

bool step_obs_is_fused(const GteParams& P, const GteData& D, int variant) {
    TmaPlan plan;
    bool ok = false;
    return fused_plan(P, D, variant, &plan, &ok) == cudaSuccess && ok;
}

// One lockstep iteration as ONE launch (transition + gather fused, see obs_tma_coop_kernel); *done = false -> the
// caller issues the two plain launches.
cudaError_t launch_fused_step_obs(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                                  const StepConsts& K, const GteStepOut& O, float* obs, int autoreset, int variant,
                                  cudaStream_t stream, bool* done) {
    TmaPlan plan;
    *done = false;
    cudaError_t e = fused_plan(P, D, variant, &plan, done);
    if (e != cudaSuccess || !*done) return e;
    FusedStep fs;
    fs.actions = actions; fs.K = K; fs.O = O; fs.autoreset = autoreset; fs.sched = nullptr;
    return launch_pdl(plan.kern, dim3(plan.grid), dim3(kCoopThreads), plan.smem, stream, P, D, S, obs, make_shape(P), 0,
                      P.n_envs, fs);
}

cudaError_t launch_obs_range(const GteParams& P, const GteData& D, const GteState& S, float* obs, int variant,
                             int env_begin, int env_end, cudaStream_t stream) {
    const ObsShape sh = make_shape(P);
    const int n_envs = env_end - env_begin;
    if (n_envs <= 0) return cudaSuccess;
    if (variant == GTE_OBS_AUTO)
        variant = obs_tma_supported(P, D) ? GTE_OBS_TMA : (obs_vec_supported(P, D) ? GTE_OBS_VEC : GTE_OBS_GENERIC);
    const int sms = num_sms();
    if (variant == GTE_OBS_GENERIC) {
        const int per_env = sh.W * sh.F;
        int G = 32;
        while (G > 1 && G / 2 >= per_env) G /= 2;
        const int64_t need = ((int64_t)n_envs * G + 255) / 256;
        const int grid = (int)(need < (int64_t)sms * 16 ? need : (int64_t)sms * 16);
        const GenericKernelFn kern = sh.dyn.general ? generic_kernel<true>(G) : generic_kernel<false>(G);
        kern<<<grid, 256, 0, stream>>>(P, D, S, obs, sh, env_begin, env_end);
        return cudaGetLastError();
    }
    if (variant == GTE_OBS_VEC) {
        if (!obs_vec_supported(P, D)) return cudaErrorInvalidValue;
        const int64_t need = ((int64_t)n_envs + 7) / 8;
        const int grid = (int)(need < (int64_t)sms * 8 ? need : (int64_t)sms * 8);
        if (sh.dyn.general) obs_vec_kernel<false, true><<<grid, 256, 0, stream>>>(P, D, S, obs, sh, env_begin, env_end);
        else if (sh.nd == 2 && sh.F % 2 == 0) obs_vec_kernel<true><<<grid, 256, 0, stream>>>(P, D, S, obs, sh, env_begin, env_end);
        else obs_vec_kernel<false><<<grid, 256, 0, stream>>>(P, D, S, obs, sh, env_begin, env_end);
        return cudaGetLastError();
    }
    if (variant == GTE_OBS_TMA) {
        if (!obs_tma_supported(P, D)) return cudaErrorInvalidValue;
        TmaPlan plan;
        cudaError_t e = plan_tma(sh, n_envs, false, &plan, stream);
        if (e != cudaSuccess) return e;
        FusedStep fs{};
        fs.sched = plan.sched;
        return launch_pdl(plan.kern, dim3(plan.grid), dim3(kCoopThreads), plan.smem, stream, P, D, S, obs, sh, env_begin, env_end, fs);
    }
    return cudaErrorInvalidValue;
}

}  // namespace gte
