// gte_launch.h — host-side launchers shared between the kernel translation units and the C-ABI.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gte_b200.h"

namespace gte {

// Launch with programmatic dependent launch allowed: the kernel may be scheduled while its predecessor in the
// stream drains, and orders itself behind it with pdl_wait() before touching anything the predecessor wrote.
// GTE_PDL=0 falls back to plain stream order.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

int num_sms();
int step_grid(int n_envs);

// A stateful dynamic feature (current_drawdown, position_age) is among the first n_dyn columns of dyn_kinds.
inline bool dyn_stateful(const GteParams& P) {
    for (int j = 0; j < P.n_dyn && j < 8; ++j) {
        const uint32_t c = ((uint32_t)P.dyn_kinds >> (4 * j)) & 15u;
        if (c == GTE_DYN_CURRENT_DRAWDOWN || c == GTE_DYN_POSITION_AGE) return true;
    }
    return false;
}
// The episode accumulators (GteState.episode_acc) run: an episode metric or a stateful dynamic feature is configured.
// Selects the ACC instantiations of the step, rollout, server and reset kernels, and rules out the fused step+gather
// launch, which has none.
inline bool acc_on(const GteParams& P) { return P.metric_kinds != 0 || dyn_stateful(P); }

cudaError_t launch_step(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                        const GteStepOut& O, int autoreset, cudaStream_t stream);
cudaError_t launch_step_range(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                              const GteStepOut& O, int autoreset, int env_begin, int env_end, int chunk_flags,
                              cudaStream_t stream, float* obs_rows, bool obs_on_host = false);
cudaError_t launch_step_host(const GteParams& P, const GteData& D, const GteState& S, const GteHostIO& io,
                             const GteStepOut& O, float* obs, int autoreset, int variant, int* mode_used,
                             cudaStream_t stream);
cudaError_t launch_reset(const GteParams& P, const GteData& D, const GteState& S, const uint8_t* mask,
                         int first, cudaStream_t stream);
cudaError_t launch_info(const GteParams& P, const GteData& D, const GteState& S, const GteInfo& I,
                        cudaStream_t stream);

// Which gather variants the shape allows (vector/TMA need 16-byte-multiple windows + window tables).
bool obs_vec_supported(const GteParams& P, const GteData& D);
bool obs_tma_supported(const GteParams& P, const GteData& D);
cudaError_t launch_obs_range(const GteParams& P, const GteData& D, const GteState& S, float* obs, int variant,
                             int env_begin, int env_end, cudaStream_t stream);
struct StepConsts;
StepConsts make_step_consts(const GteParams& P);
cudaError_t launch_fused_step_obs(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                                  const StepConsts& K, const GteStepOut& O, float* obs, int autoreset, int variant,
                                  cudaStream_t stream, bool* done);
bool step_obs_is_fused(const GteParams& P, const GteData& D, int variant);
cudaError_t launch_step_host_begin(const GteParams& P, const GteData& D, const GteState& S, const GteHostIO& io,
                                   const GteStepOut& O, float* obs, int autoreset, int variant, cudaStream_t stream);
cudaError_t launch_step_host_end(const GteHostIO& io);
// result relay (gte_relay.cu)
bool relay_supported();
cudaError_t relay_alloc(int64_t bytes, void** dev_base, void* ipc_handle);
cudaError_t relay_open(const void* ipc_handle, void** dev_base);
cudaError_t relay_release(void* dev_base, bool opened);
cudaError_t relay_push(void* peer_base, const void* src_dev, int64_t bytes, uint32_t seq, cudaEvent_t after, cudaEvent_t done);
cudaError_t relay_serve(int lane, void* own_base, int64_t bytes, uint32_t seq, void* host_dst, void* host_seq);
cudaError_t relay_unblock(void* own_base, uint32_t seq);
int default_chunks(int n_envs);
int host_io_mode(const GteParams& P, int mode);
cudaError_t serve_quiesce();
cudaError_t launch_step_obs(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                            const GteStepOut& O, float* obs, int autoreset, int variant, int n_chunks,
                            cudaStream_t stream);

cudaError_t launch_rollout(const GteParams& P, const GteData& D, const GteState& S, const void* actions,
                           int n_steps, const GteStepOut& O, float* obs, int keep_obs, int autoreset, int variant,
                           cudaStream_t stream);

}  // namespace gte
