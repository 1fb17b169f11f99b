// gte_cabi.cu — the extern "C" boundary of libgte_b200.so (see include/gte_b200.h).
// Argument validation + kernel enqueue; no allocation, no synchronisation, no hidden state except
// the thread-local last-error string.
#include <cstdio>
#include <cstring>

#include "gte_launch.h"

namespace {

thread_local char g_err[512] = "";

int fail_arg(const char* fn, const char* what) {
    std::snprintf(g_err, sizeof(g_err), "%s: bad argument: %s", fn, what);
    return GTE_ERR_ARG;
}

int check_cuda(const char* fn, cudaError_t e) {
    if (e == cudaSuccess) return GTE_OK;
    std::snprintf(g_err, sizeof(g_err), "%s: CUDA error %d (%s): %s", fn, (int)e, cudaGetErrorName(e),
                  cudaGetErrorString(e));
    return GTE_ERR_CUDA;
}

#define GTE_REQUIRE(fn, cond) do { if (!(cond)) return fail_arg(fn, #cond); } while (0)

// GteParams.n_dyn / dyn_kinds: 0 with the legacy n_dyn 0 or 2, else one kind code 1..7 per column, each at most once;
// the stateful kinds (current_drawdown, position_age) keep their state in GteState.episode_acc
const char* bad_dyn_kinds(const GteParams* p, const GteState* s) {
    if (p->n_dyn < 0 || p->n_dyn > GTE_MAX_DYN) return "dyn_kinds: n_dyn must be 0..GTE_MAX_DYN";
    const uint32_t k = (uint32_t)p->dyn_kinds;
    if (k == 0) return (p->n_dyn == 0 || p->n_dyn == 2) ? nullptr : "dyn_kinds: 0 (the defaults) needs n_dyn 0 or 2";
    if (p->n_dyn < 8 && (k >> (4 * p->n_dyn)) != 0) return "dyn_kinds: a non-zero kind beyond n_dyn";
    unsigned seen = 0;
    for (int j = 0; j < p->n_dyn; ++j) {
        const uint32_t c = (k >> (4 * j)) & 15u;
        if (c < GTE_DYN_POSITION || c > GTE_DYN_POSITION_AGE) return "dyn_kinds: kind code outside 1..7";
        if (seen & (1u << c)) return "dyn_kinds: a kind appears twice";
        seen |= 1u << c;
    }
    if ((seen & (1u << GTE_DYN_EPISODE_PROGRESS)) && p->max_episode_duration <= 0)
        return "dyn_kinds: episode_progress needs max_episode_duration > 0";
    if (gte::dyn_stateful(*p) && s->episode_acc == nullptr)
        return "dyn_kinds: current_drawdown / position_age need episode_acc";
    return nullptr;
}

// GteParams.metric_kinds: known kind bits only; the stateful kinds need GteState.episode_acc
const char* bad_metric_kinds(const GteParams* p, const GteState* s) {
    if ((p->metric_kinds & ~GTE_METRIC_KINDS_ALL) != 0) return "metric_kinds: a bit outside GTE_METRIC_KINDS_ALL";
    if ((p->metric_kinds & GTE_METRIC_KINDS_STATEFUL) != 0 && s->episode_acc == nullptr)
        return "metric_kinds: the configured kinds need episode_acc";
    return nullptr;
}

int check_common(const char* fn, const GteParams* p, const GteData* d, const GteState* s) {
    GTE_REQUIRE(fn, p != nullptr && d != nullptr && s != nullptr);
    GTE_REQUIRE(fn, p->n_envs > 0);
    GTE_REQUIRE(fn, p->n_positions > 0 && p->n_positions <= GTE_MAX_POSITIONS);
    GTE_REQUIRE(fn, p->windows >= 0);
    if (const char* why = bad_dyn_kinds(p, s)) return fail_arg(fn, why);
    GTE_REQUIRE(fn, p->n_static >= 0 && p->n_static + p->n_dyn > 0);
    GTE_REQUIRE(fn, p->n_datasets >= 1 && p->n_datasets <= GTE_MAX_DATASETS);
    GTE_REQUIRE(fn, p->initial_position_idx >= -1 && p->initial_position_idx < p->n_positions);
    GTE_REQUIRE(fn, p->episodes_between_switch >= 1);
    GTE_REQUIRE(fn, p->plan_episodes >= 0);
    GTE_REQUIRE(fn, p->t_stride >= 2);
    GTE_REQUIRE(fn, p->v0 > 0.0);
    GTE_REQUIRE(fn, p->reward_kind == GTE_REWARD_LOG_RETURN || p->reward_kind == GTE_REWARD_SIMPLE_RETURN);
    GTE_REQUIRE(fn, p->reward_lo <= p->reward_hi);
    GTE_REQUIRE(fn, d->price != nullptr && d->lengths != nullptr);
    GTE_REQUIRE(fn, p->n_static == 0 || d->features != nullptr);
    GTE_REQUIRE(fn, s->asset && s->fiat && s->interest_asset && s->interest_fiat);
    GTE_REQUIRE(fn, s->pos_idx && s->step && s->ep_start && s->dataset_idx);
    GTE_REQUIRE(fn, s->ring_clock != nullptr);
    GTE_REQUIRE(fn, p->n_dyn == 0 || (s->dyn_ring != nullptr && (reinterpret_cast<uintptr_t>(s->dyn_ring) & 15u) == 0));
    GTE_REQUIRE(fn, s->plan_cursor && s->ds_used && s->ds_episodes && s->error_flag && s->tick);
    GTE_REQUIRE(fn, p->plan_episodes == 0 || s->reset_plan != nullptr);
    if (const char* why = bad_metric_kinds(p, s)) return fail_arg(fn, why);
    GTE_REQUIRE(fn, p->n_limit_positions >= 0 && p->n_limit_positions <= p->n_positions);
    GTE_REQUIRE(fn, p->n_limit_positions == 0 || (s->limit_price && s->limit_seq && d->high && d->low));
    GTE_REQUIRE(fn, p->action_bytes == 0 || p->action_bytes == 1 || p->action_bytes == 2 || p->action_bytes == 4 || p->action_bytes == 8);
    for (int c = 0; c < 4; ++c)          // copy c starts 4c bytes before a 16-byte boundary (cp.async.bulk / ld.v4 fault otherwise)
        GTE_REQUIRE(fn, d->window_table[c] == nullptr || ((reinterpret_cast<uintptr_t>(d->window_table[c]) + 4u * c) & 15u) == 0);
    // a resident server kernel (GTE_IO_SERVER) owns the env state: every entry point but gte_step_host stops it first
    if (std::strcmp(fn, "gte_step_host") != 0)
        if (int rc = check_cuda(fn, gte::serve_quiesce())) return rc;
    return GTE_OK;
}

}  // namespace

extern "C" {

int gte_version(void) { return GTE_VERSION; }

#ifndef GTE_BUILD_ID
#define GTE_BUILD_ID "unknown"
#endif
static const char kBuildTag[] = "GTE_BUILD_ID=" GTE_BUILD_ID;     // the tag is also searched for in the file by the binding
const char* gte_build_id(void) { return kBuildTag + 13; }

const char* gte_last_error(void) { return g_err; }

int gte_reset(const GteParams* params, const GteData* data, const GteState* state, const uint8_t* mask,
              int first, void* stream) {
    if (int rc = check_common("gte_reset", params, data, state)) return rc;
    return check_cuda("gte_reset", gte::launch_reset(*params, *data, *state, mask, first,
                                                     static_cast<cudaStream_t>(stream)));
}

static int check_step_out(const char* fn, const GteParams* params, const void* actions, const GteStepOut* out,
                          bool own_results = false) {
    GTE_REQUIRE(fn, actions != nullptr && out != nullptr);
    if (params->metric_kinds != 0 && out->episode_record == nullptr)
        return fail_arg(fn, "metric_kinds: episode metrics need episode_record");
    GTE_REQUIRE(fn, own_results || (out->reward && out->terminated && out->truncated));
    GTE_REQUIRE(fn, out->metric_partials && out->metrics_step && out->block_counter);
    return GTE_OK;
}

// the gather variant a call will run, and the alignment its 128-bit / bulk stores need from obs
static int check_obs_ptr(const char* fn, const GteParams* params, const GteData* data, const float* obs, int variant) {
    GTE_REQUIRE(fn, obs != nullptr);
    int v = variant;
    if (v == GTE_OBS_AUTO)
        v = gte::obs_tma_supported(*params, *data) ? GTE_OBS_TMA : (gte::obs_vec_supported(*params, *data) ? GTE_OBS_VEC : GTE_OBS_GENERIC);
    if (params->windows > 0 && (v == GTE_OBS_VEC || v == GTE_OBS_TMA) && (reinterpret_cast<uintptr_t>(obs) & 15u) != 0)
        return fail_arg(fn, "obs must be 16-byte aligned for the vector / TMA gather");
    return GTE_OK;
}

int gte_step(const GteParams* params, const GteData* data, const GteState* state, const void* actions,
             const GteStepOut* out, int autoreset, void* stream) {
    if (int rc = check_common("gte_step", params, data, state)) return rc;
    if (int rc = check_step_out("gte_step", params, actions, out)) return rc;
    return check_cuda("gte_step", gte::launch_step(*params, *data, *state, actions, *out, autoreset,
                                                   static_cast<cudaStream_t>(stream)));
}

static int check_variant(const char* fn, const GteParams* params, const GteData* data, int variant) {
    GTE_REQUIRE(fn, variant >= GTE_OBS_AUTO && variant <= GTE_OBS_TMA);
    if (variant == GTE_OBS_VEC && !gte::obs_vec_supported(*params, *data))
        return fail_arg(fn, "GTE_OBS_VEC needs windows>0, 16-byte-multiple windows and window tables");
    if (variant == GTE_OBS_TMA && !gte::obs_tma_supported(*params, *data))
        return fail_arg(fn, "GTE_OBS_TMA needs the GTE_OBS_VEC conditions and stage buffers that fit in shared memory");
    return GTE_OK;
}

int gte_step_obs(const GteParams* params, const GteData* data, const GteState* state, const void* actions,
                 const GteStepOut* out, float* obs, int autoreset, int variant, int n_chunks, void* stream) {
    if (int rc = check_common("gte_step_obs", params, data, state)) return rc;
    if (int rc = check_step_out("gte_step_obs", params, actions, out)) return rc;
    GTE_REQUIRE("gte_step_obs", obs != nullptr && n_chunks >= 0 && n_chunks <= 16);
    if (int rc = check_variant("gte_step_obs", params, data, variant)) return rc;
    if (int rc = check_obs_ptr("gte_step_obs", params, data, obs, variant)) return rc;
    return check_cuda("gte_step_obs", gte::launch_step_obs(*params, *data, *state, actions, *out, obs, autoreset,
                                                           variant, n_chunks, static_cast<cudaStream_t>(stream)));
}

int gte_step_host(const GteParams* params, const GteData* data, const GteState* state, const GteHostIO* io,
                  const GteStepOut* out, float* obs, int autoreset, int variant, int* mode_used, void* stream) {
    if (int rc = check_common("gte_step_host", params, data, state)) return rc;
    GTE_REQUIRE("gte_step_host", io != nullptr && io->actions != nullptr && io->results != nullptr);
    if (int rc = check_step_out("gte_step_host", params, io->actions, out, true)) return rc;
    GTE_REQUIRE("gte_step_host", io->mode >= GTE_IO_AUTO && io->mode <= GTE_IO_SERVER);
    GTE_REQUIRE("gte_step_host", (reinterpret_cast<uintptr_t>(io->results) & 7u) == 0);
    GTE_REQUIRE("gte_step_host", out->seq_out == nullptr);   // the call points it into the result block itself
    GTE_REQUIRE("gte_step_host", io->obs_host == nullptr || io->obs_bytes > 0);
    if (gte::host_io_mode(*params, io->mode) == GTE_IO_COPY)
        GTE_REQUIRE("gte_step_host", io->dev_actions != nullptr && io->dev_results != nullptr &&
                                     (reinterpret_cast<uintptr_t>(io->dev_results) & 7u) == 0);
    if (int rc = check_variant("gte_step_host", params, data, variant)) return rc;
    if (int rc = check_obs_ptr("gte_step_host", params, data, obs, variant)) return rc;
    return check_cuda("gte_step_host", gte::launch_step_host(*params, *data, *state, *io, *out, obs, autoreset, variant,
                                                             mode_used, static_cast<cudaStream_t>(stream)));
}

int gte_step_host_begin(const GteParams* params, const GteData* data, const GteState* state, const GteHostIO* io,
                        const GteStepOut* out, float* obs, int autoreset, int variant, void* stream) {
    if (int rc = check_common("gte_step_host_begin", params, data, state)) return rc;
    GTE_REQUIRE("gte_step_host_begin", io != nullptr && io->actions != nullptr && io->results != nullptr);
    if (int rc = check_step_out("gte_step_host_begin", params, io->actions, out, true)) return rc;
    GTE_REQUIRE("gte_step_host_begin", io->dev_actions != nullptr && io->dev_results != nullptr);
    GTE_REQUIRE("gte_step_host_begin", ((reinterpret_cast<uintptr_t>(io->results) | reinterpret_cast<uintptr_t>(io->dev_results)) & 7u) == 0);
    GTE_REQUIRE("gte_step_host_begin", io->obs_host == nullptr && out->seq_out == nullptr);
    if (int rc = check_variant("gte_step_host_begin", params, data, variant)) return rc;
    if (int rc = check_obs_ptr("gte_step_host_begin", params, data, obs, variant)) return rc;
    return check_cuda("gte_step_host_begin", gte::launch_step_host_begin(*params, *data, *state, *io, *out, obs, autoreset,
                                                                         variant, static_cast<cudaStream_t>(stream)));
}

int gte_step_host_end(const GteHostIO* io) {
    if (io == nullptr || io->results == nullptr) return fail_arg("gte_step_host_end", "io / io->results");
    return check_cuda("gte_step_host_end", gte::launch_step_host_end(*io));
}

int gte_serve_stop(void) { return check_cuda("gte_serve_stop", gte::serve_quiesce()); }

int gte_relay_supported(void) { return gte::relay_supported() ? 1 : 0; }

int gte_relay_alloc(int64_t bytes, void** dev_base, void* ipc_handle) {
    GTE_REQUIRE("gte_relay_alloc", bytes > 0 && dev_base != nullptr && ipc_handle != nullptr);
    return check_cuda("gte_relay_alloc", gte::relay_alloc(bytes, dev_base, ipc_handle));
}

int gte_relay_open(const void* ipc_handle, void** dev_base) {
    GTE_REQUIRE("gte_relay_open", ipc_handle != nullptr && dev_base != nullptr);
    return check_cuda("gte_relay_open", gte::relay_open(ipc_handle, dev_base));
}

int gte_relay_release(void* dev_base, int opened) {
    GTE_REQUIRE("gte_relay_release", dev_base != nullptr);
    return check_cuda("gte_relay_release", gte::relay_release(dev_base, opened != 0));
}

int gte_relay_push(void* peer_base, const void* src_dev, int64_t bytes, uint32_t seq, void* after_event, void* done_event) {
    GTE_REQUIRE("gte_relay_push", peer_base != nullptr && src_dev != nullptr && bytes > 0);
    return check_cuda("gte_relay_push", gte::relay_push(peer_base, src_dev, bytes, seq, static_cast<cudaEvent_t>(after_event),
                                                        static_cast<cudaEvent_t>(done_event)));
}

int gte_relay_serve(int lane, void* own_base, int64_t bytes, uint32_t seq, void* host_dst, void* host_seq) {
    GTE_REQUIRE("gte_relay_serve", lane >= 0 && lane < 8 && own_base != nullptr && bytes > 0 && host_dst != nullptr && host_seq != nullptr);
    GTE_REQUIRE("gte_relay_serve", gte::relay_supported());
    return check_cuda("gte_relay_serve", gte::relay_serve(lane, own_base, bytes, seq, host_dst, host_seq));
}

int gte_relay_unblock(void* own_base, uint32_t seq) {
    GTE_REQUIRE("gte_relay_unblock", own_base != nullptr);
    return check_cuda("gte_relay_unblock", gte::relay_unblock(own_base, seq));
}

int gte_host_register(void* ptr, int64_t bytes) {
    GTE_REQUIRE("gte_host_register", ptr != nullptr && bytes > 0);
    return check_cuda("gte_host_register", cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
}

int gte_host_unregister(void* ptr) {
    GTE_REQUIRE("gte_host_unregister", ptr != nullptr);
    return check_cuda("gte_host_unregister", cudaHostUnregister(ptr));
}

int gte_rollout(const GteParams* params, const GteData* data, const GteState* state, const void* actions,
                int n_steps, const GteStepOut* out, float* obs, int keep_obs, int autoreset, int variant, void* stream) {
    if (int rc = check_common("gte_rollout", params, data, state)) return rc;
    if (int rc = check_step_out("gte_rollout", params, actions, out)) return rc;
    GTE_REQUIRE("gte_rollout", obs != nullptr && n_steps >= 1);
    if (int rc = check_variant("gte_rollout", params, data, variant)) return rc;
    if (int rc = check_obs_ptr("gte_rollout", params, data, obs, variant)) return rc;
    return check_cuda("gte_rollout", gte::launch_rollout(*params, *data, *state, actions, n_steps, *out, obs, keep_obs,
                                                         autoreset, variant, static_cast<cudaStream_t>(stream)));
}

int gte_gather_obs(const GteParams* params, const GteData* data, const GteState* state, float* obs,
                   int variant, void* stream) {
    if (int rc = check_common("gte_gather_obs", params, data, state)) return rc;
    GTE_REQUIRE("gte_gather_obs", obs != nullptr);
    if (int rc = check_variant("gte_gather_obs", params, data, variant)) return rc;
    if (int rc = check_obs_ptr("gte_gather_obs", params, data, obs, variant)) return rc;
    return check_cuda("gte_gather_obs", gte::launch_obs_range(*params, *data, *state, obs, variant, 0,
                                                              params->n_envs, static_cast<cudaStream_t>(stream)));
}

int gte_info(const GteParams* params, const GteData* data, const GteState* state, const GteInfo* info,
             void* stream) {
    if (int rc = check_common("gte_info", params, data, state)) return rc;
    GTE_REQUIRE("gte_info", info != nullptr);
    return check_cuda("gte_info", gte::launch_info(*params, *data, *state, *info,
                                                   static_cast<cudaStream_t>(stream)));
}

int gte_struct_size(int which) {
    switch (which) {
        case 0: return (int)sizeof(GteParams);
        case 1: return (int)sizeof(GteData);
        case 2: return (int)sizeof(GteState);
        case 3: return (int)sizeof(GteStepOut);
        case 4: return (int)sizeof(GteInfo);
        case 5: return (int)sizeof(GteHostIO);
        default: return GTE_ERR_ARG;
    }
}

int gte_step_obs_launches(const GteParams* params, const GteData* data, int variant, int n_chunks) {
    if (params == nullptr || data == nullptr || n_chunks < 0 || n_chunks > 16) return GTE_ERR_ARG;
    if (params->windows == 0) return 1;
    // (episode accumulators, gte::acc_on: the fused form is never taken, step_obs_is_fused says so)
    if (n_chunks == 0 && gte::default_chunks(params->n_envs) == 1 && gte::step_obs_is_fused(*params, *data, variant)) return 1;
    return 2 * (n_chunks == 0 ? gte::default_chunks(params->n_envs) : n_chunks);
}

int gte_default_chunks(int n_envs) { return n_envs > 0 ? gte::default_chunks(n_envs) : GTE_ERR_ARG; }

int gte_obs_variant_for(const GteParams* params, const GteData* data) {
    if (params == nullptr || data == nullptr) return GTE_ERR_ARG;
    if (gte::obs_tma_supported(*params, *data)) return GTE_OBS_TMA;
    if (gte::obs_vec_supported(*params, *data)) return GTE_OBS_VEC;
    return GTE_OBS_GENERIC;
}

}  // extern "C"
