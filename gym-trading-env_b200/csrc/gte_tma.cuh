// gte_tma.cuh — shape bookkeeping of the observation window and the sm_100a TMA / mbarrier primitives
// (inline PTX) used by the gather kernels (gte_obs.cu).
#pragma once

#include "gte_device.cuh"

namespace gte {

// floor(e / d) for e*d < 2^32 via one umulhi; magic = ceil(2^32 / d)
__device__ __forceinline__ uint32_t fast_div(uint32_t e, uint32_t magic) { return __umulhi(e, magic); }
static inline uint32_t div_magic(uint32_t d) { return (uint32_t)(((1ull << 32) + d - 1) / d); }

struct ObsShape {
    int W, F, ns, nd;            // window rows, row floats, static cols, dynamic cols
    uint32_t magicF;             // ceil(2^32 / F)
    int row_bytes, win_bytes, n_vec;
    int w_mask;                  // W-1 when W is a power of two, else -1
    DynLayout dyn;               // dynamic-column descriptor: which ring block each dynamic column reads
};

static inline ObsShape make_shape(const GteParams& P) {
    ObsShape s;
    s.W = P.windows > 0 ? P.windows : 1;
    s.ns = P.n_static;
    s.nd = P.n_dyn;
    s.F = s.ns + s.nd;
    s.magicF = div_magic((uint32_t)s.F);
    s.row_bytes = s.F * 4;
    s.win_bytes = s.W * s.row_bytes;
    s.n_vec = s.win_bytes / 16;
    s.w_mask = (s.W & (s.W - 1)) == 0 ? s.W - 1 : -1;
    s.dyn = dyn_layout(P);
    return s;
}

// byte address of the 16B-aligned copy of the window that starts at row r0 of dataset ds
__device__ __forceinline__ const char* window_src(const GteData& D, const ObsShape& sh, int ds, int r0) {
    const int64_t off = (int64_t)r0 * sh.row_bytes;
    const int c = (int)((off >> 2) & 3);
    // select without dynamic indexing (keeps the kernel parameters in the constant bank)
    const float* t = (c == 0) ? D.window_table[0] : (c == 1) ? D.window_table[1]
                   : (c == 2) ? D.window_table[2] : D.window_table[3];
    return reinterpret_cast<const char*>(t) + (int64_t)ds * D.window_table_ds_stride + off;
}

// ------------------------------------------------------------------------------------------ tma
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// TMA 1-D bulk copy shared -> global, tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace gte
