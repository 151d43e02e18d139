// hb_common.cuh -- shared device helpers for the sm_100a kernels of libhaplo_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hb {

// ---------------------------------------------------------------- SWAR byte-class masks
// Exact per-byte equality: 0x80 in every byte of w equal to the byte replicated in c4.
__device__ __forceinline__ uint32_t eq_mask(uint32_t w, uint32_t c4) {
    uint32_t t = w ^ c4;
    uint32_t m = ((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t;   // bit7 set <=> byte != 0, no cross-byte carry
    return ~m & 0x80808080u;
}
// Cheap existence test (may flag extra bytes above a true hit, never misses, zero iff no hit).
__device__ __forceinline__ uint32_t has_byte(uint32_t w, uint32_t c4) {
    uint32_t t = w ^ c4;
    return (t - 0x01010101u) & ~t & 0x80808080u;
}
constexpr uint32_t kTab4 = 0x09090909u;
constexpr uint32_t kNl4 = 0x0A0A0A0Au;

// index (0..3) of the n-th (0-based) set 0x80 flag in a 4-byte mask
__device__ __forceinline__ int nth_flag(uint32_t m, int n) {
    for (int i = 0; i < n; ++i) m &= m - 1;
    return (__ffs(m) - 1) >> 3;
}

// ---------------------------------------------------------------- mbarrier / TMA bulk (1-D)
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy (TMA, SASS UBLKCP).  src and dst 16-byte aligned, bytes % 16 == 0.
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global bulk copy (bulk async-group completion)
__device__ __forceinline__ void tma_store_1d(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- decoupled look-back words
// 64-bit status words: [63:62] flag (0 empty, 1 aggregate, 2 inclusive prefix), [61:0] payload.
constexpr uint64_t kFlagAgg = 1ull << 62;
constexpr uint64_t kFlagPre = 2ull << 62;
constexpr uint64_t kPayload = (1ull << 62) - 1;

__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// streaming 16-byte global load that does not allocate in L1
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(uint4 *p, const uint4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// ---------------------------------------------------------------- allele bytes -> bits
// bit j of the result = bit 0 of byte j of w
__device__ __forceinline__ uint32_t pack_lsb4(uint32_t w) { return ((w & 0x01010101u) * 0x01020408u) >> 24; }
// bit j of the result = byte j of w has one of bits 1..7 set (the byte is neither 0 nor 1)
__device__ __forceinline__ uint32_t pack_nz4(uint32_t w) {
    const uint32_t t = w & 0xFEFEFEFEu;
    const uint32_t nz = ((((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & 0x80808080u) >> 7;
    return (nz * 0x01020408u) >> 24;
}

// ---------------------------------------------------------------- sample subset (SampleSel, hb_internal.h)
// word s / 32 of a 128-bit block mask; s is a column of the block, 0..127
__device__ __forceinline__ uint32_t sel_word(const uint4 &m, uint32_t s) {
    const uint32_t q = s >> 5;
    return q == 0 ? m.x : q == 1 ? m.y : q == 2 ? m.z : m.w;
}
__device__ __forceinline__ bool sel_has(const uint4 &m, uint32_t s) { return (sel_word(m, s) >> (s & 31)) & 1u; }
// selected columns of the block below s
__device__ __forceinline__ uint32_t sel_rank(const uint4 &m, uint32_t s) {
    const uint32_t q = s >> 5;
    const uint32_t below = (q > 0 ? __popc(m.x) : 0) + (q > 1 ? __popc(m.y) : 0) + (q > 2 ? __popc(m.z) : 0);
    return below + __popc(sel_word(m, s) & ((1u << (s & 31)) - 1u));
}
// the plane of column s of the tile whose first column is s0 (without a subset: s0 + s)
template <bool kSubset>
__device__ __forceinline__ uint32_t sel_plane(const uint4 &m, uint32_t base, uint32_t s0, uint32_t s) {
    return kSubset ? base + sel_rank(m, s) : s0 + s;
}

}  // namespace hb
