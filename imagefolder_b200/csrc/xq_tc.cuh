// xq_tc.cuh -- the Blackwell async protocol of libxqb200 (sm_100a only): mbarrier, TMA (tensor and 1-D bulk copies),
// TMEM allocation / loads / stores, UMMA descriptors and tcgen05.mma issue, plus the host-side tensor-map encoding and
// cache and the per-device SM count.  Every kernel that speaks this protocol includes this header, so a fix to it is
// made once.
//
// Shared-memory operand layouts (all SWIZZLE_128B, 1024-byte aligned tiles; a 128-byte row holds 64 bf16 or 32 fp32):
//   "row tile"  [R rows][64 bf16]  = what one TMA box {64, R, 1} of a [.., rows, 64*k] tensor lands as:
//               byte(r, c) = r*128 + (((c >> 3) ^ (r & 7)) << 4) + (c & 7)*2
//     * as a K-major operand   (MMA K runs along the 64 columns): rows are M (or N), descriptor SBO = 1024
//     * as an MN-major operand (MMA K runs along the ROWS, M/N along the 64 columns): 8 rows = one swizzle atom,
//       SBO = 1024 (next 8 K), LBO = distance to the next 64 M/N elements (a second row tile)
//   tf32 operands (kind::tf32, the VQ search): K-major only, the same 128-byte rows holding 32 fp32 each; a K extent
//       of 32*k is k such tiles, one per 32-wide K chunk, and one MMA (K = 8) covers 32 bytes of a row
// Descriptor field meanings follow the sm_100 shared-memory matrix descriptor (start >> 4, LBO >> 4 at bit 16,
// SBO >> 4 at bit 32, version 1 at bit 46, layout type at bit 61; SWIZZLE_128B = 2).
//
// Bulk staging (no tensor map): bulk_g2s copies a contiguous global range into shared memory and completes on an mbarrier
// like a TMA load; the HBM-bound ViT kernels stream their row tiles with it (vit_kernels.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

namespace xqtc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
// non-blocking poll (try_wait may put the thread to sleep for an implementation-defined time before answering "not yet";
// an event loop that polls several barriers must not pay that for every barrier that is not ready)
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try(bar, parity)) {}
}

// ---- TMA (tensor maps are __grid_constant__ kernel parameters) ------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *map, const void *src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap *map, const void *src, int c0, int c1, int c2) {
    asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
// 1-D bulk copy of `bytes` (a multiple of 16, both addresses 16-byte aligned) global -> shared, completing on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ---- fences ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM allocation (one warp, power-of-two columns >= 32) -------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_holder) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS));
}

// ---- descriptors ------------------------------------------------------------------------------------------
// K-major SWIZZLE_128B operand: rows 128 B apart, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;                 // LBO: unused for a swizzled K-major operand one atom wide
    d |= (uint64_t)(1024 >> 4) << 32;       // SBO
    d |= (uint64_t)1 << 46;                 // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
    return d;
}
// MN-major SWIZZLE_128B operand: 64 M/N elements per 128-byte row, 8 K-rows per atom (SBO), next 64 M/N at LBO
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor, kind::f16: D = F32, A = B = BF16
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// instruction descriptor, kind::tf32: D = F32, A = B = TF32, both K-major
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMA ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
// A operand from TMEM (lane = M row, 2 bf16 per 32-bit column, K-major)
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- TMEM <-> registers (32 lanes x 32-bit, N consecutive columns per thread) ----------------------------
#define XQTC_R8(r, o) "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]), "=r"(r[o + 6]), "=r"(r[o + 7])
#define XQTC_I8(r, o) "r"(r[o + 0]), "r"(r[o + 1]), "r"(r[o + 2]), "r"(r[o + 3]), "r"(r[o + 4]), "r"(r[o + 5]), "r"(r[o + 6]), "r"(r[o + 7])

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : XQTC_R8(r, 0), XQTC_R8(r, 8), XQTC_R8(r, 16), XQTC_R8(r, 24)
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : XQTC_R8(r, 0), XQTC_R8(r, 8)
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : XQTC_R8(r, 0)
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31};"
        ::XQTC_I8(r, 0), XQTC_I8(r, 8), XQTC_I8(r, 16), XQTC_I8(r, 24), "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15};"
        ::XQTC_I8(r, 0), XQTC_I8(r, 8), "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%8], {%0, %1, %2, %3, %4, %5, %6, %7};"
                 ::XQTC_I8(r, 0), "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- CTA pair (cta_group::2): two CTAs of a 2-cluster (same TPC) issue ONE MMA with M = 256 (128 accumulator rows in each
// CTA's TMEM) and N <= 256 (each CTA stages half of the B tile).  PTX forms as in the vendored CUTLASS headers
// (cute/arch/copy_sm100_tma.hpp, cutlass/arch/barrier.h, cute/arch/tmem_allocator_sm100.hpp); verified on hardware by
// tools/gemm_probe.cu (bit-identical to cuBLAS at 131328 x 3072 x 768).
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// executed by BOTH CTAs: the bytes land in the executing CTA's shared memory and complete on the LEADER's (rank 0) barrier --
// the mbarrier address with the pair's peer bit cleared
__device__ __forceinline__ void tma_load_3d_2sm(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *leader_bar) {
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(leader_bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t *bar, uint32_t cta) {       // arrive on `bar` of cluster CTA `cta`
    asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
                 ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
__device__ __forceinline__ void umma_ss2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit2(uint64_t *bar) {                         // arrives on `bar` in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t *smem_holder) {                  // same warp id in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)), "r"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(COLS) : "memory");
}

// ---- explicit shared-memory accesses (pointers derived from the aligned dynamic-smem base are GENERIC to the compiler:
// without these it emits ST.E / LD.E generic instructions instead of STS / LDS) ------------------------------------
__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}
// advance a shared-memory matrix descriptor by `bytes` (start-address field is in 16-byte units; never carries out of it)
__device__ __forceinline__ uint64_t desc_adv(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

// one lane of a CONVERGED warp.  The single-thread tcgen05 / TMA instructions take uniform-register operands: issued
// under `if (lane == 0)` (a divergent region) the compiler wraps each one in an ELECT / BRA.U.ANY serialisation loop,
// measured at ~112 clk per tcgen05.mma whatever its shape; issued under elect.sync by a warp that runs the surrounding
// control flow uniformly they are plain predicated instructions (64 clk for M128 N128 K16 = the tensor-pipe rate).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---- misc ------------------------------------------------------------------------------------------------
// byte offset of element (row r, column c) of a [rows][64 bf16] SWIZZLE_128B row tile
__host__ __device__ __forceinline__ uint32_t rowtile_off_bf16(int r, int c) {
    return (uint32_t)(r * 128 + ((((c >> 3) ^ (r & 7)) & 7) << 4) + (c & 7) * 2);
}
// byte offset of 16-byte unit u (0..7) of row r
__host__ __device__ __forceinline__ uint32_t rowtile_unit(int r, int u) { return (uint32_t)(r * 128 + ((u ^ (r & 7)) << 4)); }

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));   // upper half <- first source
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- host side ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

// SWIZZLE_128B tensor map of rank 2 or 3 (box_inner * element size = 128 bytes; strides in bytes, inner dimension dense)
static inline bool make_map_sw128(CUtensorMap *tm, CUtensorMapDataType dt, cuuint32_t rank, void *base, const cuuint64_t *gdim,
                                  const cuuint64_t *gstr, const cuuint32_t *box) {
    PFN_encodeTiled enc = get_encode_fn();
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return enc && enc(tm, dt, rank, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// 2-D tensor map {inner, rows} with box {box_inner, box_rows}
static inline bool make_map_2d(CUtensorMap *tm, CUtensorMapDataType dt, void *base, uint64_t inner, uint64_t rows,
                               uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_rows) {
    const cuuint64_t gdim[2] = {inner, rows}, gstr[1] = {row_stride_bytes};
    const cuuint32_t box[2] = {box_inner, box_rows};
    return make_map_sw128(tm, dt, 2, base, gdim, gstr, box);
}
// 3-D tensor map {inner, rows, batch} with box {box_inner, box_rows, 1}
static inline bool make_map_3d(CUtensorMap *tm, CUtensorMapDataType dt, void *base, uint64_t inner, uint64_t rows, uint64_t batch,
                               uint64_t row_stride_bytes, uint64_t batch_stride_bytes, uint32_t box_inner, uint32_t box_rows) {
    const cuuint64_t gdim[3] = {inner, rows, batch}, gstr[2] = {row_stride_bytes, batch_stride_bytes};
    const cuuint32_t box[3] = {box_inner, box_rows, 1u};
    return make_map_sw128(tm, dt, 3, base, gdim, gstr, box);
}

// Encoded tensor maps by key (the pointers and shapes they are built from; `Key` has operator==, e.g. a std::tuple).
// Encoding is a driver call and a training step asks for the same few maps every step.  Fixed capacity, round-robin
// eviction, thread safe.
template <typename Key, typename Maps>
class MapCache {
  public:
    // the maps cached for `key`, else those make(Maps &) builds (cached only when it returns true)
    template <typename Make>
    bool get(const Key &key, Maps &out, Make make) {
        std::lock_guard<std::mutex> g(mu_);
        for (int i = 0; i < n_; ++i)
            if (keys_[i] == key) { out = maps_[i]; return true; }
        if (!make(out)) return false;
        keys_[next_] = key;
        maps_[next_] = out;
        next_ = (next_ + 1) % CAP;
        if (n_ < CAP) ++n_;
        return true;
    }

  private:
    static constexpr int CAP = 32;
    std::mutex mu_;
    Key keys_[CAP];
    Maps maps_[CAP];
    int n_ = 0, next_ = 0;
};

// multiprocessor count of the current device, queried once per device
inline cudaError_t sm_count(int *n) {
    constexpr int MAX_DEV = 64;
    static std::mutex mu;
    static int cached[MAX_DEV] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> g(mu);
    int v = dev < MAX_DEV ? cached[dev] : 0;
    if (!v) {
        e = cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        if (dev < MAX_DEV) cached[dev] = v;
    }
    *n = v;
    return cudaSuccess;
}

}  // namespace xqtc
