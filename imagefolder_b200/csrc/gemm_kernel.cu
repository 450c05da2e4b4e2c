// gemm_kernel.cu -- hand-written tcgen05 GEMM (sm_100a) with the ViT MLP's element-wise work fused into its epilogue.
//
// Path: timm `Mlp.forward` inside `Block.forward`, tokenizer/tokenizer_image/dino_enc/vision_transformer.py:336-339
//   h = GELU(fc1(y)) ; branch = fc2(h)        and its backward.
// Two entry points replace a cuBLAS GEMM + a stand-alone bias/GELU kernel each:
//   xq_vit_fc1_gelu_fwd   pre = y W1^T (bf16) ; act = GELU(pre + b1)                       [epilogue writes both]
//   xq_vit_fc2_dgelu_bwd  d_pre = (d_branch W2) * GELU'(pre + b1) ; d_b1 = colsum(d_pre)    [epilogue reads pre]
// (the other four GEMMs of the block -- fc2 forward, the two weight gradients, the fc1 input gradient -- stay plain cuBLAS calls).
//
// C[M,N] = A[M,K] . B[N,K]^T, A and B K-major (row-major as PyTorch stores activations and Linear weights), bf16 in, fp32
// accumulation in TMEM.  A CTA PAIR (cluster of 2) owns a 256 x 256 tile: one `cta_group::2` MMA, M = 256 (128 accumulator
// rows in each CTA's TMEM), N = 256 (each CTA stages half of the B tile), K = 64 per stage, 5-stage TMA ring of 32 KB per CTA,
// accumulators double-buffered in 2 x 256 TMEM columns.  Persistent: pair p keeps column block p % (N/256) for the whole kernel
// (bias slice in shared memory, bias-gradient sums in registers, the weight tile hot in L2) and walks the 256-row blocks.
// Warps 0-15 epilogue (TMEM lane quarter = warp % 4, 64 columns per warp group), warp 16 TMA producer, warp 17 MMA issuer
// (leader CTA only).  Epilogue I/O goes through a per-warp 2 KB transposition buffer so that global accesses are full
// 32-byte sectors (scattered 16-byte row stores cost 0.5 ms per output at this size); its arithmetic runs on packed fp32 pairs
// (fma.rn.f32x2 -> FFMA2 / FMUL2 / FADD2, xq_gelu.cuh) because the epilogue, not the main loop, is what bounds the fused kernels.
// Measured (tools/gemm_probe.cu, B200, M = 131328, N = 3072, K = 768): plain 0.456 ms = 1.36 PFLOP/s vs cuBLAS
// nvjet_tst_128x256_64x6_2x1_2cta 0.434 ms (ratio 1.05, bit-identical results); fused forward 0.554 ms vs 0.72 ms for
// cuBLAS + gelu_fwd_kernel; fused backward 0.670 ms vs 0.83 ms for cuBLAS + gelu_bwd_kernel (tools/mlp_gemm_bench.py).
#include "xq_common.cuh"
#include "xq_tc.cuh"
#include "xq_gelu.cuh"

#include <mutex>
#include <tuple>

namespace xq {

using namespace xqtc;
using xqv::dgelu_f2;
using xqv::gelu_f2;
using xqv::up2;

constexpr int GM_BM = 128, GM_BN = 256, GM_BK = 64;            // per CTA: 128 rows; per pair: 256 x 256
constexpr int GM_NEPI = 16;                                    // epilogue warps (4 per SM sub-partition)
constexpr int GM_THREADS = (GM_NEPI + 2) * 32;
constexpr int GM_NST = 5;
constexpr int GM_A_BYTES = GM_BM * GM_BK * 2;                  // 16 KB
constexpr int GM_ST_BYTES = 2 * GM_A_BYTES;                    // A 128 x 64 + B half 128 x 64
constexpr int GM_STG_BYTES = 2048;                             // per-warp staging: 32 rows x 32 bf16 columns
constexpr int GM_BAR_OFF = GM_NST * GM_ST_BYTES;
constexpr int GM_BIAS_OFF = GM_BAR_OFF + 256;
constexpr int GM_STG_OFF = GM_BIAS_OFF + GM_BN * 4;
constexpr int GM_SMEM = GM_STG_OFF + GM_NEPI * GM_STG_BYTES + 1024;
constexpr int GM_CW = GM_BN / (GM_NEPI / 4);                   // accumulator columns per epilogue warp group (64)

// per-warp transposition through shared memory: thread = row view (its own 64-byte row) <-> coalesced view (8 rows x 64 B per
// warp instruction: full 32-byte sectors).  16-byte chunk c of row r lives at r * 64 + ((c ^ ((r >> 1) & 3)) * 16): conflict-free
// in both views.
__device__ __forceinline__ uint32_t gm_stg_off(int r, int c) { return (uint32_t)(r * 64 + ((c ^ ((r >> 1) & 3)) << 4)); }

// this thread's 32 bf16 (16 words) of row `lane` -> staging -> global rows [0, rows_ok) of the warp's 32 (row pitch ld elements)
__device__ __forceinline__ void gm_store_rows(uint32_t stg, const uint32_t (&w)[16], __nv_bfloat16 *__restrict__ gbase, size_t ld,
                                              int rows_ok, int lane) {
#pragma unroll
    for (int c = 0; c < 4; ++c) sts128(stg + gm_stg_off(lane, c), make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]));
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = i * 8 + (lane >> 2), c = lane & 3;
        const float4 v = lds128f(stg + gm_stg_off(r, c));
        if (r < rows_ok) *reinterpret_cast<float4 *>(gbase + (size_t)r * ld + c * 8) = v;
    }
    __syncwarp();
}
// global rows -> registers in the coalesced view (rows >= rows_ok read as zero): issued one chunk AHEAD of its use
__device__ __forceinline__ void gm_prefetch_rows(uint4 (&pf)[4], const __nv_bfloat16 *__restrict__ gbase, size_t ld, int rows_ok, int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = i * 8 + (lane >> 2), c = lane & 3;
        pf[i] = make_uint4(0u, 0u, 0u, 0u);
        if (r < rows_ok) pf[i] = *reinterpret_cast<const uint4 *>(gbase + (size_t)r * ld + c * 8);
    }
}
// prefetched registers -> staging -> this thread's row
__device__ __forceinline__ void gm_load_rows(uint32_t stg, uint32_t (&w)[16], const uint4 (&pf)[4], int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = i * 8 + (lane >> 2), c = lane & 3;
        sts128(stg + gm_stg_off(r, c), pf[i]);
    }
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float4 v = lds128f(stg + gm_stg_off(lane, c));
        w[4 * c] = __float_as_uint(v.x); w[4 * c + 1] = __float_as_uint(v.y); w[4 * c + 2] = __float_as_uint(v.z); w[4 * c + 3] = __float_as_uint(v.w);
    }
    __syncwarp();
}

// EPI 1: forward  -- C = pre-activation (bf16), C2 = GELU(pre + bias) (bf16).
// EPI 2: backward -- the accumulator is d_act; C = d_act * GELU'(X + bias) with X (= C2 argument) the stored pre-activation;
//                    column sums of the ROUNDED result -> dbias (fp32 atomics, one per column per CTA at the end).
// Both epilogues apply the element-wise function to the ROUNDED bf16 value of the GEMM result, i.e. exactly what the stand-alone
// kernels compute from the tensor a library GEMM would have written.
template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GM_THREADS, 1)
mlp_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, __nv_bfloat16 *__restrict__ C,
                __nv_bfloat16 *__restrict__ C2, const float *__restrict__ bias, float *__restrict__ dbias, int M, int N, int K) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(base + GM_BAR_OFF);
    uint64_t *full = bars, *empty = bars + GM_NST, *tfull = bars + 2 * GM_NST, *tempty = bars + 2 * GM_NST + 2;
    uint32_t *tmem_holder = (uint32_t *)(bars + 2 * GM_NST + 4);
    float *sbias = (float *)(base + GM_BIAS_OFF);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    if (tid == 0) {
        // full: the leader's arrive.expect_tx + the peer's remote arrive; tempty: the 16 epilogue warps of BOTH CTAs
        for (int i = 0; i < GM_NST; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 2 * GM_NEPI); }
        mbar_fence_init();
    }
    if (warp == GM_NEPI + 1) tmem_alloc2<512>(tmem_holder);
    // schedule: pair p keeps column block nb, walks 256-row blocks mb0, mb0 + mstep, ...
    const int nN = N / GM_BN, nM = (M + 2 * GM_BM - 1) / (2 * GM_BM), nk = K / GM_BK;
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int nb = pair % nN, mstep = npairs / nN, mb0 = pair / nN;
    for (int i = tid; i < GM_BN; i += GM_THREADS) sbias[i] = bias[nb * GM_BN + i];
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem = *tmem_holder;
    if (warp == GM_NEPI) {
        // ===== TMA producer (both CTAs): own 128 rows of A, own half of the B tile; every load signals the leader's barrier =====
        if (elect_one()) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); }
        __syncwarp();
        int it = 0;
        for (int mb = mb0; mb < nM; mb += mstep) {
            const int m0 = mb * 2 * GM_BM + (int)rank * GM_BM, n0 = nb * GM_BN + (int)rank * (GM_BN / 2);
            for (int kb = 0; kb < nk; ++kb, ++it) {
                const int st = it % GM_NST;
                mbar_wait(&empty[st], ((it / GM_NST) & 1) ^ 1);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&full[st], 2 * GM_ST_BYTES);
                    else mbar_arrive_cta(&full[st], 0);
                    tma_load_3d_2sm(base + st * GM_ST_BYTES, &tmA, kb * GM_BK, m0, 0, &full[st]);      // rows >= M: zero-filled
                    tma_load_3d_2sm(base + st * GM_ST_BYTES + GM_A_BYTES, &tmB, kb * GM_BK, n0, 0, &full[st]);
                }
                __syncwarp();
            }
        }
    } else if (warp == GM_NEPI + 1) {
        // ===== MMA issuer (leader CTA; whole warp runs the control flow, one elected lane issues) =====
        if (leader) {
            const uint32_t idesc = idesc_bf16(2 * GM_BM, GM_BN, 0, 0);
            int it = 0, tc = 0;
            for (int mb = mb0; mb < nM; mb += mstep, ++tc) {
                const int as = tc & 1;
                mbar_wait(&tempty[as], ((tc >> 1) & 1) ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int st = it % GM_NST;
                    mbar_wait(&full[st], (it / GM_NST) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t ad = desc_k_sw128(smem_u32(base + st * GM_ST_BYTES));
                        const uint64_t bd = desc_k_sw128(smem_u32(base + st * GM_ST_BYTES + GM_A_BYTES));
#pragma unroll
                        for (int k = 0; k < GM_BK / 16; ++k)
                            umma_ss2(tmem + as * GM_BN, desc_adv(ad, k * 32), desc_adv(bd, k * 32), idesc, (uint32_t)(kb | k));
                        umma_commit2(&empty[st]);                         // the stage is free in BOTH CTAs once these MMAs retire
                        if (kb == nk - 1) umma_commit2(&tfull[as]);       // accumulator ready in both CTAs
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ===== epilogue: thread = one accumulator row (TMEM lane), 64 columns per warp in two chunks of 32 =====
        const int qd = warp & 3, grp = warp >> 2;
        const uint32_t lane_addr = (uint32_t)(qd * 32) << 16;
        const uint32_t stg = smem_u32(base + GM_STG_OFF + warp * GM_STG_BYTES);
        const uint32_t sb = smem_u32(sbias + grp * GM_CW);
        int tc = 0;
        float bsum[GM_CW / 32];
#pragma unroll
        for (int i = 0; i < GM_CW / 32; ++i) bsum[i] = 0.f;
        // backward: the stored pre-activation of the NEXT 32 x 32 chunk is fetched while the current one is computed (and the first
        // chunk of a tile while its MMAs are still running)
        uint4 pf[4];
        auto tile_base = [&](int mb) { return (size_t)(mb * 2 * GM_BM + (int)rank * GM_BM + qd * 32) * N + nb * GM_BN + grp * GM_CW; };
        if (EPI == 2 && mb0 < nM) gm_prefetch_rows(pf, C2 + tile_base(mb0), N, M - (mb0 * 2 * GM_BM + (int)rank * GM_BM + qd * 32), lane);
        for (int mb = mb0; mb < nM; mb += mstep, ++tc) {
            const int as = tc & 1;
            const int r0 = mb * 2 * GM_BM + (int)rank * GM_BM + qd * 32;        // first of this warp's 32 rows
            const int rows_ok = M - r0;                                          // rows < M (may be <= 0 or >= 32)
            const size_t row_w = (size_t)r0 * N + nb * GM_BN + grp * GM_CW;
            mbar_wait(&tfull[as], (tc >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < GM_CW; c0 += 32) {
                uint32_t r[32];
                tmem_ld32(tmem + lane_addr + as * GM_BN + grp * GM_CW + c0, r);
                tmem_wait_ld();
                if (c0 == GM_CW - 32) {               // this warp's share of the accumulator buffer is in registers
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cta(&tempty[as], 0);
                }
                if (EPI == 1) {
                    uint32_t wp[16], wa[16];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 b0 = lds128f(sb + (c0 + 8 * q) * 4), b1 = lds128f(sb + (c0 + 8 * q + 4) * 4);
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const uint32_t pre = pack_bf16(__uint_as_float(r[8 * q + 2 * e]), __uint_as_float(r[8 * q + 2 * e + 1]));
                            const float x0 = __uint_as_float(pre << 16) + bb[2 * e], x1 = __uint_as_float(pre & 0xffff0000u) + bb[2 * e + 1];
                            wp[4 * q + e] = pre;
                            float y0, y1;
                            up2(gelu_f2(x0, x1), y0, y1);
                            wa[4 * q + e] = pack_bf16(y0, y1);
                        }
                    }
                    gm_store_rows(stg, wp, C + row_w + c0, N, rows_ok, lane);
                    gm_store_rows(stg, wa, C2 + row_w + c0, N, rows_ok, lane);
                } else {
                    float cs[32];
                    uint32_t xin[16], wo[16];
                    gm_load_rows(stg, xin, pf, lane);
                    if (c0 + 32 < GM_CW) {
                        gm_prefetch_rows(pf, C2 + row_w + c0 + 32, N, rows_ok, lane);
                    } else if (mb + mstep < nM) {
                        gm_prefetch_rows(pf, C2 + tile_base(mb + mstep), N, M - ((mb + mstep) * 2 * GM_BM + (int)rank * GM_BM + qd * 32), lane);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 b0 = lds128f(sb + (c0 + 8 * q) * 4), b1 = lds128f(sb + (c0 + 8 * q + 4) * 4);
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            // d_act rounded to bf16 first: the stand-alone kernel reads the bf16 tensor a library GEMM wrote.
                            // Rows >= M: the zero-filled A rows give d_act = 0, so they add nothing to the bias gradient.
                            const uint32_t gh = pack_bf16(__uint_as_float(r[8 * q + 2 * e]), __uint_as_float(r[8 * q + 2 * e + 1]));
                            const uint32_t xs = xin[4 * q + e];
                            const float x0 = __uint_as_float(xs << 16) + bb[2 * e], x1 = __uint_as_float(xs & 0xffff0000u) + bb[2 * e + 1];
                            float d0, d1;
                            up2(dgelu_f2(x0, x1), d0, d1);
                            const uint32_t o = pack_bf16(__uint_as_float(gh << 16) * d0, __uint_as_float(gh & 0xffff0000u) * d1);
                            wo[4 * q + e] = o;
                            cs[8 * q + 2 * e] = __uint_as_float(o << 16);
                            cs[8 * q + 2 * e + 1] = __uint_as_float(o & 0xffff0000u);
                        }
                    }
                    gm_store_rows(stg, wo, C + row_w + c0, N, rows_ok, lane);
                    // column sums over the warp's 32 rows: transpose-reduce butterfly (31 shuffles), lane l ends with column l
                    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2, b0 = lane & 1;
                    float a[16], b_[8], c_[4], d_[2];
#pragma unroll
                    for (int j = 0; j < 16; ++j) a[j] = (b4 ? cs[16 + j] : cs[j]) + __shfl_xor_sync(0xffffffffu, b4 ? cs[j] : cs[16 + j], 16);
#pragma unroll
                    for (int j = 0; j < 8; ++j) b_[j] = (b3 ? a[8 + j] : a[j]) + __shfl_xor_sync(0xffffffffu, b3 ? a[j] : a[8 + j], 8);
#pragma unroll
                    for (int j = 0; j < 4; ++j) c_[j] = (b2 ? b_[4 + j] : b_[j]) + __shfl_xor_sync(0xffffffffu, b2 ? b_[j] : b_[4 + j], 4);
#pragma unroll
                    for (int j = 0; j < 2; ++j) d_[j] = (b1 ? c_[2 + j] : c_[j]) + __shfl_xor_sync(0xffffffffu, b1 ? c_[j] : c_[2 + j], 2);
                    bsum[c0 / 32] += (b0 ? d_[1] : d_[0]) + __shfl_xor_sync(0xffffffffu, b0 ? d_[0] : d_[1], 1);
                }
            }
        }
        if (EPI == 2) {
#pragma unroll
            for (int i = 0; i < GM_CW / 32; ++i) atomicAdd(dbias + nb * GM_BN + grp * GM_CW + i * 32 + lane, bsum[i]);
        }
    }
    tc_fence_before();
    cluster_sync_all();          // the peer's shared memory is an MMA operand until the leader's last commit: leave together
    if (warp == GM_NEPI + 1) {
        tc_fence_after();
        tmem_dealloc2<512>(tmem);
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
struct GemmMaps { CUtensorMap tmA, tmB; };

static bool gm_get_maps(const void *a, const void *b, int M, int N, int K, GemmMaps &m) {
    static MapCache<std::tuple<const void *, const void *, int, int, int>, GemmMaps> cache;
    return cache.get({a, b, M, N, K}, m, [&](GemmMaps &e) {
        return make_map_3d(&e.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, const_cast<void *>(a), K, M, 1, (uint64_t)K * 2, (uint64_t)M * K * 2, GM_BK, GM_BM) &&
               make_map_3d(&e.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, const_cast<void *>(b), K, N, 1, (uint64_t)K * 2, (uint64_t)N * K * 2, GM_BK, GM_BN / 2);
    });
}

// per-device one-time setup (function attributes are per device)
static int gm_set_attr() {
    static std::mutex mu;
    static bool attr_set[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return record_cuda_error(e, "cudaGetDevice");
    if (dev < 0 || dev >= 64) return XQ_ERR_UNSUPPORTED;
    std::lock_guard<std::mutex> g(mu);
    if (!attr_set[dev]) {
        e = cudaFuncSetAttribute(mlp_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM);
        if (e != cudaSuccess) return record_cuda_error(e, "cudaFuncSetAttribute(mlp_gemm_kernel)");
        attr_set[dev] = true;
    }
    return XQ_OK;
}

static int gm_check(const void *a, const void *b, const void *c, const void *c2, const float *bias, int M, int N, int K) {
    if (!a || !b || !c || !c2 || !bias || M <= 0 || N <= 0 || K <= 0) return XQ_ERR_ARG;
    if (N % GM_BN != 0 || K % GM_BK != 0) return XQ_ERR_UNSUPPORTED;            // the ViT widths are multiples of 256 / 64
    if ((((uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)c2 | (uintptr_t)bias) & 15) != 0) return XQ_ERR_ARG;
    return XQ_OK;
}

template <int EPI>
static int gm_launch(const void *a, const void *b, void *c, void *c2, const float *bias, float *dbias, int M, int N, int K,
                     cudaStream_t st) {
    if (int rc = gm_set_attr()) return rc;
    int n_sm = 0;
    XQ_CUDA_TRY(sm_count(&n_sm));
    const int nN = N / GM_BN, max_pairs = n_sm / 2;
    if (nN > max_pairs) return XQ_ERR_UNSUPPORTED;
    GemmMaps m;
    if (!gm_get_maps(a, b, M, N, K, m)) return XQ_ERR_UNSUPPORTED;
    const int nM = (M + 2 * GM_BM - 1) / (2 * GM_BM);
    int per_col = max_pairs / nN;                         // pairs per column block
    if (per_col > nM) per_col = nM;
    const int npairs = per_col * nN;
    mlp_gemm_kernel<EPI><<<2 * npairs, GM_THREADS, GM_SMEM, st>>>(m.tmA, m.tmB, (__nv_bfloat16 *)c, (__nv_bfloat16 *)c2, bias, dbias, M, N, K);
    XQ_LAUNCH_CHECK("mlp_gemm_kernel");
    return XQ_OK;
}

}  // namespace xq

extern "C" {

int xq_vit_fc1_gelu_fwd(const void *x, const void *w, const float *bias, void *pre, void *act, int M, int N, int K, void *stream) {
    if (int rc = xq::gm_check(x, w, pre, act, bias, M, N, K)) return rc;
    return xq::gm_launch<1>(x, w, pre, act, bias, nullptr, M, N, K, (cudaStream_t)stream);
}

int xq_vit_fc2_dgelu_bwd(const void *d_out, const void *w2t, const void *pre, const float *bias, void *d_pre, float *d_bias, int M,
                         int N, int K, void *stream) {
    if (int rc = xq::gm_check(d_out, w2t, d_pre, pre, bias, M, N, K)) return rc;
    if (!d_bias) return XQ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    XQ_CUDA_TRY(cudaMemsetAsync(d_bias, 0, sizeof(float) * (size_t)N, st));
    return xq::gm_launch<2>(d_out, w2t, d_pre, const_cast<void *>(pre), bias, d_bias, M, N, K, st);
}

}  // extern "C"
