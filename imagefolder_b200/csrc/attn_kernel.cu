// attn_kernel.cu -- tcgen05 / TMEM / TMA flash attention for the ViT blocks (head_dim 64, bf16, no mask), sm_100a.
//
// Replaces F.scaled_dot_product_attention in Attention.forward
//   (tokenizer/tokenizer_image/dino_enc/vision_transformer.py:173-197: q,k,v = qkv.reshape(B,N,3,H,hd).permute(2,0,3,1,4);
//    x = sdpa(q,k,v); x = x.transpose(1,2).reshape(B,N,C))
// reading q/k/v straight out of the packed projection [B,N,3,H,64] through ONE 3-D tensor map and writing the
// head-merged output [B,N,H*64], so that no permute / contiguous copy exists on either side.
//
// Forward, one CTA per (batch, head, 128-query tile), 2 CTAs per SM (256 TMEM columns each):
//   warp 4   TMA producer : Q tile once per tile, K / V row tiles (128 keys x 64) through 2-stage rings
//   warp 5   MMA issuer   : S = Q K^T   (kind::f16, A,B K-major smem, N = 128 or the 16-rounded tail)  -> TMEM[0,128)
//                           O += P V    (A = P from TMEM[128,192), B = V MN-major smem, N = 64)        -> TMEM[192,256)
//   warps 0-3 softmax     : one query row per thread (TMEM lane): S -> registers, running max with LAZY rescaling of O
//                           (only when the row max grows by more than 2^8), P = exp2(S*c - m*c) -> bf16 -> TMEM,
//                           epilogue O / l -> bf16 -> swizzled smem -> TMA store (rows beyond N are clipped by the map)
//   sequence lengths need not be multiples of anything: the last key block is issued with N = ceil16(valid keys) and
//   its invalid columns are masked to -inf; rows of the last query tile beyond N are zero-filled by TMA and clipped on store.
// The statistics tensor holds L2[b,h,n] = m*c + log2(l) (base-2 log-sum-exp of the SCALED scores), what backward needs.
#include "xq_common.cuh"
#include "xq_tc.cuh"

#include <mutex>
#include <tuple>

namespace xq {
using namespace xqtc;

constexpr int AT_BM = 128;          // queries per CTA
constexpr int AT_BN = 128;          // keys per block
constexpr int AT_D = 64;            // head dim
constexpr int AT_NS = 2;            // K / V ring stages
constexpr int AT_TILE = AT_BM * AT_D * 2;   // bytes of one [128][64] bf16 row tile
constexpr int AT_THREADS = 256;
constexpr float AT_LAZY = 8.0f;     // rescale O only when the scaled max grows by more than this (log2 units)

struct AttnFwdSmem {
    // offsets from the 1024-aligned base
    static constexpr int Q = 0;
    static constexpr int K = AT_TILE;
    static constexpr int V = AT_TILE * (1 + AT_NS);
    static constexpr int O = AT_TILE * (1 + 2 * AT_NS);     // output staging (the Q tile is re-loaded early for the next tile)
    static constexpr int BAR = AT_TILE * (2 + 2 * AT_NS);
    static constexpr int BYTES = BAR + 256;
};

template <int REGS>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS)); }
template <int REGS>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS)); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// Development-only clock trace (compiled in with -DXQ_ATTN_TRACE for tools/attn_trace.py; absent from libxqb200.so)
#ifdef XQ_ATTN_TRACE
__device__ long long *g_attn_trace = nullptr;
#define XQ_TR(cond, slot) do { if ((cond) && g_attn_trace && blockIdx.x == 0) g_attn_trace[(slot)] = clock64(); } while (0)
#else
#define XQ_TR(cond, slot) do { } while (0)
#endif

// PERSISTENT: gridDim.x CTAs (2 per SM) walk the (batch*head, query tile) list with stride gridDim.x; all pipeline state
// (ring stages, barrier phases) runs on across tiles, so the producer prefetches the next tile's Q / K / V while the softmax
// warps are still in the epilogue of the current one and the prologue cost (TMEM allocation, descriptor fetch, first-load
// latency) is paid once per CTA instead of once per tile.
__global__ void __launch_bounds__(AT_THREADS, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmO, float *__restrict__ lse2,
                int N, int H, int nQ /* query tiles per (b,h) handled here */, int n_tiles, float c /* softmax scale * log2(e) */) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(base + AttnFwdSmem::BAR);
    uint64_t *q_full = bars + 0;
    uint64_t *q_empty = bars + 1;
    uint64_t *k_full = bars + 2;              // [AT_NS]
    uint64_t *k_empty = bars + 2 + AT_NS;     // [AT_NS]
    uint64_t *v_full = bars + 2 + 2 * AT_NS;
    uint64_t *v_empty = bars + 2 + 3 * AT_NS;
    uint64_t *s_full = bars + 2 + 4 * AT_NS;
    uint64_t *s_free = s_full + 1;
    uint64_t *p_full = s_full + 2;
    uint64_t *pv_done = s_full + 3;
    uint64_t *o_free = s_full + 4;
    uint32_t *tmem_holder = (uint32_t *)(s_full + 5);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nK = (N + AT_BN - 1) / AT_BN;

    if (tid == 0) {
        mbar_init(q_full, 1);
        mbar_init(q_empty, 1);
        for (int i = 0; i < AT_NS; ++i) { mbar_init(&k_full[i], 1); mbar_init(&k_empty[i], 1); mbar_init(&v_full[i], 1); mbar_init(&v_empty[i], 1); }
        mbar_init(s_full, 1);
        mbar_init(s_free, 4);
        mbar_init(p_full, 4);
        mbar_init(pv_done, 1);
        mbar_init(o_free, 4);
        mbar_fence_init();
    }
    if (warp == 5) tmem_alloc<256>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_holder;
    const uint32_t tS = tmem, tP = tmem + 128, tO = tmem + 192;

    // warps 0-3 = softmax, warps 4-7 = control (4 = TMA producer, 5 = MMA issuer): the warp scheduler favours the higher
    // warp id among eligible warps, which keeps the single-thread MMA issuer from being starved by the softmax warps
    if (warp >= 4) {
        reg_dec<40>();
        if (warp == 4) {
            // ===== TMA producer (whole warp runs the loop, one elected lane issues) =====
            if (elect_one()) tma_prefetch_desc(&tmQKV);
            uint32_t it = 0, tl = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
                const int bh = t / nQ, qt = t - bh * nQ;
                const int b = bh / H, h = bh - b * H;
                const int colQ = h * AT_D, colK = (H + h) * AT_D, colV = (2 * H + h) * AT_D;
                mbar_wait(q_empty, (tl & 1) ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(q_full, AT_TILE);
                    tma_load_3d(base + AttnFwdSmem::Q, &tmQKV, colQ, qt * AT_BM, b, q_full);
                }
                __syncwarp();
                for (int j = 0; j < nK; ++j, ++it) {
                    const int st = it % AT_NS;
                    const uint32_t ph = ((it / AT_NS) & 1) ^ 1;
                    mbar_wait(&k_empty[st], ph);
                    if (elect_one()) {
                        mbar_expect_tx(&k_full[st], AT_TILE);
                        tma_load_3d(base + AttnFwdSmem::K + st * AT_TILE, &tmQKV, colK, j * AT_BN, b, &k_full[st]);
                    }
                    __syncwarp();
                    mbar_wait(&v_empty[st], ph);
                    if (elect_one()) {
                        mbar_expect_tx(&v_full[st], AT_TILE);
                        tma_load_3d(base + AttnFwdSmem::V + st * AT_TILE, &tmQKV, colV, j * AT_BN, b, &v_full[st]);
                    }
                    __syncwarp();
                }
            }
        } else if (warp == 5) {
            // ===== MMA issuer (whole warp runs the control flow, one elected lane issues: see elect_one) =====
            const uint64_t qd = desc_k_sw128(smem_u32(base + AttnFwdSmem::Q));
            uint32_t it = 0, tl = 0;
            auto issue_qk = [&](uint32_t itx, int j, bool last_of_tile) {
                const int st = itx % AT_NS;
                const int nj = (min(AT_BN, N - j * AT_BN) + 15) & ~15;
                mbar_wait(&k_full[st], (itx / AT_NS) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t kd = desc_k_sw128(smem_u32(base + AttnFwdSmem::K + st * AT_TILE));
                    const uint32_t id = idesc_bf16(AT_BM, nj, 0, 0);
#pragma unroll
                    for (int k = 0; k < AT_D / 16; ++k) umma_ss(tS, desc_adv(qd, k * 32), desc_adv(kd, k * 32), id, k > 0);
                    umma_commit(&k_empty[st]);
                    umma_commit(s_full);
                    if (last_of_tile) umma_commit(q_empty);     // every S MMA of this tile is issued: Q is dead once they retire
                }
                __syncwarp();
            };
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
                mbar_wait(q_full, tl & 1);
                if (it > 0) { mbar_wait(s_free, (it - 1) & 1); }      // the last S of the previous tile is in registers
                tc_fence_after();
                issue_qk(it, 0, nK == 1);
                for (int j = 0; j < nK; ++j, ++it) {
                    if (j + 1 < nK) {
                        mbar_wait(s_free, it & 1);          // softmax holds S_j in registers
                        tc_fence_after();
                        issue_qk(it + 1, j + 1, j + 2 == nK);
                    }
                    const int st = it % AT_NS;
                    const int nj = (min(AT_BN, N - j * AT_BN) + 15) & ~15;
                    mbar_wait(&v_full[st], (it / AT_NS) & 1);
                    mbar_wait(p_full, it & 1);              // P_j written (and O rescaled)
                    if (j == 0 && tl > 0) mbar_wait(o_free, (tl - 1) & 1);   // the epilogue has read the previous tile's O
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t vd = desc_mn_sw128(smem_u32(base + AttnFwdSmem::V + st * AT_TILE), 16384, 1024);
                        const uint32_t id = idesc_bf16(AT_BM, AT_D, 0, 1);
                        for (int k = 0; k < nj / 16; ++k) umma_ts(tO, tP + k * 8, desc_adv(vd, k * 2048), id, (j | k) != 0);
                        umma_commit(&v_empty[st]);
                        umma_commit(pv_done);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        reg_inc<216>();
        // ===== softmax: thread = query row =====
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        uint32_t it = 0, tl = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tl) {
            const int bh = t / nQ, qt = t - bh * nQ;
            const int b = bh / H, h = bh - b * H;
            const int q0 = qt * AT_BM;
            float m_used = -CUDART_INF_F;     // raw-score max the current P / O are expressed against
            float l = 0.f;
            // a warp whose 32 rows all lie beyond N (last tile of a ragged sequence) only keeps the pipeline's barriers
            // moving: its P / O rows feed rows the output tensor map clips, so their contents do not matter
            const bool warp_live = q0 + q * 32 < N;
            for (int j = 0; j < nK; ++j, ++it) {
                const int nv = min(AT_BN, N - j * AT_BN);       // valid keys in this block
                mbar_wait(s_full, it & 1);
                tc_fence_after();
                if (!warp_live) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(s_free);
                    if (j > 0) mbar_wait(pv_done, (it - 1) & 1);
                    if (lane == 0) mbar_arrive(p_full);
                    continue;
                }
                uint32_t s[128];
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    if (ch * 32 < nv) tmem_ld32(tS + lane_addr + ch * 32, *reinterpret_cast<uint32_t(*)[32]>(&s[ch * 32]));
                }
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(s_free);
                float mx4[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
                if (nv == AT_BN) {
#pragma unroll
                    for (int i = 0; i < 128; i += 4) {
                        mx4[0] = fmaxf(mx4[0], __uint_as_float(s[i]));
                        mx4[1] = fmaxf(mx4[1], __uint_as_float(s[i + 1]));
                        mx4[2] = fmaxf(mx4[2], __uint_as_float(s[i + 2]));
                        mx4[3] = fmaxf(mx4[3], __uint_as_float(s[i + 3]));
                    }
                } else {
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) {
                        if (ch * 32 < nv) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) {
                                float x = __uint_as_float(s[ch * 32 + i]);
                                if (ch * 32 + i >= nv) x = -CUDART_INF_F;
                                s[ch * 32 + i] = __float_as_uint(x);
                                mx4[i & 3] = fmaxf(mx4[i & 3], x);
                            }
                        }
                    }
                }
                const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
                if (j > 0) mbar_wait(pv_done, (it - 1) & 1);       // O and the P buffer are quiescent
                tc_fence_after();
                const bool grow = (mx - m_used) * c > AT_LAZY;     // j == 0: m_used = -inf -> true
                if (j == 0) {
                    m_used = mx;
                } else if (__any_sync(0xffffffffu, grow)) {
                    const float m_new = grow ? mx : m_used;
                    const float alpha = ex2_approx((m_used - m_new) * c);
                    l *= alpha;
                    m_used = m_new;
#pragma unroll
                    for (int c0 = 0; c0 < AT_D; c0 += 16) {
                        uint32_t o[16];
                        tmem_ld16(tO + lane_addr + c0, o);
                        tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                        tmem_st16(tO + lane_addr + c0, o);
                    }
                }
                const float mc = m_used * c;
                float sum0 = 0.f, sum1 = 0.f, sum2 = 0.f, sum3 = 0.f;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    if (ch * 32 < nv) {
                        uint32_t pk[16];
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            float p0 = ex2_approx(fmaf(__uint_as_float(s[ch * 32 + i]), c, -mc));
                            float p1 = ex2_approx(fmaf(__uint_as_float(s[ch * 32 + i + 1]), c, -mc));
                            float p2 = ex2_approx(fmaf(__uint_as_float(s[ch * 32 + i + 2]), c, -mc));
                            float p3 = ex2_approx(fmaf(__uint_as_float(s[ch * 32 + i + 3]), c, -mc));
                            sum0 += p0;
                            sum1 += p1;
                            sum2 += p2;
                            sum3 += p3;
                            pk[i >> 1] = pack_bf16(p0, p1);
                            pk[(i >> 1) + 1] = pack_bf16(p2, p3);
                        }
                        tmem_st16(tP + lane_addr + ch * 16, pk);
                    }
                }
                l += (sum0 + sum1) + (sum2 + sum3);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(p_full);
            }
            // ---- epilogue: O / l -> bf16 -> staging smem -> TMA store (rows beyond N are clipped by the tensor map)
            mbar_wait(pv_done, (it - 1) & 1);
            tc_fence_after();
            uint32_t o[64];
            tmem_ld32(tO + lane_addr, *reinterpret_cast<uint32_t(*)[32]>(&o[0]));
            tmem_ld32(tO + lane_addr + 32, *reinterpret_cast<uint32_t(*)[32]>(&o[32]));
            tmem_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(o_free);             // the next tile's first P V may overwrite O
            const float inv = 1.0f / l;
            if (q0 + row < N) lse2[(size_t)bh * N + q0 + row] = fmaf(m_used, c, log2f(l));
            uint8_t *so = base + AttnFwdSmem::O;
            const uint32_t so_a = smem_u32(so);
            if (warp == 0 && lane == 0) bulk_wait_read<0>();   // the previous tile's store has finished reading the staging tile
            named_bar_sync(1, 128);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                uint4 v;
                v.x = pack_bf16(__uint_as_float(o[8 * u + 0]) * inv, __uint_as_float(o[8 * u + 1]) * inv);
                v.y = pack_bf16(__uint_as_float(o[8 * u + 2]) * inv, __uint_as_float(o[8 * u + 3]) * inv);
                v.z = pack_bf16(__uint_as_float(o[8 * u + 4]) * inv, __uint_as_float(o[8 * u + 5]) * inv);
                v.w = pack_bf16(__uint_as_float(o[8 * u + 6]) * inv, __uint_as_float(o[8 * u + 7]) * inv);
                sts128(so_a + rowtile_unit(row, u), v);
            }
            fence_async_smem();
            named_bar_sync(2, 128);
            if (warp == 0 && lane == 0) {
                tma_store_3d(&tmO, so, h * AT_D, q0, b);
                bulk_commit();
            }
        }
        if (warp == 0 && lane == 0) bulk_wait<0>();
    }
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc<256>(tmem);
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------
struct AttnMaps { CUtensorMap tmQKV, tmO; };

// per-device one-time setup (function attributes are per device)
struct AttnDevState { bool fwd_attr = false, bwd_attr = false, prep_attr = false; };
static int attn_dev_state(AttnDevState **out) {
    static std::mutex mu;
    static AttnDevState states[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return xq::record_cuda_error(e, "cudaGetDevice");
    if (dev < 0 || dev >= 64) return XQ_ERR_UNSUPPORTED;
    std::lock_guard<std::mutex> g(mu);
    *out = &states[dev];
    return XQ_OK;
}

static bool get_fwd_maps(const void *qkv, void *out, int B, int N, int H, AttnMaps &m) {
    static MapCache<std::tuple<const void *, const void *, int, int, int>, AttnMaps> cache;
    return cache.get({qkv, out, B, N, H}, m, [&](AttnMaps &e) {
        const uint64_t W = (uint64_t)3 * H * AT_D, Wo = (uint64_t)H * AT_D;
        return make_map_3d(&e.tmQKV, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, const_cast<void *>(qkv), W, N, B, W * 2, (uint64_t)N * W * 2, AT_D, AT_BM) &&
               make_map_3d(&e.tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, out, Wo, N, B, Wo * 2, (uint64_t)N * Wo * 2, AT_D, AT_BM);
    });
}

// =====================================================================================================================
// Backward.  One CTA per (batch, head, 128-key block), 1 CTA per SM, looping over the query blocks i:
//     S^T  = K Q_i^T              (M = keys on TMEM lanes, N = queries)            TMEM [0,128)
//     dP^T = V dO_i^T                                                              TMEM [128,256)
//     P^T  = exp2(S^T c - L2[q])            -> bf16 -> TMEM [448,512)
//     dS^T = P^T o (dP^T - delta[q])        -> bf16 -> TMEM (over dP^T) and, transposed view, smem (MN-major A operand)
//     dV  += P^T dO_i   (A from TMEM, B = dO tile MN-major)                        TMEM [256,320)
//     dK  += dS^T Q_i   (A from TMEM, B = Q tile MN-major)                         TMEM [320,384)
//     dQ_i = dS K       (A = dS smem MN-major, B = K tile MN-major)                TMEM [384,448) -> fp32 smem -> TMA reduce-add
// With keys on the lanes, the softmax statistics L2[q] / delta[q] are per COLUMN: broadcast reads from shared memory.
// The query tail is cheap (it is the MMA N / K extent, rounded to 16); `scale` is folded into the dK epilogue and the
// dQ conversion.  dQ is accumulated across the key blocks of a (batch, head) in an fp32 workspace by TMA reduce-add
// and converted to bf16 into dqkv by attn_dq_convert_kernel.
// Warp-specialised, 24 warps (warp % 4 = TMEM lane quarter; "half" = 64 of the block's 128 queries):
//   wgE  warps 0-7    P^T = exp2(...)                  one warpgroup per query half   (the MUFU work)
//   wgD  warps 8-15   dS^T = P^T o (dP^T - delta)      one warpgroup per query half, written to TMEM (dK operand) and
//                                                      smem (dQ operand)              (the FMA work)
//   ctl  warps 16-19  16 = TMA producer, 17 = MMA issuer
//   wgQ  warps 20-23  drains each dQ_i partial: TMEM -> fp32 smem -> TMA reduce-add
// The exp2 of block i+1 (MUFU pipe) overlaps the dS arithmetic of block i (FMA pipe), the dQ drain never sits on either's
// critical path, and every sub-partition holds two warps of each elementwise role (latency hiding).  wgD reads P^T back
// from TMEM as bf16 (the same rounded values the dV MMA consumes).
// =====================================================================================================================
constexpr int AB_THREADS = 768;

constexpr int AB_QS = 3;            // Q / dO ring stages (a stage is released only when dK_i retires: 2 stages starve the MMAs)

struct AttnBwdSmem {
    static constexpr int K = 0;                             // 2 buffers (item parity): the next item's K / V are prefetched
    static constexpr int V = 2 * AT_TILE;                   // 2 buffers
    static constexpr int Q = 4 * AT_TILE;                   // AB_QS stages
    static constexpr int DO = (4 + AB_QS) * AT_TILE;        // AB_QS stages
    static constexpr int DS = (4 + 2 * AB_QS) * AT_TILE;    // 2 row tiles (one per query half)
    static constexpr int DQ = (6 + 2 * AB_QS) * AT_TILE;    // fp32 staging: ONE row tile [128][32 fp32] (two passes per dQ_i)
    static constexpr int STAT = (7 + 2 * AB_QS) * AT_TILE;  // lse[AB_QS][128], delta[AB_QS][128]
    static constexpr int BAR = STAT + AB_QS * 1024;
    static constexpr int BYTES = BAR + 256;
};

// dV / dK epilogue of one item: the thread's accumulator row (64 fp32 in TMEM at `taddr`) * mul -> bf16 -> 128 contiguous bytes
// of the packed gradient, and the column sums of the ROUNDED values of the warp's 32 rows -> qkv-bias gradient.  The sums are a
// transpose-reduce butterfly over the warp (lane = row): 62 shuffles, after which lane l holds columns c0 and c0 + 1,
// c0 = 32 b4 + 16 b3 + 8 b2 + 4 b1 + 2 b0 (bits of l) -> 2 atomics per lane.  The row is read 8 + 8 columns at a time (column j
// with column j + 32: the first butterfly step is fused with the rounding), so ~50 registers are live; `freed` is signalled as
// soon as the last columns have left TMEM.  Rows beyond N hold zeros (masked keys) and are not stored.
__device__ __forceinline__ void bwd_epilogue_rows(uint32_t taddr, float mul, __nv_bfloat16 *__restrict__ dst_row, bool row_ok,
                                                  float *__restrict__ g_bias_cols, int lane, uint64_t *freed) {
    float a[32], b[16], c[8], d[4];
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2, b0 = lane & 1;
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
        uint32_t lo[8], hi[8];
        tmem_ld8(taddr + c8 * 8, lo);
        tmem_ld8(taddr + 32 + c8 * 8, hi);
        tmem_wait_ld();
        if (c8 == 3) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(freed);
        }
        uint32_t wl[4], wh[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            wl[e] = pack_bf16(__uint_as_float(lo[2 * e]) * mul, __uint_as_float(lo[2 * e + 1]) * mul);
            wh[e] = pack_bf16(__uint_as_float(hi[2 * e]) * mul, __uint_as_float(hi[2 * e + 1]) * mul);
        }
        if (row_ok) {
            *reinterpret_cast<uint4 *>(dst_row + c8 * 8) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
            *reinterpret_cast<uint4 *>(dst_row + 32 + c8 * 8) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
        }
        if (g_bias_cols) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float l0 = __uint_as_float(wl[e] << 16), l1 = __uint_as_float(wl[e] & 0xffff0000u);
                const float h0 = __uint_as_float(wh[e] << 16), h1 = __uint_as_float(wh[e] & 0xffff0000u);
                a[c8 * 8 + 2 * e] = (b4 ? h0 : l0) + __shfl_xor_sync(0xffffffffu, b4 ? l0 : h0, 16);
                a[c8 * 8 + 2 * e + 1] = (b4 ? h1 : l1) + __shfl_xor_sync(0xffffffffu, b4 ? l1 : h1, 16);
            }
        }
    }
    if (g_bias_cols) {
#pragma unroll
        for (int j = 0; j < 16; ++j) b[j] = (b3 ? a[16 + j] : a[j]) + __shfl_xor_sync(0xffffffffu, b3 ? a[j] : a[16 + j], 8);
#pragma unroll
        for (int j = 0; j < 8; ++j) c[j] = (b2 ? b[8 + j] : b[j]) + __shfl_xor_sync(0xffffffffu, b2 ? b[j] : b[8 + j], 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) d[j] = (b1 ? c[4 + j] : c[j]) + __shfl_xor_sync(0xffffffffu, b1 ? c[j] : c[4 + j], 2);
        const float s0 = (b0 ? d[2] : d[0]) + __shfl_xor_sync(0xffffffffu, b0 ? d[0] : d[2], 1);
        const float s1 = (b0 ? d[3] : d[1]) + __shfl_xor_sync(0xffffffffu, b0 ? d[1] : d[3], 1);
        const int c0 = (b4 ? 32 : 0) + (b3 ? 16 : 0) + (b2 ? 8 : 0) + (b1 ? 4 : 0) + (b0 ? 2 : 0);
        atomicAdd(g_bias_cols + c0, s0);
        atomicAdd(g_bias_cols + c0 + 1, s1);
    }
}

__global__ void __launch_bounds__(AB_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                const __grid_constant__ CUtensorMap tmDQ, const float *__restrict__ lseP, const float *__restrict__ deltaP,
                __nv_bfloat16 *__restrict__ dqkv, float *__restrict__ g_bias, int N, int H, int nK, int Npad, int n_items, float c,
                float scale) {
    extern __shared__ uint8_t smem_raw[];
    XQ_TR(threadIdx.x == 0, 16 * 30 + 4);
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(base + AttnBwdSmem::BAR);
    uint64_t *kv_full = bars + 19;    // [2] K / V buffers (item parity)
    uint64_t *q_full = bars + 1;      // [AB_QS] stages
    uint64_t *q_empty = bars + 4;     // [AB_QS]
    uint64_t *s_full = bars + 7;      // S^T_i in TMEM                      (MMA commit)
    uint64_t *s_free = bars + 8;      // S^T_i in wgE's registers           (4 warps)
    uint64_t *p_full = bars + 9;      // P^T_i (bf16) in TMEM               (4 warps of wgE)
    uint64_t *p_read = bars + 10;     // P^T_i in wgD's registers           (4 warps of wgD)
    uint64_t *dv_done = bars + 11;    // dV MMAs of block i retired         (MMA commit)
    uint64_t *dp_full = bars + 12;    // dP^T_i in TMEM                     (MMA commit)
    uint64_t *ds_full = bars + 13;    // dS_i in TMEM and smem              (4 warps of wgD)
    uint64_t *dq_full = bars + 14;    // dQ_i partial in TMEM               (MMA commit)
    uint64_t *dq_free = bars + 15;    // dQ_i drained                       (4 warps of wgQ)
    uint64_t *dkv_done = bars + 16;   // dV / dK of the item complete          (MMA commit)
    uint64_t *kv_free = bars + 21;    // [2] last MMA reading this K / V buffer retired (MMA commit): it may be reloaded
    uint64_t *dkv_free = bars + 18;   // dV / dK of the item in registers      (4 warps of wgE0 + 4 of wgD0)
    uint32_t *tmem_holder = (uint32_t *)(bars + 23);
    float *s_lse = (float *)(base + AttnBwdSmem::STAT);          // [AB_QS][128]
    float *s_delta = s_lse + AB_QS * 128;                        // [AB_QS][128]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // PERSISTENT: the CTA walks items (batch*head, key block) blockIdx.x, + gridDim.x, ...; every pipeline below keeps running
    // across item boundaries on one global query-block counter g (barrier parities are functions of g, or of the item count n
    // for the per-item barriers), so that the dQ drain and the dK / dV epilogue of item n overlap the first blocks of item n+1
    // and no CTA launch / barrier init / TMEM allocation sits between items.
    struct Item { int bh, b, h, k0, colQ, colK, colV; };
    auto item_at = [&](int it) {
        Item t;
        t.bh = it / nK;
        t.b = t.bh / H; t.h = t.bh - t.b * H;
        t.k0 = (it - t.bh * nK) * AT_BN;
        t.colQ = t.h * AT_D; t.colK = (H + t.h) * AT_D; t.colV = (2 * H + t.h) * AT_D;
        return t;
    };
    const int nQ = Npad / AT_BM;

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_free[i], 1); }
        for (int i = 0; i < AB_QS; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
        mbar_init(s_full, 1); mbar_init(s_free, 8);
        mbar_init(p_full, 8); mbar_init(p_read, 8);
        mbar_init(dv_done, 1); mbar_init(dp_full, 1);
        mbar_init(ds_full, 8); mbar_init(dq_full, 1);
        mbar_init(dq_free, 4); mbar_init(dkv_done, 1);
        mbar_init(dkv_free, 8);
        mbar_fence_init();
    }
    if (warp == 17) tmem_alloc<512>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_holder;
    const uint32_t tS = tmem, tDP = tmem + 128, tDV = tmem + 256, tDK = tmem + 320, tDQ = tmem + 384, tP = tmem + 448;
    XQ_TR(tid == 0, 16 * 30 + 2);
    // queries of block i, rounded up to the MMA granularity
    auto nq_of = [&](int i) { return (min(AT_BM, N - i * AT_BM) + 15) & ~15; };
    const int qd = warp & 3;                         // TMEM lane quarter of this warp
    const int krow = qd * 32 + lane;                 // row of the 128-row tile this thread owns (a key, or a query in wgQ)
    const uint32_t lane_addr = (uint32_t)(qd * 32) << 16;

    // register budget (768 threads x 80 at launch = 61440): 4 compute warpgroups x 88 + control 72 + wgQ 56 = 6 x 80
    if (warp >= 16 && warp < 20) {
        reg_dec<72>();
        if (warp == 16) {
            // ===== TMA producer (whole warp runs the loop, one elected lane issues) =====
            if (elect_one()) {
                tma_prefetch_desc(&tmQKV);
                tma_prefetch_desc(&tmDO);
            }
            __syncwarp();
            // K / V of item n live in buffer n & 1; the next item's pair is requested while this item's third query block is being
            // loaded (by then the last dQ MMA of item n-1, the previous user of that buffer, has all but retired), i.e. two to
            // three blocks before its first MMA needs it: a TMA tile load was measured at ~5 k clk here.
            auto load_kv = [&](int it, int n) {
                const Item T = item_at(it);
                const int kb = n & 1;
                if (n >= 2) mbar_wait(&kv_free[kb], ((n >> 1) - 1) & 1);
                if (elect_one()) {
                    mbar_expect_tx(&kv_full[kb], 2 * AT_TILE);
                    tma_load_3d(base + AttnBwdSmem::K + kb * AT_TILE, &tmQKV, T.colK, T.k0, T.b, &kv_full[kb]);
                    tma_load_3d(base + AttnBwdSmem::V + kb * AT_TILE, &tmQKV, T.colV, T.k0, T.b, &kv_full[kb]);
                }
                __syncwarp();
            };
            if ((int)blockIdx.x < n_items) load_kv(blockIdx.x, 0);
            for (int it = blockIdx.x, n = 0; it < n_items; it += gridDim.x, ++n) {
                const Item T = item_at(it);
                const int pre = min(2, nQ - 1);
                for (int i = 0; i < nQ; ++i) {
                    const int g = n * nQ + i, st = g % AB_QS;
                    mbar_wait(&q_empty[st], ((g / AB_QS) & 1) ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(&q_full[st], 2 * AT_TILE + 1024);
                        tma_load_3d(base + AttnBwdSmem::Q + st * AT_TILE, &tmQKV, T.colQ, i * AT_BM, T.b, &q_full[st]);
                        tma_load_3d(base + AttnBwdSmem::DO + st * AT_TILE, &tmDO, T.h * AT_D, i * AT_BM, T.b, &q_full[st]);
                        bulk_g2s(s_lse + st * 128, lseP + (size_t)T.bh * Npad + i * AT_BM, 512, &q_full[st]);
                        bulk_g2s(s_delta + st * 128, deltaP + (size_t)T.bh * Npad + i * AT_BM, 512, &q_full[st]);
                    }
                    __syncwarp();
                    if (i == pre && it + (int)gridDim.x < n_items) load_kv(it + gridDim.x, n + 1);
                }
            }
        } else if (warp == 17) {
            // ===== MMA issuer (whole warp runs the control flow, one elected lane issues: see elect_one) =====
            // program order per query block i:   S^T_{i+1}  |  dV += P^T_i dO_i  |  dK += dS^T_i Q_i ; dP^T_{i+1} ; dQ_i = dS_i K
            // (S^T_{i+1} only needs S^T_i to have left TMEM, so wgE never waits for it; dP^T_{i+1} is queued right behind
            //  dK_i -- which reads dS^T_i out of the same columns -- so wgD gets it back after two MMA groups)
            const uint64_t kd_k0 = desc_k_sw128(smem_u32(base + AttnBwdSmem::K)), vd_k0 = desc_k_sw128(smem_u32(base + AttnBwdSmem::V));
            const uint64_t kd_mn0 = desc_mn_sw128(smem_u32(base + AttnBwdSmem::K), 16384, 1024);
            const uint64_t qd_k0 = desc_k_sw128(smem_u32(base + AttnBwdSmem::Q)), dd_k0 = desc_k_sw128(smem_u32(base + AttnBwdSmem::DO));
            const uint64_t qd_mn0 = desc_mn_sw128(smem_u32(base + AttnBwdSmem::Q), 16384, 1024);
            const uint64_t dd_mn0 = desc_mn_sw128(smem_u32(base + AttnBwdSmem::DO), 16384, 1024);
            const uint64_t dsd = desc_mn_sw128(smem_u32(base + AttnBwdSmem::DS), AT_TILE, 1024);
            const uint32_t id_acc = idesc_bf16(AT_BN, AT_D, 0, 1);     // A from TMEM (K-major), B MN-major
            const uint32_t id_dq = idesc_bf16(AT_BM, AT_D, 1, 1);      // A, B MN-major smem
            auto issue_s = [&](int i, int g, int kb) {
                if (elect_one()) {
                    const uint64_t qdk = desc_adv(qd_k0, (g % AB_QS) * AT_TILE), kd_k = desc_adv(kd_k0, kb * AT_TILE);
                    const uint32_t id = idesc_bf16(AT_BN, nq_of(i), 0, 0);
#pragma unroll
                    for (int k = 0; k < AT_D / 16; ++k) umma_ss(tS, desc_adv(kd_k, k * 32), desc_adv(qdk, k * 32), id, k > 0);
                    umma_commit(s_full);
                }
                __syncwarp();
            };
            auto issue_dp = [&](int i, int g, int kb) {
                if (elect_one()) {
                    const uint64_t ddk = desc_adv(dd_k0, (g % AB_QS) * AT_TILE), vd_k = desc_adv(vd_k0, kb * AT_TILE);
                    const uint32_t id = idesc_bf16(AT_BN, nq_of(i), 0, 0);
#pragma unroll
                    for (int k = 0; k < AT_D / 16; ++k) umma_ss(tDP, desc_adv(vd_k, k * 32), desc_adv(ddk, k * 32), id, k > 0);
                    umma_commit(dp_full);
                }
                __syncwarp();
            };
            // one flat pipeline over (item n, query block i), global block counter g: the S^T and dP^T MMAs of the NEXT block are
            // issued one block ahead also across an item boundary (the next item's K / V sit in the other buffer)
            if ((int)blockIdx.x < n_items) {
                mbar_wait(&kv_full[0], 0);
                mbar_wait(&q_full[0], 0);
                tc_fence_after();
                issue_s(0, 0, 0);
                issue_dp(0, 0, 0);
            }
            for (int it = blockIdx.x, n = 0; it < n_items; it += gridDim.x, ++n) {
                const int g0 = n * nQ, kb = n & 1;
                const bool next_item = it + (int)gridDim.x < n_items;
                const uint64_t kd_mn = desc_adv(kd_mn0, kb * AT_TILE);
                for (int i = 0; i < nQ; ++i) {
                    const int g = g0 + i, st = g % AB_QS;
                    const int ks = nq_of(i) / 16;
                    const uint64_t qd_mn = desc_adv(qd_mn0, st * AT_TILE), dd_mn = desc_adv(dd_mn0, st * AT_TILE);
                    const bool last = i + 1 == nQ;
                    const bool more = !last || next_item;
                    const int ni = last ? 0 : i + 1, nkb = last ? kb ^ 1 : kb;      // the block after this one
                    if (more) {
                        if (last) mbar_wait(&kv_full[nkb], ((n + 1) >> 1) & 1);
                        mbar_wait(s_free, g & 1);
                        mbar_wait(&q_full[(g + 1) % AB_QS], ((g + 1) / AB_QS) & 1);
                        tc_fence_after();
                        issue_s(ni, g + 1, nkb);
                    }
                    mbar_wait(p_full, g & 1);
                    XQ_TR(g < 30 && lane == 0, 16 * g + 0);
                    if (i == 0 && n > 0) mbar_wait(dkv_free, (n - 1) & 1);   // the previous item's dV / dK have left TMEM
                    tc_fence_after();
                    if (elect_one()) {
                        for (int k = 0; k < ks; ++k)      // dV += P^T dO : 16 queries per k-step
                            umma_ts(tDV, tP + k * 8, desc_adv(dd_mn, k * 2048), id_acc, (uint32_t)(i | k));   // P^T: 8 columns per k-step, contiguous
                        umma_commit(dv_done);
                    }
                    __syncwarp();
                    mbar_wait(ds_full, g & 1);
                    XQ_TR(g < 30 && lane == 0, 16 * g + 1);
                    tc_fence_after();
                    if (elect_one()) {
                        for (int k = 0; k < ks; ++k)      // dK += dS^T Q : each query half keeps its dS^T (bf16) over the start of its own dP^T columns
                            umma_ts(tDK, tDP + (k >> 2) * 64 + (k & 3) * 8, desc_adv(qd_mn, k * 2048), id_acc, (uint32_t)(i | k));
                        umma_commit(&q_empty[st]);        // Q_i / dO_i tiles are dead once dV_i and dK_i retire
                        if (last) umma_commit(dkv_done);
                    }
                    __syncwarp();
                    if (more) issue_dp(ni, g + 1, nkb);   // in program order behind dK_g, the last reader of these TMEM columns
                    if (g > 0) { mbar_wait(dq_free, (g - 1) & 1); tc_fence_after(); }
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < AT_BN / 16; ++k)    // dQ_i = dS K : A = dS [M = q (2 row tiles), K = keys], B = K tile
                            umma_ss(tDQ, desc_adv(dsd, k * 2048), desc_adv(kd_mn, k * 2048), id_dq, k > 0);
                        umma_commit(dq_full);
                        if (last) umma_commit(&kv_free[kb]);     // every MMA that reads this item's K / V has been issued
                    }
                    __syncwarp();
                    XQ_TR(g < 30 && lane == 0, 16 * g + 2);
                }
            }
        }
    } else if (warp < 8) {
        reg_inc<88>();
        // ===== wgE (warps 0-7): P^T = exp2(S^T c - L2[q]); thread = (key row, query half hf): the MUFU warpgroups =====
        const int hf = warp >> 2;
        // epilogue of item n (hf == 0 warps): dV (TMEM) -> registers (the accumulator is then free) -> bf16 -> global
        auto epilogue_dv = [&](int it_e, int n_e) {
            const Item E = item_at(it_e);
            XQ_TR(n_e == 0 && tid == 0, 16 * 30 + 5);
            mbar_wait(dkv_done, n_e & 1);
            tc_fence_after();
            XQ_TR(n_e == 0 && tid == 0, 16 * 30 + 6);
            bwd_epilogue_rows(tDV + lane_addr, 1.0f, dqkv + ((size_t)E.b * N + E.k0 + krow) * (size_t)(3 * H * AT_D) + E.colV,
                              E.k0 + krow < N, g_bias ? g_bias + E.colV : nullptr, lane, dkv_free);
            XQ_TR(n_e == 0 && tid == 0, 16 * 30 + 8);
        };
        for (int it = blockIdx.x, n = 0; it < n_items; it += gridDim.x, ++n) {
        const Item T = item_at(it);
        const bool key_ok = T.k0 + krow < N;
        const bool keys_full = T.k0 + AT_BN <= N;    // warp-uniform: no key of this block needs masking
        for (int i = 0; i < nQ; ++i) {
            const int gq = n * nQ + i, st = gq % AB_QS;
            const int nqr = nq_of(i);
            mbar_wait(&q_full[st], (gq / AB_QS) & 1);               // statistics of this query block are in smem
            mbar_wait(s_full, gq & 1);
            XQ_TR(gq < 30 && warp == 0 && lane == 0, 16 * gq + 4);
            tc_fence_after();
            const uint32_t l4 = smem_u32(s_lse + st * 128 + hf * 64);
            const bool fast = keys_full && nqr == AT_BM;
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {                        // 2 chunks of 32 queries
                const int col = hf * 64 + ch * 32;
                uint32_t sb[32];
                if (col < nqr) tmem_ld32(tS + lane_addr + col, sb);
                tmem_wait_ld();
                if (ch == 1) {                                      // this half of S^T_i has left TMEM
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(s_free);
                }
                uint32_t pk[16];
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    const float4 L = lds128f(l4 + (ch * 8 + g) * 16);
                    float p0 = ex2_approx(fmaf(__uint_as_float(sb[4 * g + 0]), c, -L.x));
                    float p1 = ex2_approx(fmaf(__uint_as_float(sb[4 * g + 1]), c, -L.y));
                    float p2 = ex2_approx(fmaf(__uint_as_float(sb[4 * g + 2]), c, -L.z));
                    float p3 = ex2_approx(fmaf(__uint_as_float(sb[4 * g + 3]), c, -L.w));
                    if (!fast) {
                        const bool ok = key_ok && (col < nqr);
                        p0 = ok ? p0 : 0.f; p1 = ok ? p1 : 0.f; p2 = ok ? p2 : 0.f; p3 = ok ? p3 : 0.f;
                    }
                    pk[2 * g] = pack_bf16(p0, p1);
                    pk[2 * g + 1] = pack_bf16(p2, p3);
                }
                if (ch == 0 && gq > 0) {                            // the P buffer is free: dV_{g-1} retired and wgD holds P_{g-1}
                    mbar_wait(dv_done, (gq - 1) & 1);
                    mbar_wait(p_read, (gq - 1) & 1);
                    tc_fence_after();
                }
                tmem_st16(tP + lane_addr + hf * 32 + ch * 16, pk);
            }
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_full);
            XQ_TR(gq < 30 && warp == 0 && lane == 0, 16 * gq + 5);
            // the previous item's dV: its last dK MMA retires about now (this P^T was computed a block ahead), and the first dV
            // MMA of this item waits for the accumulator to be in our registers (dkv_free)
            if (hf == 0 && i == 0 && n > 0) epilogue_dv(it - gridDim.x, n - 1);
        }
        }
        if (hf == 0 && n_items > (int)blockIdx.x) {
            const int n_last = (n_items - 1 - (int)blockIdx.x) / (int)gridDim.x;
            epilogue_dv(blockIdx.x + n_last * gridDim.x, n_last);
        }
    } else if (warp < 16) {
        reg_inc<88>();
        // ===== wgD (warps 8-15): dS^T = P^T o (dP^T - delta[q]); thread = (key row, query half hf): the FMA warpgroups =====
        const int hf = (warp - 8) >> 2;
        const uint32_t dsrow = smem_u32(base + AttnBwdSmem::DS + hf * AT_TILE);
        // epilogue of item n (hf == 0 warps): dK (TMEM) -> registers -> * scale -> bf16 -> global
        auto epilogue_dk = [&](int it_e, int n_e) {
            const Item E = item_at(it_e);
            mbar_wait(dkv_done, n_e & 1);
            tc_fence_after();
            bwd_epilogue_rows(tDK + lane_addr, scale, dqkv + ((size_t)E.b * N + E.k0 + krow) * (size_t)(3 * H * AT_D) + E.colK,
                              E.k0 + krow < N, g_bias ? g_bias + E.colK : nullptr, lane, dkv_free);
        };
        for (int it = blockIdx.x, n = 0; it < n_items; it += gridDim.x, ++n) {
        for (int i = 0; i < nQ; ++i) {
            const int gq = n * nQ + i, st = gq % AB_QS;
            const int nqr = nq_of(i);
            // the previous item's dK: these warps would only wait for P^T of this block here (wgE is still computing it)
            if (hf == 0 && i == 0 && n > 0) epilogue_dk(it - gridDim.x, n - 1);
            mbar_wait(&q_full[st], (gq / AB_QS) & 1);
            mbar_wait(p_full, gq & 1);
            XQ_TR(gq < 30 && warp == 8 && lane == 0, 16 * gq + 8);
            tc_fence_after();
            uint32_t pk[32];                                          // this half of P^T as written by wgE: 2 bf16 per word
            tmem_ld32(tP + lane_addr + hf * 32, pk);
            tmem_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_read);
            mbar_wait(dp_full, gq & 1);
            XQ_TR(gq < 30 && warp == 8 && lane == 0, 16 * gq + 9);
            // the dS operand tile in shared memory is single-buffered (the second buffer went to the K / V prefetch): dQ_{g-1},
            // its last reader, must have retired
            if (gq > 0) mbar_wait(dq_full, (gq - 1) & 1);
            tc_fence_after();
            const uint32_t d4 = smem_u32(s_delta + st * 128 + hf * 64);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {                          // 16 queries per chunk
                const int col = hf * 64 + ch * 16;
                uint32_t dp[16], o8[8];
                if (col < nqr) {
                    tmem_ld16(tDP + lane_addr + col, dp);
                    tmem_wait_ld();
                } else {                                              // beyond the block's queries: P = 0, dS = 0
#pragma unroll
                    for (int e = 0; e < 16; ++e) dp[e] = 0u;
                }
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const float4 Dl = lds128f(d4 + (ch * 4 + g) * 16);
                    const uint32_t w0 = pk[ch * 8 + g * 2], w1 = pk[ch * 8 + g * 2 + 1];
                    const float d0 = __uint_as_float(w0 << 16) * (__uint_as_float(dp[g * 4 + 0]) - Dl.x);
                    const float d1 = __uint_as_float(w0 & 0xffff0000u) * (__uint_as_float(dp[g * 4 + 1]) - Dl.y);
                    const float d2 = __uint_as_float(w1 << 16) * (__uint_as_float(dp[g * 4 + 2]) - Dl.z);
                    const float d3 = __uint_as_float(w1 & 0xffff0000u) * (__uint_as_float(dp[g * 4 + 3]) - Dl.w);
                    o8[g * 2 + 0] = pack_bf16(d0, d1);
                    o8[g * 2 + 1] = pack_bf16(d2, d3);
                }
                // dS^T for the dK MMA (TMEM, over this thread's own, already consumed, dP^T columns) ...
                tmem_st8(tDP + lane_addr + hf * 64 + ch * 8, o8);
                // ... and dS for the dQ MMA (smem, MN-major: row = key, this half's 64 queries along the row)
                sts128(dsrow + rowtile_unit(krow, ch * 2), make_uint4(o8[0], o8[1], o8[2], o8[3]));
                sts128(dsrow + rowtile_unit(krow, ch * 2 + 1), make_uint4(o8[4], o8[5], o8[6], o8[7]));
                XQ_TR(gq < 30 && warp == 8 && lane == 0 && ch < 3, 16 * gq + 13 + ch);
            }
            XQ_TR(gq < 30 && warp == 8 && lane == 0, 16 * gq + 11);
            fence_async_smem();
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(ds_full);
            XQ_TR(gq < 30 && warp == 8 && lane == 0, 16 * gq + 10);
        }
        }
        if (hf == 0 && n_items > (int)blockIdx.x) {
            const int n_last = (n_items - 1 - (int)blockIdx.x) / (int)gridDim.x;
            epilogue_dk(blockIdx.x + n_last * gridDim.x, n_last);
        }
    } else {
        reg_dec<56>();
        // ===== wgQ (warps 20-23): dQ_i partial (TMEM lanes = queries) -> fp32 smem row tiles -> TMA reduce-add =====
        const uint32_t stg = smem_u32(base + AttnBwdSmem::DQ);
        const bool issuer = tid == 20 * 32;
        for (int it = blockIdx.x, n = 0; it < n_items; it += gridDim.x, ++n) {
        const int bh = it / nK;
        for (int i = 0; i < nQ; ++i) {
            const int gq = n * nQ + i;
            mbar_wait(dq_full, gq & 1);
            tc_fence_after();
#pragma unroll
            for (int hfc = 0; hfc < 2; ++hfc) {       // 32 head-dim columns per pass through the staging tile
                uint32_t r[32];
                tmem_ld32(tDQ + lane_addr + hfc * 32, r);
                tmem_wait_ld();
                if (hfc == 1) {                       // the whole accumulator has left TMEM: the next dQ MMA may start
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(dq_free);
                }
                if (issuer) bulk_wait_read<0>();     // the previous reduce has finished reading the staging tile
                named_bar_sync(4, 128);
#pragma unroll
                for (int u = 0; u < 8; ++u) sts128(stg + rowtile_unit(krow, u), make_uint4(r[4 * u], r[4 * u + 1], r[4 * u + 2], r[4 * u + 3]));
                fence_async_smem();
                named_bar_sync(5, 128);
                if (issuer) {
#ifndef XQ_ATTN_EXP_NODQ      // experiment switch (tools/): time the kernel without the dQ reduce traffic
                    tma_reduce_add_3d(&tmDQ, base + AttnBwdSmem::DQ, hfc * 32, i * AT_BM, bh);
#endif
                    bulk_commit();
                }
            }
            XQ_TR(gq < 30 && qd == 0 && lane == 0, 16 * gq + 12);
        }
        }
        if (issuer) bulk_wait<0>();
    }
    __syncthreads();
    XQ_TR(tid == 0, 16 * 30 + 3);
    if (warp == 17) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}


// Backward pre-pass, one launch.  256 threads = 32 rows x 8 lanes (16 B of a 64-wide head row each); a CTA works on 128-row
// blocks of one (batch, head), four row passes per block with all loads issued up front.
//   * delta[q] = sum_d dO[q][d] O[q][d]  and the lse copied into the 128-padded layout the main kernel's TMA reads (+inf pads);
//   * the fp32 dQ accumulator rows are zeroed here (they are this kernel's rows anyway; saves a 400 MB memset node);
//   * NT > 0 -- the last (N mod 128) keys when they are few (<= AB_KTAIL_MAX; 513 = 4*128 + 1): a whole CTA of attn_bwd_kernel,
//     five query blocks of full-size MMAs, for one or two key rows is 20 % of that kernel's work at N = 513.  Those keys are
//     handled here on CUDA cores instead, since dO[q] is in registers already (one more 16 B load for q):
//         s = c q.k_t ; p = exp2(s - L2[q]) ; dp = dO[q].v_t ; ds = p (dp - delta[q])
//         dV[t] += p dO[q] ; dK[t] += ds q  (registers; one CTA owns the whole (batch, head), so it also writes the rounded
//         dK / dV rows of those keys and their share of the qkv-bias gradient) ; ds[q][t] -> dsT.
//     attn_dq_convert_kernel folds  dQ[q] += sum_t ds[q][t] k_t  in while it converts the accumulator.
// grid: NT == 0 -> (Npad / 128, B*H);  NT > 0 -> (1, B*H), the CTA loops over the row blocks.
constexpr int AB_KTAIL_MAX = 4;
constexpr int AB_PREP_ROWS = 128;

__device__ __forceinline__ void unpack8(const uint4 &w, float (&f)[8]) {
    const uint32_t x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { f[2 * e] = __uint_as_float(x[e] << 16); f[2 * e + 1] = __uint_as_float(x[e] & 0xffff0000u); }
}

template <int NT>
__global__ void __launch_bounds__(256, 2)
attn_bwd_prep_kernel(const __nv_bfloat16 *__restrict__ qkv, const __nv_bfloat16 *__restrict__ out, const __nv_bfloat16 *__restrict__ dout,
                     const float *__restrict__ lse2, float *__restrict__ lseP, float *__restrict__ deltaP, float *__restrict__ dq_acc,
                     float *__restrict__ dsT, __nv_bfloat16 *__restrict__ dqkv, float *__restrict__ g_bias, int N, int H, int Npad,
                     float c, float scale) {
    constexpr int NTA = NT > 0 ? NT : 1;
    __shared__ float red[NT > 0 ? 8 : 1][2][NTA][AT_D];
    __shared__ __align__(16) float skv[2][NTA][AT_D];
    const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
    const int lane = threadIdx.x & 31, sub = threadIdx.x & 7, rloc = threadIdx.x >> 3;
    const int n0 = N - NT;
    const size_t W = (size_t)3 * H * AT_D;
    const __nv_bfloat16 *qb = qkv + (size_t)b * N * W + h * AT_D + sub * 8;
    const size_t ob = (size_t)b * N * H * AT_D + h * AT_D + sub * 8;
    float aK[NTA][8], aV[NTA][8];
    if constexpr (NT > 0) {
        // tail key / value rows as fp32 in shared memory: [t][d]; 16 threads per t (8 for k, 8 for v), 16 B of bf16 each
        if (threadIdx.x < NT * 16) {
            const int t = threadIdx.x >> 4, isv = (threadIdx.x >> 3) & 1;
            float f[8];
            unpack8(*reinterpret_cast<const uint4 *>(qb + (size_t)(n0 + t) * W + (size_t)(1 + isv) * H * AT_D), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) skv[isv][t][sub * 8 + e] = f[e];
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) {
#pragma unroll
            for (int e = 0; e < 8; ++e) aK[t][e] = aV[t][e] = 0.f;
        }
        __syncthreads();
    }
    constexpr int PASSES = AB_PREP_ROWS / 32;
    // NT > 0: the CTA walks the row blocks of its (batch, head) with the next block's rows in flight (cp.async into a two-stage
    // shared buffer; every thread reads back only the 16-byte slots it copied itself, so the wait_group is the only sync needed)
    extern __shared__ uint4 prep_stage[];                                  // [2 stages][3: O, dO, q][PASSES][256 threads]
    auto prefetch = [&](int blk, int stg) {
#pragma unroll
        for (int ps = 0; ps < PASSES; ++ps) {
            const int n = blk * AB_PREP_ROWS + ps * 32 + rloc;
            const int nc = n < N ? n : N - 1;
            uint4 *dst = prep_stage + ((size_t)(stg * 3) * PASSES + ps) * 256 + threadIdx.x;
            cp_async16(dst, out + ob + (size_t)nc * H * AT_D);
            cp_async16(dst + PASSES * 256, dout + ob + (size_t)nc * H * AT_D);
            cp_async16(dst + 2 * PASSES * 256, qb + (size_t)nc * W);
        }
        cp_async_commit();
    };
    if constexpr (NT > 0) prefetch(blockIdx.x, 0);
    int stg = 0;
    for (int blk = blockIdx.x; blk * AB_PREP_ROWS < Npad; blk += gridDim.x, stg ^= 1) {
        uint4 ow[PASSES], gw[PASSES], qw[PASSES];
        float lq[PASSES];
#pragma unroll
        for (int ps = 0; ps < PASSES; ++ps) {
            const int n = blk * AB_PREP_ROWS + ps * 32 + rloc;
            const int nc = n < N ? n : N - 1;                              // pads: load the last row, results discarded below
            if constexpr (NT == 0) {
                ow[ps] = *reinterpret_cast<const uint4 *>(out + ob + (size_t)nc * H * AT_D);
                gw[ps] = *reinterpret_cast<const uint4 *>(dout + ob + (size_t)nc * H * AT_D);
            }
            lq[ps] = lse2[(size_t)bh * N + nc];
        }
        if constexpr (NT > 0) {
            if ((blk + (int)gridDim.x) * AB_PREP_ROWS < Npad) { prefetch(blk + gridDim.x, stg ^ 1); cp_async_wait<1>(); }
            else cp_async_wait<0>();
        }
#pragma unroll
        for (int ps = 0; ps < PASSES; ++ps) {
            const int n = blk * AB_PREP_ROWS + ps * 32 + rloc;             // < Npad
            const bool live = n < N;
            float ov[8], gv[8];
            if constexpr (NT > 0) {
                const uint4 *src = prep_stage + ((size_t)(stg * 3) * PASSES + ps) * 256 + threadIdx.x;
                ow[ps] = src[0];
                gw[ps] = src[PASSES * 256];
                qw[ps] = src[2 * PASSES * 256];
            }
            unpack8(ow[ps], ov);
            unpack8(gw[ps], gv);
            float dl = 0.f;
#pragma unroll
            for (int e = 0; e < 8; ++e) dl = fmaf(ov[e], gv[e], dl);
            dl += __shfl_xor_sync(0xffffffffu, dl, 1);
            dl += __shfl_xor_sync(0xffffffffu, dl, 2);
            dl += __shfl_xor_sync(0xffffffffu, dl, 4);
            if (!live) dl = 0.f;
            if (sub == 0) {
                deltaP[(size_t)bh * Npad + n] = dl;
                lseP[(size_t)bh * Npad + n] = live ? lq[ps] : CUDART_INF_F;
            }
            if (live) {
                float4 *z = reinterpret_cast<float4 *>(dq_acc + ((size_t)bh * N + n) * AT_D + sub * 8);
                z[0] = make_float4(0.f, 0.f, 0.f, 0.f);
                z[1] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if constexpr (NT > 0) {
                float qv[8];
                unpack8(qw[ps], qv);
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    float sx = 0.f, pd = 0.f;
                    const float4 k0 = *reinterpret_cast<const float4 *>(&skv[0][t][sub * 8]), k1 = *reinterpret_cast<const float4 *>(&skv[0][t][sub * 8 + 4]);
                    const float4 v0 = *reinterpret_cast<const float4 *>(&skv[1][t][sub * 8]), v1 = *reinterpret_cast<const float4 *>(&skv[1][t][sub * 8 + 4]);
                    const float kt[8] = {k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w}, vt[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                    for (int e = 0; e < 8; ++e) { sx = fmaf(qv[e], kt[e], sx); pd = fmaf(gv[e], vt[e], pd); }
#pragma unroll
                    for (int o = 4; o > 0; o >>= 1) {
                        sx += __shfl_xor_sync(0xffffffffu, sx, o);
                        pd += __shfl_xor_sync(0xffffffffu, pd, o);
                    }
                    const float p = live ? ex2_approx(fmaf(sx, c, -lq[ps])) : 0.f;
                    const float ds = p * (pd - dl);
#pragma unroll
                    for (int e = 0; e < 8; ++e) { aV[t][e] = fmaf(p, gv[e], aV[t][e]); aK[t][e] = fmaf(ds, qv[e], aK[t][e]); }
                    if (sub == 0 && live) dsT[((size_t)bh * N + n) * NT + t] = ds;
                }
            }
        }
    }
    if constexpr (NT > 0) {
        // the 4 row slots of a warp share `sub`: xor-shuffle over 8, 16; then the 8 warps' partials through shared memory (plain
        // stores: shared-memory float atomics are CAS loops, and 8 warps on the same 128 words serialise badly)
        const int warp = threadIdx.x >> 5;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float a = aK[t][e], v = aV[t][e];
                a += __shfl_xor_sync(0xffffffffu, a, 8);  v += __shfl_xor_sync(0xffffffffu, v, 8);
                a += __shfl_xor_sync(0xffffffffu, a, 16); v += __shfl_xor_sync(0xffffffffu, v, 16);
                if (lane < 8) { red[warp][0][t][sub * 8 + e] = a; red[warp][1][t][sub * 8 + e] = v; }
            }
        }
        __syncthreads();
        // dK (scaled) / dV rows of the tail keys -> packed gradient (+ their share of the qkv-bias gradient: sums of the ROUNDED values)
        if (threadIdx.x < 2 * AT_D) {
            const int which = threadIdx.x / AT_D, d = threadIdx.x - which * AT_D;
            float bsum = 0.f;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                float sum = 0.f;
#pragma unroll
                for (int w8 = 0; w8 < 8; ++w8) sum += red[w8][which][t][d];
                const __nv_bfloat16 val = __float2bfloat16(sum * (which == 0 ? scale : 1.0f));
                dqkv[((size_t)b * N + n0 + t) * W + (size_t)(1 + which) * H * AT_D + h * AT_D + d] = val;
                bsum += __bfloat162float(val);
            }
            if (g_bias) atomicAdd(g_bias + (size_t)(1 + which) * H * AT_D + h * AT_D + d, bsum);
        }
    }
}

// dq_acc fp32 [B*H][N][64] (+ the tail keys' contribution sum_t ds[q][t] k_t) * scale -> dqkv[b][n][0][h][:] bf16 ; optionally the
// q-part of the qkv-bias gradient (column sums of the rounded values).  grid = (ceil(N / 128), B*H), 256 threads = 32 rows x 8
// column groups, four row passes with the loads issued up front: a block never mixes heads.
constexpr int AB_CONV_ROWS = 128;

__global__ void __launch_bounds__(256)
attn_dq_convert_kernel(const float *__restrict__ dq_acc, const __nv_bfloat16 *__restrict__ qkv, const float *__restrict__ dsT,
                       __nv_bfloat16 *__restrict__ dqkv, float *__restrict__ g_bias, int N, int H, int n0, int nt, float scale) {
    __shared__ float red[8][AT_D];
    __shared__ float skt[AB_KTAIL_MAX][AT_D];
    const int part = threadIdx.x & 7, rloc = threadIdx.x >> 3;
    const int bhh = blockIdx.y;
    const int hh = bhh % H, bb = bhh / H;
    constexpr int PASSES = AB_CONV_ROWS / 32;
    float4 x0[PASSES], x1[PASSES];
#pragma unroll
    for (int ps = 0; ps < PASSES; ++ps) {
        const int n = blockIdx.x * AB_CONV_ROWS + ps * 32 + rloc;
        const size_t rowid = (size_t)bhh * N + (n < N ? n : N - 1);
        x0[ps] = *reinterpret_cast<const float4 *>(dq_acc + rowid * AT_D + part * 8);
        x1[ps] = *reinterpret_cast<const float4 *>(dq_acc + rowid * AT_D + part * 8 + 4);
    }
    if (nt > 0) {
        for (int i = threadIdx.x; i < nt * AT_D; i += 256) {
            const int t = i / AT_D, d = i - t * AT_D;
            skt[t][d] = __bfloat162float(qkv[(((size_t)bb * N + n0 + t) * 3 * H + H + hh) * AT_D + d]);
        }
        __syncthreads();
    }
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = 0.f;
#pragma unroll
    for (int ps = 0; ps < PASSES; ++ps) {
        const int n = blockIdx.x * AB_CONV_ROWS + ps * 32 + rloc;
        if (n < N) {
            const size_t rowid = (size_t)bhh * N + n;
            float x[8] = {x0[ps].x, x0[ps].y, x0[ps].z, x0[ps].w, x1[ps].x, x1[ps].y, x1[ps].z, x1[ps].w};
            for (int t = 0; t < nt; ++t) {
                const float ds = dsT[rowid * nt + t];
#pragma unroll
                for (int e = 0; e < 8; ++e) x[e] = fmaf(ds, skt[t][part * 8 + e], x[e]);
            }
            uint4 o;
            o.x = pack_bf16(x[0] * scale, x[1] * scale);
            o.y = pack_bf16(x[2] * scale, x[3] * scale);
            o.z = pack_bf16(x[4] * scale, x[5] * scale);
            o.w = pack_bf16(x[6] * scale, x[7] * scale);
            *reinterpret_cast<uint4 *>(dqkv + (((size_t)bb * N + n) * 3 * H + hh) * AT_D + part * 8) = o;
            const uint32_t w[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) { v[2 * e] += __uint_as_float(w[e] << 16); v[2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u); }
        }
    }
    if (!g_bias) return;
    // rows of a warp: lanes with equal `part` are 8 apart -> xor-shuffle over 8, 16; then 8 warps through shared memory
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        v[e] += __shfl_xor_sync(0xffffffffu, v[e], 8);
        v[e] += __shfl_xor_sync(0xffffffffu, v[e], 16);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane < 8) {
#pragma unroll
        for (int e = 0; e < 8; ++e) red[warp][lane * 8 + e] = v[e];
    }
    __syncthreads();
    if (threadIdx.x < AT_D) {
        float acc = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) acc += red[w8][threadIdx.x];
        atomicAdd(g_bias + hh * AT_D + threadIdx.x, acc);
    }
}

struct AttnBwdMaps { CUtensorMap tmQKV, tmDO, tmDQ; };

static bool get_bwd_maps(const void *qkv, const void *dout, void *acc, int B, int N, int H, AttnBwdMaps &m) {
    static MapCache<std::tuple<const void *, const void *, const void *, int, int, int>, AttnBwdMaps> cache;
    return cache.get({qkv, dout, acc, B, N, H}, m, [&](AttnBwdMaps &e) {
        const uint64_t W = (uint64_t)3 * H * AT_D, Wo = (uint64_t)H * AT_D;
        return make_map_3d(&e.tmQKV, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, const_cast<void *>(qkv), W, N, B, W * 2, (uint64_t)N * W * 2, AT_D, AT_BM) &&
               make_map_3d(&e.tmDO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, const_cast<void *>(dout), Wo, N, B, Wo * 2, (uint64_t)N * Wo * 2, AT_D, AT_BM) &&
               make_map_3d(&e.tmDQ, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, acc, AT_D, N, (uint64_t)B * H, AT_D * 4, (uint64_t)N * AT_D * 4, 32, AT_BM);
    });
}

// keys handled by attn_bwd_prep_kernel<NT> instead of a key block of attn_bwd_kernel (0 = none)
static int attn_bwd_ktail(int N) {
    const int r = N % AT_BN;
    return (N > AT_BN && r != 0 && r <= AB_KTAIL_MAX) ? r : 0;
}

static size_t attn_bwd_ws_layout(int B, int N, int H, size_t *off_lse, size_t *off_delta, size_t *off_dst) {
    const size_t Npad = ((size_t)N + AT_BM - 1) / AT_BM * AT_BM;
    const size_t acc = align_up((size_t)B * H * N * AT_D * sizeof(float), 1024);
    const size_t st = align_up((size_t)B * H * Npad * sizeof(float), 1024);
    const size_t dst = align_up((size_t)B * H * N * attn_bwd_ktail(N) * sizeof(float), 1024);    // dsT [B*H][N][nt]
    if (off_lse) *off_lse = acc;
    if (off_delta) *off_delta = acc + st;
    if (off_dst) *off_dst = acc + 2 * st;
    return acc + 2 * st + dst;
}

}  // namespace xq

extern "C" {

#ifdef XQ_ATTN_TRACE
int xq_dev_set_attn_trace(void *dev_ptr) {
    long long *p = (long long *)dev_ptr;
    return cudaMemcpyToSymbol(xq::g_attn_trace, &p, sizeof(p)) == cudaSuccess ? 0 : -3;
}
#endif

size_t xq_vit_attn_bwd_workspace_bytes(int B, int N, int H) {
    if (B <= 0 || N <= 0 || H <= 0) return 0;
    return xq::attn_bwd_ws_layout(B, N, H, nullptr, nullptr, nullptr);
}

int xq_vit_attn_bwd(const void *qkv, const void *out, const void *d_out, const float *lse2, void *dqkv, float *g_bias, int B, int N,
                    int H, int head_dim, float scale, void *workspace, size_t workspace_bytes, void *stream) {
    using namespace xq;
    if (!qkv || !out || !d_out || !lse2 || !dqkv || !workspace || B <= 0 || N <= 0 || H <= 0) return XQ_ERR_ARG;
    if (head_dim != AT_D) return XQ_ERR_UNSUPPORTED;
    if (((uintptr_t)qkv & 15) || ((uintptr_t)out & 15) || ((uintptr_t)d_out & 15) || ((uintptr_t)dqkv & 15) || ((uintptr_t)workspace & 255))
        return XQ_ERR_ARG;
    size_t off_lse, off_delta, off_dst;
    if (workspace_bytes < attn_bwd_ws_layout(B, N, H, &off_lse, &off_delta, &off_dst)) return XQ_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    float *acc = (float *)workspace;
    float *lseP = (float *)((char *)workspace + off_lse);
    float *deltaP = (float *)((char *)workspace + off_delta);
    float *dsT = (float *)((char *)workspace + off_dst);
    AttnBwdMaps m;
    if (!get_bwd_maps(qkv, d_out, acc, B, N, H, m)) return XQ_ERR_UNSUPPORTED;
    const int nt = attn_bwd_ktail(N);                                     // few trailing keys: CUDA-core kernel, not a key block
    const int nK = nt ? N / AT_BN : (N + AT_BN - 1) / AT_BN;
    const int Npad = (N + AT_BM - 1) / AT_BM * AT_BM;
    if ((long long)B * H > 65535) return XQ_ERR_UNSUPPORTED;
    if (g_bias) XQ_CUDA_TRY(cudaMemsetAsync(g_bias, 0, (size_t)3 * H * AT_D * sizeof(float), st));
    const float c2 = scale * 1.4426950408889634f;
    AttnDevState *ds = nullptr;
    if (int rc = attn_dev_state(&ds)) return rc;
    {
        dim3 grid(nt ? 1u : (unsigned)(Npad / AB_PREP_ROWS), (unsigned)(B * H));
        const __nv_bfloat16 *qp = (const __nv_bfloat16 *)qkv, *op = (const __nv_bfloat16 *)out, *gp = (const __nv_bfloat16 *)d_out;
        __nv_bfloat16 *dp = (__nv_bfloat16 *)dqkv;
        constexpr int PS = 2 * 3 * (AB_PREP_ROWS / 32) * 256 * 16;             // the NT > 0 variants' two-stage row buffer
        if (!ds->prep_attr) {
            XQ_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_prep_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS));
            XQ_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_prep_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS));
            XQ_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_prep_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS));
            XQ_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_prep_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS));
            ds->prep_attr = true;
        }
        switch (nt) {
        case 0: attn_bwd_prep_kernel<0><<<grid, 256, 0, st>>>(qp, op, gp, lse2, lseP, deltaP, acc, dsT, dp, g_bias, N, H, Npad, c2, scale); break;
        case 1: attn_bwd_prep_kernel<1><<<grid, 256, PS, st>>>(qp, op, gp, lse2, lseP, deltaP, acc, dsT, dp, g_bias, N, H, Npad, c2, scale); break;
        case 2: attn_bwd_prep_kernel<2><<<grid, 256, PS, st>>>(qp, op, gp, lse2, lseP, deltaP, acc, dsT, dp, g_bias, N, H, Npad, c2, scale); break;
        case 3: attn_bwd_prep_kernel<3><<<grid, 256, PS, st>>>(qp, op, gp, lse2, lseP, deltaP, acc, dsT, dp, g_bias, N, H, Npad, c2, scale); break;
        default: attn_bwd_prep_kernel<4><<<grid, 256, PS, st>>>(qp, op, gp, lse2, lseP, deltaP, acc, dsT, dp, g_bias, N, H, Npad, c2, scale); break;
        }
        XQ_LAUNCH_CHECK("attn_bwd_prep_kernel");
    }
    const size_t smem = AttnBwdSmem::BYTES + 1024;
    if (!ds->bwd_attr) {
        XQ_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ds->bwd_attr = true;
    }
    const long long items = (long long)B * H * nK;          // (batch*head, key block) work items of the persistent grid
    if (items > 0x7fffffffLL) return XQ_ERR_ARG;
    int n_sm = 0;
    XQ_CUDA_TRY(sm_count(&n_sm));
    const unsigned ctas = (unsigned)(items < n_sm ? items : n_sm);
    attn_bwd_kernel<<<ctas, AB_THREADS, smem, st>>>(m.tmQKV, m.tmDO, m.tmDQ, lseP, deltaP, (__nv_bfloat16 *)dqkv, g_bias, N, H, nK, Npad,
                                                    (int)items, c2, scale);
    XQ_LAUNCH_CHECK("attn_bwd_kernel");
    {
        dim3 grid((unsigned)((N + AB_CONV_ROWS - 1) / AB_CONV_ROWS), (unsigned)(B * H));
        attn_dq_convert_kernel<<<grid, 256, 0, st>>>(acc, (const __nv_bfloat16 *)qkv, dsT, (__nv_bfloat16 *)dqkv, g_bias, N, H, N - nt, nt, scale);
        XQ_LAUNCH_CHECK("attn_dq_convert_kernel");
    }
    return XQ_OK;
}

int xq_vit_attn_fwd(const void *qkv, void *out, float *lse2, int B, int N, int H, int head_dim, float scale, void *stream) {
    using namespace xq;
    if (!qkv || !out || !lse2 || B <= 0 || N <= 0 || H <= 0) return XQ_ERR_ARG;
    if (head_dim != AT_D) return XQ_ERR_UNSUPPORTED;
    if (((uintptr_t)qkv & 15) || ((uintptr_t)out & 15)) return XQ_ERR_ARG;
    AttnMaps m;
    if (!get_fwd_maps(qkv, out, B, N, H, m)) return XQ_ERR_UNSUPPORTED;
    const int nQ = (N + AT_BM - 1) / AT_BM;      // query tiles; the last one may be ragged
    const size_t smem = AttnFwdSmem::BYTES + 1024;
    AttnDevState *ds = nullptr;
    if (int rc = attn_dev_state(&ds)) return rc;
    int n_sm = 0;
    XQ_CUDA_TRY(sm_count(&n_sm));
    if (!ds->fwd_attr) {
        XQ_CUDA_TRY(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ds->fwd_attr = true;
    }
    const long long tiles = (long long)B * H * nQ;
    if (tiles > 0x7fffffffLL) return XQ_ERR_ARG;
    const int grid = (int)(tiles < 2LL * n_sm ? tiles : 2LL * n_sm);
    const float c = scale * 1.4426950408889634f;
    attn_fwd_kernel<<<grid, AT_THREADS, smem, (cudaStream_t)stream>>>(m.tmQKV, m.tmO, lse2, N, H, nQ, (int)tiles, c);
    XQ_LAUNCH_CHECK("attn_fwd_kernel");
    return XQ_OK;
}

}  // extern "C"
