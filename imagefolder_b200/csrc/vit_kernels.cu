// vit_kernels.cu -- HBM-bound glue kernels of the ViT encoder/decoder blocks (sm_100a).
//
// The reference block (dino_enc/vision_transformer.py:336-339) is
//     x = x + drop_path(ls1(attn(norm1(x))));   x = x + drop_path(ls2(mlp(norm2(x))))
// with the residual stream in fp32 and GEMM operands in bf16 under autocast.  Eager PyTorch spends
// one kernel per arrow (LayerNorm, cast, LayerScale mul, DropPath mul, add, GELU ...), each a full
// HBM round trip.  Here the whole non-GEMM glue between two GEMMs is ONE pass:
//
//   residual_ln_fwd : x_new = x + rowscale[b] * gamma_ls[d] * branch[m,d]      (fp32 stream, bf16 branch)
//                     y     = LayerNorm(x_new) * w + b  -> bf16 (next GEMM operand), mean / rstd saved
//   residual_ln_bwd : G = g_xnew + LN^T(g_y);  g_branch = G * rowscale * gamma_ls -> bf16;
//                     d ln_w, d ln_b, d gamma_ls column sums (per-CTA partials, reduced deterministically)
//   gelu_fwd / gelu_bwd : exact (erf) GELU on bf16, 16-byte vectors
//
// Algorithmic bytes per element (row x channel): fwd 4 (x) + 2 (branch) + 4 (x_new) + 2 (y) = 12 B;
// bwd 4 (g_xnew) + 2 (g_y) + 4 (x_new) + 2 (branch) + 4 (G) + 2 (g_branch) = 18 B.
// These TUs do not carry index decisions, so they are built with the default -fmad=true.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/xqb200.h"
#include "xq_gelu.cuh"
#include "xq_tc.cuh"

namespace xqv {
using namespace xqtc;

constexpr int WARPS = 8;
constexpr int THREADS = WARPS * 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct bf16x4 { __nv_bfloat162 a, b; };

__device__ __forceinline__ float4 load_bf16x4(const __nv_bfloat16 *p) {
    bf16x4 v = *reinterpret_cast<const bf16x4 *>(p);
    float2 lo = __bfloat1622float2(v.a), hi = __bfloat1622float2(v.b);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ void store_bf16x4(__nv_bfloat16 *p, float4 f) {
    bf16x4 v;
    v.a = __floats2bfloat162_rn(f.x, f.y);
    v.b = __floats2bfloat162_rn(f.z, f.w);
    *reinterpret_cast<bf16x4 *>(p) = v;
}

// One warp handles FR = 2 rows (loads of both issued before any arithmetic); NV = D / 128 float4 chunks per lane.
//   x_new = x + rowscale * gamma_ls * (branch + branch_bias)
constexpr int FR = 2;
template <int NV>
__global__ void __launch_bounds__(THREADS)
residual_ln_fwd_kernel(const float *__restrict__ x, const __nv_bfloat16 *__restrict__ branch,
                       const float *__restrict__ branch_bias, const float *__restrict__ ls_gamma,
                       const float *__restrict__ rowscale, int rows_per_sample, const float *__restrict__ ln_w,
                       const float *__restrict__ ln_b, float eps, int M, float *__restrict__ x_out,
                       __nv_bfloat16 *__restrict__ y, float *__restrict__ mean_out, float *__restrict__ rstd_out) {
    constexpr int D = NV * 128;
    const int lane = threadIdx.x & 31;
    const int rbase = (blockIdx.x * WARPS + (threadIdx.x >> 5)) * FR;
    if (rbase >= M) return;
    float4 v[FR][NV], bv[FR][NV];
    bool ok[FR];
#pragma unroll
    for (int u = 0; u < FR; ++u) {
        ok[u] = rbase + u < M;
        const size_t base = (size_t)(ok[u] ? rbase + u : rbase) * D;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int col = (i * 32 + lane) * 4;
            v[u][i] = *reinterpret_cast<const float4 *>(x + base + col);
            bv[u][i] = branch ? load_bf16x4(branch + base + col) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
#pragma unroll
    for (int u = 0; u < FR; ++u) {
        if (!ok[u]) continue;
        const int row = rbase + u;
        const size_t base = (size_t)row * D;
        if (branch) {
            const float s = rowscale ? rowscale[row / rows_per_sample] : 1.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int col = (i * 32 + lane) * 4;
                float4 b = bv[u][i];
                if (branch_bias) {
                    float4 bb = *reinterpret_cast<const float4 *>(branch_bias + col);
                    b.x += bb.x; b.y += bb.y; b.z += bb.z; b.w += bb.w;
                }
                float4 g = ls_gamma ? *reinterpret_cast<const float4 *>(ls_gamma + col) : make_float4(1.f, 1.f, 1.f, 1.f);
                v[u][i].x += s * g.x * b.x; v[u][i].y += s * g.y * b.y; v[u][i].z += s * g.z * b.z; v[u][i].w += s * g.w * b.w;
            }
        }
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) sum += v[u][i].x + v[u][i].y + v[u][i].z + v[u][i].w;
        const float mean = warp_sum(sum) * (1.f / D);
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            float a = v[u][i].x - mean, b = v[u][i].y - mean, c = v[u][i].z - mean, d = v[u][i].w - mean;
            sq += a * a + b * b + c * c + d * d;
        }
        const float rstd = rsqrtf(warp_sum(sq) * (1.f / D) + eps);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int col = (i * 32 + lane) * 4;
            if (x_out) *reinterpret_cast<float4 *>(x_out + base + col) = v[u][i];
            if (y) {
                float4 w = *reinterpret_cast<const float4 *>(ln_w + col);
                float4 b = *reinterpret_cast<const float4 *>(ln_b + col);
                float4 o;
                o.x = (v[u][i].x - mean) * rstd * w.x + b.x; o.y = (v[u][i].y - mean) * rstd * w.y + b.y;
                o.z = (v[u][i].z - mean) * rstd * w.z + b.z; o.w = (v[u][i].w - mean) * rstd * w.w + b.w;
                store_bf16x4(y + base + col, o);
            }
        }
        if (lane == 0 && mean_out) { mean_out[row] = mean; rstd_out[row] = rstd; }
    }
}

// ---- TMA-bulk staged streaming skeleton -------------------------------------------------------------------------
// tools/mb/stream_mb.cu (B200): a persistent 1-CTA-per-SM kernel whose producer warp stages row tiles into shared memory
// with 1-D bulk copies (bulk_g2s, completing on an mbarrier) and whose consumer warps each own one row of the tile, with tiles
// handed out by an atomic counter, streams at 6.7-6.8 TB/s INCLUDING register-resident column sums -- the same rate as a
// flat copy -- where the best register-load loop (grid-stride, software-pipelined) reaches 5.7-6.0 and the previous
// warp-per-row LayerNorm backward 4.5.  No registers are spent on loads in flight and the memory system always has
// NST-1 tiles outstanding.

// Backward.  grid = #SMs, 1 CTA / SM, warp 0 = producer, LNB_TR consumer warps (one tile row each), LNB_NST stages.
// Stage layout: x_out [TR][D] f32 | g_xout [TR][D] f32 | g_y [TR][D] bf16 | branch [TR][D] bf16 | mean, rstd, scale [TR].
// A lane owns columns (i*32 + lane)*4 .. +3, i < NV, for EVERY row it sees, so ln_w / ls_gamma and the four column
// partial sums (d ln_w, d ln_b, sum G*s*branch, sum G*s) live in registers for the whole kernel.
//   g_xout may be null (no later residual gradient), g_y may be null (LN output unused).
constexpr int NACC = 4;
constexpr int LNB_TR = 8;
constexpr int LNB_THREADS = (LNB_TR + 1) * 32;
__host__ __device__ inline size_t lnb_stage_bytes(int D) { return (size_t)LNB_TR * D * 12 + 128; }
__host__ __device__ inline int lnb_stages(int D) { return lnb_stage_bytes(D) * 3 <= 225 * 1024 ? 3 : 2; }

template <int NV>
__global__ void __launch_bounds__(LNB_THREADS, 1)
residual_ln_bwd_kernel(const float *__restrict__ g_xout, const __nv_bfloat16 *__restrict__ g_y,
                       const float *__restrict__ x_out, const float *__restrict__ mean_in,
                       const float *__restrict__ rstd_in, const float *__restrict__ ln_w,
                       const __nv_bfloat16 *__restrict__ branch, const float *__restrict__ branch_bias,
                       const float *__restrict__ ls_gamma, const float *__restrict__ rowscale, int rows_per_sample,
                       int M, float *__restrict__ g_x, __nv_bfloat16 *__restrict__ g_branch,
                       float *__restrict__ part, int *__restrict__ counter, int nst) {
    constexpr int D = NV * 128;
    constexpr int TR = LNB_TR;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full[3], empty[3];
    __shared__ int tile_of[3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (M + TR - 1) / TR;
    const size_t stage_bytes = lnb_stage_bytes(D);
    auto st_x = [&](int st) { return reinterpret_cast<float *>(smem + st * stage_bytes); };
    auto st_r = [&](int st) { return reinterpret_cast<float *>(smem + st * stage_bytes + (size_t)TR * D * 4); };
    auto st_gy = [&](int st) { return reinterpret_cast<__nv_bfloat16 *>(smem + st * stage_bytes + (size_t)TR * D * 8); };
    auto st_br = [&](int st) { return reinterpret_cast<__nv_bfloat16 *>(smem + st * stage_bytes + (size_t)TR * D * 10); };
    auto st_sc = [&](int st) { return reinterpret_cast<float *>(smem + st * stage_bytes + (size_t)TR * D * 12); };
    if (threadIdx.x == 0) {
        for (int i = 0; i < nst; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], TR); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ---------------- producer ----------------
        for (int it = 0;; ++it) {
            const int st = it % nst;
            mbar_wait(&empty[st], ((it / nst) & 1) ^ 1);
            int tile = 0;
            if (lane == 0) tile = it == 0 ? (int)blockIdx.x : (int)gridDim.x + atomicAdd(counter, 1);
            tile = __shfl_sync(0xffffffffu, tile, 0);
            if (tile >= ntiles) {
                if (lane == 0) { tile_of[st] = tile; mbar_arrive(&full[st]); mbar_arrive(&full[st]); }
                break;
            }
            const int r0 = tile * TR, nr = min(TR, M - r0);
            if (lane == 0) {
                tile_of[st] = tile;
                const uint32_t b4 = (uint32_t)nr * D * 4, b2 = (uint32_t)nr * D * 2;
                mbar_expect_tx(&full[st], b4 + (g_xout ? b4 : 0) + (g_y ? b2 : 0) + (branch ? b2 : 0));
                bulk_g2s(st_x(st), x_out + (size_t)r0 * D, b4, &full[st]);
                if (g_y) bulk_g2s(st_gy(st), g_y + (size_t)r0 * D, b2, &full[st]);
                if (g_xout) bulk_g2s(st_r(st), g_xout + (size_t)r0 * D, b4, &full[st]);
                if (branch) bulk_g2s(st_br(st), branch + (size_t)r0 * D, b2, &full[st]);
            }
            if (lane < nr) {
                float *sc = st_sc(st);
                sc[lane] = mean_in[r0 + lane];
                sc[TR + lane] = rstd_in[r0 + lane];
                sc[2 * TR + lane] = (branch && rowscale) ? rowscale[(r0 + lane) / rows_per_sample] : 1.f;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[st]);
        }
    } else {
        // ---------------- consumers ----------------
        const int cw = warp - 1;
        float4 w4[NV], gm4[NV], a0[NV], a1[NV], a2[NV], a3[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int col = (i * 32 + lane) * 4;
            w4[i] = g_y ? *reinterpret_cast<const float4 *>(ln_w + col) : make_float4(0.f, 0.f, 0.f, 0.f);
            gm4[i] = (branch && ls_gamma) ? *reinterpret_cast<const float4 *>(ls_gamma + col) : make_float4(1.f, 1.f, 1.f, 1.f);
            a0[i] = a1[i] = a2[i] = a3[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int it = 0;; ++it) {
            const int st = it % nst;
            mbar_wait(&full[st], (it / nst) & 1);
            const int tile = tile_of[st];
            if (tile >= ntiles) break;
            const int row = tile * TR + cw;
            if (row < M) {
                const float *sc = st_sc(st);
                const float mean = sc[cw], rstd = sc[TR + cw], s_row = sc[2 * TR + cw];
                const float *xs = st_x(st) + (size_t)cw * D;
                const float *rs = st_r(st) + (size_t)cw * D;
                const __nv_bfloat16 *gys = st_gy(st) + (size_t)cw * D;
                const __nv_bfloat16 *brs = st_br(st) + (size_t)cw * D;
                // two passes over the row in SHARED memory (x-hat and g*w are recomputed in pass 2 instead of being kept
                // in 48 more registers; shared-memory bandwidth is nowhere near binding here)
                float c1 = 0.f, c2 = 0.f;
                if (g_y) {
#pragma unroll
                    for (int i = 0; i < NV; ++i) {
                        const int col = (i * 32 + lane) * 4;
                        const float4 xv = *reinterpret_cast<const float4 *>(xs + col);
                        const float4 xh = make_float4((xv.x - mean) * rstd, (xv.y - mean) * rstd, (xv.z - mean) * rstd,
                                                      (xv.w - mean) * rstd);
                        const float4 g = load_bf16x4(gys + col);
                        a0[i].x += g.x * xh.x; a0[i].y += g.y * xh.y; a0[i].z += g.z * xh.z; a0[i].w += g.w * xh.w;
                        a1[i].x += g.x; a1[i].y += g.y; a1[i].z += g.z; a1[i].w += g.w;
                        const float4 gw = make_float4(g.x * w4[i].x, g.y * w4[i].y, g.z * w4[i].z, g.w * w4[i].w);
                        c1 += gw.x + gw.y + gw.z + gw.w;
                        c2 += gw.x * xh.x + gw.y * xh.y + gw.z * xh.z + gw.w * xh.w;
                    }
                    c1 = warp_sum(c1) * (1.f / D);
                    c2 = warp_sum(c2) * (1.f / D);
                }
                const size_t base = (size_t)row * D;
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const int col = (i * 32 + lane) * 4;
                    float4 G = g_xout ? *reinterpret_cast<const float4 *>(rs + col) : make_float4(0.f, 0.f, 0.f, 0.f);
                    if (g_y) {
                        const float4 xv = *reinterpret_cast<const float4 *>(xs + col);
                        const float4 xh = make_float4((xv.x - mean) * rstd, (xv.y - mean) * rstd, (xv.z - mean) * rstd,
                                                      (xv.w - mean) * rstd);
                        const float4 g = load_bf16x4(gys + col);
                        G.x += rstd * (g.x * w4[i].x - c1 - xh.x * c2);
                        G.y += rstd * (g.y * w4[i].y - c1 - xh.y * c2);
                        G.z += rstd * (g.z * w4[i].z - c1 - xh.z * c2);
                        G.w += rstd * (g.w * w4[i].w - c1 - xh.w * c2);
                    }
                    if (g_x) *reinterpret_cast<float4 *>(g_x + base + col) = G;
                    if (branch) {
                        const float4 bv = load_bf16x4(brs + col);
                        const float4 Gs = make_float4(G.x * s_row, G.y * s_row, G.z * s_row, G.w * s_row);
                        a2[i].x += Gs.x * bv.x; a2[i].y += Gs.y * bv.y; a2[i].z += Gs.z * bv.z; a2[i].w += Gs.w * bv.w;
                        a3[i].x += Gs.x; a3[i].y += Gs.y; a3[i].z += Gs.z; a3[i].w += Gs.w;
                        if (g_branch)
                            store_bf16x4(g_branch + base + col,
                                         make_float4(Gs.x * gm4[i].x, Gs.y * gm4[i].y, Gs.z * gm4[i].z, Gs.w * gm4[i].w));
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
        }
        // park the register sums in the stage memory -- but only once EVERY consumer warp is past its last real tile
        // (a fast warp sees the sentinel while a slow one still reads its row): named barrier over the consumer warps
        asm volatile("bar.sync 1, %0;" ::"n"(LNB_TR * 32) : "memory");
        float *red = reinterpret_cast<float *>(smem) + (size_t)cw * NACC * D;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int col = (i * 32 + lane) * 4;
            *reinterpret_cast<float4 *>(red + 0 * D + col) = a0[i];
            *reinterpret_cast<float4 *>(red + 1 * D + col) = a1[i];
            *reinterpret_cast<float4 *>(red + 2 * D + col) = a2[i];
            *reinterpret_cast<float4 *>(red + 3 * D + col) = a3[i];
        }
    }
    __syncthreads();
    const float *red = reinterpret_cast<const float *>(smem);
    float *outp = part + (size_t)blockIdx.x * NACC * D;
    for (int e = threadIdx.x; e < NACC * D; e += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < TR; ++w) a += red[(size_t)w * NACC * D + e];
        outp[e] = a;
    }
}

// sums the CTA partials and finishes the four vectors:
//   d ln_w = P0 ; d ln_b = P1 ; d gamma_ls = P2 + bias * P3 ; d branch_bias = gamma_ls * P3
// one thread per column, 8 independent loads in flight per accumulator (the serial version was latency-bound)
__global__ void reduce_parts_kernel(const float *__restrict__ part, int nblocks, int D, const float *__restrict__ ls_gamma,
                                    const float *__restrict__ branch_bias, float *__restrict__ g_ln_w,
                                    float *__restrict__ g_ln_b, float *__restrict__ g_ls_gamma,
                                    float *__restrict__ g_branch_bias) {
    __shared__ float sh[NACC][8][32];
    const int lane = threadIdx.x & 31, sub = threadIdx.x >> 5;       // 8 sub-ranges of the block list per column
    const int d = blockIdx.x * 32 + lane;
    float p[NACC] = {0.f, 0.f, 0.f, 0.f};
    if (d < D) {
        for (int b = sub; b < nblocks; b += 8) {
#pragma unroll
            for (int q = 0; q < NACC; ++q) p[q] += part[((size_t)b * NACC + q) * D + d];
        }
    }
#pragma unroll
    for (int q = 0; q < NACC; ++q) sh[q][sub][lane] = p[q];
    __syncthreads();
    if (sub == 0 && d < D) {
#pragma unroll
        for (int q = 0; q < NACC; ++q) {
            float a = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) a += sh[q][w][lane];
            p[q] = a;
        }
        if (g_ln_w) g_ln_w[d] = p[0];
        if (g_ln_b) g_ln_b[d] = p[1];
        if (g_ls_gamma) g_ls_gamma[d] = p[2] + (branch_bias ? branch_bias[d] * p[3] : 0.f);
        if (g_branch_bias) g_branch_bias[d] = (ls_gamma ? ls_gamma[d] : 1.f) * p[3];
    }
}

// erf via Abramowitz-Stegun 7.1.28:  erf(a) = 1 - (1 + a1 a + ... + a6 a^6)^-16,  |abs err| <= 3e-7 (far below the bf16
// output rounding).  ONE special-function op (the reciprocal) per element -- the 7.1.26 form used before needed exp and
// reciprocal, and the kernel was bound by the 16-lane/clk MUFU pipe, not by HBM.
__device__ __forceinline__ float erf_as(float z) {
    const float a = fabsf(z);
    float p = fmaf(a, 0.0000430638f, 0.0002765672f);
    p = fmaf(p, a, 0.0001520143f);
    p = fmaf(p, a, 0.0092705272f);
    p = fmaf(p, a, 0.0422820123f);
    p = fmaf(p, a, 0.0705230784f);
    p = fmaf(p, a, 1.0f);
    p = p * p; p = p * p; p = p * p; p = p * p;          // ^16 (overflows to +inf for |z| > ~9 -> erf = 1, as it should)
    return copysignf(1.0f - rcp_fast(p), z);
}
// y = gelu(x + bias).  A thread owns column chunk c (8 bf16 = 16 B) and walks rows with a grid stride, RU rows
// per iteration so that RU independent 16-byte loads are in flight (one load per iteration leaves HBM idle).
constexpr int GELU_RU = 4;
__device__ __forceinline__ void load_bias8(const float *bias, int c, float (&bb)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) bb[k] = 0.f;
    if (bias) {
        float4 b0 = *reinterpret_cast<const float4 *>(bias + c * 8), b1 = *reinterpret_cast<const float4 *>(bias + c * 8 + 4);
        bb[0] = b0.x; bb[1] = b0.y; bb[2] = b0.z; bb[3] = b0.w; bb[4] = b1.x; bb[5] = b1.y; bb[6] = b1.z; bb[7] = b1.w;
    }
}
__global__ void gelu_fwd_kernel(const uint4 *__restrict__ x, const float *__restrict__ bias, uint4 *__restrict__ y,
                                int M, int C8) {
    // NON-persistent: one CTA per GELU_RU rows.  tools/mb/stream_mb.cu on B200: fresh small CTAs stream at 6.1 TB/s where
    // the persistent grid-stride form of the same loop reaches 5.4 (lock-step load/store phases + SM imbalance).
    const int row0 = blockIdx.x * GELU_RU;
    for (int c = threadIdx.x; c < C8; c += blockDim.x) {
        float bb[8];
        load_bias8(bias, c, bb);
        uint4 v[GELU_RU];
#pragma unroll
        for (int u = 0; u < GELU_RU; ++u)
            if (row0 + u < M) v[u] = x[(size_t)(row0 + u) * C8 + c];
#pragma unroll
        for (int u = 0; u < GELU_RU; ++u) {
            if (row0 + u >= M) continue;
            __nv_bfloat162 *p = reinterpret_cast<__nv_bfloat162 *>(&v[u]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float2 f = __bfloat1622float2(p[k]);
                p[k] = __floats2bfloat162_rn(gelu_f(f.x + bb[2 * k]), gelu_f(f.y + bb[2 * k + 1]));
            }
            y[(size_t)(row0 + u) * C8 + c] = v[u];
        }
    }
}

// gx = gy * gelu'(x + bias); column sums of gx (= d bias) accumulate per thread, one atomicAdd per column
// per CTA at the end (g_bias must be zeroed by the caller).
constexpr int GELU_BWD_RU = 2;
__global__ void gelu_bwd_kernel(const uint4 *__restrict__ x, const float *__restrict__ bias, const uint4 *__restrict__ gy,
                                uint4 *__restrict__ gx, float *__restrict__ g_bias, int M, int C8) {
    // persistent (the column sums stay in registers, one atomicAdd per column per CTA) and SOFTWARE-PIPELINED: the loads
    // of iteration i+1 are issued before the math / stores of iteration i, so a warp always has loads in flight.
    constexpr int RU = GELU_BWD_RU;
    const int step = gridDim.x * RU;
    for (int c = threadIdx.x; c < C8; c += blockDim.x) {
        float bb[8], acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        load_bias8(bias, c, bb);
        uint4 v[RU], g[RU], vn[RU], gn[RU];
        int row0 = blockIdx.x * RU;
#pragma unroll
        for (int u = 0; u < RU; ++u)
            if (row0 + u < M) { v[u] = x[(size_t)(row0 + u) * C8 + c]; g[u] = gy[(size_t)(row0 + u) * C8 + c]; }
        for (; row0 < M; row0 += step) {
            const int nxt = row0 + step;
#pragma unroll
            for (int u = 0; u < RU; ++u)
                if (nxt + u < M) { vn[u] = x[(size_t)(nxt + u) * C8 + c]; gn[u] = gy[(size_t)(nxt + u) * C8 + c]; }
#pragma unroll
            for (int u = 0; u < RU; ++u) {
                if (row0 + u >= M) continue;
                __nv_bfloat162 *p = reinterpret_cast<__nv_bfloat162 *>(&v[u]);
                __nv_bfloat162 *q = reinterpret_cast<__nv_bfloat162 *>(&g[u]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float2 f = __bfloat1622float2(p[k]), h = __bfloat1622float2(q[k]);
                    float r0 = h.x * dgelu_f(f.x + bb[2 * k]), r1 = h.y * dgelu_f(f.y + bb[2 * k + 1]);
                    acc[2 * k] += r0; acc[2 * k + 1] += r1;
                    p[k] = __floats2bfloat162_rn(r0, r1);
                }
                gx[(size_t)(row0 + u) * C8 + c] = v[u];
            }
#pragma unroll
            for (int u = 0; u < RU; ++u) { v[u] = vn[u]; g[u] = gn[u]; }
        }
        if (g_bias) {
#pragma unroll
            for (int k = 0; k < 8; ++k) atomicAdd(g_bias + c * 8 + k, acc[k]);
        }
    }
}

// dq, dk, dv: each [M, C] bf16 dense (what the SDPA backward returns for q/k/v views of a packed
// [M, 3C] projection) -> dqkv [M, 3C], and (optionally) g_bias [3C] = column sums of dqkv = the gradient of the
// qkv projection bias, which autograd would otherwise compute with one more full pass over dqkv.
// Same TMA-bulk staged skeleton as residual_ln_bwd_kernel: warp 0 stages PACK_TR rows of the three sources per tile,
// consumer warp w copies row w (a lane owns 16-byte column chunks j*32 + lane of the PACKED row) and keeps the column
// sums in registers; one atomicAdd per column per CTA at the end (g_bias zeroed by the launcher).
constexpr int PACK_TR = 8;
constexpr int PACK_NST = 4;
constexpr int PACK_NCH = 12;                 // 16-byte chunks per lane: 3*C/8 <= 384  (C <= 1024)
constexpr int PACK_THREADS = (PACK_TR + 1) * 32;
__global__ void __launch_bounds__(PACK_THREADS, 1)
pack_qkv_kernel(const uint4 *__restrict__ dq, const uint4 *__restrict__ dk, const uint4 *__restrict__ dv,
                uint4 *__restrict__ out, float *__restrict__ g_bias, int *__restrict__ counter, int M, int C8) {
    constexpr int TR = PACK_TR, NST = PACK_NST;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full[NST], empty[NST];
    __shared__ int tile_of[NST];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (M + TR - 1) / TR, per_row = 3 * C8;
    const uint32_t src_row = (uint32_t)C8 * 16;                    // bytes of one source row
    const size_t stage_bytes = (size_t)3 * TR * src_row;           // [3][TR][C8] uint4
    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], TR); }
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0;; ++it) {
                const int st = it % NST;
                mbar_wait(&empty[st], ((it / NST) & 1) ^ 1);
                const int tile = it == 0 ? (int)blockIdx.x : (int)gridDim.x + atomicAdd(counter, 1);
                tile_of[st] = tile;
                if (tile >= ntiles) { mbar_arrive(&full[st]); break; }
                const int r0 = tile * TR, nr = min(TR, M - r0);
                unsigned char *dst = smem + st * stage_bytes;
                mbar_expect_tx(&full[st], 3u * nr * src_row);
                bulk_g2s(dst, dq + (size_t)r0 * C8, nr * src_row, &full[st]);
                bulk_g2s(dst + (size_t)TR * src_row, dk + (size_t)r0 * C8, nr * src_row, &full[st]);
                bulk_g2s(dst + (size_t)2 * TR * src_row, dv + (size_t)r0 * C8, nr * src_row, &full[st]);
            }
        }
    } else {
        const int cw = warp - 1;
        float acc[PACK_NCH][8];
#pragma unroll
        for (int j = 0; j < PACK_NCH; ++j)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[j][k] = 0.f;
        for (int it = 0;; ++it) {
            const int st = it % NST;
            mbar_wait(&full[st], (it / NST) & 1);
            const int tile = tile_of[st];
            if (tile >= ntiles) break;
            const int row = tile * TR + cw;
            if (row < M) {
                const unsigned char *base = smem + st * stage_bytes + (size_t)cw * src_row;
#pragma unroll
                for (int j = 0; j < PACK_NCH; ++j) {
                    const int c = j * 32 + lane;
                    if (c < per_row) {
                        const int which = c / C8, cc = c - which * C8;
                        const uint4 v = *reinterpret_cast<const uint4 *>(base + (size_t)which * TR * src_row + (size_t)cc * 16);
                        out[(size_t)row * per_row + c] = v;
                        if (g_bias) {
                            const __nv_bfloat162 *p = reinterpret_cast<const __nv_bfloat162 *>(&v);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                float2 f = __bfloat1622float2(p[k]);
                                acc[j][2 * k] += f.x; acc[j][2 * k + 1] += f.y;
                            }
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
        }
        if (g_bias) {
            asm volatile("bar.sync 1, %0;" ::"n"(PACK_TR * 32) : "memory");   // every consumer is past its last tile
            float *red = reinterpret_cast<float *>(smem) + (size_t)cw * per_row * 8;
#pragma unroll
            for (int j = 0; j < PACK_NCH; ++j) {
                const int c = j * 32 + lane;
                if (c < per_row)
#pragma unroll
                    for (int k = 0; k < 8; ++k) red[c * 8 + k] = acc[j][k];
            }
        }
    }
    if (g_bias) {
        __syncthreads();
        const float *red = reinterpret_cast<const float *>(smem);
        for (int e = threadIdx.x; e < per_row * 8; e += blockDim.x) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < TR; ++w) t += red[(size_t)w * per_row * 8 + e];
            atomicAdd(g_bias + e, t);
        }
    }
}

// Patch embedding as a GEMM (timm PatchEmbed: Conv2d(kernel = stride = p) -> flatten -> NLC, vision_transformer.py:
// patch_embed): non-overlapping patches make im2col a pure permutation, so the conv is
//   tokens[B*gh*gw, D] = patches[B*gh*gw, Cin*p*p] @ W[D, Cin*p*p]^T + b .
// This kernel writes `patches` in bf16 (GEMM operand) from the fp32 NCHW image: 4 pixels (16 B in, 8 B out) per thread,
// output-major indexing -> fully coalesced stores, 64-byte-segment loads.  (cuDNN's implicit-GEMM for Cin = 3 pads the
// channel dimension to 8 and adds two layout conversions: 4.3 ms per step at B = 256 vs 0.1 ms here + a 0.06 ms GEMM.)
__global__ void patchify_kernel(const float *__restrict__ x, __nv_bfloat16 *__restrict__ out, int Cin, int H, int W, int p,
                                size_t total4) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int p4 = p >> 2, gw = W / p, gh = H / p;
    size_t t = i;
    const int kx4 = (int)(t % p4); t /= p4;
    const int ky = (int)(t % p); t /= p;
    const int c = (int)(t % Cin); t /= Cin;
    const int px = (int)(t % gw); t /= gw;
    const int py = (int)(t % gh); t /= gh;
    const size_t b = t;
    const float4 v = *reinterpret_cast<const float4 *>(x + ((b * Cin + c) * H + (size_t)py * p + ky) * W + (size_t)px * p + kx4 * 4);
    store_bf16x4(out + i * 4, v);
}

// persistent grids = (SM count) x (CTAs of this kernel that are actually co-resident on one SM); 0 if the device query fails
template <typename K>
static int persistent_grid(K kernel, int threads, size_t smem = 0) {
    int sms = 0, per_sm = 1;
    if (sm_count(&sms) != cudaSuccess) return 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    return sms * per_sm;
}

// Token assembly (dinov2.py:151-170 / 318-336): the encoder / decoder build their input sequence as
//   [prefix | image tokens | latent tokens] + positional / level embeddings
// with cat + add + cat + add over [B, T, D] fp32 tensors.  Everything except ONE block of rows (the patch tokens in the
// encoder, the quantised latents in the decoder) is batch-independent, so the sequence is
//   out[b, t, :] = table[t, :] + (t0 <= t < t0 + Ls ? src[b, t - t0, :] : 0)
// where `table` [T, D] is the module's own assembly evaluated once on a zero input of batch 1 (host side, autograd intact).
// fwd: one pass (read src, write out).  bwd: ONE read of g produces d_src (cast to the source dtype) and d_table = sum_b g.
template <typename TS>
__global__ void assemble_fwd_kernel(const TS *__restrict__ src, const float *__restrict__ table, int Ls, int T, int D4, int t0,
                                    float *__restrict__ out, size_t total4) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int d4 = (int)(i % D4);
    const size_t bt = i / D4;
    const int t = (int)(bt % T);
    const size_t b = bt / T;
    float4 v = *reinterpret_cast<const float4 *>(table + ((size_t)t * D4 + d4) * 4);
    if (t >= t0 && t < t0 + Ls) {
        const size_t so = ((b * Ls + (t - t0)) * D4 + d4) * 4;
        float4 sv;
        if (sizeof(TS) == 2) sv = load_bf16x4(reinterpret_cast<const __nv_bfloat16 *>(src) + so);
        else sv = *reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(src) + so);
        v.x += sv.x; v.y += sv.y; v.z += sv.z; v.w += sv.w;
    }
    *reinterpret_cast<float4 *>(out + i * 4) = v;
}

template <typename TS>
__global__ void assemble_bwd_kernel(const float *__restrict__ g, int B, int Ls, int T, int D4, int t0, TS *__restrict__ d_src,
                                    float *__restrict__ d_table) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;      // (t, d4)
    if (i >= T * D4) return;
    const int t = i / D4, d4 = i - t * D4;
    const bool in_src = d_src && t >= t0 && t < t0 + Ls;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t stride = (size_t)T * D4 * 4;
    const float *gp = g + ((size_t)t * D4 + d4) * 4;
    for (int b0 = 0; b0 < B; b0 += 8) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            v[u] = (b0 + u < B) ? *reinterpret_cast<const float4 *>(gp + (size_t)(b0 + u) * stride) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
            if (in_src && b0 + u < B) {
                const size_t so = (((size_t)(b0 + u) * Ls + (t - t0)) * D4 + d4) * 4;
                if (sizeof(TS) == 2) store_bf16x4(reinterpret_cast<__nv_bfloat16 *>(d_src) + so, v[u]);
                else *reinterpret_cast<float4 *>(reinterpret_cast<float *>(d_src) + so) = v[u];
            }
        }
    }
    if (d_table) *reinterpret_cast<float4 *>(d_table + ((size_t)t * D4 + d4) * 4) = acc;
}

}  // namespace xqv

using namespace xqv;

#define XQV_DISPATCH(D, ...)                  \
    switch (D) {                               \
        case 384: { constexpr int NV = 3; __VA_ARGS__; break; }   \
        case 768: { constexpr int NV = 6; __VA_ARGS__; break; }   \
        case 1024: { constexpr int NV = 8; __VA_ARGS__; break; }  \
        default: return XQ_ERR_UNSUPPORTED;    \
    }

extern "C" {

// The TMA-staged kernels (LayerNorm backward, pack) run 1 CTA / SM: their tiles fill the shared memory.
size_t xq_vit_ln_bwd_workspace_bytes(int D) {
    int sms = 0;
    if (sm_count(&sms) != cudaSuccess) return 0;      // xq_vit_residual_ln_bwd reports the error
    return sizeof(float) * (size_t)sms * NACC * D + 256;
}

int xq_vit_residual_ln_fwd(const float *x, const void *branch, const float *branch_bias, const float *ls_gamma,
                           const float *rowscale, int rows_per_sample, const float *ln_w, const float *ln_b, float eps,
                           int M, int D, float *x_out, void *y, float *mean, float *rstd, void *stream) {
    if (!x || M <= 0 || (y && (!ln_w || !ln_b)) || (!x_out && !y)) return XQ_ERR_ARG;
    if (branch && rowscale && rows_per_sample <= 0) return XQ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int grid = (M + WARPS * FR - 1) / (WARPS * FR);
    XQV_DISPATCH(D, (residual_ln_fwd_kernel<NV><<<grid, THREADS, 0, st>>>(
                        x, (const __nv_bfloat16 *)branch, branch_bias, ls_gamma, rowscale, rows_per_sample, ln_w, ln_b,
                        eps, M, x_out, (__nv_bfloat16 *)y, mean, rstd)));
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_residual_ln_bwd(const float *g_xout, const void *g_y, const float *x_out, const float *mean,
                           const float *rstd, const float *ln_w, const void *branch, const float *branch_bias,
                           const float *ls_gamma, const float *rowscale, int rows_per_sample, int M, int D, float *g_x,
                           void *g_branch, float *g_ln_w, float *g_ln_b, float *g_ls_gamma, float *g_branch_bias,
                           void *workspace, size_t workspace_bytes, void *stream) {
    if (!x_out || !mean || !rstd || M <= 0 || !workspace) return XQ_ERR_ARG;
    if (g_y && !ln_w) return XQ_ERR_ARG;
    if (branch && rowscale && rows_per_sample <= 0) return XQ_ERR_ARG;
    int sms = 0;
    if (sm_count(&sms) != cudaSuccess) return XQ_ERR_CUDA;
    if (workspace_bytes < sizeof(float) * (size_t)sms * NACC * D + 256) return XQ_ERR_WORKSPACE;
    const int ntiles = (M + LNB_TR - 1) / LNB_TR;
    const int grid = sms < ntiles ? sms : ntiles;
    cudaStream_t st = (cudaStream_t)stream;
    float *part = (float *)workspace;
    int *counter = (int *)((char *)workspace + sizeof(float) * (size_t)sms * NACC * D);   // dynamic tile counter
    if (cudaMemsetAsync(counter, 0, sizeof(int), st) != cudaSuccess) return XQ_ERR_CUDA;
    const int nst = lnb_stages(D);
    size_t smem = lnb_stage_bytes(D) * nst;
    if (smem < sizeof(float) * (size_t)LNB_TR * NACC * D) smem = sizeof(float) * (size_t)LNB_TR * NACC * D;
    XQV_DISPATCH(D, {
        if (cudaFuncSetAttribute(residual_ln_bwd_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return XQ_ERR_CUDA;
        residual_ln_bwd_kernel<NV><<<grid, LNB_THREADS, smem, st>>>(
            g_xout, (const __nv_bfloat16 *)g_y, x_out, mean, rstd, ln_w, (const __nv_bfloat16 *)branch, branch_bias,
            ls_gamma, rowscale, rows_per_sample, M, g_x, (__nv_bfloat16 *)g_branch, part, counter, nst);
    });
    if (cudaGetLastError() != cudaSuccess) return XQ_ERR_CUDA;
    reduce_parts_kernel<<<(D + 31) / 32, 256, 0, st>>>(part, grid, D, ls_gamma, branch_bias, g_ln_w, g_ln_b,
                                                        branch ? g_ls_gamma : nullptr, branch ? g_branch_bias : nullptr);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

size_t xq_vit_pack_workspace_bytes(void) { return 256; }

int xq_vit_pack_qkv(const void *dq, const void *dk, const void *dv, void *dqkv, float *g_bias, size_t M, int C,
                    void *workspace, size_t workspace_bytes, void *stream) {
    if (!dq || !dk || !dv || !dqkv || M == 0 || M > 0x7fffffffu || C <= 0 || (C & 7) || !workspace) return XQ_ERR_ARG;
    if (workspace_bytes < 256) return XQ_ERR_WORKSPACE;
    if (3 * (C / 8) > PACK_NCH * 32) return XQ_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const int C8 = C / 8;
    int *counter = (int *)workspace;     // dynamic tile counter, reset on the stream before each launch
    if (cudaMemsetAsync(counter, 0, sizeof(int), st) != cudaSuccess) return XQ_ERR_CUDA;
    if (g_bias && cudaMemsetAsync(g_bias, 0, sizeof(float) * 3 * (size_t)C, st) != cudaSuccess) return XQ_ERR_CUDA;
    int sms = 0;
    if (sm_count(&sms) != cudaSuccess) return XQ_ERR_CUDA;
    const int ntiles = (int)((M + PACK_TR - 1) / PACK_TR);
    const int grid = sms < ntiles ? sms : ntiles;
    size_t smem = (size_t)PACK_NST * 3 * PACK_TR * C8 * 16;
    const size_t red = sizeof(float) * (size_t)PACK_TR * 3 * C8 * 8;
    if (smem < red) smem = red;
    if (cudaFuncSetAttribute(pack_qkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return XQ_ERR_CUDA;
    pack_qkv_kernel<<<grid, PACK_THREADS, smem, st>>>((const uint4 *)dq, (const uint4 *)dk, (const uint4 *)dv,
                                                      (uint4 *)dqkv, g_bias, counter, (int)M, C8);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_assemble_fwd(const void *src, int src_is_bf16, const float *table, int B, int Ls, int T, int D, int t0, float *out,
                        void *stream) {
    if (!src || !table || !out || B <= 0 || Ls <= 0 || T <= 0 || D <= 0 || (D & 3) || t0 < 0 || t0 + Ls > T) return XQ_ERR_ARG;
    const size_t total4 = (size_t)B * T * (D / 4);
    const unsigned grid = (unsigned)((total4 + 255) / 256);
    if (src_is_bf16)
        assemble_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16 *)src, table, Ls, T, D / 4, t0, out, total4);
    else
        assemble_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float *)src, table, Ls, T, D / 4, t0, out, total4);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_assemble_bwd(const float *g, int B, int Ls, int T, int D, int t0, void *d_src, int src_is_bf16, float *d_table,
                        void *stream) {
    if (!g || (!d_src && !d_table) || B <= 0 || Ls <= 0 || T <= 0 || D <= 0 || (D & 3) || t0 < 0 || t0 + Ls > T) return XQ_ERR_ARG;
    const int n = T * (D / 4);
    if (src_is_bf16)
        assemble_bwd_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(g, B, Ls, T, D / 4, t0, (__nv_bfloat16 *)d_src, d_table);
    else
        assemble_bwd_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(g, B, Ls, T, D / 4, t0, (float *)d_src, d_table);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_patchify(const float *x, void *patches, int B, int Cin, int H, int W, int p, void *stream) {
    if (!x || !patches || B <= 0 || Cin <= 0 || H <= 0 || W <= 0 || p <= 0) return XQ_ERR_ARG;
    if ((p & 3) || H % p || W % p) return XQ_ERR_UNSUPPORTED;
    const size_t total4 = (size_t)B * Cin * H * W / 4;
    patchify_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, (__nv_bfloat16 *)patches, Cin, H, W,
                                                                                       p, total4);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_gelu_fwd(const void *x, const float *bias, void *y, int M, int C, void *stream) {
    if (!x || !y || M <= 0 || C <= 0 || (C & 7)) return XQ_ERR_ARG;
    int C8 = C / 8;
    int threads = C8 >= 384 ? 384 : (C8 >= 192 ? 192 : 128);
    int grid = (M + GELU_RU - 1) / GELU_RU;
    gelu_fwd_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>((const uint4 *)x, bias, (uint4 *)y, M, C8);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

int xq_vit_gelu_bwd(const void *x, const float *bias, const void *gy, void *gx, float *g_bias, int M, int C, void *stream) {
    if (!x || !gy || !gx || M <= 0 || C <= 0 || (C & 7)) return XQ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int C8 = C / 8;
    int threads = C8 >= 384 ? 384 : (C8 >= 192 ? 192 : 128);
    int grid = persistent_grid(gelu_bwd_kernel, threads);
    if (grid == 0) return XQ_ERR_CUDA;
    if ((M + GELU_BWD_RU - 1) / GELU_BWD_RU < grid) grid = (M + GELU_BWD_RU - 1) / GELU_BWD_RU;
    if (g_bias && cudaMemsetAsync(g_bias, 0, sizeof(float) * (size_t)C, st) != cudaSuccess) return XQ_ERR_CUDA;
    gelu_bwd_kernel<<<grid, threads, 0, st>>>((const uint4 *)x, bias, (const uint4 *)gy, (uint4 *)gx, g_bias, M, C8);
    return cudaGetLastError() == cudaSuccess ? XQ_OK : XQ_ERR_CUDA;
}

}  // extern "C"
