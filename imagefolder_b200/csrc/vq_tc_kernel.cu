// vq_tc_kernel.cu -- tcgen05 / TMEM / TMA version of the fused VQ search (sm_100a).
//
// Same contract and same BIT-EXACT results as vq_search_kernel (vq_kernels.cu), reached differently:
//
//   screening   the -2<z,c> inner products of a 128-row x 256-code tile are computed by ONE thread issuing
//               tf32 tensor-core MMAs (operands in 128B-swizzled shared memory: rows written by the CTA,
//               code tiles streamed by TMA), accumulators in TMEM (2 x 256 columns, double buffered);
//   epilogue    4 warps read their TMEM lanes (32 columns at a time), take the maximum of each
//               32-code group with FMNMX3 trees and remember, per row, the few groups whose maximum is
//               within W of the running maximum (a push is ~10 instructions; no per-element scan);
//   rescoring   only the codes of those groups (1.1 groups per row on average) are re-scored with the
//               canonical fp32 arithmetic (fmaf chain, d = (zz+ee) - 2 dot, first index on ties) -> the index
//               equals the exact kernel's and the oracle's: the true argmin provably lies in a kept group.
//
// Error bound (codebook_norm=1, |z| = |c| = 1 up to 1e-6): TF32 operands carry <= 2^-10 relative error
// each, so |dot_tf32 - dot| <= 2^-9 * sum|z_k c_k| <= 1.96e-3.  We use eps = 2.5e-3 and keep every code with
// score >= running_max - (2 eps + 2e-6)  (the 2e-6 covers the fp32 rounding of zz + ee in the canonical key).
//
// Roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 = epilogue
// (TMEM lane quadrant = warp_id % 4).  Pipelines: full/empty mbarriers per smem stage (TMA <-> MMA),
// tmem_full/tmem_empty per accumulator stage (MMA <-> epilogue).  The PTX protocol is in xq_tc.cuh.
#include <tuple>

#include "xq_common.cuh"
#include "xq_tc.cuh"

namespace xq {
using namespace xqtc;

static long long *g_vq_tc_trace = nullptr;     // in-kernel clock trace buffer (development builds only)

constexpr int TC_BM = 128;       // rows per CTA  (UMMA M)
constexpr int TC_BN = 128;       // codes per tile (UMMA N); 2 accumulator stages = 256 TMEM columns -> 2 CTAs / SM
constexpr int TC_THREADS = 192;
constexpr int TC_CAP = 16;       // candidate-group slots per row
constexpr float TC_EPS = 2.5e-3f;
constexpr float TC_W = 2.0f * TC_EPS + 2e-6f;

// byte offset of element (row, k) inside a K-major SWIZZLE_128B operand made of 32-float (128 B) K chunks
__device__ __forceinline__ uint32_t sw128_off(int row, int k, int rows_per_chunk) {
    int kc = k >> 5, kk = k & 31;
    return (uint32_t)(kc * rows_per_chunk * 128 + row * 128 + (((kk >> 2) ^ (row & 7)) << 4) + ((kk & 3) << 2));
}

// remember a candidate group: its best score, its runner-up score and the code holding the best score;
// compacts the list when it is full
__device__ __forceinline__ void cand_push(float m1, float m2, int code, float *c1, float *c2, int *cv, int &cnt,
                                          int &overflow, float thr) {
    if (cnt == TC_CAP) {  // drop groups that fell below the threshold since they were stored
        int w = 0;
        for (int e = 0; e < TC_CAP; ++e)
            if (c1[e] >= thr) { c1[w] = c1[e]; c2[w] = c2[e]; cv[w] = cv[e]; ++w; }
        cnt = w;
    }
    if (cnt < TC_CAP) { c1[cnt] = m1; c2[cnt] = m2; cv[cnt] = code; ++cnt; }
    else overflow = 1;
}

struct TcSmem {
    float *A;        // [C/32][128][32]  swizzled
    float *B;        // [NSTAGE][C/32][256][32] swizzled (TMA)
    float *cand_s;   // [128][CAP] best score of the group
    float *cand_s2;  // [128][CAP] runner-up score of the group
    int *cand_v;     // [128][CAP] code with the best score (group = code >> 5)
    float *zz, *red;
    int *idx;
    uint64_t *full, *empty, *tfull, *tempty;
    uint32_t *tmem_ptr;
};

static size_t tc_smem_bytes(int C, int nstage) {
    size_t b = 1024;                                        // alignment slack
    b += (size_t)TC_BM * C * 4;                             // A
    b += (size_t)nstage * TC_BN * C * 4;                    // B
    b += (size_t)TC_BM * TC_CAP * 12;                       // candidates
    b += (size_t)TC_BM * 4 * 2 + 32 * 4;                    // zz, idx, red
    b += 8 * (2 * 8 + 4) + 16;                              // barriers + tmem ptr
    return b;
}

__global__ void __launch_bounds__(TC_THREADS, 2)
vq_search_tc_kernel(const __grid_constant__ CUtensorMap tmB, const float *__restrict__ z, const float *__restrict__ E,
                    const float *__restrict__ En, const float *__restrict__ ee, int N, int C, int HW, int V, int Vpad,
                    int nstage, int ste_value, int64_t *__restrict__ idx_out, float *__restrict__ out,
                    float *__restrict__ partial, float *__restrict__ hist, long long *__restrict__ dbg) {
    extern __shared__ uint8_t smem_raw[];
    // dbg (optional, CTA 0 only): [0] start, [1] after prologue; per tile t: [8+4t+0] mma waited tempty,
    // [+1] mma waited full, [+2] mma issued+committed, [+3] epilogue warp 2 done with tile
    const bool trace = dbg && blockIdx.x == 0;
    if (trace && threadIdx.x == 0) dbg[0] = clock64();
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    TcSmem s;
    s.A = (float *)base;
    s.B = (float *)(base + (size_t)TC_BM * C * 4);
    uint8_t *p = base + (size_t)TC_BM * C * 4 + (size_t)nstage * TC_BN * C * 4;
    s.cand_s = (float *)p; p += (size_t)TC_BM * TC_CAP * 4;
    s.cand_s2 = (float *)p; p += (size_t)TC_BM * TC_CAP * 4;
    s.cand_v = (int *)p; p += (size_t)TC_BM * TC_CAP * 4;
    s.zz = (float *)p; p += TC_BM * 4;
    s.idx = (int *)p; p += TC_BM * 4;
    s.red = (float *)p; p += 32 * 4;
    s.full = (uint64_t *)p; p += 8 * 8;
    s.empty = (uint64_t *)p; p += 8 * 8;
    s.tfull = (uint64_t *)p; p += 2 * 8;
    s.tempty = (uint64_t *)p; p += 2 * 8;
    s.tmem_ptr = (uint32_t *)p;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row0 = blockIdx.x * TC_BM;
    const int KC = C >> 5;                       // 128-byte K chunks
    const int T = Vpad / TC_BN;
    const uint32_t stage_bytes = (uint32_t)TC_BN * C * 4;

    if (tid == 0) {
        for (int i = 0; i < nstage; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 4); }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<2 * TC_BN>(s.tmem_ptr);
    // rows: coalesced load of the raw NCHW tile into the swizzled A operand (consecutive threads = consecutive
    // rows of one channel), then one thread per row normalises in place with the canonical chain
    for (int i = tid; i < C * TC_BM; i += TC_THREADS) {
        const int k = i / TC_BM, r = i - k * TC_BM;
        const int n = row0 + r;
        float x = 0.f;
        if (n < N) {
            const int b = n / HW, pp = n - b * HW;
            x = z[((size_t)b * C + k) * HW + pp];
        }
        *(float *)((uint8_t *)s.A + sw128_off(r, k, TC_BM)) = x;
    }
    __syncthreads();
    if (tid < TC_BM) {
        float ss = 0.f, zz = 0.f;
        for (int k = 0; k < C; ++k) { float x = *(const float *)((const uint8_t *)s.A + sw128_off(tid, k, TC_BM)); ss = fmaf(x, x, ss); }
        const float den = fmaxf(sqrtf(ss), XQ_EPS);
        for (int k = 0; k < C; ++k) {
            float *pa = (float *)((uint8_t *)s.A + sw128_off(tid, k, TC_BM));
            float x = *pa / den;
            zz = fmaf(x, x, zz);
            *pa = x;
        }
        s.zz[tid] = zz;
    }
    fence_async_smem();            // generic-proxy stores to A -> visible to the async proxy (the MMAs)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s.tmem_ptr;
    if (trace && threadIdx.x == 0) dbg[1] = clock64();

    if (warp == 0) {
        // ===== TMA producer (whole warp runs the loop, one elected lane issues) =====
        for (int t = 0; t < T; ++t) {
            const int st = t % nstage;
            mbar_wait(&s.empty[st], ((t / nstage) & 1) ^ 1);
            if (elect_one()) {
                mbar_expect_tx(&s.full[st], stage_bytes);
                float *dst = s.B + (size_t)st * TC_BN * C;
                for (int kc = 0; kc < KC; ++kc)
                    tma_load_2d(dst + (size_t)kc * TC_BN * 32, &tmB, kc * 32, t * TC_BN, &s.full[st]);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ===== MMA issuer (whole warp runs the control flow, one elected lane issues) =====
        const uint32_t idesc = idesc_tf32(TC_BM, TC_BN);
        const uint32_t a_addr = smem_u32(s.A);
        for (int t = 0; t < T; ++t) {
            const int st = t % nstage, as = t & 1;
            mbar_wait(&s.tempty[as], ((t >> 1) & 1) ^ 1);
            if (trace && lane == 0 && t < 60) dbg[8 + 4 * t + 0] = clock64();
            mbar_wait(&s.full[st], (t / nstage) & 1);
            if (trace && lane == 0 && t < 60) dbg[8 + 4 * t + 1] = clock64();
            tc_fence_after();
            if (elect_one()) {
                const uint32_t b_addr = smem_u32(s.B + (size_t)st * TC_BN * C);
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * TC_BN);
                for (int kc = 0; kc < KC; ++kc) {
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) {
                        uint64_t ad = desc_k_sw128(a_addr + kc * TC_BM * 128 + k4 * 32);
                        uint64_t bd = desc_k_sw128(b_addr + kc * TC_BN * 128 + k4 * 32);
                        umma_tf32(d_tmem, ad, bd, idesc, (kc | k4) ? 1u : 0u);
                    }
                }
                umma_commit(&s.empty[st]);    // smem stage free once these MMAs retire
                umma_commit(&s.tfull[as]);    // accumulator ready
            }
            __syncwarp();
            if (trace && lane == 0 && t < 60) dbg[8 + 4 * t + 2] = clock64();
        }
    } else {
        // ===== epilogue: one thread per row (TMEM lane) =====
        const int q = warp & 3;
        const int row = q * 32 + lane;
        float runmax = -CUDART_INF_F, thr = -CUDART_INF_F;
        int cnt = 0, overflow = 0;
        float *cs = s.cand_s + row * TC_CAP;
        float *cs2 = s.cand_s2 + row * TC_CAP;
        int *cv = s.cand_v + row * TC_CAP;
        for (int t = 0; t < T; ++t) {
            const int as = t & 1;
            mbar_wait(&s.tfull[as], (t >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * TC_BN);
            const int vt = t * TC_BN;
            float v[TC_BN / 32][32];
#pragma unroll
            for (int g = 0; g < TC_BN / 32; ++g) {         // issue all loads, wait once
                uint32_t r[32];
                tmem_ld32(taddr + g * 32, r);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[g][j] = __uint_as_float(r[j]);
            }
            tmem_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&s.tempty[as]);     // the accumulator stage is free as soon as it is in registers
#pragma unroll
            for (int g = 0; g < TC_BN / 32; ++g) {
                float m = v[g][0];
#pragma unroll
                for (int j = 1; j < 32; ++j) m = fmaxf(m, v[g][j]);
                if (m >= thr) {          // rare per row (~ln(#groups) times); branch-free, ILP-friendly body
                    const int cbase = vt + g * 32;
                    float m1 = m;
                    if (cbase + 32 > V) {            // last tile only: padding rows must not take part
                        m1 = -CUDART_INF_F;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            if (cbase + j >= V) v[g][j] = -CUDART_INF_F;
                            m1 = fmaxf(m1, v[g][j]);
                        }
                    }
                    if (m1 >= thr) {
                        // argmax (first index) by a min-tree over (value == max ? j : 32); and how many codes of the
                        // group lie within W of the group's own maximum (1 => the group can hold only ONE candidate)
                        const float lo = m1 - TC_W;
                        int ia = 32, ib = 32, ic = 32, id = 32;
                        int na = 0, nb = 0, nc = 0, nd = 0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            ia = min(ia, v[g][j + 0] == m1 ? j + 0 : 32);
                            ib = min(ib, v[g][j + 1] == m1 ? j + 1 : 32);
                            ic = min(ic, v[g][j + 2] == m1 ? j + 2 : 32);
                            id = min(id, v[g][j + 3] == m1 ? j + 3 : 32);
                            na += v[g][j + 0] >= lo;
                            nb += v[g][j + 1] >= lo;
                            nc += v[g][j + 2] >= lo;
                            nd += v[g][j + 3] >= lo;
                        }
                        const int i1 = min(min(ia, ib), min(ic, id));
                        const int nW = (na + nb) + (nc + nd);
                        if (m1 > runmax) { runmax = m1; thr = runmax - TC_W; }
                        // second slot: m1 again when several codes are within W of it (forces rescoring), else -inf
                        cand_push(m1, nW > 1 ? m1 : -CUDART_INF_F, cbase + i1, cs, cs2, cv, cnt, overflow, thr);
                    }
                }
            }

            if (trace && warp == 2 && lane == 0 && t < 60) dbg[8 + 4 * t + 3] = clock64();
        }
        if (trace && warp == 2 && lane == 0) dbg[2] = clock64();
        // exact canonical rescoring, warp-cooperative: for every (row, candidate group) of this warp, lane j
        // scores code j of the group against the row (row values broadcast from smem, the 32 code rows are one
        // contiguous 32*C*4-byte block of En), then a (d, code) lexicographic warp-argmin picks the winner.
        float best_d = CUDART_INF_F;
        int best_v = 0x7fffffff;
        // A row whose candidate set {codes with approximate score >= final threshold} has exactly ONE element needs
        // no rescoring: the true argmin provably lies in that set.  (~90 % of rows.)
        int n_live = 0, multi = 0, uniq = 0;
        for (int e = 0; e < cnt; ++e)
            if (cs[e] >= thr) { ++n_live; uniq = cv[e]; multi |= (cs2[e] >= thr); }
        const bool need = overflow || multi || n_live != 1;
        if (!need) best_v = uniq;
        const unsigned need_mask = __ballot_sync(0xffffffffu, need);
        const unsigned any_overflow = __ballot_sync(0xffffffffu, overflow != 0);
        for (int r = 0; r < 32; ++r) {
            if (!((need_mask >> r) & 1u)) continue;
            const int rrow = q * 32 + r;
            const int rcnt = __shfl_sync(0xffffffffu, cnt, r);
            const float rthr = __shfl_sync(0xffffffffu, thr, r);
            const float rzz = s.zz[rrow];
            float rb_d = CUDART_INF_F;
            int rb_v = 0x7fffffff;
            const int ngroups = ((any_overflow >> r) & 1u) ? (V + 31) / 32 : rcnt;   // overflow: scan every group
            for (int e = 0; e < ngroups; ++e) {
                int gid;
                if ((any_overflow >> r) & 1u) gid = e;
                else {
                    if (s.cand_s[rrow * TC_CAP + e] < rthr) continue;     // warp-uniform
                    gid = s.cand_v[rrow * TC_CAP + e] >> 5;
                }
                const int code = (gid << 5) + lane;
                float d = CUDART_INF_F;
                if (code < V) {
                    const float4 *en4 = reinterpret_cast<const float4 *>(En + (size_t)code * C);
                    float dot = 0.f;
                    for (int k4 = 0; k4 < C / 4; ++k4) {
                        float4 ev = en4[k4];
                        // A(rrow, 4*k4 .. 4*k4+3) is one 16-byte chunk of the swizzled operand (broadcast read)
                        const float4 av = *reinterpret_cast<const float4 *>((const uint8_t *)s.A + sw128_off(rrow, 4 * k4, TC_BM));
                        dot = fmaf(av.x, ev.x, dot);
                        dot = fmaf(av.y, ev.y, dot);
                        dot = fmaf(av.z, ev.z, dot);
                        dot = fmaf(av.w, ev.w, dot);
                    }
                    d = fmaf(-2.0f, dot, rzz + ee[code]);
                }
                int cv_ = code;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    float od = __shfl_xor_sync(0xffffffffu, d, o);
                    int oc = __shfl_xor_sync(0xffffffffu, cv_, o);
                    if (od < d || (od == d && oc < cv_)) { d = od; cv_ = oc; }
                }
                if (d < rb_d || (d == rb_d && cv_ < rb_v)) { rb_d = d; rb_v = cv_; }
            }
            if (lane == r) { best_d = rb_d; best_v = rb_v; }
        }
        s.idx[row] = best_v;
        if (trace && warp == 2 && lane == 0) dbg[4] = clock64();
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc<2 * TC_BN>(tmem_base);
    // ---- common epilogue: z_q = normalised code (xqgan_model.py:769-771).  En[v] (prep kernel) holds exactly
    // E[v] / max(|E[v]|, eps) computed with the canonical chain, i.e. the bits the exact kernel recomputes here.
    float sq = 0.f;
    if (tid < TC_BM && row0 + tid < N) {
        const int n = row0 + tid;
        int v = s.idx[tid];
        if (v < 0 || v >= V) v = 0;
        const float *qn = En + (size_t)v * C;
        const int b = n / HW, pp = n - b * HW;
        float *op = out + (size_t)b * C * HW + pp;
#pragma unroll 4
        for (int k = 0; k < C; ++k) {
            float qv = qn[k];
            float zn = *(const float *)((const uint8_t *)s.A + sw128_off(tid, k, TC_BM));
            float df = qv - zn;
            sq = fmaf(df, df, sq);
            op[(size_t)k * HW] = ste_value ? zn + df : qv;
        }
        idx_out[n] = (int64_t)v;
        if (hist) atomicAdd(hist + v, 1.0f);
    }
    sq = block_sum(sq, s.red);
    if (tid == 0 && partial) partial[blockIdx.x] = sq;
    if (trace && tid == 0) dbg[3] = clock64();
}

// row-major normalised codebook En[Vpad][C] (+ ee[Vpad]); padded rows are zero
__global__ void codebook_prep_rowmajor_kernel(const float *__restrict__ E, int V, int C, int Vpad, float *__restrict__ En,
                                              float *__restrict__ ee) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= Vpad) return;
    if (v >= V) {
        for (int k = 0; k < C; ++k) En[(size_t)v * C + k] = 0.f;
        ee[v] = CUDART_INF_F;
        return;
    }
    const float *e = E + (size_t)v * C;
    float ss = 0.f;
    for (int k = 0; k < C; ++k) ss = fmaf(e[k], e[k], ss);
    float den = fmaxf(sqrtf(ss), XQ_EPS);
    float s2 = 0.f;
    for (int k = 0; k < C; ++k) {
        float x = e[k] / den;
        En[(size_t)v * C + k] = x;
        s2 = fmaf(x, x, s2);
    }
    ee[v] = s2;
}

__global__ void finalize_mse_tc_kernel(const float *__restrict__ partial, int n, double inv_count, float beta,
                                       float *__restrict__ loss) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 32) acc += (double)partial[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) {
        float mse = (float)(acc * inv_count);
        loss[0] = mse;
        loss[1] = beta * mse;
    }
}

size_t vq_tc_workspace_bytes(int B, int C, int HW, int V) {
    size_t Vp = ((size_t)V + TC_BN - 1) / TC_BN * TC_BN;
    size_t ctas = ((size_t)B * HW + TC_BM - 1) / TC_BM;
    return align_up(sizeof(float) * Vp * C, 1024) + align_up(sizeof(float) * Vp, 256) + align_up(sizeof(float) * ctas, 256);
}

bool vq_tc_supported(int C, int V, int codebook_norm) {
    return codebook_norm && (C == 32 || C == 64) && V >= 1;
}

// returns XQ_OK, or an error; XQ_ERR_UNSUPPORTED lets the caller fall back to the exact CUDA-core kernel
int vq_tc_forward(const float *z, const float *E, int B, int C, int HW, int V, int ste_value, float beta, int64_t *idx,
                  float *out, float *loss, float *hist, void *workspace, size_t workspace_bytes, cudaStream_t stream) {
    if (!vq_tc_supported(C, V, 1)) return XQ_ERR_UNSUPPORTED;
    if (workspace_bytes < vq_tc_workspace_bytes(B, C, HW, V)) return XQ_ERR_WORKSPACE;
    if (((uintptr_t)workspace & 127) != 0) return XQ_ERR_UNSUPPORTED;   // TMA global address alignment
    const int Vp = (V + TC_BN - 1) / TC_BN * TC_BN;
    const int N = B * HW;
    char *ws = (char *)workspace;
    float *En = (float *)ws;
    ws += align_up(sizeof(float) * (size_t)Vp * C, 1024);
    float *ee = (float *)ws;
    ws += align_up(sizeof(float) * (size_t)Vp, 256);
    float *partial = (float *)ws;
    const int nstage = (C == 32) ? 4 : 3;
    const size_t smem = tc_smem_bytes(C, nstage);
    if (smem > 227 * 1024) return XQ_ERR_UNSUPPORTED;

    // the tensor map depends only on (workspace pointer, Vp, C): encode it once per distinct triple
    static MapCache<std::tuple<const void *, int, int>, CUtensorMap> maps;
    CUtensorMap tm;
    if (!maps.get({En, Vp, C}, tm, [&](CUtensorMap &m) {
            return make_map_2d(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, En, C, Vp, (uint64_t)C * sizeof(float), 32, TC_BN);
        }))
        return XQ_ERR_UNSUPPORTED;

    codebook_prep_rowmajor_kernel<<<(Vp + 127) / 128, 128, 0, stream>>>(E, V, C, Vp, En, ee);
    XQ_LAUNCH_CHECK("codebook_prep_rowmajor_kernel");
    XQ_CUDA_TRY(cudaFuncSetAttribute(vq_search_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ctas = (N + TC_BM - 1) / TC_BM;
    long long *dbg = g_vq_tc_trace;          // nullptr unless a development build set it (xq_dev_set_vq_trace, -DXQ_VQ_TC_TRACE)
    vq_search_tc_kernel<<<ctas, TC_THREADS, smem, stream>>>(tm, z, E, En, ee, N, C, HW, V, Vp, nstage, ste_value, idx, out,
                                                           loss ? partial : nullptr, hist, dbg);
    XQ_LAUNCH_CHECK("vq_search_tc_kernel");
    if (loss) {
        finalize_mse_tc_kernel<<<1, 32, 0, stream>>>(partial, ctas, 1.0 / ((double)N * (double)C), beta, loss);
        XQ_LAUNCH_CHECK("finalize_mse_tc_kernel");
    }
    return XQ_OK;
}

#ifdef XQ_VQ_TC_TRACE
extern "C" int xq_dev_set_vq_trace(void *dev_ptr) { xq::g_vq_tc_trace = (long long *)dev_ptr; return 0; }   // tools/vq_tc_trace.py
#endif

}  // namespace xq
