// umma_probe.cu -- dev tool: checks, on a real B200, every tcgen05 / TMA operand flavour the attention kernels rely on
// (descriptor encodings cannot be verified without the hardware).  Build: nvcc -gencode arch=compute_100a,code=sm_100a
// -O2 -o tools/mb/umma_probe tools/umma_probe.cu -lcuda ; run on the GPU box; prints PASS/FAIL per flavour.
//
//   T0  SS  A K-major [128x64], B K-major [N x64]          D[128xN]  = A B^T          (S = Q K^T), N = 128 and 16
//   T1  TS  A in TMEM [128x128 bf16], B MN-major [128x64]  D[128x64] = A B            (O = P V, dV = P^T dO, dK = dS^T Q)
//   T2  SS  A MN-major [M=128 x K=128] (2 row tiles), B MN-major [128x64]  D = A B    (dQ = dS K)
//   T3  TMA 3-D load with OOB rows, TMA 3-D store with clipping, TMA 3-D fp32 reduce-add
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include "../imagefolder_b200/csrc/xq_tc.cuh"

using namespace xqtc;
typedef __nv_bfloat16 bf16;

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1); } } while (0)

// test: 0 = SS KK, 1 = TS MN, 2 = SS MNMN.  variant bit0: swap LBO/SBO in MN descriptors
__global__ void __launch_bounds__(128, 1) probe_kernel(int test, int N, int variant, const bf16 *A, const bf16 *Bm, float *D) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = base;                 // up to 2 row tiles of 128 rows = 32 KB
    uint8_t *sB = base + 32768;         // 16 KB
    uint64_t *bar = (uint64_t *)(base + 49152);
    uint32_t *tptr = (uint32_t *)(base + 49152 + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc<512>(tptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tptr;
    if (test == 0) {
        // A [128][64] row-major -> K-major row tile ; B [N][64] -> K-major row tile (rows >= N zero)
        for (int i = tid; i < 128 * 64; i += 128) {
            int r = i >> 6, c = i & 63;
            *(bf16 *)(sA + rowtile_off_bf16(r, c)) = A[i];
            *(bf16 *)(sB + rowtile_off_bf16(r, c)) = r < N ? Bm[i] : __float2bfloat16(0.f);
        }
    } else if (test == 1) {
        // A [128][128] -> TMEM cols 256.. (2 bf16 / column) ; B [128 k][64 n] -> MN-major row tile
        uint32_t r0[32], r1[32];
        const int row = warp * 32 + lane;
        for (int c = 0; c < 32; ++c) {
            r0[c] = pack_bf16(__bfloat162float(A[row * 128 + 2 * c]), __bfloat162float(A[row * 128 + 2 * c + 1]));
            r1[c] = pack_bf16(__bfloat162float(A[row * 128 + 64 + 2 * c]), __bfloat162float(A[row * 128 + 64 + 2 * c + 1]));
        }
        const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + 256;
        tmem_st32(ta, r0);
        tmem_st32(ta + 32, r1);
        tmem_wait_st();
        for (int i = tid; i < 128 * 64; i += 128) {
            int k = i >> 6, n = i & 63;
            *(bf16 *)(sB + rowtile_off_bf16(k, n)) = Bm[i];
        }
    } else {
        // A [128 m][128 k] -> MN-major: element (m, k) in row tile (m >> 6), row k, column m & 63 ; B as test 1
        for (int i = tid; i < 128 * 128; i += 128) {
            int m = i >> 7, k = i & 127;
            *(bf16 *)(sA + (m >> 6) * 16384 + rowtile_off_bf16(k, m & 63)) = A[i];
        }
        for (int i = tid; i < 128 * 64; i += 128) {
            int k = i >> 6, n = i & 63;
            *(bf16 *)(sB + rowtile_off_bf16(k, n)) = Bm[i];
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {
        if (test == 0) {
            const uint32_t id = idesc_bf16(128, N, 0, 0);
            for (int k = 0; k < 4; ++k)
                umma_ss(tmem, desc_k_sw128(smem_u32(sA) + k * 32), desc_k_sw128(smem_u32(sB) + k * 32), id, k > 0);
        } else if (test == 1) {
            const uint32_t id = idesc_bf16(128, 64, 0, 1);
            for (int k = 0; k < 8; ++k) {
                uint64_t bd = (variant & 1) ? desc_mn_sw128(smem_u32(sB) + k * 2048, 1024, 16384)
                                            : desc_mn_sw128(smem_u32(sB) + k * 2048, 16384, 1024);
                umma_ts(tmem, tmem + 256 + k * 8, bd, id, k > 0);
            }
        } else {
            const uint32_t id = idesc_bf16(128, 64, 1, 1);
            for (int k = 0; k < 8; ++k) {
                uint64_t ad = (variant & 1) ? desc_mn_sw128(smem_u32(sA) + k * 2048, 1024, 16384)
                                            : desc_mn_sw128(smem_u32(sA) + k * 2048, 16384, 1024);
                uint64_t bd = (variant & 1) ? desc_mn_sw128(smem_u32(sB) + k * 2048, 1024, 16384)
                                            : desc_mn_sw128(smem_u32(sB) + k * 2048, 16384, 1024);
                umma_ss(tmem, ad, bd, id, k > 0);
            }
        }
        umma_commit(bar);
    }
    mbar_wait(bar, 0);
    tc_fence_after();
    const int ND = test == 0 ? N : 64;
    const int row = warp * 32 + lane;
    for (int c0 = 0; c0 < ND; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c0, r);
        tmem_wait_ld();
        for (int j = 0; j < 16; ++j) D[row * ND + c0 + j] = __uint_as_float(r[j]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

// TMA probe: load box (col0,row0,b) -> dump ; store tile ; reduce-add fp32
__global__ void __launch_bounds__(128, 1)
tma_probe_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmOut,
                 const __grid_constant__ CUtensorMap tmAcc, int col0, int row0, int b, uint8_t *dump) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sT = base;              // 16 KB bf16 row tile
    uint8_t *sF = base + 16384;      // 16 KB fp32 [128][32] row tile
    uint64_t *bar = (uint64_t *)(base + 32768);
    const int tid = threadIdx.x;
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(bar, 16384);
        tma_load_3d(sT, &tmIn, col0, row0, b, bar);
    }
    mbar_wait(bar, 0);
    for (int i = tid; i < 16384; i += 128) dump[i] = sT[i];
    __syncthreads();
    // store: row r holds value (r*64 + c) mod 251 + 1 as bf16
    for (int i = tid; i < 128 * 64; i += 128) {
        int r = i >> 6, c = i & 63;
        *(bf16 *)(sT + rowtile_off_bf16(r, c)) = __float2bfloat16((float)((r * 64 + c) % 251 + 1));
        if (c < 32) {
            // fp32 row tile: 16-byte unit = 4 floats
            uint32_t off = r * 128 + ((((c >> 2) ^ (r & 7)) & 7) << 4) + (c & 3) * 4;
            *(float *)(sF + off) = (float)(r * 32 + c);
        }
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
        tma_store_3d(&tmOut, sT, col0, row0, b);
        tma_reduce_add_3d(&tmAcc, sF, 0, row0, b);
        tma_reduce_add_3d(&tmAcc, sF, 32, row0, b);
        tma_reduce_add_3d(&tmAcc, sF, 0, row0, b);
        bulk_commit();
        bulk_wait<0>();
    }
    __syncthreads();
}

// timing: `reps` back-to-back MMAs of one flavour (same operands, accumulating), one commit; clocks measured by the issuer
//   flavour 0: SS K x K, N = n   1: TS (A tmem) x B MN-major, N = 64   2: SS A MN x B MN, N = 64   3: SS K x K with B = 64-row half tile
__global__ void __launch_bounds__(128, 1) mma_time_kernel(int flavour, int n, int reps, long long *out) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = base, *sB = base + 32768;
    uint64_t *bar = (uint64_t *)(base + 49152);
    uint32_t *tptr = (uint32_t *)(base + 49152 + 16);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc<512>(tptr);
    for (int i = tid; i < 49152 / 4; i += 128) ((uint32_t *)base)[i] = 0x3c003c00u;   // finite bf16 values
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tptr;
    if (tid == 0) {
        long long t0 = clock64();
        for (int r = 0; r < reps; ++r) {
            const int k = r & 3;
            if (flavour == 0) umma_ss(tmem, desc_k_sw128(smem_u32(sA) + k * 32), desc_k_sw128(smem_u32(sB) + k * 32), idesc_bf16(128, n, 0, 0), 1);
            else if (flavour == 1) umma_ts(tmem, tmem + 256 + k * 8, desc_mn_sw128(smem_u32(sB) + k * 2048, 16384, 1024), idesc_bf16(128, 64, 0, 1), 1);
            else if (flavour == 2) umma_ss(tmem, desc_mn_sw128(smem_u32(sA) + k * 2048, 16384, 1024), desc_mn_sw128(smem_u32(sB) + k * 2048, 16384, 1024), idesc_bf16(128, 64, 1, 1), 1);
            else umma_ss(tmem, desc_k_sw128(smem_u32(sA) + k * 32), desc_mn_sw128(smem_u32(sB) + k * 2048, 16384, 1024), idesc_bf16(128, n, 0, 1), 1);
        }
        long long t1 = clock64();
        umma_commit(bar);
        mbar_wait(bar, 0);
        long long t2 = clock64();
        out[0] = t1 - t0;
        out[1] = t2 - t0;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

// same measurement, but the WHOLE warp runs the loop and only the MMA is predicated by elect.sync (CUTLASS style)
template <int flavour>
__global__ void __launch_bounds__(128, 1) mma_time_kernel_elect(int n, int reps, long long *out) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = base, *sB = base + 32768;
    uint64_t *bar = (uint64_t *)(base + 49152);
    uint32_t *tptr = (uint32_t *)(base + 49152 + 16);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc<512>(tptr);
    for (int i = tid; i < 49152 / 4; i += 128) ((uint32_t *)base)[i] = 0x3c003c00u;
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tptr;
    if (warp == 1) {
        const uint64_t ad = desc_k_sw128(smem_u32(sA)), bd = desc_k_sw128(smem_u32(sB));
        const uint64_t amn = desc_mn_sw128(smem_u32(sA), 16384, 1024), bmn = desc_mn_sw128(smem_u32(sB), 16384, 1024);
        long long t0 = clock64();
        for (int r = 0; r < reps; r += 4) {
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (flavour == 0) umma_ss(tmem, ad + 2 * k, bd + 2 * k, idesc_bf16(128, n, 0, 0), 1);
                    else if (flavour == 1) umma_ts(tmem, tmem + 256 + k * 8, bmn + 128 * k, idesc_bf16(128, n, 0, 1), 1);
                    else if (flavour == 2) umma_ss(tmem, amn + 128 * k, bmn + 128 * k, idesc_bf16(128, n, 1, 1), 1);
                    else umma_ts(tmem, tmem + 256 + k * 8, bd + 2 * k, idesc_bf16(128, n, 0, 0), 1);
                }
            }
            __syncwarp();
        }
        long long t1 = clock64();
        if (elect_one()) umma_commit(bar);
        __syncwarp();
        mbar_wait(bar, 0);
        long long t2 = clock64();
        if (tid == 32) { out[0] = t1 - t0; out[1] = t2 - t0; }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

static float bf(bf16 x) { return __bfloat162float(x); }

int main() {
    srand(1);
    int fails = 0;
    const size_t SMEM = 49152 + 64 + 1024;
    CK(cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    bf16 *dA, *dB;
    float *dD;
    CK(cudaMalloc(&dA, 128 * 128 * 2));
    CK(cudaMalloc(&dB, 128 * 64 * 2));
    CK(cudaMalloc(&dD, 128 * 128 * 4));
    std::vector<bf16> hA(128 * 128), hB(128 * 64);
    std::vector<float> hD(128 * 128);
    for (auto &x : hA) x = __float2bfloat16((float)(rand() % 7 - 3));
    for (auto &x : hB) x = __float2bfloat16((float)(rand() % 5 - 2));
    CK(cudaMemcpy(dA, hA.data(), hA.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, hB.data(), hB.size() * 2, cudaMemcpyHostToDevice));
    // T0
    for (int N : {128, 16, 64}) {
        CK(cudaMemset(dD, 0, 128 * 128 * 4));
        probe_kernel<<<1, 128, SMEM>>>(0, N, 0, dA, dB, dD);
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(hD.data(), dD, 128 * N * 4, cudaMemcpyDeviceToHost));
        double err = 0;
        for (int m = 0; m < 128; ++m)
            for (int n = 0; n < N; ++n) {
                float ref = 0;
                for (int k = 0; k < 64; ++k) ref += bf(hA[m * 64 + k]) * bf(hB[n * 64 + k]);   // A read as [128][64]
                err = fmax(err, fabs(ref - hD[m * N + n]));
            }
        printf("T0 SS K-major x K-major  N=%3d  max|err| = %g  %s\n", N, err, err == 0 ? "PASS" : "FAIL");
        fails += err != 0;
    }
    for (int variant = 0; variant < 1; ++variant) {   // variant 1 (LBO/SBO swapped) faults on hardware: the encoding in xq_tc.cuh is the right one
        // T1
        CK(cudaMemset(dD, 0, 128 * 128 * 4));
        probe_kernel<<<1, 128, SMEM>>>(1, 64, variant, dA, dB, dD);
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(hD.data(), dD, 128 * 64 * 4, cudaMemcpyDeviceToHost));
        double err = 0;
        for (int m = 0; m < 128; ++m)
            for (int n = 0; n < 64; ++n) {
                float ref = 0;
                for (int k = 0; k < 128; ++k) ref += bf(hA[m * 128 + k]) * bf(hB[k * 64 + n]);
                err = fmax(err, fabs(ref - hD[m * 64 + n]));
            }
        printf("T1 TS A(TMEM) x B MN-major variant %d  max|err| = %g  %s\n", variant, err, err == 0 ? "PASS" : "FAIL");
        if (variant == 0) fails += err != 0;
        // T2
        CK(cudaMemset(dD, 0, 128 * 128 * 4));
        probe_kernel<<<1, 128, SMEM>>>(2, 64, variant, dA, dB, dD);
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(hD.data(), dD, 128 * 64 * 4, cudaMemcpyDeviceToHost));
        err = 0;
        for (int m = 0; m < 128; ++m)
            for (int n = 0; n < 64; ++n) {
                float ref = 0;
                for (int k = 0; k < 128; ++k) ref += bf(hA[m * 128 + k]) * bf(hB[k * 64 + n]);
                err = fmax(err, fabs(ref - hD[m * 64 + n]));
            }
        printf("T2 SS A MN-major x B MN-major variant %d  max|err| = %g  %s\n", variant, err, err == 0 ? "PASS" : "FAIL");
        if (variant == 0) fails += err != 0;
    }
    // T3: TMA
    {
        const int B = 3, N = 200, H = 2, W = 3 * H * 64;   // qkv-like [B][N][3*H*64]
        std::vector<bf16> hq((size_t)B * N * W);
        for (size_t i = 0; i < hq.size(); ++i) hq[i] = __float2bfloat16((float)(i % 509) - 254.f);
        bf16 *dq, *dout;
        float *dacc;
        uint8_t *ddump;
        CK(cudaMalloc(&dq, hq.size() * 2));
        CK(cudaMalloc(&dout, (size_t)B * N * H * 64 * 2));
        CK(cudaMalloc(&dacc, (size_t)B * H * N * 64 * 4));
        CK(cudaMalloc(&ddump, 16384));
        CK(cudaMemcpy(dq, hq.data(), hq.size() * 2, cudaMemcpyHostToDevice));
        CK(cudaMemset(dout, 0, (size_t)B * N * H * 64 * 2));
        CK(cudaMemset(dacc, 0, (size_t)B * H * N * 64 * 4));
        CUtensorMap tmIn, tmOut, tmAcc;
        bool ok = make_map_3d(&tmIn, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, dq, W, N, B, (uint64_t)W * 2, (uint64_t)N * W * 2, 64, 128);
        ok = ok && make_map_3d(&tmOut, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, dout, H * 64, N, B, (uint64_t)H * 64 * 2, (uint64_t)N * H * 64 * 2, 64, 128);
        ok = ok && make_map_3d(&tmAcc, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dacc, 64, N, B * H, 256, (uint64_t)N * 256, 32, 128);
        printf("T3 tensor maps encode: %s\n", ok ? "ok" : "FAILED");
        if (!ok) return 1;
        CK(cudaFuncSetAttribute(tma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 34816 + 1024));
        const int col0 = (1 * H + 1) * 64, row0 = 128, b = 1;      // k of head 1, second row block (rows 128..199 valid)
        tma_probe_kernel<<<1, 128, 34816 + 1024>>>(tmIn, tmOut, tmAcc, col0, row0, b, ddump);
        CK(cudaDeviceSynchronize());
        std::vector<uint8_t> hd(16384);
        CK(cudaMemcpy(hd.data(), ddump, 16384, cudaMemcpyDeviceToHost));
        int bad = 0;
        for (int r = 0; r < 128; ++r)
            for (int c = 0; c < 64; ++c) {
                float want = row0 + r < N ? bf(hq[((size_t)b * N + row0 + r) * W + col0 + c]) : 0.f;
                float got = bf(*(bf16 *)(hd.data() + rowtile_off_bf16(r, c)));
                bad += want != got;
            }
        printf("T3a TMA 3-D load (swizzle + OOB zero fill): mismatches = %d  %s\n", bad, bad == 0 ? "PASS" : "FAIL");
        fails += bad != 0;
        // store check: tmOut is [B][N][H*64]; the store used col0 (=192) which is outside H*64 = 128 -> fully clipped?  use separate run
        std::vector<bf16> ho((size_t)B * N * H * 64);
        CK(cudaMemcpy(ho.data(), dout, ho.size() * 2, cudaMemcpyDeviceToHost));
        int nz = 0;
        for (auto &x : ho) nz += bf(x) != 0.f;
        printf("T3b TMA store fully out of range in dim0 (col0=%d >= %d): nonzeros written = %d  %s\n", col0, H * 64, nz, nz == 0 ? "PASS" : "FAIL");
        fails += nz != 0;
        std::vector<float> hacc((size_t)B * H * N * 64);
        CK(cudaMemcpy(hacc.data(), dacc, hacc.size() * 4, cudaMemcpyDeviceToHost));
        bad = 0;
        for (int bh = 0; bh < B * H; ++bh)
            for (int n = 0; n < N; ++n)
                for (int c = 0; c < 64; ++c) {
                    float want = 0.f;
                    if (bh == b && n >= row0) { int r = n - row0; want = (c < 32 ? 2.f : 1.f) * (float)(r * 32 + (c & 31)); }
                    bad += hacc[((size_t)bh * N + n) * 64 + c] != want;
                }
        printf("T3c TMA fp32 reduce-add (3 ops, clipped rows): mismatches = %d  %s\n", bad, bad == 0 ? "PASS" : "FAIL");
        fails += bad != 0;
        // second run: store in range
        CK(cudaMemset(dacc, 0, (size_t)B * H * N * 64 * 4));
        tma_probe_kernel<<<1, 128, 34816 + 1024>>>(tmIn, tmOut, tmAcc, 64, row0, b, ddump);
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(ho.data(), dout, ho.size() * 2, cudaMemcpyDeviceToHost));
        bad = 0;
        for (int bb = 0; bb < B; ++bb)
            for (int n = 0; n < N; ++n)
                for (int c = 0; c < H * 64; ++c) {
                    float want = 0.f;
                    if (bb == b && n >= row0 && c >= 64) { int r = n - row0; want = bf(__float2bfloat16((float)((r * 64 + (c - 64)) % 251 + 1))); }
                    bad += bf(ho[((size_t)bb * N + n) * H * 64 + c]) != want;
                }
        printf("T3d TMA 3-D store (row clipping at N): mismatches = %d  %s\n", bad, bad == 0 ? "PASS" : "FAIL");
        fails += bad != 0;
    }
    {
        long long *dout, hout[2];
        CK(cudaMalloc(&dout, 16));
        CK(cudaFuncSetAttribute(mma_time_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        struct { int fl, n; const char *name; } cases[] = {
            {0, 128, "SS  A K-major x B K-major   M128 N128 K16"}, {0, 64, "SS  A K-major x B K-major   M128 N64  K16"},
            {0, 16, "SS  A K-major x B K-major   M128 N16  K16"}, {1, 64, "TS  A tmem    x B MN-major  M128 N64  K16"},
            {2, 64, "SS  A MN-major x B MN-major M128 N64  K16"}, {3, 64, "SS  A K-major x B MN-major  M128 N64  K16"}};
        for (auto &c : cases)
            for (int reps : {64, 256}) {
                mma_time_kernel<<<1, 128, SMEM>>>(c.fl, c.n, reps, dout);
                CK(cudaDeviceSynchronize());
                CK(cudaMemcpy(hout, dout, 16, cudaMemcpyDeviceToHost));
                printf("T4 %-58s reps %3d: issue %6.1f clk/MMA, issue+drain %6.1f clk/MMA\n", c.name, reps, (double)hout[0] / reps, (double)hout[1] / reps);
            }
    }
    {
        long long *dout, hout[2];
        CK(cudaMalloc(&dout, 16));
        CK(cudaFuncSetAttribute(mma_time_kernel_elect<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        CK(cudaFuncSetAttribute(mma_time_kernel_elect<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        CK(cudaFuncSetAttribute(mma_time_kernel_elect<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        CK(cudaFuncSetAttribute(mma_time_kernel_elect<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        struct { int fl, n; const char *name; } ec[] = {{0, 128, "SS K x K   N128"}, {0, 64, "SS K x K   N64"}, {0, 16, "SS K x K   N16"},
            {1, 64, "TS tmem x B MN-major N64"}, {2, 64, "SS A MN x B MN N64"}, {3, 64, "TS tmem x B K-major N64"}, {3, 128, "TS tmem x B K-major N128"}};
        for (auto &c : ec)
            for (int reps : {64, 256}) {
                if (c.fl == 0) mma_time_kernel_elect<0><<<1, 128, SMEM>>>(c.n, reps, dout);
                if (c.fl == 1) mma_time_kernel_elect<1><<<1, 128, SMEM>>>(c.n, reps, dout);
                if (c.fl == 2) mma_time_kernel_elect<2><<<1, 128, SMEM>>>(c.n, reps, dout);
                if (c.fl == 3) mma_time_kernel_elect<3><<<1, 128, SMEM>>>(c.n, reps, dout);
                CK(cudaDeviceSynchronize());
                CK(cudaMemcpy(hout, dout, 16, cudaMemcpyDeviceToHost));
                printf("T5 elect.sync issue, %-28s reps %3d: issue %6.1f clk/MMA, issue+drain %6.1f clk/MMA\n", c.name, reps,
                       (double)hout[0] / reps, (double)hout[1] / reps);
            }
    }
    printf("umma_probe: %s (%d failing checks)\n", fails ? "FAILED" : "ALL PASS", fails);
    return 0;
}
