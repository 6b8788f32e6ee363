// tnq_gemm_f64.cu -- batched float64 GEMM on the FP64 tensor cores (DMMA), the float64 / complex128 sibling of
// tnq_gemm_tf32x3:
//
//     C[b] (M x N, row major, ldc)  (=|+=)  A[b] (M x K, row major, lda) * B[b]^T  (B[b] is N x K, ldb)
//
// tcgen05 has no f64 kind; the FP64 tensor-core instruction of sm_100a is the warp-level
// mma.sync.aligned.m8n8k4.row.col.f64 (one DMMA.8x8x4 in SASS).  Its A fragment (8 x 4, row) and B fragment
// (4 x 8, col) are one double per lane at [lane / 4][lane % 4] of an operand stored K-contiguous, so A and B
// (both K-major here) are read the same way.
//
// Kernel anatomy (one 128 x 128 output tile per CTA, 8 warps of 64 x 32 each, 32 DMMA per k-step of 4):
//   cp.async ring of 3 stages of BK = 16 doubles: 16-byte copies when K, lda / ldb, the batch strides and the base
//   addresses allow (two doubles), 8-byte copies otherwise; out-of-range rows and k are zero-filled by the copy;
//   shared rows padded to 20 doubles, so that each half-warp's fragment loads hit 32 distinct banks;
//   accumulators in registers (64 doubles a lane), written once at the end (double2 stores where aligned).
// Determinism: every output is the sum over its k-blocks in increasing k, in one fixed order per lane.  Split-K
// (two halves of the k-range, C zeroed, both halves added with red.global.add.f64) only when a launch covers at
// most half the SMs; 0 + x + y == 0 + y + x, so the result does not depend on which half lands first.
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "tneq_b200.h"

extern int tnq_internal_fail(const std::string& msg);
extern int tnq_internal_cuda_fail(cudaError_t e, const char* what);
extern void tnq_internal_count_launch();

namespace {

constexpr int BM = 128, BN = 128, BK = 16;           // tile; BK doubles = 128 bytes
constexpr int STAGES = 3;
constexpr int LDS = BK + 4;                          // padded shared row (doubles)
constexpr int THREADS = 256;
constexpr int STAGE_ELEMS = (BM + BN) * LDS;
constexpr size_t SMEM_BYTES = sizeof(double) * STAGES * STAGE_ELEMS;   // 120 KB

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// `bytes` (8 or 16) from global to shared; src_bytes = 0 writes zeros (the address must still be valid)
template <int BYTES>
__device__ __forceinline__ void cp_async(uint32_t dst, const double* src, bool valid) {
    const int n = valid ? BYTES : 0;
    if constexpr (BYTES == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// one BK-wide k-block of a 128-row operand tile into shared memory (rows >= rows_left or k >= k_left: zeros)
template <bool VEC>
__device__ __forceinline__ void load_tile(double* dst, const double* __restrict__ src, long long ld, long long rows_left,
                                          long long k_left, const double* any_valid) {
    const uint32_t base = smem_u32(dst);
    if constexpr (VEC) {                             // 128 rows x 8 chunks of two doubles
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = threadIdx.x + i * THREADS, row = c >> 3, k = (c & 7) * 2;
            const bool ok = row < rows_left && k < k_left;
            cp_async<16>(base + (uint32_t)(row * LDS + k) * 8, ok ? src + row * ld + k : any_valid, ok);
        }
    } else {                                         // 128 rows x 16 doubles
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int e = threadIdx.x + i * THREADS, row = e >> 4, k = e & 15;
            const bool ok = row < rows_left && k < k_left;
            cp_async<8>(base + (uint32_t)(row * LDS + k) * 8, ok ? src + row * ld + k : any_valid, ok);
        }
    }
}

template <bool VEC>
__global__ void __launch_bounds__(THREADS, 1)
    tnq_gemm_f64_kernel(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ C, long long M,
                        long long N, long long K, long long lda, long long ldb, long long ldc, long long sA, long long sB,
                        long long sC, int accumulate, int splitk, int c_vec) {
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp >> 2, wn = warp & 3;         // 2 x 4 warps of 64 x 32
    const long long m0 = (long long)blockIdx.y * BM, n0 = (long long)blockIdx.x * BN;
    const long long bz = splitk > 1 ? 0 : blockIdx.z;
    long long kbeg = 0, kend = K;
    if (splitk > 1) {                                // two halves, the split on a k-block boundary
        const long long half = ((K + 2 * BK - 1) / (2 * BK)) * BK;
        kbeg = blockIdx.z ? half : 0;
        kend = blockIdx.z ? K : half;
    }
    const double* a = A + bz * sA + m0 * lda + kbeg;
    const double* b = B + bz * sB + n0 * ldb + kbeg;
    const long long ra = M - m0, rb = N - n0;
    const int nkb = (int)((kend - kbeg + BK - 1) / BK);

    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto load_stage = [&](int kb) {
        double* s = smem + (kb % STAGES) * STAGE_ELEMS;
        const long long k0 = (long long)kb * BK, kl = kend - kbeg - k0;
        load_tile<VEC>(s, a + k0, lda, ra, kl, A);
        load_tile<VEC>(s + BM * LDS, b + k0, ldb, rb, kl, B);
    };
#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nkb) load_stage(s);
        cp_commit();
    }
    for (int kb = 0; kb < nkb; ++kb) {
        cp_wait<STAGES - 2>();
        __syncthreads();                             // stage kb landed for every thread; stage kb - 1 is free
        if (kb + STAGES - 1 < nkb) load_stage(kb + STAGES - 1);
        cp_commit();
        const double* as = smem + (kb % STAGES) * STAGE_ELEMS + (wm * 64 + (lane >> 2)) * LDS + (lane & 3);
        const double* bs = smem + (kb % STAGES) * STAGE_ELEMS + BM * LDS + (wn * 32 + (lane >> 2)) * LDS + (lane & 3);
#pragma unroll
        for (int kk = 0; kk < BK; kk += 4) {
            double fa[8], fb[4];
#pragma unroll
            for (int i = 0; i < 8; ++i) fa[i] = as[i * 8 * LDS + kk];
#pragma unroll
            for (int j = 0; j < 4; ++j) fb[j] = bs[j * 8 * LDS + kk];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
        }
    }
    cp_wait<0>();

    // epilogue: lane holds C[row][col], C[row][col + 1] of every 8 x 8 sub-tile
    double* c = C + bz * sC;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const long long row = m0 + wm * 64 + i * 8 + (lane >> 2);
        if (row >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long col = n0 + wn * 32 + j * 8 + (lane & 3) * 2;
            double* p = c + row * ldc + col;
            if (splitk > 1) {
                if (col < N) atomicAdd(p, acc[i][j][0]);
                if (col + 1 < N) atomicAdd(p + 1, acc[i][j][1]);
            } else if (c_vec && col + 1 < N) {
                double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
                if (accumulate) {
                    const double2 o = *reinterpret_cast<const double2*>(p);
                    v.x += o.x, v.y += o.y;
                }
                *reinterpret_cast<double2*>(p) = v;
            } else {
                if (col < N) p[0] = accumulate ? p[0] + acc[i][j][0] : acc[i][j][0];
                if (col + 1 < N) p[1] = accumulate ? p[1] + acc[i][j][1] : acc[i][j][1];
            }
        }
    }
}

}  // namespace

extern "C" int tnq_gemm_f64(const double* A, const double* B, double* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                            int64_t ldb, int64_t ldc, int64_t batch, int64_t strideA, int64_t strideB, int64_t strideC,
                            int accumulate, void* stream) {
    if (!A || !B || !C || M <= 0 || N <= 0 || K <= 0 || batch <= 0)
        return tnq_internal_fail("tnq_gemm_f64: bad arguments");
    if ((((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 7)) return tnq_internal_fail("tnq_gemm_f64: pointers must be 8-byte aligned");
    if (batch > 65535) return tnq_internal_fail("tnq_gemm_f64: batch too large for one launch (max 65535)");
    const long long mt = (M + BM - 1) / BM, nt = (N + BN - 1) / BN;
    if (mt > 65535) return tnq_internal_fail("tnq_gemm_f64: M too large for one launch");
    const bool vec = !((K & 1) || (lda & 1) || (ldb & 1) || (batch > 1 && ((strideA & 1) || (strideB & 1))) ||
                       (((uintptr_t)A | (uintptr_t)B) & 15));
    const int c_vec = !((ldc & 1) || (batch > 1 && (strideC & 1)) || ((uintptr_t)C & 15));
    cudaStream_t st = (cudaStream_t)stream;
    // split-K by two when the tiles would leave more than half of the SMs idle and the k-loop is long
    const int splitk = (batch == 1 && !accumulate && mt * nt <= 74 && K >= 64 * BK) ? 2 : 1;
    if (splitk > 1) {
        cudaError_t e0 = ldc == N ? cudaMemsetAsync(C, 0, sizeof(double) * (size_t)M * (size_t)N, st)
                                  : cudaMemset2DAsync(C, sizeof(double) * (size_t)ldc, 0, sizeof(double) * (size_t)N, (size_t)M, st);
        if (e0 != cudaSuccess) return tnq_internal_cuda_fail(e0, "cudaMemsetAsync(tnq_gemm_f64 split-K)");
    }
    auto kern = vec ? tnq_gemm_f64_kernel<true> : tnq_gemm_f64_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, "cudaFuncSetAttribute(tnq_gemm_f64)");
    dim3 grid((unsigned)nt, (unsigned)mt, (unsigned)(splitk > 1 ? splitk : batch));
    kern<<<grid, THREADS, SMEM_BYTES, st>>>(A, B, C, M, N, K, lda, ldb, ldc, strideA, strideB, strideC, accumulate, splitk,
                                            c_vec);
    tnq_internal_count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, "tnq_gemm_f64 launch");
    return 0;
}
