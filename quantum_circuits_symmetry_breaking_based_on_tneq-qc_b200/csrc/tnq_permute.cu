// tnq_permute.cu -- index permutation / merge / split of dense tensors (HBM-bound), and the
// complex <-> 2x2-real expansion used to feed complex contractions to the real GEMM.
//
// In the reference every pairwise contraction inside torch.einsum is "permute, reshape, bmm,
// reshape, permute" (tneq_qc/contractor/greedy_strategy.py:940,959 -> ATen); the reference's own
// micro-benchmarks single the permute out as a first-class cost
// (tools/stage3_memory_permute/test_transpose_cost.py).  Here it is one kernel per operand:
//
//   tnq_permute_f32      out (compact, row major over out_dims) <- in viewed through per-dimension
//                        strides.  `vec` trailing elements (1, 2 or 4 floats: a complex number is
//                        vec = 2) move together.  Two code paths:
//                          direct : the innermost moving dimension is contiguous on both sides
//                                   -> fully coalesced vector copy;
//                          tiled  : otherwise a 32 x 32 tile is transposed through shared memory
//                                   (padded, conflict free) so that BOTH the global reads and the
//                                   global writes of every warp are contiguous.
//                        conj != 0 negates the second float of every pair (complex conjugate).
//   tnq_cplx_expand_f32  Qx[..., ri, ..., ro] = E[ri][ro][c] * Q[..., c]  (E = 2x2 real form of a
//                        complex number), permuted into GEMM operand layout in the same pass.
//   tnq_cplx_fold_f32    the adjoint of the expansion (gradient path).
// Every kernel is a template on the element type; the _f64 entry points are the same kernels on doubles
// (float64 / complex128 networks): strides count doubles, vectors are at most two doubles (16 bytes), so a
// complex128 number is vec = 2 and conj negates the second double of each 16-byte pair.
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "tneq_b200.h"

extern int tnq_internal_fail(const std::string& msg);
extern int tnq_internal_cuda_fail(cudaError_t e, const char* what);
extern void tnq_internal_count_launch();

namespace {

constexpr int MAXD = 12;

struct Dims {
    int nd;
    long long size[MAXD];     // output extents (in units of vec elements for the last dim)
    long long istride[MAXD];  // input stride (floats) of each output dimension
};

template <typename T, int VEC>
struct VecT;
template <>
struct VecT<float, 1> { using type = float; };
template <>
struct VecT<float, 2> { using type = float2; };
template <>
struct VecT<float, 4> { using type = float4; };
template <>
struct VecT<double, 1> { using type = double; };
template <>
struct VecT<double, 2> { using type = double2; };

template <typename T>
struct Pair;
template <>
struct Pair<float> { using type = float2; };
template <>
struct Pair<double> { using type = double2; };

template <int VEC, typename V>
__device__ __forceinline__ V conj_vec(V v, int conj) {
    if constexpr (VEC == 2) {
        if (conj) v.y = -v.y;
    } else if constexpr (VEC == 4) {
        if (conj) v.y = -v.y, v.w = -v.w;
    }
    return v;
}

// direct path: one thread per output vector; the innermost dimension is contiguous in the input
template <typename T, int VEC>
__global__ void __launch_bounds__(256) permute_direct_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                             Dims d, long long total, int conj) {
    using V = typename VecT<T, VEC>::type;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long rem = i, off = 0;
#pragma unroll 1
        for (int k = d.nd - 1; k >= 0; --k) {
            const long long q = rem / d.size[k];
            off += (rem - q * d.size[k]) * d.istride[k];
            rem = q;
        }
        V v = __ldg(reinterpret_cast<const V*>(in + off));
        reinterpret_cast<V*>(out)[i] = conj_vec<VEC>(v, conj);
    }
}

// tiled path: dimension `da` is the one that is contiguous in the INPUT, the last dimension is
// contiguous in the OUTPUT; 32 x 32 vectors go through shared memory.
template <typename T, int VEC>
__global__ void __launch_bounds__(256) permute_tiled_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                            Dims d, int da, long long ostride_a, long long tiles_a,
                                                            long long tiles_b, long long ntiles, int conj) {
    using V = typename VecT<T, VEC>::type;
    __shared__ V tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    const int db = d.nd - 1;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        // tile index -> (other dims..., tile_a, tile_b)
        long long rem = t;
        const long long tb = rem % tiles_b;
        rem /= tiles_b;
        const long long ta = rem % tiles_a;
        rem /= tiles_a;
        long long ioff = 0, ooff = 0, ostr = 1;
        // output strides are compact: compute on the fly from the innermost dimension outwards
        long long ostride[MAXD];
        for (int k = d.nd - 1; k >= 0; --k) {
            ostride[k] = ostr;
            ostr *= d.size[k];
        }
        for (int k = d.nd - 2; k >= 0; --k) {
            if (k == da) continue;
            const long long q = rem / d.size[k];
            const long long idx = rem - q * d.size[k];
            ioff += idx * d.istride[k];
            ooff += idx * ostride[k];
            rem = q;
        }
        const long long a0 = ta * 32, b0 = tb * 32;
        // read: lanes along a (contiguous in the input), rows along b
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const long long a = a0 + tx, b = b0 + j;
            if (a < d.size[da] && b < d.size[db])
                tile[j][tx] = __ldg(reinterpret_cast<const V*>(in + ioff + a * d.istride[da] + b * d.istride[db]));
        }
        __syncthreads();
        // write: lanes along b (contiguous in the output), rows along a
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const long long a = a0 + j, b = b0 + tx;
            if (a < d.size[da] && b < d.size[db])
                reinterpret_cast<V*>(out)[ooff + a * ostride_a + b] = conj_vec<VEC>(tile[tx][j], conj);
        }
        __syncthreads();
    }
}

// tiled path for scalar elements with 16-byte accesses on BOTH sides: a 64 x 64 float tile, float4 global loads along
// a (contiguous in the input), float4 global stores along b (contiguous in the output), transposed through a
// [64][65] shared tile with scalar accesses (two-way bank conflicts at most).  Used when extents, strides and
// pointers are multiples of four floats -- the batch-into-K transpositions of the bond-64 gradient GEMMs.
__global__ void __launch_bounds__(256) permute_tiled64_kernel(const float* __restrict__ in, float* __restrict__ out, Dims d,
                                                              int da, long long ostride_a, long long tiles_a, long long tiles_b,
                                                              long long ntiles) {
    __shared__ float tile[64][65];
    const int x = threadIdx.x & 15, y = threadIdx.x >> 4;     // 16 float4 columns x 16 rows
    const int db = d.nd - 1;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        long long rem = t;
        const long long tb = rem % tiles_b;
        rem /= tiles_b;
        const long long ta = rem % tiles_a;
        rem /= tiles_a;
        long long ioff = 0, ooff = 0, ostr = 1;
        long long ostride[MAXD];
        for (int k = d.nd - 1; k >= 0; --k) {
            ostride[k] = ostr;
            ostr *= d.size[k];
        }
        for (int k = d.nd - 2; k >= 0; --k) {
            if (k == da) continue;
            const long long q = rem / d.size[k];
            const long long idx = rem - q * d.size[k];
            ioff += idx * d.istride[k];
            ooff += idx * ostride[k];
            rem = q;
        }
        const long long a0 = ta * 64, b0 = tb * 64;
#pragma unroll
        for (int j = y; j < 64; j += 16) {          // rows along b, float4 along a
            const long long a = a0 + 4 * x, b = b0 + j;
            if (a < d.size[da] && b < d.size[db]) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(in + ioff + a + b * d.istride[db]));
                tile[j][4 * x] = v.x, tile[j][4 * x + 1] = v.y, tile[j][4 * x + 2] = v.z, tile[j][4 * x + 3] = v.w;
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = y; j < 64; j += 16) {          // rows along a, float4 along b
            const long long a = a0 + j, b = b0 + 4 * x;
            if (a < d.size[da] && b < d.size[db]) {
                float4 v;
                v.x = tile[4 * x][j], v.y = tile[4 * x + 1][j], v.z = tile[4 * x + 2][j], v.w = tile[4 * x + 3][j];
                *reinterpret_cast<float4*>(out + ooff + a * ostride_a + b) = v;
            }
        }
        __syncthreads();
    }
}

// Qx[o] = sign * Q[i(o)] with the two extra output dimensions ri (dim pa) and ro (dim pb):
// c = ri ^ ro, sign = -1 for (ri, ro) = (1, 0); conj flips the sign of c = 1.
template <typename T>
__global__ void __launch_bounds__(256) cplx_expand_kernel(const T* __restrict__ in, T* __restrict__ out, Dims d,
                                                          long long total, int pa, int pb, int conj) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long rem = i, off = 0;
        int ri = 0, ro = 0;
#pragma unroll 1
        for (int k = d.nd - 1; k >= 0; --k) {
            const long long q = rem / d.size[k];
            const long long idx = rem - q * d.size[k];
            if (k == pa)
                ri = (int)idx;
            else if (k == pb)
                ro = (int)idx;
            else
                off += idx * d.istride[k];
            rem = q;
        }
        const int c = ri ^ ro;
        T v = __ldg(in + off + c);
        if ((ri == 1 && ro == 0) != (conj && c == 1)) v = -v;
        out[i] = v;
    }
}

// adjoint: dQ[..., c] = sum_{ri ^ ro = c} sign * dQx[..., ri, ..., ro]; `d` describes dQ (the last
// dimension is c, extent 2) and istride the strides of dQx for the other dimensions.
template <typename T>
__global__ void __launch_bounds__(256) cplx_fold_kernel(const T* __restrict__ in, T* __restrict__ out, Dims d,
                                                        long long total, long long sa, long long sb, int conj,
                                                        int accumulate) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long rem = i, off = 0;
        int c = 0;
#pragma unroll 1
        for (int k = d.nd - 1; k >= 0; --k) {
            const long long q = rem / d.size[k];
            const long long idx = rem - q * d.size[k];
            if (k == d.nd - 1)
                c = (int)idx;
            else
                off += idx * d.istride[k];
            rem = q;
        }
        T v;
        if (c == 0)
            v = __ldg(in + off) + __ldg(in + off + sa + sb);          // (0,0) + (1,1)
        else
            v = __ldg(in + off + sb) - __ldg(in + off + sa);          // (0,1) - (1,0)
        if (conj && c == 1) v = -v;
        out[i] = accumulate ? out[i] + v : v;
    }
}

// ---- contraction of a big tensor with a tiny one over ONE index (+ the complex component) -----------------------------
// The state folding of the large-bond sweep: Bs[c,e,f] = sum_d G[c,d,e,f] s[d] (tneq_qc/contractor/greedy_strategy.py:
// the circuit-state operands of every group, "cdef,...,d,i->..."), complex data in the 2x2-real form:
//     out[a, c, ro] = sum_{d, ri} P[a, d, c, ri] * Q[d, ri, ro]          P: [A][D][C][2] in place, Q: [D][2][2]
// The generic route was transposition (2 x 134 MB at bond 64) + a GEMM with N = 2 (a 128-wide tensor-core tile for two
// columns); here P is read ONCE, coalesced along c, Q sits in shared memory.
template <typename T>
__global__ void __launch_bounds__(256) fold_vec_kernel(const T* __restrict__ P, const T* __restrict__ Q,
                                                      T* __restrict__ out, long long A, int D, long long C) {
    using T2 = typename Pair<T>::type;
    extern __shared__ __align__(16) unsigned char q_raw[];
    T* q = reinterpret_cast<T*>(q_raw);              // [D][4]
    for (int i = threadIdx.x; i < D * 4; i += blockDim.x) q[i] = __ldg(Q + i);
    __syncthreads();
    const long long total = A * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long a = i / C, c = i - a * C;
        const T2* src = reinterpret_cast<const T2*>(P) + a * D * C + c;
        T o0 = 0, o1 = 0;
#pragma unroll 8
        for (int d = 0; d < D; ++d) {
            const T2 v = __ldg(src + (long long)d * C);
            o0 = fma(v.x, q[4 * d], fma(v.y, q[4 * d + 2], o0));
            o1 = fma(v.x, q[4 * d + 1], fma(v.y, q[4 * d + 3], o1));
        }
        T2 o;
        o.x = o0, o.y = o1;
        reinterpret_cast<T2*>(out)[i] = o;
    }
}

// the adjoint (an outer product accumulated in place): T[a, d, c, ri] += sum_ro P[a, c, ro] * Q[d, ri, ro]
template <typename E>
__global__ void __launch_bounds__(256) outer_acc_kernel(const E* __restrict__ P, const E* __restrict__ Q,
                                                       E* __restrict__ T, long long A, int D, long long C) {
    using E2 = typename Pair<E>::type;
    extern __shared__ __align__(16) unsigned char q_raw[];
    E* q = reinterpret_cast<E*>(q_raw);              // [D][4]
    for (int i = threadIdx.x; i < D * 4; i += blockDim.x) q[i] = __ldg(Q + i);
    __syncthreads();
    const long long total = A * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long a = i / C, c = i - a * C;
        const E2 p = __ldg(reinterpret_cast<const E2*>(P) + i);
        E2* dst = reinterpret_cast<E2*>(T) + a * D * C + c;
#pragma unroll 8
        for (int d = 0; d < D; ++d) {
            E2 t = dst[(long long)d * C];
            t.x = fma(p.x, q[4 * d], fma(p.y, q[4 * d + 1], t.x));
            t.y = fma(p.x, q[4 * d + 2], fma(p.y, q[4 * d + 3], t.y));
            dst[(long long)d * C] = t;
        }
    }
}

int fill_dims(Dims& d, int ndim, const int64_t* out_dims, const int64_t* in_strides) {
    if (ndim < 1 || ndim > MAXD) return tnq_internal_fail("tnq_permute: between 1 and 12 dimensions are supported");
    d.nd = ndim;
    for (int k = 0; k < ndim; ++k) {
        if (out_dims[k] <= 0) return tnq_internal_fail("tnq_permute: non-positive extent");
        d.size[k] = out_dims[k];
        d.istride[k] = in_strides[k];
    }
    return 0;
}

// Q of fold_vec / outer_acc sits in dynamic shared memory (16 D bytes in float32, 32 D in float64): above the default
// 48 KB per block (float32: 3072 < D <= 4096, float64: 1536 < D <= 4096) a launch fails unless the kernel opts in to more
template <typename Kernel>
int allow_smem(Kernel kern, size_t bytes, const std::string& what) {
    if (bytes <= 48 * 1024) return 0;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return e == cudaSuccess ? 0 : tnq_internal_cuda_fail(e, what.c_str());
}

int grid_for(long long work, int per_block) {
    long long g = (work + per_block - 1) / per_block;
    const long long cap = 148LL * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}


template <typename T>
int permute_impl(const T* in, T* out, int ndim, const int64_t* out_dims, const int64_t* in_strides, int vec, int conj,
                 void* stream, const char* name) {
    const std::string nm(name);
    constexpr int ES = (int)sizeof(T);
    constexpr int VMAX = 16 / ES;                    // widest vector: 16 bytes
    if (!in || !out || !out_dims || !in_strides) return tnq_internal_fail(nm + ": bad arguments");
    if (vec != 1 && vec != 2 && vec != 4) return tnq_internal_fail(nm + ": vec must be 1, 2 or 4");
    if (vec > VMAX) return tnq_internal_fail(nm + ": vec must be 1 or 2");
    if (conj && vec == 1) return tnq_internal_fail(nm + ": conj needs vec >= 2 (interleaved complex)");
    Dims d;
    if (int rc = fill_dims(d, ndim, out_dims, in_strides)) return rc;
    if (((uintptr_t)in | (uintptr_t)out) & (uintptr_t)(vec * ES - 1))
        return tnq_internal_fail(nm + ": pointers must be aligned to the vector width");
    long long total = 1;
    for (int k = 0; k < ndim; ++k) {
        if (k < ndim - 1 && vec > 1 && (d.istride[k] % vec)) return tnq_internal_fail(nm + ": stride not a multiple of vec");
        total *= d.size[k];
    }
    if (vec > 1 && (d.size[ndim - 1] % vec || d.istride[ndim - 1] != 1))
        return tnq_internal_fail(nm + ": the last dimension must be contiguous and a multiple of vec");
    // ---- canonical form (all in elements): drop extent-1 dimensions, merge neighbours that are adjacent in the input
    // in the same order as in the output (stride[k] == stride[k+1] * size[k+1]): a (.., 64, 2) pair of (index, re/im)
    // becomes one run of 128 contiguous floats, so that a true transposition finds a long input-contiguous dimension
    // for its shared-memory tiles instead of falling back to strided scalar loads (measured on the 537 MB
    // intermediates of the bond-64 sweep: 0.5 TB/s before, see DESIGN section 4)
    {
        int m = 0;
        for (int k = 0; k < d.nd; ++k) {
            if (d.size[k] == 1) continue;
            d.size[m] = d.size[k], d.istride[m] = d.istride[k];
            ++m;
        }
        if (m == 0) d.size[0] = 1, d.istride[0] = 1, m = 1;      // a single element
        d.nd = m;
        for (int k = d.nd - 2; k >= 0; --k) {
            if (d.istride[k] == d.istride[k + 1] * d.size[k + 1]) {
                d.size[k] = d.size[k] * d.size[k + 1];
                d.istride[k] = d.istride[k + 1];
                for (int j = k + 1; j < d.nd - 1; ++j) d.size[j] = d.size[j + 1], d.istride[j] = d.istride[j + 1];
                d.nd -= 1;
            }
        }
    }
    // ---- widest vector that keeps the meaning: the last dimension contiguous in the input, its extent and every
    // other stride a multiple of the width, both pointers aligned (a requested vec = 2 with conj stays >= 2)
    if (d.istride[d.nd - 1] == 1) {
        for (int w = VMAX; w > vec; w >>= 1) {
            bool ok = d.size[d.nd - 1] % w == 0 && !(((uintptr_t)in | (uintptr_t)out) & (uintptr_t)(w * ES - 1));
            for (int k = 0; k < d.nd - 1 && ok; ++k) ok = d.istride[k] % w == 0;
            if (ok) {
                vec = w;
                break;
            }
        }
    }
    // fold the innermost `vec` elements into one vector
    if (vec > 1) {
        d.size[d.nd - 1] /= vec;
        d.istride[d.nd - 1] = vec;
        total /= vec;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // drop a trailing dimension of extent 1 left by the folding (pure complex scalar per element)
    int da = -1;
    if (d.size[d.nd - 1] == 1 && d.nd > 1) d.nd -= 1;
    for (int k = 0; k < d.nd; ++k)
        if (d.istride[k] == vec && d.size[k] > 1) da = k;
    const bool direct = d.istride[d.nd - 1] == vec || d.size[d.nd - 1] == 1 || da < 0 || d.size[d.nd - 1] < 8 ||
                        d.size[da] < 8;
    if (direct) {
        const int grid = grid_for(total, 256 * 4);
        if (vec == 1) permute_direct_kernel<T, 1><<<grid, 256, 0, st>>>(in, out, d, total, conj);
        if (vec == 2) permute_direct_kernel<T, 2><<<grid, 256, 0, st>>>(in, out, d, total, conj);
        if constexpr (VMAX == 4)
            if (vec == 4) permute_direct_kernel<T, 4><<<grid, 256, 0, st>>>(in, out, d, total, conj);
    } else {
        long long ostride_a = 1;
        for (int k = d.nd - 1; k > da; --k) ostride_a *= d.size[k];
        if constexpr (sizeof(T) == 4) {
            bool wide = vec == 1 && !conj && d.size[da] % 4 == 0 && d.size[d.nd - 1] % 4 == 0 && ostride_a % 4 == 0 &&
                        d.size[da] >= 32 && d.size[d.nd - 1] >= 32 && !(((uintptr_t)in | (uintptr_t)out) & 15);
            for (int k = 0; k < d.nd && wide; ++k)
                if (k != da) wide = d.istride[k] % 4 == 0;
            if (wide) {
                long long os = 1;                    // every output stride above the last dimension is a multiple of four
                for (int k = d.nd - 1; k >= 1 && wide; --k) {
                    os *= d.size[k];
                    wide = os % 4 == 0;
                }
            }
            if (wide) {
                const long long tiles_a = (d.size[da] + 63) / 64, tiles_b = (d.size[d.nd - 1] + 63) / 64;
                long long ntiles = tiles_a * tiles_b;
                for (int k = 0; k < d.nd - 1; ++k)
                    if (k != da) ntiles *= d.size[k];
                permute_tiled64_kernel<<<grid_for(ntiles, 1), 256, 0, st>>>(in, out, d, da, ostride_a, tiles_a, tiles_b, ntiles);
                tnq_internal_count_launch();
                cudaError_t e64 = cudaGetLastError();
                if (e64 != cudaSuccess) return tnq_internal_cuda_fail(e64, (nm + " launch").c_str());
                return 0;
            }
        }
        const long long tiles_a = (d.size[da] + 31) / 32, tiles_b = (d.size[d.nd - 1] + 31) / 32;
        long long ntiles = tiles_a * tiles_b;
        for (int k = 0; k < d.nd - 1; ++k)
            if (k != da) ntiles *= d.size[k];
        const int grid = grid_for(ntiles, 1);
        if (vec == 1) permute_tiled_kernel<T, 1><<<grid, 256, 0, st>>>(in, out, d, da, ostride_a, tiles_a, tiles_b, ntiles, conj);
        if (vec == 2) permute_tiled_kernel<T, 2><<<grid, 256, 0, st>>>(in, out, d, da, ostride_a, tiles_a, tiles_b, ntiles, conj);
        if constexpr (VMAX == 4)
            if (vec == 4) permute_tiled_kernel<T, 4><<<grid, 256, 0, st>>>(in, out, d, da, ostride_a, tiles_a, tiles_b, ntiles, conj);
    }
    tnq_internal_count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, (nm + " launch").c_str());
    return 0;
}

template <typename T>
int cplx_expand_impl(const T* in, T* out, int ndim, const int64_t* out_dims, const int64_t* in_strides, int ri_dim,
                     int ro_dim, int conj, void* stream, const char* name) {
    const std::string nm(name);
    if (!in || !out) return tnq_internal_fail(nm + ": bad arguments");
    Dims d;
    if (int rc = fill_dims(d, ndim, out_dims, in_strides)) return rc;
    if (ri_dim < 0 || ro_dim < 0 || ri_dim >= ndim || ro_dim >= ndim || ri_dim == ro_dim || d.size[ri_dim] != 2 ||
        d.size[ro_dim] != 2)
        return tnq_internal_fail(nm + ": ri/ro must be two distinct output dimensions of extent 2");
    long long total = 1;
    for (int k = 0; k < ndim; ++k) total *= d.size[k];
    cplx_expand_kernel<T><<<grid_for(total, 256 * 4), 256, 0, (cudaStream_t)stream>>>(in, out, d, total, ri_dim, ro_dim, conj);
    tnq_internal_count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, (nm + " launch").c_str());
    return 0;
}

template <typename T>
int cplx_fold_impl(const T* in, T* out, int ndim, const int64_t* out_dims, const int64_t* in_strides, int64_t ri_stride,
                   int64_t ro_stride, int conj, int accumulate, void* stream, const char* name) {
    const std::string nm(name);
    if (!in || !out) return tnq_internal_fail(nm + ": bad arguments");
    Dims d;
    if (int rc = fill_dims(d, ndim, out_dims, in_strides)) return rc;
    if (d.size[ndim - 1] != 2) return tnq_internal_fail(nm + ": the last output dimension must be (re, im)");
    long long total = 1;
    for (int k = 0; k < ndim; ++k) total *= d.size[k];
    cplx_fold_kernel<T><<<grid_for(total, 256 * 4), 256, 0, (cudaStream_t)stream>>>(in, out, d, total, ri_stride, ro_stride,
                                                                                    conj, accumulate);
    tnq_internal_count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, (nm + " launch").c_str());
    return 0;
}

// fold_vec (OUTER = false) / outer_acc (OUTER = true): P, out / T hold (re, im) pairs, 2 * sizeof(T)-byte aligned
template <typename T, bool OUTER>
int fold_impl(const T* P, const T* Q, T* out, int64_t A, int64_t D, int64_t C, void* stream, const char* name) {
    const std::string nm(name);
    if (!P || !Q || !out || A <= 0 || D <= 0 || C <= 0 || D > 4096) return tnq_internal_fail(nm + ": bad arguments");
    if (((uintptr_t)P | (uintptr_t)out) & (2 * sizeof(T) - 1))
        return tnq_internal_fail(nm + (sizeof(T) == 4 ? ": pointers must be 8-byte aligned" : ": pointers must be 16-byte aligned"));
    const size_t smem = sizeof(T) * 4 * (size_t)D;
    auto kern = OUTER ? outer_acc_kernel<T> : fold_vec_kernel<T>;
    if (int rc = allow_smem(kern, smem, "cudaFuncSetAttribute(" + nm + ")")) return rc;
    kern<<<grid_for(A * C, 256), 256, smem, (cudaStream_t)stream>>>(P, Q, out, A, (int)D, C);
    tnq_internal_count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, (nm + " launch").c_str());
    return 0;
}

}  // namespace

extern "C" {

int tnq_permute_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                    int vec, int conj, void* stream) {
    return permute_impl(in, out, ndim, out_dims, in_strides, vec, conj, stream, "tnq_permute_f32");
}

int tnq_permute_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                    int vec, int conj, void* stream) {
    return permute_impl(in, out, ndim, out_dims, in_strides, vec, conj, stream, "tnq_permute_f64");
}

int tnq_cplx_expand_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                        int ri_dim, int ro_dim, int conj, void* stream) {
    return cplx_expand_impl(in, out, ndim, out_dims, in_strides, ri_dim, ro_dim, conj, stream, "tnq_cplx_expand_f32");
}

int tnq_cplx_expand_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                        int ri_dim, int ro_dim, int conj, void* stream) {
    return cplx_expand_impl(in, out, ndim, out_dims, in_strides, ri_dim, ro_dim, conj, stream, "tnq_cplx_expand_f64");
}

int tnq_cplx_fold_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                      int64_t ri_stride, int64_t ro_stride, int conj, int accumulate, void* stream) {
    return cplx_fold_impl(in, out, ndim, out_dims, in_strides, ri_stride, ro_stride, conj, accumulate, stream,
                          "tnq_cplx_fold_f32");
}

int tnq_cplx_fold_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                      int64_t ri_stride, int64_t ro_stride, int conj, int accumulate, void* stream) {
    return cplx_fold_impl(in, out, ndim, out_dims, in_strides, ri_stride, ro_stride, conj, accumulate, stream,
                          "tnq_cplx_fold_f64");
}

int tnq_fold_vec_f32(const float* P, const float* Q, float* out, int64_t A, int64_t D, int64_t C, void* stream) {
    return fold_impl<float, false>(P, Q, out, A, D, C, stream, "tnq_fold_vec_f32");
}

int tnq_fold_vec_f64(const double* P, const double* Q, double* out, int64_t A, int64_t D, int64_t C, void* stream) {
    return fold_impl<double, false>(P, Q, out, A, D, C, stream, "tnq_fold_vec_f64");
}

int tnq_outer_acc_f32(const float* P, const float* Q, float* T, int64_t A, int64_t D, int64_t C, void* stream) {
    return fold_impl<float, true>(P, Q, T, A, D, C, stream, "tnq_outer_acc_f32");
}

int tnq_outer_acc_f64(const double* P, const double* Q, double* T, int64_t A, int64_t D, int64_t C, void* stream) {
    return fold_impl<double, true>(P, Q, T, A, D, C, stream, "tnq_outer_acc_f64");
}

}  // extern "C"
