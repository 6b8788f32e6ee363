// tnq_sgdg.cu -- the Stiefel-manifold SGD step (Cayley transform) of the reference optimizer for ALL
// cores of a network in one launch: one CTA per core, every matrix in shared memory.
//
// Reference: tneq_qc/backends/backend_pytorch.py:349-468 (_sgdg_step), per core ~20 small torch
// kernels (norm, 4 mm, inverse, ...); for the 46 cores of the 24-qubit two-layer network that is
// ~1000 launches per optimizer step, far more than the fused contraction itself.
//
// Per core (p viewed as d x D, d = product of the first half of its dims; Stiefel case d <= D;
// ^H is the conjugate transpose, the plain transpose for real cores):
//   X  = p / (||p||_row + 1e-8)                              V  = momentum * V - g^H
//   MX = V X      XMX = X MX      W^ = MX - 1/2 X^H XMX      W = W^ - W^H
//   alpha = min(lr, 1 / (||W||_1 + 1e-8))                    (||.||_1 = max column sum of moduli)
//   Y  = (I - alpha/2 W)^-1 (I + alpha/2 W) X^H              p_new = Y^H        V_new = W X^H
// The 1 % random QR retraction of the reference (backend_pytorch.py:382) is decided on the host.
//
// The kernel is a template on the element type: float, double, and complex numbers in float and in double
// (interleaved (re, im) pairs, Cx below).
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "tneq_b200.h"

extern int tnq_internal_fail(const std::string& msg);
extern int tnq_internal_cuda_fail(cudaError_t e, const char* what);
extern void tnq_internal_count_launch();

namespace {

constexpr int SG_THREADS = 128;

template <class R>
struct __align__(2 * sizeof(R)) Cx {
    R re, im;
};

template <class E> struct RealOf { using type = E; };
template <class R> struct RealOf<Cx<R>> { using type = R; };
template <class E> using real_t = typename RealOf<E>::type;

template <class R> __device__ __forceinline__ Cx<R> operator+(Cx<R> a, Cx<R> b) { return {a.re + b.re, a.im + b.im}; }
template <class R> __device__ __forceinline__ Cx<R> operator-(Cx<R> a, Cx<R> b) { return {a.re - b.re, a.im - b.im}; }
template <class R> __device__ __forceinline__ Cx<R> operator-(Cx<R> a) { return {-a.re, -a.im}; }
template <class R> __device__ __forceinline__ Cx<R> operator*(R s, Cx<R> a) { return {s * a.re, s * a.im}; }
template <class R> __device__ __forceinline__ Cx<R> operator/(Cx<R> a, R s) { return {a.re / s, a.im / s}; }
template <class R> __device__ __forceinline__ Cx<R> operator*(Cx<R> a, Cx<R> b) {
    return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re};
}
template <class R> __device__ __forceinline__ Cx<R>& operator*=(Cx<R>& a, Cx<R> b) { return a = a * b; }

// a * b + c
__device__ __forceinline__ float madd(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double madd(double a, double b, double c) { return fma(a, b, c); }
template <class R> __device__ __forceinline__ Cx<R> madd(Cx<R> a, Cx<R> b, Cx<R> c) {
    return {madd(a.re, b.re, madd(-a.im, b.im, c.re)), madd(a.re, b.im, madd(a.im, b.re, c.im))};
}
template <class R> __device__ __forceinline__ R cj(R x) { return x; }
template <class R> __device__ __forceinline__ Cx<R> cj(Cx<R> z) { return {z.re, -z.im}; }
// |z|^2 + acc
template <class R> __device__ __forceinline__ R norm2_acc(R x, R acc) { return madd(x, x, acc); }
template <class R> __device__ __forceinline__ R norm2_acc(Cx<R> z, R acc) { return madd(z.re, z.re, madd(z.im, z.im, acc)); }
// |z| (the modulus, as torch.abs)
template <class R> __device__ __forceinline__ R mag(R x) { return fabs(x); }
template <class R> __device__ __forceinline__ R mag(Cx<R> z) { return hypot(z.re, z.im); }
// pivot size |re| + |im| (LAPACK's cabs1): I - a/2 W with skew-Hermitian W has all singular values >= 1
template <class R> __device__ __forceinline__ R pivmag(R x) { return fabs(x); }
template <class R> __device__ __forceinline__ R pivmag(Cx<R> z) { return fabs(z.re) + fabs(z.im); }
template <class R> __device__ __forceinline__ R recip(R x) { return R(1) / x; }
template <class R> __device__ __forceinline__ Cx<R> recip(Cx<R> z) {
    const R s = R(1) / madd(z.re, z.re, z.im * z.im);
    return {z.re * s, -z.im * s};
}
template <class E> __device__ __forceinline__ E from_real(real_t<E> x) { return E{x}; }

// Shared-memory matrices of maxd x (maxd + 1) elements.  With 8- and 16-byte elements T shares V's buffer (V is
// dead once MX = V X is formed): six buffers, so that width 64 fits the opt-in 227 KB of an sm_100 block in 8 bytes
// and width 48 in 16 bytes.  float32 keeps its separate T (seven buffers; width 64 fits either way).
template <class E> __host__ __device__ constexpr int sg_buffers() { return sizeof(E) == 4 ? 7 : 6; }

// C[m x n] = A[m x k] * B[k x n], all row major in shared memory with leading dimension ld; at / bt: the operand
// is read conjugate-transposed
template <class E>
__device__ __forceinline__ void mm(E* C, const E* A, const E* B, int m, int k, int n, int ld, bool at = false,
                                   bool bt = false) {
    for (int i = threadIdx.x; i < m * n; i += blockDim.x) {
        const int r = i / n, c = i % n;
        E s = from_real<E>(0);
        for (int j = 0; j < k; ++j) s = madd(at ? cj(A[j * ld + r]) : A[r * ld + j], bt ? cj(B[c * ld + j]) : B[j * ld + c], s);
        C[r * ld + c] = s;
    }
    __syncthreads();
}

template <class E>
__global__ void __launch_bounds__(SG_THREADS)
tnq_sgdg_kernel(E* const* __restrict__ params, const E* const* __restrict__ grads, E* const* __restrict__ vel,
                const int* __restrict__ rows, const int* __restrict__ cols, int maxd, real_t<E> lr, real_t<E> momentum,
                E* pbase, const E* gbase, E* vbase, const long long* __restrict__ offs) {
    using R = real_t<E>;
    constexpr int nb = sg_buffers<E>();
    extern __shared__ __align__(16) unsigned char sg_smem[];
    E* sm = reinterpret_cast<E*>(sg_smem);
    const int d = rows[blockIdx.x], D = cols[blockIdx.x];      // p is d x D with d <= D; W is D x D
    const int ld = maxd + 1, sz = maxd * ld;
    E *X = sm, *V = sm + sz, *MX = sm + 2 * sz, *T = sm + (nb == 7 ? 3 : 1) * sz, *W = sm + (nb - 3) * sz,
      *L = sm + (nb - 2) * sz, *Rm = sm + (nb - 1) * sz;
    __shared__ R red[SG_THREADS];
    __shared__ R s_alpha;
    __shared__ int piv;
    // flat form: three base pointers + a static table of element offsets [3][ncores] (params | grads | velocity)
    E* p = offs ? pbase + offs[blockIdx.x] : params[blockIdx.x];
    const E* g = offs ? gbase + offs[gridDim.x + blockIdx.x] : grads[blockIdx.x];
    E* v = offs ? vbase + offs[2 * gridDim.x + blockIdx.x] : vel[blockIdx.x];
    const R eps = R(1e-8);
    // X (d x D) = row-normalised p ; V (D x d) = momentum * V - g^H
    for (int r = threadIdx.x; r < d; r += blockDim.x) {
        R nrm = 0;
        for (int c = 0; c < D; ++c) nrm = norm2_acc(p[r * D + c], nrm);
        nrm = sqrt(nrm) + eps;
        for (int c = 0; c < D; ++c) X[r * ld + c] = p[r * D + c] / nrm;
    }
    for (int i = threadIdx.x; i < D * d; i += blockDim.x) {
        const int r = i / d, c = i % d;
        V[r * ld + c] = momentum * v[i] - cj(g[c * D + r]);
    }
    __syncthreads();
    mm(MX, V, X, D, d, D, ld);                 // MX   = V X        (D x D)
    mm(T, X, MX, d, D, D, ld);                 // XMX  = X MX       (d x D)
    mm(W, X, T, D, d, D, ld, /*at=*/true);     // XXMX = X^H XMX    (D x D, into W temporarily)
    for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
        const int r = i / D, c = i % D;
        L[r * ld + c] = MX[r * ld + c] - R(0.5) * W[r * ld + c];   // W^
    }
    __syncthreads();
    for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
        const int r = i / D, c = i % D;
        W[r * ld + c] = L[r * ld + c] - cj(L[c * ld + r]);
    }
    __syncthreads();
    // ||W||_1 = max over columns of the column sum of moduli
    R best = 0;
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        R s = 0;
        for (int r = 0; r < D; ++r) s += mag(W[r * ld + c]);
        best = fmax(best, s);
    }
    red[threadIdx.x] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        R m = 0;
        for (int i = 0; i < blockDim.x; ++i) m = fmax(m, red[i]);
        s_alpha = fmin(R(0.5) * R(2) / (m + eps), lr);
    }
    __syncthreads();
    const R ha = R(0.5) * s_alpha;
    // L = I - a/2 W  (inverted into Rm by Gauss-Jordan), MX <- I + a/2 W
    for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
        const int r = i / D, c = i % D;
        const E id = from_real<E>(r == c ? R(1) : R(0));
        L[r * ld + c] = id - ha * W[r * ld + c];
        MX[r * ld + c] = id + ha * W[r * ld + c];
        Rm[r * ld + c] = id;
    }
    __syncthreads();
    for (int k = 0; k < D; ++k) {              // Gauss-Jordan with partial pivoting
        if (threadIdx.x == 0) {
            int bi = k;
            R bv = pivmag(L[k * ld + k]);
            for (int r = k + 1; r < D; ++r)
                if (pivmag(L[r * ld + k]) > bv) bv = pivmag(L[r * ld + k]), bi = r;
            piv = bi;
        }
        __syncthreads();
        if (piv != k) {
            for (int c = threadIdx.x; c < D; c += blockDim.x) {
                E t0 = L[k * ld + c];
                L[k * ld + c] = L[piv * ld + c];
                L[piv * ld + c] = t0;
                t0 = Rm[k * ld + c];
                Rm[k * ld + c] = Rm[piv * ld + c];
                Rm[piv * ld + c] = t0;
            }
        }
        __syncthreads();
        const E inv = recip(L[k * ld + k]);
        __syncthreads();
        for (int c = threadIdx.x; c < D; c += blockDim.x) {
            L[k * ld + c] *= inv;
            Rm[k * ld + c] *= inv;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
            const int r = i / D, c = i % D;
            if (r == k) continue;
            const E f = L[r * ld + k];
            // column k of L is read by every thread of this sweep: it is cleared afterwards
            if (c != k) L[r * ld + c] = madd(-f, L[k * ld + c], L[r * ld + c]);
            Rm[r * ld + c] = madd(-f, Rm[k * ld + c], Rm[r * ld + c]);
        }
        __syncthreads();
        for (int r = threadIdx.x; r < D; r += blockDim.x)
            if (r != k) L[r * ld + k] = from_real<E>(0);
        __syncthreads();
    }
    mm(T, Rm, MX, D, D, D, ld);                      // T = L^-1 (I + a/2 W)     (D x D)
    mm(L, T, X, D, D, d, ld, false, /*bt=*/true);    // Y = T X^H                (D x d)
    mm(Rm, W, X, D, D, d, ld, false, /*bt=*/true);   // V_new = W X^H            (D x d)
    for (int i = threadIdx.x; i < d * D; i += blockDim.x) {
        const int r = i / D, c = i % D;
        p[i] = cj(L[c * ld + r]);                    // p_new = Y^H              (d x D)
    }
    for (int i = threadIdx.x; i < D * d; i += blockDim.x) v[i] = Rm[(i / d) * ld + i % d];
}

// Width check, shared-memory opt-in and the launch; table != nullptr selects the flat form.
template <class E>
int sgdg_launch(const char* name, int max_allowed, E* const* params, const E* const* grads, E* const* velocity,
                const int* rows, const int* cols, int ncores, int max_cols, real_t<E> lr, real_t<E> momentum, E* pbase,
                const E* gbase, E* vbase, const int64_t* table, void* stream) {
    if (max_cols < 1 || max_cols > max_allowed)
        return tnq_internal_fail(std::string(name) + ": matrix width must be between 1 and " + std::to_string(max_allowed));
    const int d = max_cols;
    const size_t smem = sizeof(E) * sg_buffers<E>() * (size_t)d * (d + 1);
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(tnq_sgdg_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, "cudaFuncSetAttribute(sgdg)");
    tnq_sgdg_kernel<E><<<ncores, SG_THREADS, smem, (cudaStream_t)stream>>>(params, grads, velocity, rows, cols, d, lr,
                                                                            momentum, pbase, gbase, vbase,
                                                                            reinterpret_cast<const long long*>(table));
    tnq_internal_count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return tnq_internal_cuda_fail(e, (std::string(name) + " launch").c_str());
    return 0;
}

template <class E, class P>
int sgdg_step(const char* name, int max_allowed, P* const* params, const P* const* grads, P* const* velocity,
              const int* rows, const int* cols, int ncores, int max_cols, real_t<E> lr, real_t<E> momentum, void* stream) {
    if (!params || !grads || !velocity || !rows || !cols || ncores <= 0)
        return tnq_internal_fail(std::string(name) + ": bad arguments");
    return sgdg_launch<E>(name, max_allowed, reinterpret_cast<E* const*>(params),
                          reinterpret_cast<const E* const*>(grads), reinterpret_cast<E* const*>(velocity), rows, cols,
                          ncores, max_cols, lr, momentum, nullptr, nullptr, nullptr, nullptr, stream);
}

template <class E, class P>
int sgdg_step_flat(const char* name, int max_allowed, P* params, const P* grads, P* velocity, const int64_t* offsets,
                   const int* rows, const int* cols, int ncores, int max_cols, real_t<E> lr, real_t<E> momentum,
                   void* stream) {
    if (!params || !grads || !velocity || !offsets || !rows || !cols || ncores <= 0)
        return tnq_internal_fail(std::string(name) + ": bad arguments");
    return sgdg_launch<E>(name, max_allowed, nullptr, nullptr, nullptr, rows, cols, ncores, max_cols, lr, momentum,
                          reinterpret_cast<E*>(params), reinterpret_cast<const E*>(grads),
                          reinterpret_cast<E*>(velocity), offsets, stream);
}

}  // namespace

extern "C" int tnq_sgdg_step(float* const* params, const float* const* grads, float* const* velocity, const int* rows,
                             const int* cols, int ncores, int max_cols, float lr, float momentum, void* stream) {
    return sgdg_step<float>("tnq_sgdg_step", TNQ_SGDG_MAX_COLS, params, grads, velocity, rows, cols, ncores, max_cols,
                            lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_flat(float* params, const float* grads, float* velocity, const int64_t* offsets,
                                  const int* rows, const int* cols, int ncores, int max_cols, float lr, float momentum,
                                  void* stream) {
    return sgdg_step_flat<float>("tnq_sgdg_step_flat", TNQ_SGDG_MAX_COLS, params, grads, velocity, offsets, rows, cols,
                                 ncores, max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_c64(float* const* params, const float* const* grads, float* const* velocity,
                                 const int* rows, const int* cols, int ncores, int max_cols, float lr, float momentum,
                                 void* stream) {
    return sgdg_step<Cx<float>>("tnq_sgdg_step_c64", TNQ_SGDG_MAX_COLS_C64, params, grads, velocity, rows, cols,
                                ncores, max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_flat_c64(float* params, const float* grads, float* velocity, const int64_t* offsets,
                                      const int* rows, const int* cols, int ncores, int max_cols, float lr,
                                      float momentum, void* stream) {
    return sgdg_step_flat<Cx<float>>("tnq_sgdg_step_flat_c64", TNQ_SGDG_MAX_COLS_C64, params, grads, velocity, offsets,
                                     rows, cols, ncores, max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_f64(double* const* params, const double* const* grads, double* const* velocity,
                                 const int* rows, const int* cols, int ncores, int max_cols, double lr, double momentum,
                                 void* stream) {
    return sgdg_step<double>("tnq_sgdg_step_f64", TNQ_SGDG_MAX_COLS_F64, params, grads, velocity, rows, cols, ncores,
                             max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_flat_f64(double* params, const double* grads, double* velocity, const int64_t* offsets,
                                      const int* rows, const int* cols, int ncores, int max_cols, double lr,
                                      double momentum, void* stream) {
    return sgdg_step_flat<double>("tnq_sgdg_step_flat_f64", TNQ_SGDG_MAX_COLS_F64, params, grads, velocity, offsets,
                                  rows, cols, ncores, max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_c128(double* const* params, const double* const* grads, double* const* velocity,
                                  const int* rows, const int* cols, int ncores, int max_cols, double lr,
                                  double momentum, void* stream) {
    return sgdg_step<Cx<double>>("tnq_sgdg_step_c128", TNQ_SGDG_MAX_COLS_C128, params, grads, velocity, rows, cols,
                                 ncores, max_cols, lr, momentum, stream);
}

extern "C" int tnq_sgdg_step_flat_c128(double* params, const double* grads, double* velocity, const int64_t* offsets,
                                       const int* rows, const int* cols, int ncores, int max_cols, double lr,
                                       double momentum, void* stream) {
    return sgdg_step_flat<Cx<double>>("tnq_sgdg_step_flat_c128", TNQ_SGDG_MAX_COLS_C128, params, grads, velocity,
                                      offsets, rows, cols, ncores, max_cols, lr, momentum, stream);
}
