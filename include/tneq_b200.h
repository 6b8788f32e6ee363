/*
 * tneq_b200 C ABI  --  libtneq_b200.so
 *
 * Drop-in boundary for ONE path of the reference (tneq_qc): contracting a QCTN
 * against a batch of measurement matrices (probabilities / loss / core
 * gradients).  The reference has no FFI for this path: its boundary is the two
 * Python plug-in registries BackendFactory.register_backend
 * (tneq_qc/backends/backend_factory.py:91-100) and
 * StrategyCompiler.register_strategy (tneq_qc/contractor/compiler.py:38-54).
 * The Python host code in this repository implements those two interfaces and
 * calls the functions below through ctypes; every entry point names the
 * reference code it replaces.  INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *   - plain C types only; all device memory is owned by the caller (PyTorch);
 *   - every function returns 0 on success, non-zero on error; the message is
 *     available from tnq_last_error() (thread local);
 *   - all work is enqueued on the CUDA stream passed in (a cudaStream_t cast to
 *     void*); no hidden synchronisation; a plan is used by one host thread at a
 *     time and belongs to the CUDA device that was current at creation;
 *   - there is no CPU fallback: without a CUDA device every call fails.
 */
#ifndef TNEQ_B200_H
#define TNEQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TNQ_MAX_INPUTS 192
#define TNQ_MAX_OUTPUTS 128
#define TNQ_CHAIN_MAX_QUBITS 64

typedef struct tnq_plan tnq_plan_t;

/* Launch geometry chosen for a plan at a given batch (reported for bench/roofline). */
typedef struct tnq_run_info {
    int32_t tile_samples;     /* samples per tile (S) */
    int32_t grid;             /* CTAs of the BODY kernel */
    int32_t frame_in_smem;    /* 1: per-tile working set lives in shared memory */
    int32_t launches;         /* kernels launched by one tnq_plan_run */
    int64_t smem_bytes;       /* dynamic shared memory per CTA */
    int64_t workspace_bytes;  /* scratch the caller must provide */
} tnq_run_info_t;

/* Library / device sanity: 0 when a CUDA device of compute capability 10.x is current. */
int tnq_device_check(void);

/*
 * A plan is one compiled contraction program: the complete qubit sweep of
 * GreedyStrategy.compute_fn (tneq_qc/contractor/greedy_strategy.py:45-598)
 * -- optionally followed by the fused loss of
 * EngineSiamese.contract_with_compiled_strategy_for_gradient
 * (tneq_qc/core/engine_siamese.py:441-530) and the reverse sweep that
 * torch.autograd.grad performs in BackendPyTorch.compute_value_and_grad
 * (tneq_qc/backends/backend_pytorch.py:107-166).
 * `blob` is the int64 encoding produced by contractor/vm_program.py.
 */
int tnq_plan_create(const int64_t* blob, int64_t nwords, tnq_plan_t** out);
void tnq_plan_destroy(tnq_plan_t* plan);

int tnq_plan_num_inputs(const tnq_plan_t* plan);
int tnq_plan_num_outputs(const tnq_plan_t* plan);
int tnq_plan_query(const tnq_plan_t* plan, int64_t nsamples, tnq_run_info_t* info);

/*
 * Run the plan on `nsamples` samples (= batch size x 2 when measurements are
 * stacked (B,2,K,K), engine_siamese.py:683-719).
 *   in_ptrs[i]        device pointer of input slot i (cores, circuit states,
 *                     per-qubit measurement matrices, optional grad seed);
 *   in_stride_hi/lo   for batched inputs: element offset of sample s is
 *                     (s / nb) * hi + (s % nb) * lo  (nb is stored in the plan);
 *   out_ptrs[j]       device pointer of output slot j (batched outputs are
 *                     [nsamples, elems] row-major; shared ones [elems]);
 *   scalars           host array {log_scale, 1/count}: the summed TNTensor
 *                     log-scale and the mean weight of the fused loss;
 *   workspace         device scratch of at least tnq_plan_query().workspace_bytes.
 */
int tnq_plan_run(tnq_plan_t* plan, int64_t nsamples, const void* const* in_ptrs,
                 const int64_t* in_stride_hi, const int64_t* in_stride_lo, void* const* out_ptrs,
                 const double* scalars, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Register-resident sweep for single-layer MPS networks (the reference's default graph,
 * QCTNHelper.generate_example_graph(graph_type="mps")), float32, edge rank K in {2,3,4}: the whole
 * greedy sweep greedy_strategy.py:461-598 -- and for mode != 0 the loss engine_siamese.py:490-530 and
 * the reverse sweep -- in one kernel with the K x K environment in registers.
 *   cores[q]  q < n-1 : [K][K][K][K]   states[q] : [K]   mx[q] : sample b at mx[q] + b * mx_stride[q], [K][K]
 *   mode 0: values[B]                       mode 1: values[B] (optional), *loss, grads[q] (fused loss)
 *   mode 2: grads[q] seeded by seed[B] = d loss / d value (torch.autograd route)
 */
int64_t tnq_mps_chain_workspace_bytes(int K, int n, int64_t B);
int tnq_mps_chain(int K, int n, const float* const* cores, const float* const* states, const float* const* mx,
                  const int64_t* mx_stride, int64_t B, int mode, const float* seed, float* values, float* loss,
                  float* const* grads, double log_scale, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * The same sweep (forward values) with the measurement matrices generated IN REGISTERS from x: opt-in fusion of
 * EngineSiamese.generate_data (tneq_qc/core/engine_siamese.py:59-111 weights and Hermite recurrence, :133-254)
 * into the contraction (SURVEY 8f2).  phi_k(x) = w_k sqrt(exp(-x^2/2)) He_k(x), Mx = phi phi^T / scale[q] with
 * scale[q] = max over the batch of |phi phi^T| (TNTensor.auto_scale, tn_tensor.py:72-85) computed by a first
 * kernel.  The sweep reads n floats per sample instead of n K^2.
 *   x: sample b, qubit q at x[b * xs_b + q * xs_q];  weights[K] (host);  scale[n] (device, out)
 *   values[B]: contraction of the scaled matrices; the true value is values * prod_q scale[q].
 */
int tnq_mps_chain_x(int K, int n, const float* const* cores, const float* const* states, const float* x, int64_t xs_b,
                    int64_t xs_q, const float* weights, int64_t B, float* scale, float* values, void* stream);

/*
 * sample() with prefix environments for single-layer MPS networks (SURVEY 8f3; replaces the n full forwards at batch
 * num_samples x grid_size of EngineSiamese.sample, tneq_qc/core/engine_siamese.py:740-915: grid expansion :802-822,
 * forward :842-847, inverse CDF :855-905).  One thread per sample walks the chain once: left environment in
 * registers, right environments (identity measurements) shared, the value linear in the measurement matrix of the
 * qubit being sampled, cumulative sum / search / interpolation / generate_data of the sampled value on the device.
 *   grid_x[G]; mx_grid[G][K][K] = generate_data(grid_x); u[S][n] uniform numbers in the reference's draw order
 *   (one (S,1) draw per qubit; qubit q of sample s at u[s*n + q]); weights[K] (host) -> samples[S][n].
 */
int tnq_mps_chain_sample(int K, int n, const float* const* cores, const float* const* states, int64_t S, int G,
                         const float* grid_x, const float* mx_grid, const float* u, const float* weights, float* samples,
                         void* stream);

/*
 * Warp-level sweep for TWO-LAYER merged MPS networks (QCTN.merge(mps_n, mps_n), reference
 * tneq_qc/core/qctn.py:1296-1506; BASELINE cfg3), float32, edge rank K in {2,3}, n >= 3: the greedy
 * sweep greedy_strategy.py:461-598 with its rank-6 environment kept in shared memory by the warp that
 * owns the sample -- and for mode != 0 the loss engine_siamese.py:490-530 and the reverse sweep -- in
 * one kernel (csrc/tnq_ladder.cu).
 *   cores_a[q], cores_x[q], q < n-1 : first / second layer core on wires (q, q+1), [K][K][K][K]
 *   states[q] : [K]     mx[q] : sample b at mx[q] + b * mx_stride[q], [K][K]
 *   mode 0: values[B]      mode 1: values[B] (optional), *loss, grads_a[q], grads_x[q] (fused loss)
 *   mode 2: grads seeded by seed[B] = d loss / d value (torch.autograd route)
 * workspace: tnq_mps_ladder_workspace_bytes(K, n, B, mode) bytes (per-warp checkpoints and
 * gradient slices; bounded by the number of resident warps, not by B).
 */
int64_t tnq_mps_ladder_workspace_bytes(int K, int n, int64_t B, int mode);
/*
 * The same sweep, second generation (csrc/tnq_ladder2.cu, edge rank 3; tnq_mps_ladder dispatches K = 3 here):
 * a lane is a sample, tiles of 32/R samples per 4-warp CTA (R = 1, 2, 4, 8 picked from B and the SM count),
 * core tensors as uniform operands from constant memory, the rank-6 environment kept in registers (phase C of
 * a step fused with phase A of the next), T2 the only per-sample state checkpointed to HBM, the environment
 * re-derived in the reverse sweep.  Same arguments and modes as tnq_mps_ladder.  The constant pool is one
 * per device: launches must be stream-ordered with each other (one stream, or events between streams).
 *   tnq_mps_ladder2_geometry: out[6] = {R, samples per tile, tiles, CTAs, dynamic shared bytes, warps per CTA} for (n, B, mode).
 */
int64_t tnq_mps_ladder2_workspace_bytes(int n, int64_t B, int mode);
int tnq_mps_ladder2_geometry(int n, int64_t B, int mode, int64_t* out);
int tnq_mps_ladder2(int n, const float* const* cores_a, const float* const* cores_x, const float* const* states,
                    const float* const* mx, const int64_t* mx_stride, int64_t B, int mode, const float* seed,
                    float* values, float* loss, float* const* grads_a, float* const* grads_x, double log_scale,
                    void* workspace, int64_t workspace_bytes, void* stream);
int tnq_mps_ladder(int K, int n, const float* const* cores_a, const float* const* cores_x,
                   const float* const* states, const float* const* mx, const int64_t* mx_stride, int64_t B, int mode,
                   const float* seed, float* values, float* loss, float* const* grads_a, float* const* grads_x,
                   double log_scale, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Large-bond-dimension regime: one pairwise contraction of the sweep as a batched GEMM on the
 * tcgen05 tensor cores with fp32-faithful 3xTF32 arithmetic (replaces the bmm that torch.einsum
 * dispatches for greedy_strategy.py:940,959 when the bond dimension is 64-128):
 *     C[b] (M x N, row major, ldc) (=|+=) A[b] (M x K, row major, lda) * B[b]^T,  B[b] is N x K (ldb)
 * Operands whose K, leading dimensions, batch strides (multiples of 4 floats) and base addresses
 * (16 bytes) are aligned take 16-byte loads; anything else works through guarded scalar loads.
 * A batch stride of 0 shares that operand across the batch.
 */
int tnq_gemm_tf32x3(const float* A, const float* B, float* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                    int64_t ldb, int64_t ldc, int64_t batch, int64_t strideA, int64_t strideB, int64_t strideC,
                    int accumulate, void* stream);
/*
 * The same contraction in float64 (float64 / complex128 networks at large bond dimension) on the FP64 tensor
 * cores (mma.sync m8n8k4 f64, csrc/tnq_gemm_f64.cu), same arguments with leading dimensions and batch strides
 * in doubles.  Any M, N, K >= 1; 16-byte loads where K, lda / ldb, the batch strides (even) and the base
 * addresses (16 bytes) allow, 8-byte loads otherwise; pointers 8-byte aligned.  Deterministic: a fixed
 * summation order per output (a long k-loop on few tiles is split in two halves added with red.global.add.f64).
 */
int tnq_gemm_f64(const double* A, const double* B, double* C, int64_t M, int64_t N, int64_t K, int64_t lda,
                 int64_t ldb, int64_t ldc, int64_t batch, int64_t strideA, int64_t strideB, int64_t strideC,
                 int accumulate, void* stream);
/* Launch resources of one variant of the GEMM kernel: out[4] = {registers per thread, max threads per block,
 * static shared bytes, threads per block the launch uses}. */
/*
 * Batch-into-K GEMM (the gradients of shared tensors: the sample index joins the contracted indices,
 * torch.autograd through torch.einsum in the reference, tneq_qc/core/engine_siamese.py:476,537):
 *   C[m, n] = sum_{b, k} A_b[m, k] * B_b[n, k],  K = batch x Kin.
 * An operand is K-major and contiguous, X[rows][batch * Kin] (x_mn = 0), or MN-major IN PLACE,
 * X[batch][x_tiles][Kin][128] with rows = 128 x_tiles (x_mn = 1): read through a 5-D tensor map and consumed by the
 * tensor core through MN-major shared-memory descriptors, i.e. without the transposition.  -2: not expressible, nothing launched.
 */
int tnq_gemm_tf32x3_bk(const float* A, int a_mn, int64_t a_tiles, const float* B, int b_mn, int64_t b_tiles, float* C,
                       int64_t M, int64_t N, int64_t batch, int64_t Kin, void* stream);
/*
 * Contraction of a big tensor with a tiny one over ONE index and the complex component -- the circuit-state operands
 * of every greedy group ("cdef,...,d,i->...": Bs[c,e,f] = sum_d G[c,d,e,f] s[d], tneq_qc/contractor/greedy_strategy.py:690-990)
 * at large bond dimension, complex data in the 2x2-real form -- and its adjoint, both in ONE pass over the big tensor
 * (the generic route: a transposition of the 134 MB core plus a GEMM with two columns):
 *   tnq_fold_vec_f32 : out[a, c, ro]  = sum_{d, ri} P[a, d, c, ri] * Q[d, ri, ro]      P [A][D][C][2], Q [D][2][2]
 *   tnq_outer_acc_f32: T[a, d, c, ri] += sum_ro     P[a, c, ro]    * Q[d, ri, ro]      P [A][C][2],    T [A][D][C][2]
 * D <= 4096 (Q is staged in shared memory); P, out and T 8-byte aligned.
 * The _f64 versions: the same on doubles (complex128), P, out and T 16-byte aligned.
 */
int tnq_fold_vec_f32(const float* P, const float* Q, float* out, int64_t A, int64_t D, int64_t C, void* stream);
int tnq_outer_acc_f32(const float* P, const float* Q, float* T, int64_t A, int64_t D, int64_t C, void* stream);
int tnq_fold_vec_f64(const double* P, const double* Q, double* out, int64_t A, int64_t D, int64_t C, void* stream);
int tnq_outer_acc_f64(const double* P, const double* Q, double* T, int64_t A, int64_t D, int64_t C, void* stream);
int tnq_gemm_kernel_attrs(int aligned, int smallk, int* out);
/*
 * The same GEMM with the index permutation of the A operand done by the TMA unit: A is a strided 4-level VIEW
 * (rows m = r1 * R0 + r0, contraction index k = k1 * K0 + k0, element at A + r1*sR1 + r0*sR0 + k1*sK1 + k0, strides in
 * floats), e.g. the B x chi^3 intermediate [b, i, j, (k,l)] of the bond-64 sweep read as rows (b, j) x K (i, k, l)
 * without the explicit transposition the reference's einsum performs (permute + reshape + bmm,
 * tneq_qc/contractor/greedy_strategy.py:940,959).  B: N x K row major (ldb); C: M x N row major (ldc).
 * Returns -2 WITHOUT launching when the view is not expressible as a tensor map (alignment; K0 % 32; R0 neither a
 * multiple nor a divisor of 128; K <= 256): the caller then transposes with tnq_permute_f32 and calls tnq_gemm_tf32x3.
 */
int tnq_gemm_tf32x3_view(const float* A, int64_t R1, int64_t R0, int64_t sR1, int64_t sR0, int64_t K1, int64_t K0,
                         int64_t sK1, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t N, void* stream);

/*
 * Index permutation / merge / split of a dense fp32 tensor (what torch.einsum does around every
 * bmm, greedy_strategy.py:940,959; cf. tools/stage3_memory_permute/test_transpose_cost.py).
 * `out` is compact row-major over out_dims[ndim]; in_strides[d] is the stride, in floats, of
 * output dimension d in `in`.  The innermost `vec` floats (1, 2 = one complex number, or 4)
 * move together and must be contiguous on both sides.  conj != 0 negates the imaginary parts.
 * tnq_permute_f64: the same for float64 tensors, strides in doubles, vec 1 or 2 (2 = one complex128 number).
 */
int tnq_permute_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                    int vec, int conj, void* stream);
int tnq_permute_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                    int vec, int conj, void* stream);

/*
 * Complex -> 2x2-real expansion fused with a permutation:
 *   out[..., ri, ..., ro] = E[ri][ro][c] * in[..., c],  E = [[re, im], [-im, re]]
 * ri_dim / ro_dim are the positions of the two extra (extent-2) output dimensions; their
 * in_strides entries are ignored; `in`'s (re, im) pair is contiguous.  conj conjugates `in`.
 * tnq_cplx_fold_f32 is its adjoint (gradient path): out[..., c] (=|+=) sum over ri ^ ro == c.
 * The _f64 versions: the same on doubles (complex128 in, float64 out), strides in doubles.
 */
int tnq_cplx_expand_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                        int ri_dim, int ro_dim, int conj, void* stream);
int tnq_cplx_fold_f32(const float* in, float* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                      int64_t ri_stride, int64_t ro_stride, int conj, int accumulate, void* stream);
int tnq_cplx_expand_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                        int ri_dim, int ro_dim, int conj, void* stream);
int tnq_cplx_fold_f64(const double* in, double* out, int ndim, const int64_t* out_dims, const int64_t* in_strides,
                      int64_t ri_stride, int64_t ro_stride, int conj, int accumulate, void* stream);

/*
 * The optimizer step of the reference's default method ('sgdg': SGD on the Stiefel manifold by a
 * Cayley transform, backend_pytorch.py:349-468) for all cores of a network in one launch.
 * Core i is a row-major rows[i] x cols[i] float32 matrix (rows = product of the first half of its
 * dims, backend_pytorch.py:364-368) with rows[i] <= cols[i] <= TNQ_SGDG_MAX_COLS; velocity[i] is the
 * cols[i] x rows[i] momentum buffer.  params and velocity are updated in place; the pointer tables
 * and rows/cols are DEVICE arrays of ncores entries.  The reference's 1 % random QR retraction
 * (backend_pytorch.py:382) is the caller's business.
 */
#define TNQ_SGDG_MAX_COLS 64
int tnq_sgdg_step(float* const* params, const float* const* grads, float* const* velocity, const int* rows,
                  const int* cols, int ncores, int max_cols, float lr, float momentum, void* stream);
/* The same step when parameters, gradients and momentum buffers each live in ONE buffer (the fused
 * contraction routes return the gradients that way): `offsets` is a DEVICE table [3][ncores] of element
 * offsets (params | grads | velocity) that is static per network, so a step needs no host-to-device
 * traffic and no host synchronisation. */
int tnq_sgdg_step_flat(float* params, const float* grads, float* velocity, const int64_t* offsets, const int* rows,
                       const int* cols, int ncores, int max_cols, float lr, float momentum, void* stream);

/*
 * One-shot all-reduce of the packed gradient + loss buffer of one training step over NVLink peer
 * memory (replaces the per-core blocking collectives of DataParallelTrainer.sync_gradients,
 * tneq_qc/distributed/parallel/data_parallel.py:194-204 / comm/comm_torch.py:292-318).
 *   peer_bufs_dev : DEVICE array of `world` pointers, entry r = rank r's symmetric buffer as mapped
 *                   into this process (torch.distributed._symmetric_memory: buffer_ptrs_dev); every
 *                   buffer has tnq_allreduce_oneshot_words(nmax) zero-initialised 32-bit words
 *   out[0, na+nb) = scale * sum over ranks of (src_a[0,na) ++ src_b[0,nb)), summed in rank order on
 *   every rank (bit-identical results).  All ranks must call it the same number of times.
 * A peer that does not arrive within the timeout (default 600 000 ms; tnq_allreduce_set_timeout_ms) does
 * not kill the context: out[] is filled with NaN, word 33 of this rank's symmetric buffer receives the
 * epoch of the failed call and word 34 the first missing rank; the caller raises or falls back to NCCL.
 */
int64_t tnq_allreduce_oneshot_words(int64_t nmax);
int tnq_allreduce_set_timeout_ms(int64_t ms);
int tnq_allreduce_oneshot(const uint64_t* peer_bufs_dev, int rank, int world, int64_t nmax, const float* src_a,
                          int64_t na, const float* src_b, int64_t nb, float* out, float scale, void* stream);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t tnq_launch_count(void);

const char* tnq_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* TNEQ_B200_H */
