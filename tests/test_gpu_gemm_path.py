"""The large-bond-dimension route (permute kernels + tcgen05 3xTF32 GEMM) against the oracle.

TNQ_FORCE_GEMM_PATH=1 sends small networks down the same route that bond dimension 64-128 takes,
so that the CPU oracle can still check every number."""
import os

import pytest
import torch

import tneq_b200
from oracle import qctn_oracle as oc
from helpers import well_conditioned_case, upcast, clone_mx, rel_err, mps_f64, NOISE_FACTOR

pytestmark = pytest.mark.gpu
H = tneq_b200.QCTNHelper


def _to_dev(x, dev):
    if isinstance(x, oc.TNT):
        return tneq_b200.TNTensor(x.tensor.to(dev), x.scale, x.log_scale)
    return x.to(dev)


@pytest.fixture
def force_gemm_path():
    os.environ["TNQ_FORCE_GEMM_PATH"] = "1"
    yield
    os.environ.pop("TNQ_FORCE_GEMM_PATH", None)


@pytest.mark.parametrize("kind,n,K,B,dtype", [("mps", 5, 4, 24, "float32"), ("mps", 4, 8, 10, "float32"),
                                             ("mps", 5, 4, 12, "complex64"), ("mps", 4, 8, 6, "complex64"),
                                             ("tree", 6, 4, 9, "float32"), ("mps", 3, 16, 5, "complex64")])
def test_gemm_path_matches_oracle(kind, n, K, B, dtype, built_lib, force_gemm_path):
    graph = H.generate_example_graph(n=n, graph_type=kind, dim_char=str(K))
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, B, dtype)
    td64 = torch.complex128 if "complex" in dtype else torch.float64
    want = oc.forward(graph, cores, states, clone_mx(mxs))
    c64 = {k: v.to(td64) for k, v in cores.items()}
    s64 = [s.to(td64) for s in states]
    tl, tg = oc.loss_and_grads(graph, c64, s64, [upcast(m, td64) for m in clone_mx(mxs)])
    wl, wg = oc.loss_and_grads(graph, cores, states, clone_mx(mxs))
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype=dtype)
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    dev = torch.device("cuda:0")
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.to(dev).requires_grad_(True)
    st = [s.to(dev) for s in states]
    launches0 = tneq_b200._lib.launch_count()
    got = eng.contract_with_compiled_strategy(q, st, [_to_dev(m, dev) for m in clone_mx(mxs)])
    fn = eng._compiled(q, st, [_to_dev(m, dev) for m in clone_mx(mxs)], True, "symmetric")
    assert next(iter(fn.plans.values())).use_gemm_path and tneq_b200._lib.launch_count() > launches0
    assert got.shape == want.shape
    # complex dtypes return |amplitude|^2 (reference quirk D10): the amplitude's 1e-5 bound doubles
    truth = oc.forward(graph, c64, s64, [upcast(m, td64) for m in clone_mx(mxs)])
    tol_p = 2e-5 if "complex" in dtype else 1e-5
    assert rel_err(got.double(), truth) < max(tol_p, NOISE_FACTOR * rel_err(want.double(), truth))
    for fused in (True, False):
        loss, grads = eng.contract_with_compiled_strategy_for_gradient(
            q, st, [_to_dev(m, dev) for m in clone_mx(mxs)], fused=fused)
        assert abs(loss.item() - wl.item()) <= 1e-5 * abs(wl.item())
        for g_, w, t in zip(grads, wg, tg):
            assert g_.shape == w.shape and g_.dtype == w.dtype
            ref_err = rel_err(w.to(td64), t)
            assert rel_err(g_.to(td64), t) < max(1e-5, NOISE_FACTOR * ref_err), (fused, rel_err(g_.to(td64), t), ref_err)


def _unitary_cores(q, K, dtype=torch.complex64, seed=0):
    torch.manual_seed(seed)
    for c in q.cores:
        m = torch.randn(K * K, K * K, dtype=torch.complex128, device="cuda")
        qm, _ = torch.linalg.qr(m)
        q.cores_weights[c] = qm.reshape(K, K, K, K).to(dtype)
        del m, qm


def _last_states(K, n, dtype=torch.complex64):
    st = [torch.zeros(K, dtype=dtype, device="cuda") for _ in range(n)]
    for s in st:
        s[-1] = 1.0
    return st


@pytest.mark.parametrize("K,n,B", [(32, 6, 3), (64, 6, 3), (64, 16, 2), (128, 4, 2)])
def test_large_bond_normalisation(K, n, B, built_lib):
    """KAT-1 at bond dimensions the CPU oracle cannot reach (32, 64 -- also at BASELINE cfg4's 16
    qubits -- and 128, complex64): unitary cores (QR in complex128, then cast) + identity
    measurements => value 1 for every sample, to the north-star tolerance of 1e-5.
    The tensor core adds into its fp32 accumulator with truncation; tnq_gemm.cu drains the
    accumulator after every k-block and sums the partial results round-to-nearest (its header)."""
    graph = H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype="complex64")
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    q = tneq_b200.QCTN(graph)
    _unitary_cores(q, K)
    st = _last_states(K, n)
    eye = torch.eye(K, dtype=torch.complex64, device="cuda").expand(B, K, K)
    got = eng.contract_with_compiled_strategy(q, st, [eye] * n)
    fn = eng._compiled(q, st, [eye] * n, True, "symmetric")
    assert next(iter(fn.plans.values())).use_gemm_path
    assert torch.allclose(got.cpu(), torch.ones(B), atol=1e-5), got


@pytest.mark.parametrize("K,n,B", [(64, 5, 4), (128, 3, 2)])
def test_large_bond_identity_circuit(K, n, B, built_lib):
    """KAT-2 at bond 64 / 128: identity cores, states e_{K-1} => amplitude = prod_q M_q[b, K-1, K-1]
    (complex dtypes report |amplitude|^2, reference quirk D10)."""
    graph = H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype="complex64")
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    q = tneq_b200.QCTN(graph)
    ident = torch.eye(K * K, dtype=torch.complex64, device="cuda").reshape(K, K, K, K)
    for c in q.cores:
        q.cores_weights[c] = ident
    st = _last_states(K, n)
    torch.manual_seed(1)
    mx = []
    for _ in range(n):
        h = torch.randn(B, K, K, dtype=torch.complex64, device="cuda") / (2.0 * K ** 0.5)
        mx.append(torch.eye(K, dtype=torch.complex64, device="cuda") + 0.3 * (h + h.transpose(1, 2).conj()))
    got = eng.contract_with_compiled_strategy(q, st, mx)
    amp = torch.ones(B, dtype=torch.complex128, device="cuda")
    for m in mx:
        amp = amp * m[:, K - 1, K - 1].to(torch.complex128)
    want = (amp.real ** 2 + amp.imag ** 2).cpu()
    assert rel_err(got.double().cpu(), want) < 2e-5      # |amplitude|^2: the amplitude's 1e-5 doubles


@pytest.mark.parametrize("K,n,B", [(32, 6, 6), (64, 5, 4)])
def test_large_bond_loss_and_gradients_vs_float64(K, n, B, built_lib):
    """Values, loss and core gradients at bond 32 / 64 against a complex128 contraction of the same
    network on the GPU (torch.autograd for the gradients): 1e-5 relative, gradients per tensor
    relative to the largest entry."""
    graph = H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype="complex64")
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    q = tneq_b200.QCTN(graph)
    _unitary_cores(q, K, seed=3)
    for c in q.cores:
        q.cores_weights[c].requires_grad_(True)
    st = _last_states(K, n)
    torch.manual_seed(4)
    mx = []
    for _ in range(n):                      # I + 0.1 H: keeps the value O(1) (a random unitary's overlap is ~K^-n)
        h = torch.randn(B, K, K, dtype=torch.complex64, device="cuda") / (2.0 * K ** 0.5)
        mx.append(torch.eye(K, dtype=torch.complex64, device="cuda") + 0.1 * (h + h.transpose(1, 2).conj()))
    got = eng.contract_with_compiled_strategy(q, st, mx)
    loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, st, mx)
    fn = eng._compiled(q, st, mx, True, "symmetric")
    assert next(iter(fn.plans.values())).use_gemm_path
    c128 = [q.cores_weights[c].detach().to(torch.complex128).requires_grad_(True) for c in q.cores]
    amp = mps_f64(c128, [s.to(torch.complex128) for s in st], [m.to(torch.complex128) for m in mx])
    val = amp.real ** 2 + amp.imag ** 2
    assert rel_err(got.double().cpu(), val.detach().cpu()) < 2e-5
    want_loss = -(torch.log(torch.clamp(val, min=1e-10))).mean()
    want_grads = torch.autograd.grad(want_loss, c128)
    # loss = -mean(log value): its ABSOLUTE error is the relative error of the values
    assert abs(loss.item() - want_loss.item()) <= 1e-5 * max(abs(want_loss.item()), 1.0)
    for g, w in zip(grads, want_grads):
        assert g.shape == w.shape
        assert rel_err(g.to(torch.complex128).cpu(), w.cpu()) < 1e-5, rel_err(g.to(torch.complex128).cpu(), w.cpu())


def test_permute_kernel_paths(built_lib):
    """direct and tiled code paths of tnq_permute_f32, real and complex (vec = 2), against torch."""
    import ctypes
    from ctypes import c_int64, c_void_p
    from tneq_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(0)
    cases = [((6, 40, 50), (2, 1, 0), 1), ((3, 33, 65, 2), (2, 0, 1, 3), 2), ((64, 64, 64), (1, 2, 0), 1),
             ((5, 7, 9, 4), (0, 2, 1, 3), 4), ((130, 70), (1, 0), 1), ((8, 3, 3, 2), (0, 2, 1, 3), 2),
             # neighbours that merge into one input-contiguous run (the batch-into-K transposition of the bond-64
             # gradient GEMMs), vector widening (vec 2 -> 4), extent-1 dimensions, plain copies
             ((5, 6, 12, 16, 2), (1, 3, 4, 0, 2), 1), ((3, 5, 7, 8, 2), (0, 2, 1, 3, 4), 2), ((3, 5, 7, 6, 2), (0, 2, 1, 3, 4), 2),
             ((1, 5, 1, 4), (2, 0, 1, 3), 1), ((4,), (0,), 1), ((7, 9, 8), (0, 1, 2), 1), ((2, 40, 3, 36, 2), (2, 3, 4, 0, 1), 1),
             # the 64 x 64 float4 tile path (extents and strides multiples of four), with ragged tile edges
             ((3, 100, 5, 72), (2, 3, 0, 1), 1), ((4, 64, 2, 68, 2), (1, 3, 4, 0, 2), 1), ((132, 260), (1, 0), 1)]
    for shape, perm, vec in cases:
        x = torch.randn(*shape, device="cuda")
        want = x.permute(*perm).contiguous()
        out = torch.empty_like(want)
        dims = list(want.shape)
        st = [x.stride(p) for p in perm]
        n = len(dims)
        _lib.check(lib.tnq_permute_f32(c_void_p(x.data_ptr()), c_void_p(out.data_ptr()), n, (c_int64 * n)(*dims),
                                       (c_int64 * n)(*st), vec, 0, c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        assert torch.equal(out, want), (shape, perm, vec)
    # conjugation rides along for interleaved complex data
    z = torch.randn(9, 11, 5, dtype=torch.complex64, device="cuda")
    x = torch.view_as_real(z)
    want = torch.view_as_real(z.permute(2, 0, 1).conj().resolve_conj().contiguous())
    out = torch.empty_like(want)
    dims, st = list(want.shape), [x.stride(2), x.stride(0), x.stride(1), 1]
    _lib.check(lib.tnq_permute_f32(c_void_p(x.data_ptr()), c_void_p(out.data_ptr()), 4, (c_int64 * 4)(*dims),
                                   (c_int64 * 4)(*st), 2, 1, c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(out, want)


def _ptr(t):
    from ctypes import c_void_p
    return c_void_p(t.data_ptr())


def _ptr_stream():
    from ctypes import c_void_p
    return c_void_p(torch.cuda.current_stream().cuda_stream)


# The fold kernels sum 2 D float32 products in sequence: their rounding error relative to the largest output grows
# like sqrt(D) (a float32 emulation of the kernel's order on the CPU gives 4.2e-7 at D = 64 and 2.7e-6 at D = 4096).
def _fold_bound(D):
    return 1e-6 * max(1.0, (D / 64) ** 0.5)


@pytest.mark.parametrize("A,D,C", [(1, 1, 1), (3, 2, 5), (7, 3, 1), (5, 64, 129), (1, 128, 257), (3, 4096, 33), (2, 4096, 1)])
def test_fold_vec_and_outer_acc_vs_float64(A, D, C, built_lib):
    """tnq_fold_vec_f32 and tnq_outer_acc_f32 (include/tneq_b200.h) against float64 einsum: odd A and C, C = 1, D
    from 1 to 4096 (above D = 3072 Q needs more than the default 48 KB of shared memory), outer_acc into a nonzero T."""
    from tneq_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(A * 1000 + D + C)
    stream = _ptr_stream()
    P = torch.randn(A, D, C, 2, device="cuda")
    Q = torch.randn(D, 2, 2, device="cuda")
    out = torch.full((A, C, 2), float("nan"), device="cuda")
    launches = _lib.launch_count()
    _lib.check(lib.tnq_fold_vec_f32(_ptr(P), _ptr(Q), _ptr(out), A, D, C, stream))
    want = torch.einsum("adcr,dro->aco", P.double(), Q.double())
    torch.cuda.synchronize()
    assert _lib.launch_count() == launches + 1
    assert rel_err(out.double(), want) < _fold_bound(D), rel_err(out.double(), want)
    # the adjoint: T[a, d, c, ri] += sum_ro P[a, c, ro] Q[d, ri, ro], accumulated into a nonzero T
    Pa = torch.randn(A, C, 2, device="cuda")
    T0 = torch.randn(A, D, C, 2, device="cuda")
    T = T0.clone()
    _lib.check(lib.tnq_outer_acc_f32(_ptr(Pa), _ptr(Q), _ptr(T), A, D, C, stream))
    want = T0.double() + torch.einsum("acO,drO->adcr", Pa.double(), Q.double())
    torch.cuda.synchronize()
    assert rel_err(T.double(), want) < 1e-6, rel_err(T.double(), want)


def _expand_ref(z, ri, ro, conj):
    """out[..., ri, ..., ro] = E[ri][ro] of z[...] (E = [[re, im], [-im, re]]), the two extent-2 dimensions inserted
    at output positions ri < ro, in float64."""
    z = z.conj() if conj else z
    E = torch.stack([torch.stack([z.real, z.imag], -1), torch.stack([-z.imag, z.real], -1)], -2)   # [..., 2, 2]
    nd = z.dim() + 2
    order = [i for i in range(nd) if i not in (ri, ro)]          # output positions of z's dimensions
    perm = [0] * nd
    for src, dst in enumerate(order + [ri, ro]):
        perm[dst] = src
    return E.permute(*perm)


@pytest.mark.parametrize("shape,ri,ro", [((3, 5), 2, 3), ((3, 5), 0, 2), ((4, 1, 7), 1, 4), ((33, 65), 0, 1), ((2, 3, 5), 1, 3)])
@pytest.mark.parametrize("conj", [0, 1])
def test_cplx_expand_and_fold_vs_float64(shape, ri, ro, conj, built_lib):
    """tnq_cplx_expand_f32 (complex -> 2x2 real form fused with a permutation) and its adjoint tnq_cplx_fold_f32 against
    float64: ri and ro at different output positions, a transposed (strided) input, conj, fold with accumulate."""
    from tneq_b200 import _lib
    lib = _lib.load()
    from ctypes import c_int64
    torch.manual_seed(sum(shape) * 10 + ri + ro + conj)
    stream = _ptr_stream()
    zt = torch.randn(*reversed(shape), dtype=torch.complex64, device="cuda")
    z = zt.permute(*reversed(range(len(shape))))                  # z[...] read through strides
    x = torch.view_as_real(zt)                                     # memory of z: (re, im) innermost
    nd = len(shape) + 2
    zdims = [i for i in range(nd) if i not in (ri, ro)]
    dims = [0] * nd
    st = [0] * nd
    for k, pos in enumerate(zdims):
        dims[pos], st[pos] = shape[k], x.stride(len(shape) - 1 - k)
    dims[ri] = dims[ro] = 2
    out = torch.empty(dims, device="cuda")
    _lib.check(lib.tnq_cplx_expand_f32(_ptr(x), _ptr(out), nd, (c_int64 * nd)(*dims), (c_int64 * nd)(*st), ri, ro, conj,
                                       stream))
    want = _expand_ref(z.to(torch.complex128), ri, ro, conj)
    torch.cuda.synchronize()
    assert torch.equal(out.double(), want), (shape, ri, ro, conj)
    # adjoint: dz[..., c] = sum_{ri ^ ro = c} sign * G[..., ri, ..., ro] in z's dimension order, added, then written
    G = torch.randn(dims, device="cuda")
    fdims = list(shape) + [2]
    fst = [G.stride(pos) for pos in zdims] + [0]
    g64 = G.double()
    sel = lambda a, b: g64.select(ro, b).select(ri, a)             # ri < ro: select ro first
    im = sel(0, 1) - sel(1, 0)
    F = torch.stack([sel(0, 0) + sel(1, 1), -im if conj else im], -1)
    prev = torch.randn(fdims, device="cuda")
    got = prev.clone()
    for acc, want in ((1, prev.double() + F), (0, F)):
        _lib.check(lib.tnq_cplx_fold_f32(_ptr(G), _ptr(got), nd - 1, (c_int64 * (nd - 1))(*fdims),
                                         (c_int64 * (nd - 1))(*fst), G.stride(ri), G.stride(ro), conj, acc, stream))
        torch.cuda.synchronize()
        assert rel_err(got.double(), want) < 1e-6, (acc, rel_err(got.double(), want))
