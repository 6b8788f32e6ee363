"""The large-bond route in float64 / complex128: tnq_gemm_f64 (FP64 tensor cores), the _f64 layout kernels, and the
whole route against float64 references.

float64 arithmetic leaves ~1e-16 per operation; the bounds below are reasoned, not fitted: exact answers where the
inputs make every product and sum exact, 1e-13 of the largest entry for a GEMM against the CPU, 1e-12 where a small
network is compared with the CPU oracle, 1e-10 of the largest entry for bond 32-128 (dozens of chained contractions
of K up to 16 384, each amplifying the last one's rounding by at most its condition).  A float32-grade error (1e-7 and
up) fails all of them."""
import itertools
import os
from ctypes import c_int64, c_void_p

import pytest
import torch

import tneq_b200
from helpers import LARGE_BOND_CASES, clone_mx, elem_rel_err, record_routes, rel_err, well_conditioned_case
from oracle import qctn_oracle as oc
from test_gpu_gemm_path import _expand_ref
from test_gpu_large_bond import _degree_identity, _engine, _errors, _loss_err, _measurements, _network, _yardstick
from test_oracle_golden import GOLDEN, fresh_mx, load_case
from tneq_b200 import _lib
from tneq_b200.contractor.gemm_path import GemmPathRunner

pytestmark = pytest.mark.gpu
H = tneq_b200.QCTNHelper


def _p(t):
    return c_void_p(t.data_ptr())


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- 1. tnq_gemm_f64 ------------------------------------------------------------------------------------------------
def _operand(batch, rows, K, ld, stride, fill):
    """(CPU view [batch][rows][K] with row stride ld and batch stride `stride` (0: shared), its device copy with the
    same memory layout)."""
    n = (0 if stride == 0 else (batch - 1) * stride) + (rows - 1) * ld + K
    flat = fill(n)
    return torch.as_strided(flat, (batch, rows, K), (stride, ld, 1)), flat.cuda()


def _run_gemm(M, N, K, fill, lda=None, ldb=None, ldc=None, batch=1, sA=None, sB=None, sC=None, acc=False):
    """tnq_gemm_f64 on operands laid out as asked; returns (C on the CPU, float64 CPU reference, device C)."""
    lda, ldb, ldc = lda or K, ldb or K, ldc or N
    sA = (M - 1) * lda + K if sA is None else sA
    sB = (N - 1) * ldb + K if sB is None else sB
    sC = (M - 1) * ldc + N if sC is None else sC
    a, da = _operand(batch, M, K, lda, sA, fill)
    b, db = _operand(batch, N, K, ldb, sB, fill)
    c0, dc = _operand(batch, M, N, ldc, sC, fill)
    want = torch.matmul(a, b.transpose(1, 2)) + (c0 if acc else 0)
    n0 = _lib.launch_count()
    _lib.check(_lib.load().tnq_gemm_f64(_p(da), _p(db), _p(dc), M, N, K, lda, ldb, ldc, batch, sA, sB, sC, int(acc),
                                        _stream()))
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1
    got = torch.as_strided(dc.cpu(), (batch, M, N), (sC, ldc, 1))
    return got, want, dc


def _ints(lo=-8, hi=9):
    return lambda n: torch.randint(lo, hi, (n,), dtype=torch.float64)


def _normal(n):
    return torch.randn(n, dtype=torch.float64)


SIZES = (1, 7, 16, 127, 129, 1000)


def test_gemm_f64_exact_on_integers(built_lib):
    """Integer entries in [-8, 8]: every product and partial sum is an integer below 2^53, so any summation order gives
    the exact answer -- bit-equal for every M, N, K in {1, 7, 16, 127, 129, 1000}."""
    torch.manual_seed(0)
    for M, N, K in itertools.product(SIZES, SIZES, SIZES):
        got, want, _ = _run_gemm(M, N, K, _ints())
        assert torch.equal(got, want), (M, N, K)


LAYOUTS = [
    # M, N, K, extra arguments
    (1000, 1000, 1000, {}),
    (129, 127, 1000, {}),
    (7, 129, 16, {}),
    (127, 129, 4096, {}),                                   # 2 output tiles, long k-loop: split-K
    (129, 7, 4099, {}),                                     # split-K with odd K (8-byte loads)
    (127, 129, 127, dict(lda=131, ldb=129, ldc=133)),       # odd leading dimensions everywhere
    (16, 16, 16, dict(lda=17, ldb=19, ldc=21)),
    (129, 127, 129, dict(batch=5, sA=129 * 129 + 3, sB=127 * 129 + 5, sC=129 * 127 + 7)),   # odd batch strides
    (64, 33, 128, dict(batch=3, sB=0)),                     # B shared across the batch
    (129, 127, 1000, dict(acc=True)),                       # C += A B^T (no split-K)
    (127, 129, 4096, dict(acc=True)),
    (7, 16, 127, dict(batch=4, acc=True, ldc=17, sC=7 * 17 + 1)),
]


@pytest.mark.parametrize("M,N,K,kw", LAYOUTS, ids=[f"{m}x{n}x{k}-{'-'.join(kw) or 'plain'}" for m, n, k, kw in LAYOUTS])
def test_gemm_f64_random_vs_cpu(M, N, K, kw, built_lib):
    """Random normal entries against float64 torch.matmul on the CPU: 1e-13 of the largest entry; integers bit-equal
    in the same layout (catches an index error that random data would only blur)."""
    torch.manual_seed(M + N + K)
    got, want, _ = _run_gemm(M, N, K, _normal, **kw)
    assert rel_err(got, want) <= 1e-13, rel_err(got, want)
    got, want, _ = _run_gemm(M, N, K, _ints(), **kw)
    assert torch.equal(got, want)


# the GEMMs of one cfg4 step in complex128 (16 qubits, bond 64, B = 256): the three forward shapes and the two
# core-gradient shapes (64 output tiles: split-K)
CFG4 = [(16384, 8192, 128, 1), (4096, 128, 128, 256), (16384, 128, 8192, 1), (128, 8192, 16384, 1), (8192, 128, 16384, 1)]


@pytest.mark.parametrize("M,N,K,batch", CFG4, ids=[f"{m}x{n}x{k}-b{b}" for m, n, k, b in CFG4])
def test_gemm_f64_cfg4_shapes(M, N, K, batch, built_lib):
    """cfg4's shapes on the device: 256 sampled (batch, row) pairs against float64 torch.matmul
    on the CPU to 1e-13 of the largest entry, and two launches bit-identical."""
    torch.manual_seed(1)
    g = torch.Generator(device="cuda").manual_seed(2)
    A = torch.randn(batch, M, K, dtype=torch.float64, device="cuda", generator=g)
    B = torch.randn(batch, N, K, dtype=torch.float64, device="cuda", generator=g)
    C = [torch.empty(batch, M, N, dtype=torch.float64, device="cuda") for _ in range(2)]
    for c in C:
        _lib.check(_lib.load().tnq_gemm_f64(_p(A), _p(B), _p(c), M, N, K, K, K, N, batch, M * K, N * K, M * N, 0,
                                            _stream()))
    torch.cuda.synchronize()
    assert torch.equal(C[0], C[1])
    bs = torch.randint(0, batch, (256,))
    rows = torch.randint(0, M, (256,))
    a = A[bs.cuda(), rows.cuda()].cpu()
    want = a @ B[0].cpu().T if batch == 1 else torch.einsum("rk,rnk->rn", a, B[bs.cuda()].cpu())
    got = C[0][bs.cuda(), rows.cuda()].cpu()
    assert rel_err(got, want) <= 1e-13, rel_err(got, want)


# ---- 2. the _f64 layout kernels ---------------------------------------------------------------------------------------
PERMUTES = [((6, 40, 50), (2, 1, 0), 1), ((3, 33, 65, 2), (2, 0, 1, 3), 2), ((64, 64, 64), (1, 2, 0), 1),
            ((130, 70), (1, 0), 1), ((8, 3, 3, 2), (0, 2, 1, 3), 2), ((5, 6, 12, 16, 2), (1, 3, 4, 0, 2), 1),
            ((3, 5, 7, 8, 2), (0, 2, 1, 3, 4), 2), ((1, 5, 1, 4), (2, 0, 1, 3), 1), ((4,), (0,), 1),
            ((7, 9, 8), (0, 1, 2), 1), ((3, 100, 5, 72), (2, 3, 0, 1), 1), ((40, 50, 2), (1, 0, 2), 2)]


def test_permute_f64_bit_exact(built_lib):
    """tnq_permute_f64 through its direct and tiled paths (scalars, complex128 pairs, merged runs, extent-1 dimensions,
    plain copies), and with conj, against torch: bit-exact."""
    torch.manual_seed(0)
    lib = _lib.load()
    for shape, perm, vec in PERMUTES:
        x = torch.randn(*shape, dtype=torch.float64, device="cuda")
        want = x.permute(*perm).contiguous()
        out = torch.empty_like(want)
        dims, st, n = list(want.shape), [x.stride(p) for p in perm], len(perm)
        _lib.check(lib.tnq_permute_f64(_p(x), _p(out), n, (c_int64 * n)(*dims), (c_int64 * n)(*st), vec, 0, _stream()))
        torch.cuda.synchronize()
        assert torch.equal(out, want), (shape, perm, vec)
    for shape, perm in (((9, 11, 5), (2, 0, 1)), ((40, 50), (1, 0)), ((3, 4), (0, 1))):
        z = torch.randn(*shape, dtype=torch.complex128, device="cuda")
        x = torch.view_as_real(z)
        want = torch.view_as_real(z.permute(*perm).conj().resolve_conj().contiguous())
        out = torch.empty_like(want)
        n = len(shape) + 1
        dims, st = list(want.shape), [x.stride(p) for p in perm] + [1]
        _lib.check(lib.tnq_permute_f64(_p(x), _p(out), n, (c_int64 * n)(*dims), (c_int64 * n)(*st), 2, 1, _stream()))
        torch.cuda.synchronize()
        assert torch.equal(out, want), (shape, perm)


@pytest.mark.parametrize("shape,ri,ro", [((3, 5), 2, 3), ((3, 5), 0, 2), ((4, 1, 7), 1, 4), ((33, 65), 0, 1)])
@pytest.mark.parametrize("conj", [0, 1])
def test_cplx_expand_and_fold_f64(shape, ri, ro, conj, built_lib):
    """tnq_cplx_expand_f64 (bit-exact, conj negating the second double of each pair) and its adjoint tnq_cplx_fold_f64
    (two terms per output: 1e-14, with and without accumulate) against complex128 torch."""
    lib = _lib.load()
    torch.manual_seed(sum(shape) * 10 + ri + ro + conj)
    zt = torch.randn(*reversed(shape), dtype=torch.complex128, device="cuda")
    z = zt.permute(*reversed(range(len(shape))))
    x = torch.view_as_real(zt)
    nd = len(shape) + 2
    zdims = [i for i in range(nd) if i not in (ri, ro)]
    dims, st = [0] * nd, [0] * nd
    for k, pos in enumerate(zdims):
        dims[pos], st[pos] = shape[k], x.stride(len(shape) - 1 - k)
    dims[ri] = dims[ro] = 2
    out = torch.empty(dims, dtype=torch.float64, device="cuda")
    _lib.check(lib.tnq_cplx_expand_f64(_p(x), _p(out), nd, (c_int64 * nd)(*dims), (c_int64 * nd)(*st), ri, ro, conj,
                                       _stream()))
    torch.cuda.synchronize()
    assert torch.equal(out, _expand_ref(z, ri, ro, conj))
    G = torch.randn(dims, dtype=torch.float64, device="cuda")
    fdims = list(shape) + [2]
    fst = [G.stride(pos) for pos in zdims] + [0]
    sel = lambda a, b: G.select(ro, b).select(ri, a)
    im = sel(0, 1) - sel(1, 0)
    F = torch.stack([sel(0, 0) + sel(1, 1), -im if conj else im], -1)
    prev = torch.randn(fdims, dtype=torch.float64, device="cuda")
    got = prev.clone()
    for acc, want in ((1, prev + F), (0, F)):
        _lib.check(lib.tnq_cplx_fold_f64(_p(G), _p(got), nd - 1, (c_int64 * (nd - 1))(*fdims), (c_int64 * (nd - 1))(*fst),
                                         G.stride(ri), G.stride(ro), conj, acc, _stream()))
        torch.cuda.synchronize()
        assert rel_err(got, want) <= 1e-14, (acc, rel_err(got, want))


def _dyadic(*shape):
    """Multiples of 2^-10 in [-1, 1]: the 2 D-term sums of the fold kernels are exact in float64 for D <= 4096."""
    return torch.randint(-1024, 1025, shape, dtype=torch.float64, device="cuda") / 1024.0


@pytest.mark.parametrize("A,D,C", [(1, 1, 1), (3, 2, 5), (5, 64, 129), (3, 1536, 7), (3, 1537, 7), (2, 4096, 33)])
def test_fold_vec_and_outer_acc_f64(A, D, C, built_lib):
    """tnq_fold_vec_f64 and tnq_outer_acc_f64 against float64 einsum to 1e-14 of the largest output: D from 1 to 4096
    (above D = 1536 Q needs more than the default 48 KB of shared memory in float64), outer_acc into a nonzero T.
    Dyadic inputs (exact sums), then normal ones at the same shape."""
    lib = _lib.load()
    torch.manual_seed(A * 1000 + D + C)
    for make in (_dyadic, lambda *s: torch.randn(*s, dtype=torch.float64, device="cuda")):
        P, Q = make(A, D, C, 2), make(D, 2, 2)
        out = torch.full((A, C, 2), float("nan"), dtype=torch.float64, device="cuda")
        n0 = _lib.launch_count()
        _lib.check(lib.tnq_fold_vec_f64(_p(P), _p(Q), _p(out), A, D, C, _stream()))
        want = torch.einsum("adcr,dro->aco", P.cpu(), Q.cpu())
        torch.cuda.synchronize()
        assert _lib.launch_count() == n0 + 1
        # normal inputs: 2 D terms summed in sequence leave ~eps sqrt(D) relative to the largest output, ~1e-15 at
        # D = 4096
        assert rel_err(out.cpu(), want) <= 1e-14, rel_err(out.cpu(), want)
        Pa, T0 = make(A, C, 2), make(A, D, C, 2)
        T = T0.clone()
        _lib.check(lib.tnq_outer_acc_f64(_p(Pa), _p(Q), _p(T), A, D, C, _stream()))
        want = T0.cpu() + torch.einsum("acO,drO->adcr", Pa.cpu(), Q.cpu())
        torch.cuda.synchronize()
        assert rel_err(T.cpu(), want) <= 1e-14, rel_err(T.cpu(), want)


# ---- 3. the forced GEMM path on small networks --------------------------------------------------------------------
def _to_dev(x):
    if isinstance(x, oc.TNT):
        return tneq_b200.TNTensor(x.tensor.cuda(), x.scale, x.log_scale)
    return x.cuda()


def _run_engine(graph, K, dtype, cores, states, mxs):
    """(values, fused loss, fused grads, autograd loss, autograd grads, whether the GEMM path ran) of a fresh engine."""
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype=dtype)
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.cuda().requires_grad_(True)
    st = [s.cuda() for s in states]
    val = eng.contract_with_compiled_strategy(q, st, [_to_dev(m) for m in clone_mx(mxs)])
    fn = eng._compiled(q, st, [_to_dev(m) for m in clone_mx(mxs)], True, "symmetric")
    gemm = next(iter(fn.plans.values())).use_gemm_path
    out = [val.detach().cpu()]
    for fused in (True, False):
        loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, st, [_to_dev(m) for m in clone_mx(mxs)],
                                                                       fused=fused)
        out += [loss.detach().cpu(), [g.detach().cpu() for g in grads]]
    torch.cuda.synchronize()
    return (*out, gemm)


def _assert_close(got, want, tol, what):
    """values (relative to the largest), loss, gradients (each relative to its largest entry) of two runs"""
    val, l1, g1, l2, g2, _ = got
    wval, wloss, wgrads = want
    assert val.shape == wval.shape
    errs = [rel_err(val, wval), _loss_err(l1, wloss), _loss_err(l2, wloss)]
    errs += [rel_err(a, w) for gs in (g1, g2) for a, w in zip(gs, wgrads)]
    for gs in (g1, g2):
        assert [a.dtype for a in gs] == [w.dtype for w in wgrads]
    print(f"[{what}] worst error {max(errs):.2e}")
    assert max(errs) <= tol, (what, errs)


def test_forced_gemm_path_reference_fixture(monkeypatch, built_lib):
    """The reference's own float64 fixture (tests/golden/mps5_k2_f64.npz: 5-qubit MPS, K = 2) on the GEMM path:
    values, loss and gradients (fused and autograd) within 1e-12."""
    monkeypatch.setenv("TNQ_FORCE_GEMM_PATH", "1")
    c = load_case(os.path.join(GOLDEN, "mps5_k2_f64.npz"))
    got = _run_engine(c["graph"], c["K"], c["dtype"], c["cores"], c["states"], fresh_mx(c))
    assert got[-1]
    _assert_close(got, (c["probabilities"], c["loss"], c["grads"]), 1e-12, "mps5_k2_f64 fixture")


def _graph(kind, n, K):
    if kind == "merged":
        q0 = tneq_b200.QCTN(H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K)))
        return tneq_b200.QCTN.merge(q0, q0).graph
    return H.generate_example_graph(n=n, graph_type=kind, dim_char=str(K))


@pytest.mark.parametrize("kind,n,K,B", [("mps", 5, 4, 12), ("mps", 6, 3, 10), ("merged", 4, 2, 8), ("tree", 6, 4, 9)])
@pytest.mark.parametrize("dtype", ["float64", "complex128"])
def test_forced_gemm_path_vs_oracle_and_vm(kind, n, K, B, dtype, monkeypatch, built_lib):
    """MPS, two-layer merged and tree networks in float64 and complex128 on the GEMM path, against the CPU oracle in
    float64 and against the shared-memory VM route in the same process: values, loss, gradients within 1e-12."""
    graph = _graph(kind, n, K)
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, B, dtype)
    want = oc.forward(graph, cores, states, clone_mx(mxs))
    wl, wg = oc.loss_and_grads(graph, cores, states, clone_mx(mxs))
    monkeypatch.setenv("TNQ_FORCE_GEMM_PATH", "1")
    got = _run_engine(graph, K, dtype, cores, states, mxs)
    assert got[-1]
    monkeypatch.delenv("TNQ_FORCE_GEMM_PATH")
    vm = _run_engine(graph, K, dtype, cores, states, mxs)
    assert not vm[-1]
    _assert_close(got, (want, wl, wg), 1e-12, f"{kind} {dtype} GEMM path vs oracle")
    _assert_close(got, (vm[0], vm[1], vm[2]), 1e-12, f"{kind} {dtype} GEMM path vs VM")


# ---- 6. the headline case: float64 bond 9 / complex128 bond 7, natural route, only _f64 kernels ---------------------
class _Spy:
    """The library with every tnq_* entry point that is called recorded by name."""

    def __init__(self, lib):
        self._lib, self.called = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if not name.startswith("tnq_") or name in ("tnq_last_error", "tnq_launch_count", "tnq_device_check"):
            return fn

        def call(*args):
            self.called.append(name)
            return fn(*args)
        return call


@pytest.mark.parametrize("dtype,K", [("float64", 9), ("complex128", 7)])
def test_big_float64_cores_launch_only_f64_kernels(dtype, K, monkeypatch, built_lib):
    """A 4-qubit MPS whose cores exceed the shared-memory VM (float64 bond 9, complex128 bond 7) runs on the GEMM path
    without TNQ_FORCE_GEMM_PATH, launches only _f64 kernels, and matches the CPU oracle within 1e-12."""
    monkeypatch.delenv("TNQ_FORCE_GEMM_PATH", raising=False)
    spy = _Spy(_lib.load())
    monkeypatch.setattr(_lib, "load", lambda: spy)
    graph = H.generate_example_graph(n=4, graph_type="mps", dim_char=str(K))
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, 5, dtype)
    want = oc.forward(graph, cores, states, clone_mx(mxs))
    wl, wg = oc.loss_and_grads(graph, cores, states, clone_mx(mxs))
    n0 = spy._lib.tnq_launch_count()
    got = _run_engine(graph, K, dtype, cores, states, mxs)
    assert got[-1] and spy._lib.tnq_launch_count() > n0
    called = set(spy.called)
    assert "tnq_gemm_f64" in called and all(c.endswith("_f64") for c in called), sorted(called)
    _assert_close(got, (want, wl, wg), 1e-12, f"{dtype} bond {K}")


# ---- 4. large bond against the complex128 / float64 yardstick ---------------------------------------------------------
F64_CASES = [({"complex64": "complex128", "float32": "float64"}[c[0]],) + tuple(c[1:4]) for c in LARGE_BOND_CASES]
_F32_OF = {"complex128": "complex64", "float64": "float32"}


@pytest.mark.parametrize("dtype,chi,n,B", F64_CASES, ids=[f"{c[0]}-chi{c[1]}-n{c[2]}-B{c[3]}" for c in F64_CASES])
def test_large_bond_f64_vs_yardstick(dtype, chi, n, B, monkeypatch, built_lib):
    """Bond 32-128, B from 2 to 256 (the batch sizes of helpers.LARGE_BOND_CASES): values, loss and gradients within
    1e-10 of the largest entry of helpers.mps_f64; fused and autograd gradients within 1e-12 of each other; no view or
    in-place GEMM variant; the float32 route on the same inputs within its 1e-5 of the float64 one."""
    torch.cuda.empty_cache()
    routes = record_routes(monkeypatch, GemmPathRunner)
    eng, q, st = _network(dtype, chi, n, seed=3)
    mx = _measurements(dtype, chi, n, B, seed=4)
    truth = _yardstick(q, st, mx)
    got = _engine(eng, q, st, mx, fused=True)
    assert not [k for k in routes if k[0] in ("view", "bk")], dict(routes)
    if dtype == "complex128":
        assert routes[("fold_vec",)] and routes[("outer_acc",)]
    ev, el, eg = _errors(got, truth)
    auto = _engine(eng, q, st, mx, fused=False)
    ea = max(rel_err(a, b) for a, b in zip(auto[2], got[2]))
    eng32, q32, st32 = _network(_F32_OF[dtype], chi, n, seed=3)
    f32 = _engine(eng32, q32, st32, [m.to(getattr(torch, _F32_OF[dtype])) for m in mx])
    fv, fl, fg = _errors(f32, got)
    print(f"[{dtype} chi={chi} n={n} B={B}] vs yardstick: value {ev:.2e} loss {el:.2e} grad {eg:.2e}; fused vs autograd "
          f"{ea:.2e}; float32 route vs float64 route: value {fv:.2e} loss {fl:.2e} grad {fg:.2e}; "
          f"peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    assert got[0].dtype == torch.float64 and all(g.dtype == getattr(torch, dtype) for g in got[2])
    assert ev <= 1e-10 and el <= 1e-10 and eg <= 1e-10, (ev, el, eg)
    assert ea <= 1e-12, ea
    tol_v = 2e-5 if dtype == "complex128" else 1e-5
    assert fv < tol_v and fl <= 1e-5 and fg < 1e-5, (fv, fl, fg)


# ---- 5. cfg4 in complex128 at full shape ----------------------------------------------------------------------------
def test_cfg4_complex128_full_shape(built_lib):
    """cfg4 (16 qubits, bond 64, B = 256) in complex128: KAT-1 (unitary cores, identity measurements: value 1, loss 0)
    to 1e-12; the degree identity sum Re(conj(dL/dG) G) = -4 per core to 1e-10; the batch split 100 + 156 against the
    full batch to 1e-12 (values per sample, sample-weighted loss and gradients)."""
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    chi, n, B = 64, 16, 256
    eng, q, st = _network("complex128", chi, n, seed=11)
    eye = torch.eye(chi, dtype=torch.complex128, device="cuda").expand(B, chi, chi).contiguous()
    val, loss, grads = _engine(eng, q, st, [eye] * n)
    e_val = elem_rel_err(val, torch.ones(B, dtype=torch.float64, device="cuda"))
    e_id = _degree_identity(q, grads, True)
    print(f"[cfg4 c128 KAT-1] value {e_val:.2e} loss {abs(loss.item()):.2e} degree identity {e_id:.2e}")
    assert val.shape == (B,) and val.dtype == torch.float64
    assert e_val <= 1e-12 and abs(loss.item()) <= 1e-12 and e_id <= 1e-10
    mx = _measurements("complex128", chi, n, B, seed=12)
    val, loss, grads = _engine(eng, q, st, mx)
    assert 1e-3 < val.min().item() and val.max().item() < 1e3
    e_id = _degree_identity(q, grads, True)
    halves = [_engine(eng, q, st, [m[lo:hi].contiguous() for m in mx]) for lo, hi in ((0, 100), (100, 256))]
    (v1, l1, g1), (v2, l2, g2) = halves
    w1, w2 = 100 / B, 156 / B
    e_val = elem_rel_err(torch.cat([v1, v2]), val)
    e_loss = _loss_err(w1 * l1 + w2 * l2, loss)
    e_grad = max(rel_err(w1 * a + w2 * b, g) for a, b, g in zip(g1, g2, grads))
    print(f"[cfg4 c128 I + eps H] degree identity {e_id:.2e}; batch 100 + 156 vs 256: value {e_val:.2e} "
          f"loss {e_loss:.2e} grad {e_grad:.2e}; peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    assert e_id <= 1e-10 and e_val <= 1e-12 and e_loss <= 1e-12 and e_grad <= 1e-12, (e_id, e_val, e_loss, e_grad)
