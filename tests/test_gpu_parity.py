"""GPU parity: the CUDA path (through the engine API and the C ABI) against the oracle.

Tolerance (BASELINE.json north_star): probabilities and gradients within 1e-5
relative for float32 / complex64.  "Relative" is measured per tensor against its
largest magnitude for gradients (elements near zero carry no relative
information in float32) and per sample for probabilities; both sides compute in
float32 with different summation orders, so the oracle in float64 is used as
the common yardstick where stated.
"""
import pytest
import torch

import tneq_b200
from oracle import qctn_oracle as oc
from helpers import make_case, well_conditioned_case, upcast, clone_mx, rel_err, elem_rel_err, NOISE_FACTOR

pytestmark = pytest.mark.gpu

H = tneq_b200.QCTNHelper


def _graph(kind, n, K):
    if kind == "merged":
        q = tneq_b200.QCTN(H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K)))
        return tneq_b200.QCTN.merge(q, q).graph
    return H.generate_example_graph(n=n, graph_type=kind, dim_char=str(K))


def _to_dev(x, dev):
    if isinstance(x, oc.TNT):
        return tneq_b200.TNTensor(x.tensor.to(dev), x.scale, x.log_scale)
    return x.to(dev)


def _engine(dtype, K, built_lib):
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype=dtype)
    return be, tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)


CASES = [
    ("mps", 6, 3, 37, "float32", "a"),
    ("mps", 16, 3, 300, "float32", "a"),
    ("mps", 5, 2, 33, "float64", "a"),
    ("mps", 6, 3, 19, "complex64", "a"),
    ("mps", 5, 2, 8, "complex128", "a"),
    ("tree", 6, 2, 65, "float32", "a"),
    ("tree", 7, 3, 21, "float32", "a"),
    ("wall", 4, 2, 16, "float32", "a"),
    ("merged", 4, 2, 50, "float32", "a"),
    ("merged", 6, 3, 40, "float32", "a"),
    ("merged", 4, 2, 9, "complex64", "a"),
    ("mps", 6, 3, 10, "float32", "ab"),
    ("mps", 4, 4, 130, "float32", "a"),
    ("mps", 2, 2, 70, "float32", "a"),
    ("mps", 24, 2, 1000, "float32", "a"),
]


@pytest.fixture(params=["default-route", "vm-only"])
def route(request):
    """single-layer MPS float32 networks take the register-resident chain kernel by default;
    'vm-only' forces the same cases through the generic contraction VM as well."""
    import os
    if request.param == "vm-only":
        os.environ["TNQ_NO_CHAIN"] = "1"
    yield request.param
    os.environ.pop("TNQ_NO_CHAIN", None)


@pytest.mark.parametrize("kind,n,K,B,dtype,mode", CASES)
def test_forward_and_training_step(kind, n, K, B, dtype, mode, built_lib, route):
    """Probabilities, loss and core gradients of the CUDA path vs the oracle on the same inputs.
    Tolerance 1e-5 relative (north_star) for float32/complex64, measured per tensor against its
    largest entry, on well-conditioned samples (see helpers.well_conditioned_case); 1e-11 for
    float64/complex128.  The float64 oracle on the same float32 inputs is the common yardstick:
    the CUDA path must be as close to it as the reference's own float32 arithmetic is."""
    graph = _graph(kind, n, K)
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, B, dtype, mode=mode)
    single = dtype in ("float32", "complex64")
    tol = 1e-5 if single else 1e-11
    td64 = torch.complex128 if "complex" in dtype else torch.float64
    want = oc.forward(graph, cores, states, clone_mx(mxs))
    c64 = {k: v.to(td64) for k, v in cores.items()}
    s64 = [s.to(td64) for s in states]
    truth = oc.forward(graph, c64, s64, [upcast(m, td64) for m in clone_mx(mxs)])
    be, eng = _engine(dtype, K, built_lib)
    dev = torch.device("cuda:0")
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.to(dev).requires_grad_(True)
    st = [s.to(dev) for s in states]
    got = eng.contract_with_compiled_strategy(q, st, [_to_dev(m, dev) for m in clone_mx(mxs)])
    bound = next(iter(eng._compiled(q, st, [_to_dev(m, dev) for m in clone_mx(mxs)], True, "symmetric").plans.values()))
    expect_chain = route == "default-route" and kind == "mps" and dtype == "float32" and mode == "a" and K <= 4
    assert bool(bound.chain_rank) == expect_chain
    assert got.shape == want.shape and got.dtype == want.dtype
    assert rel_err(got, want) < tol
    assert elem_rel_err(got.double(), truth) < max(tol, NOISE_FACTOR * elem_rel_err(want.double(), truth))

    if mode == "ab":
        return
    wl, wg = oc.loss_and_grads(graph, cores, states, clone_mx(mxs))
    tl, tg = oc.loss_and_grads(graph, c64, s64, [upcast(m, td64) for m in clone_mx(mxs)])
    for fused in (True, False):   # fused device program, then the torch.autograd route
        loss, grads = eng.contract_with_compiled_strategy_for_gradient(
            q, st, [_to_dev(m, dev) for m in clone_mx(mxs)], fused=fused)
        assert abs(loss.item() - wl.item()) <= tol * abs(wl.item())
        assert len(grads) == len(wg)
        for g, w, t in zip(grads, wg, tg):
            assert g.shape == w.shape and g.dtype == w.dtype
            ref_err = rel_err(w.to(td64), t)
            assert rel_err(g.to(td64), t) < max(tol, NOISE_FACTOR * ref_err), (fused, rel_err(g.to(td64), t), ref_err)
            assert rel_err(g, w) < max(tol, NOISE_FACTOR * ref_err)


def test_kat_normalisation_identity_measurements(built_lib):
    """KAT-1: orthogonal cores + identity on every qubit => value == 1 for every sample."""
    for kind, n, K in [("mps", 8, 3), ("merged", 4, 2), ("tree", 6, 2)]:
        graph = _graph(kind, n, K)
        names, table, nq, cores, states, mxs = make_case(graph, K, 5, "float32", tnt=False, identity_q=range(64))
        be, eng = _engine("float32", K, built_lib)
        q = tneq_b200.QCTN(graph, backend=be)
        for k, v in cores.items():
            q.cores_weights[k] = v.cuda()
        got = eng.contract_with_compiled_strategy(q, [s.cuda() for s in states], [m.cuda() for m in mxs])
        assert torch.allclose(got.cpu(), torch.ones(5), atol=2e-6)


def test_kat_identity_circuit(built_lib):
    """KAT-2: identity cores, states e_{K-1} => P_b = prod_q Mx_q[b, K-1, K-1]."""
    K, n, B = 3, 6, 11
    graph = _graph("mps", n, K)
    names, table, nq, cores, states, mxs = make_case(graph, K, B, "float64", tnt=False)
    be, eng = _engine("float64", K, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    for k in q.cores:
        q.cores_weights[k] = torch.eye(K * K, dtype=torch.float64).reshape(K, K, K, K).cuda()
    got = eng.contract_with_compiled_strategy(q, [s.cuda() for s in states], [m.cuda() for m in mxs])
    want = torch.ones(B, dtype=torch.float64)
    for m in mxs:
        want = want * m[:, K - 1, K - 1]
    assert rel_err(got, want) < 1e-12


def test_conditional_probability_identity(built_lib):
    """The only numeric assertion of the reference's own test file
    (tests/test_probabilities.py:84-87): P(t|c) == P(t,c) / P(c), atol 1e-5."""
    K, n, B = 2, 4, 6
    graph = _graph("mps", n, K)
    names, table, nq, cores, states, mxs = make_case(graph, K, B, "float32", tnt=False)
    be, eng = _engine("float32", K, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.cuda()
    st = [s.cuda() for s in states]
    m = [x.cuda() for x in mxs]
    joint = eng.calculate_marginal_probability(q, st, [m[0], m[1]], [0, 1])
    marg = eng.calculate_marginal_probability(q, st, [m[0]], [0])
    cond = eng.calculate_conditional_probability(q, st, [m[0], m[1]], [0, 1], [1])
    assert torch.allclose(cond, joint / (marg + 1e-10), atol=1e-5)


def test_sampling_shape_and_bounds(built_lib):
    """tests/test_probabilities.py:296-333: shape (S, n) and -5 <= samples <= 5."""
    K, n = 3, 4
    graph = _graph("mps", n, K)
    be, eng = _engine("float32", K, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    st = [s.cuda() for s in oc.unit_states(n, K)]
    samples = eng.sample(q, st, num_samples=50, K=K, bounds=[-5, 5], grid_size=40)
    assert tuple(samples.shape) == (50, n)
    assert (samples >= -5).all() and (samples <= 5).all()


def test_sampling_linear_method_equals_grid_method(built_lib):
    """SURVEY 8f3: sample(method='linear') -- K^2 contractions per sample and qubit instead of grid_size, using the
    exact linearity of the value in one qubit's measurement matrix -- draws the same samples as the reference's
    grid procedure (method='grid') from the same random numbers, on a chain, a two-layer and a tree network; and
    it launches far fewer contractions' worth of samples."""
    for kind, n, K in (("mps", 6, 3), ("merged", 4, 3), ("tree", 6, 2)):
        graph = _graph(kind, n, K)
        be, eng = _engine("float32", K, built_lib)
        torch.manual_seed(5)
        names, table, nq = oc.parse_graph(graph)
        cores = oc.random_cores(table)
        q = tneq_b200.QCTN(graph, backend=be)
        for k, v in cores.items():
            q.cores_weights[k] = v.cuda()
        st = [s.cuda() for s in oc.unit_states(nq, K)]
        out = {}
        for method in ("grid", "linear"):
            torch.manual_seed(77)
            torch.cuda.manual_seed(77)
            out[method] = eng.sample(q, st, num_samples=64, K=K, bounds=[-5, 5], grid_size=60, method=method)
        assert tuple(out["linear"].shape) == (64, nq)
        assert (out["linear"] - out["grid"]).abs().max().item() < 2e-3, kind


def test_sampling_prefix_environments_equal_contraction_methods(built_lib):
    """SURVEY 8f3: sample(method='prefix') -- one kernel launch, a thread per sample, left environment cached in
    registers, shared right environments (tnq_mps_chain_sample) -- draws the same samples from the same random
    numbers as the reference's procedure (method='grid': one full forward per qubit at batch S x G) and as
    method='linear', for K = 2, 3, 4, TNTensor and plain cores; 'auto' picks it for a single-layer MPS and
    falls back to 'linear' (same draws) elsewhere."""
    for n, K, G, S in ((6, 3, 60, 64), (4, 2, 33, 70), (5, 4, 50, 40), (2, 3, 25, 9)):
        graph = _graph("mps", n, K)
        be, eng = _engine("float32", K, built_lib)
        torch.manual_seed(5 + n)
        names, table, nq = oc.parse_graph(graph)
        cores = oc.random_cores(table)
        q = tneq_b200.QCTN(graph, backend=be)
        for k, v in cores.items():
            q.cores_weights[k] = v.cuda()
        st = [s.cuda() for s in oc.unit_states(nq, K)]
        out = {}
        launches = {}
        for method in ("grid", "linear", "prefix", "auto"):
            torch.manual_seed(77)
            torch.cuda.manual_seed(77)
            l0 = tneq_b200._lib.launch_count()
            out[method] = eng.sample(q, st, num_samples=S, K=K, bounds=[-5, 5], grid_size=G, method=method)
            launches[method] = tneq_b200._lib.launch_count() - l0
        assert tuple(out["prefix"].shape) == (S, nq)
        assert launches["prefix"] == 1 and launches["auto"] == 1 and launches["grid"] >= nq
        assert (out["prefix"] >= -5).all() and (out["prefix"] <= 5).all()
        # float32 round-off in the running sums moves a sample by ~1e-6 of the grid spacing (the bulk agrees to
        # ~1e-6; where a grid cell carries almost no probability the reference's own formula (u - c0) / (c1 - c0 + 1e-10)
        # divides two round-off-sized numbers, hence a bound in units of the cell).  A flipped `cdf < u` comparison is
        # NOT continuous: the formula extrapolates from the first CDF value not below u, so a flip moves y by
        # dx (1 - d[idx+1] / d[idx+2]).  It needs u within the running sums' round-off of a CDF value, which these few
        # draws do not meet; tests/test_gpu_register_kernels.py checks such flips at 227 559 draws.
        cell = 10.0 / (G - 1)
        for other in ("grid", "linear"):
            diff = (out["prefix"] - out[other]).abs()
            assert diff.median().item() < 1e-5 and diff.max().item() < 0.05 * cell, (n, K, other, diff.max().item())
        assert torch.equal(out["auto"], out["prefix"])
    # another network family: 'auto' = 'linear', with the draws made up front
    graph = _graph("merged", 4, 3)
    be, eng = _engine("float32", 3, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    st = [s.cuda() for s in oc.unit_states(4, 3)]
    res = {}
    for method in ("linear", "auto"):
        torch.manual_seed(3)
        torch.cuda.manual_seed(3)
        res[method] = eng.sample(q, st, num_samples=32, K=3, bounds=[-5, 5], grid_size=30, method=method)
    assert (res["auto"] - res["linear"]).abs().max().item() < 1e-5
    with pytest.raises(NotImplementedError):
        eng.sample(q, st, num_samples=4, K=3, grid_size=10, method="prefix")


def test_large_batch_and_ragged_tail(built_lib):
    """Batch sizes that are not a multiple of the tile, and one bigger than a wave."""
    K, n = 3, 8
    graph = _graph("mps", n, K)
    for B in (1, 127, 20011):
        names, table, nq, cores, states, mxs = make_case(graph, K, B, "float32", tnt=True, seed=B)
        want = oc.forward(graph, cores, states, clone_mx(mxs))
        be, eng = _engine("float32", K, built_lib)
        q = tneq_b200.QCTN(graph, backend=be)
        for k, v in cores.items():
            q.cores_weights[k] = v.cuda()
        got = eng.contract_with_compiled_strategy(q, [s.cuda() for s in states],
                                                  [_to_dev(m, torch.device("cuda:0")) for m in clone_mx(mxs)])
        assert rel_err(got, want) < 2e-5


@pytest.mark.parametrize("n,K,B", [(16, 3, 1000), (6, 2, 130), (5, 4, 77), (2, 3, 9)])
def test_contract_from_x_fused_generate_data(n, K, B, built_lib):
    """SURVEY 8f2: EngineSiamese.contract_from_x (generate_data fused into the chain kernel, tnq_mps_chain_x)
    against the oracle's generate_data (engine_siamese.py:133-254) + forward, and against this package's own
    unfused route; the per-qubit TNTensor scales (tn_tensor.py:72-85) are reproduced too."""
    graph = _graph("mps", n, K)
    torch.manual_seed(n * 7 + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table)
    states = oc.unit_states(nq, K)
    x = torch.randn(B, nq)
    mx, _ = oc.generate_data(x, K, torch.float32, "TNTensor")
    want = oc.forward(graph, cores, states, clone_mx(mx))
    truth = oc.forward(graph, {k: v.double() for k, v in cores.items()}, [s.double() for s in states],
                       [upcast(m, torch.float64) for m in clone_mx(mx)])
    be, eng = _engine("float32", K, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.cuda()
    st = [s.cuda() for s in states]
    launches0 = tneq_b200._lib.launch_count()
    got = eng.contract_from_x(q, st, x.cuda(), K=K)
    assert tneq_b200._lib.launch_count() == launches0 + 2, "scale kernel + fused chain kernel"
    assert got.shape == want.shape
    assert rel_err(got, want) < 1e-5
    assert elem_rel_err(got.double(), truth) < max(1e-5, NOISE_FACTOR * elem_rel_err(want.double(), truth))
    res = eng.contract_from_x(q, st, x.cuda(), K=K, ret_type="TNTensor")
    ref_scale = 1.0
    for m in mx:
        ref_scale *= m.scale
    assert abs(res.scale - ref_scale) <= 1e-5 * ref_scale
    unfused = eng.contract_with_compiled_strategy(q, st, eng.generate_data(x.cuda(), K=K, ret_type="TNTensor")[0])
    assert rel_err(got, unfused) < 1e-5


def test_contract_from_x_other_networks_take_the_usual_route(built_lib):
    K, n, B = 3, 5, 40
    graph = _graph("merged", n, K)
    names, table, nq, cores, states, mxs = make_case(graph, K, B, "float32")
    be, eng = _engine("float32", K, built_lib)
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.cuda()
    st = [s.cuda() for s in states]
    torch.manual_seed(3)
    x = torch.randn(B, nq).cuda()
    a = eng.contract_from_x(q, st, x, K=K)
    b = eng.contract_with_compiled_strategy(q, st, eng.generate_data(x, K=K, ret_type="TNTensor")[0])
    assert torch.equal(a, b)
