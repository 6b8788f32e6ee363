"""GPU parity of the Stiefel/Cayley optimizer kernel (csrc/tnq_sgdg.cu) for complex64, float64 and complex128
cores (tnq_sgdg_step_{c64,f64,c128} and their _flat siblings) against the oracle's restatement of
backend_pytorch.py:349-468 evaluated in float64 / complex128, and against the reference's own float64 steps."""
import random

import pytest
import torch

from oracle import qctn_oracle as oc

pytestmark = pytest.mark.gpu

DTYPES = [torch.complex64, torch.float64, torch.complex128]
# relative (Frobenius) error of one step against the float64 / complex128 oracle
TOL = {torch.complex64: 2e-5, torch.float64: 1e-12, torch.complex128: 1e-12}
# p p^H = X X^H (= I up to the 1e-8 of the row normalisation)
ORTHO = {torch.complex64: 1e-4, torch.float64: 1e-12, torch.complex128: 1e-12}
WIDEST = {torch.complex64: (8, 8, 8, 8), torch.float64: (8, 8, 8, 8), torch.complex128: (48, 48)}
DEV = torch.device("cuda:0")


def _wide(dtype):
    return torch.complex128 if dtype.is_complex else torch.float64


def _rel(a, b):
    return ((a.to(b.dtype).cpu() - b).norm() / max(b.norm(), 1e-30)).item()


def _stiefel_cores(shape, ncores, dtype):
    """Cores whose matrix has orthonormal rows up to a row scale, in the oracle's precision."""
    from tneq_b200.optim import steps
    rows, cols = steps._matrix_shape(shape)
    out = []
    for _ in range(ncores):
        q, _r = torch.linalg.qr(torch.randn(cols, cols, dtype=_wide(dtype)))
        out.append((q[:rows] * (1 + 0.1 * torch.rand(rows, 1, dtype=torch.float64))).reshape(shape).contiguous())
    return out


def _quiet_seed(ndraws, start):
    """A Python-random seed whose next ndraws draws fire no QR retraction."""
    return next(s for s in range(start, start + 10000)
                if (random.seed(s) or True) and all(random.randint(1, 101) != 1 for _ in range(ndraws)))


def _firing_seed(ndraws):
    return next(s for s in range(10000) if (random.seed(s) or True) and any(random.randint(1, 101) == 1 for _ in range(ndraws)))


def _cases():
    # (core shape, number of cores): 2-leg-per-side MPS cores of rank 2/3/4, a rectangular edge core, a plain matrix,
    # a wide rectangular matrix, the widest matrix of the dtype
    shapes = [((2, 2, 2, 2), 5), ((3, 3, 3, 3), 46), ((4, 4, 4, 4), 7), ((3, 3, 3), 3), ((8, 8), 2), ((4, 16), 2)]
    return [pytest.param(dt, s, n, id=f"{str(dt)[6:]}-{'x'.join(map(str, s))}x{n}")
            for dt in DTYPES for s, n in shapes + [(WIDEST[dt], 2)]]


@pytest.mark.parametrize("dtype,shape,ncores", _cases())
def test_sgdg_kernel_matches_oracle(built_lib, dtype, shape, ncores):
    """Four consecutive steps with momentum 0.9, each started from the kernel's previous point: parameters and momentum
    against the oracle, orthonormal rows, one launch per step, fresh tensors."""
    from tneq_b200.optim import steps
    from tneq_b200 import _lib
    torch.manual_seed(hash(shape) % 1000 + DTYPES.index(dtype))
    rows, cols = steps._matrix_shape(shape)
    params = [p.to(dtype).to(DEV) for p in _stiefel_cores(shape, ncores, dtype)]
    st_w, st_g = {}, {}
    hp = dict(learning_rate=0.05, momentum=0.9, stiefel=True)
    for it in range(4):
        grads64 = [0.3 * torch.randn(shape, dtype=_wide(dtype)) for _ in range(ncores)]
        grads = [g.to(dtype).to(DEV) for g in grads64]
        start = [p.detach().cpu().to(_wide(dtype)) for p in params]
        if st_g.get("momentum_buffer"):
            st_w["momentum_buffer"] = [v.cpu().to(_wide(dtype)) for v in st_g["momentum_buffer"]]
        seed = _quiet_seed(ncores, 1000 * it)
        random.seed(seed)
        want, st_w = oc.sgdg_step(start, grads64, st_w, lr=0.05, momentum=0.9)
        random.seed(seed)
        before = _lib.launch_count()
        old_ptrs = [p.data_ptr() for p in params]
        got, st_g = steps.optimizer_update(list(params), grads, st_g, "sgdg", hp)
        assert _lib.launch_count() == before + 1, "all cores must go through ONE kernel launch"
        for a, b, o in zip(got, want, old_ptrs):
            assert a.dtype == dtype and a.shape == b.shape and a.data_ptr() != o, "fresh tensors like the reference"
            assert _rel(a, b) < TOL[dtype], f"step {it}: param err {_rel(a, b):.2e}"
        for a, b in zip(st_g["momentum_buffer"], st_w["momentum_buffer"]):
            assert a.dtype == dtype and _rel(a, b) < TOL[dtype], f"step {it}: momentum err {_rel(a, b):.2e}"
        for a, x in zip(got, start):
            # the step is a unitary map of X = p / (||p||_row + 1e-8), so p_new p_new^H = X X^H: the identity, up to
            # the reference's 1e-8 in the row norm (its own rows come out 1e-8 short of unit norm too)
            m = a.reshape(rows, cols).to(_wide(dtype)).cpu()
            x = x.reshape(rows, cols)
            x = x / (x.norm(dim=1, keepdim=True) + 1e-8)
            assert (m @ m.conj().T - x @ x.conj().T).abs().max().item() < ORTHO[dtype]
            assert (m @ m.conj().T - torch.eye(rows, dtype=m.dtype)).abs().max().item() < 1e-4
        params = [g.detach() for g in got]


def test_sgdg_kernel_matches_reference_fixture_f64(built_lib):
    """The float64 kernel against three consecutive steps of the REAL reference (tests/golden/sgdg_f64.npz, written by
    oracle/make_golden.py from backend_pytorch.py:349-468, momentum 0.5), including a fired QR retraction, within the
    oracle's own bound of 1e-12."""
    import os
    from test_oracle_golden import load_sgdg
    from tneq_b200.optim import steps
    from tneq_b200 import _lib
    path = os.path.join(os.path.dirname(__file__), "golden", "sgdg_f64.npz")
    params, grads, want, lr, momentum, seed, dtype = load_sgdg(path)
    assert dtype == "float64"
    params = [p.to(DEV) for p in params]
    assert all(steps.sgdg_kernel_eligible(p.dtype, p.shape, "cuda") for p in params)
    state = {}
    random.seed(seed)
    for k in range(3):
        before = _lib.launch_count()
        params, state = steps.optimizer_update(list(params), [g.to(DEV) for g in grads[k]], state, "sgdg",
                                               dict(learning_rate=lr, momentum=momentum, stiefel=True))
        assert _lib.launch_count() == before + 1
        params = [p.detach() for p in params]
        for a, b in zip(params, want[k]):
            assert (a.cpu() - b).abs().max() <= 1e-12 * b.abs().max(), (k, (a.cpu() - b).abs().max().item())


def _views_of_one_buffer(ncores, shape, dtype):
    """Gradients as the contraction routes return them: views of ONE buffer; complex ones are view_as_complex views
    of one REAL buffer."""
    n = ncores * int(torch.tensor(shape).prod())
    if dtype.is_complex:
        real = 0.3 * torch.randn(2 * n, dtype=dtype.to_real(), device=DEV)
        flat = torch.view_as_complex(real.view(n, 2))
    else:
        real = flat = 0.3 * torch.randn(n, dtype=dtype, device=DEV)
    views = list(flat.view(ncores, *shape).unbind(0))
    assert all(v._base is real for v in views)
    return views


@pytest.mark.parametrize("dtype", DTYPES, ids=[str(d)[6:] for d in DTYPES])
def test_sgdg_flat_gradients_take_the_table_free_launch(built_lib, dtype):
    """Gradients that are views of one buffer take tnq_sgdg_step_flat_*: results torch.equal to the pointer-table
    launch over 5 steps with momentum, one launch per step, and from the second step on no host synchronisation
    (torch.cuda.set_sync_debug_mode("error")).  The torch route synchronises there: the negative control."""
    from tneq_b200.optim import steps
    from tneq_b200 import _lib
    torch.manual_seed(11)
    shape, ncores = (3, 3, 3, 3), 46
    params = [oc.init_random_core([9, 9], dtype).reshape(shape).to(DEV) for _ in range(ncores)]
    pa, pb = [p.clone() for p in params], [p.clone() for p in params]
    sa, sb = {}, {}
    hp = dict(learning_rate=0.05, momentum=0.9, stiefel=True)
    for it in range(5):
        views = _views_of_one_buffer(ncores, shape, dtype)
        separate = [v.clone() for v in views]
        seed = _quiet_seed(ncores, 100 * it)
        random.seed(seed)
        before = _lib.launch_count()
        old = [p.data_ptr() for p in pa]
        torch.cuda.synchronize()
        if it > 0:
            torch.cuda.set_sync_debug_mode("error")
        try:
            ga, sa = steps.optimizer_update(list(pa), views, sa, "sgdg", hp)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert _lib.launch_count() == before + 1 and "_flat_offs" in sa
        random.seed(seed)
        gb, sb = steps.optimizer_update(list(pb), separate, sb, "sgdg", hp)
        assert "_flat_offs" not in sb
        for a, b, o in zip(ga, gb, old):
            assert a.dtype == dtype and a.data_ptr() != o and torch.equal(a, b)
        for a, b in zip(sa["momentum_buffer"], sb["momentum_buffer"]):
            assert a.dtype == dtype and torch.equal(a, b)
        pa, pb = [g.detach() for g in ga], [g.detach() for g in gb]
    random.seed(_quiet_seed(ncores, 0))
    torch.cuda.set_sync_debug_mode("error")
    try:
        with pytest.raises(RuntimeError):
            steps.optimizer_update(list(pa), views, {}, "sgdg", dict(hp, device_kernel=False))
    finally:
        torch.cuda.set_sync_debug_mode("default")


def test_sgdg_kernel_qr_retraction_and_tntensor_c64(built_lib):
    """complex64 TNTensor cores keep their scale, and a seed that fires the 1 % QR retraction still matches the
    oracle."""
    from tneq_b200.optim import steps
    from tneq_b200 import _lib
    import tneq_b200 as tb
    torch.manual_seed(3)
    seed = _firing_seed(6)
    params64 = [oc.init_random_core([9, 9], torch.complex128).reshape(3, 3, 3, 3) * 1.3 for _ in range(6)]
    grads64 = [torch.randn(3, 3, 3, 3, dtype=torch.complex128) for _ in range(6)]
    random.seed(seed)
    want, _ = oc.sgdg_step([p.clone() for p in params64], grads64, {}, lr=0.02, momentum=0.0)
    random.seed(seed)
    tnts = [tb.TNTensor((p / 2.0).to(torch.complex64).to(DEV), 2.0) for p in params64]
    before = _lib.launch_count()
    got, _ = steps.optimizer_update(tnts, [(2.0 * g).to(torch.complex64).to(DEV) for g in grads64], {}, "sgdg",
                                    dict(learning_rate=0.02))
    assert _lib.launch_count() == before + 1
    for a, b in zip(got, want):
        assert isinstance(a, tb.TNTensor) and a.tensor.requires_grad and a.scale == 2.0
        assert _rel((a.tensor.detach() * a.scale), b) < TOL[torch.complex64]


@pytest.mark.parametrize("dtype,wide", [(torch.complex64, (9, 9, 9, 9)), (torch.complex128, (7, 7, 7, 7))],
                         ids=["complex64", "complex128"])
def test_sgdg_mixed_widths(built_lib, dtype, wide):
    """A network with one core wider than its dtype's maximum: the narrow cores take one launch, the wide one takes
    torch, and all match the oracle over three steps with momentum."""
    from tneq_b200.optim import steps
    from tneq_b200 import _lib
    torch.manual_seed(5)
    shapes = [(3, 3, 3, 3)] * 2 + [wide] + [(3, 3, 3, 3)] * 2 + [(3, 3, 3)]
    assert [steps.sgdg_kernel_eligible(dtype, s, "cuda") for s in shapes] == [True, True, False, True, True, True]
    params = [_stiefel_cores(s, 1, dtype)[0].to(dtype).to(DEV) for s in shapes]
    st_w, st_g = {}, {}
    for it in range(3):
        grads64 = [0.3 * torch.randn(s, dtype=_wide(dtype)) for s in shapes]
        start = [p.detach().cpu().to(_wide(dtype)) for p in params]
        if st_g.get("momentum_buffer"):
            st_w["momentum_buffer"] = [v.cpu().to(_wide(dtype)) for v in st_g["momentum_buffer"]]
        seed = _quiet_seed(len(shapes), 500 * it)
        random.seed(seed)
        want, st_w = oc.sgdg_step(start, grads64, st_w, lr=0.05, momentum=0.9)
        random.seed(seed)
        before = _lib.launch_count()
        got, st_g = steps.optimizer_update(list(params), [g.to(dtype).to(DEV) for g in grads64], st_g, "sgdg",
                                           dict(learning_rate=0.05, momentum=0.9))
        assert _lib.launch_count() == before + 1
        for a, b in zip(got, want):
            assert _rel(a, b) < TOL[dtype], f"step {it}: {_rel(a, b):.2e}"
        params = [g.detach() for g in got]


def _train(dtype, merged, kernel, monkeypatch, steps_n=10):
    """steps_n training steps of a 6-qubit K = 3 network through the public API on one well-conditioned batch (samples
    near the loss clamp or whose value nearly cancels turn rounding differences into loss differences of any size,
    helpers.well_conditioned_case); returns the losses, the launches of each optimizer step and the optimizer state."""
    import tneq_b200 as tb
    from tneq_b200 import _lib
    from tneq_b200.optim import steps
    from helpers import well_conditioned_case
    if not kernel:
        monkeypatch.setattr(steps, "sgdg_kernel_eligible", lambda *a: False)
    n, K, B = 6, 3, 64
    random.seed(42)
    be = tb.BackendFactory.create_backend("b200", device="cuda:0", dtype=str(dtype)[6:])
    eng = tb.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    graph = tb.QCTNHelper.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))
    if merged:
        one = tb.QCTN(graph, backend=be)
        graph = tb.QCTN.merge(one, one).graph
    _, _, nq, cores, states, mxs = well_conditioned_case(graph, K, B, str(dtype)[6:], seed=3)
    q = tb.QCTN(graph, backend=be)
    for name, core in cores.items():
        q.cores_weights[name] = core.to(DEV).requires_grad_(True)
    states = [s.to(DEV) for s in states]
    opt = tb.Optimizer(method="sgdg", learning_rate=0.02, max_iter=steps_n, engine=eng, momentum=0.9, stiefel=True,
                       verbose=False)
    losses, launches = [], []
    for step in range(steps_n):
        data = [tb.TNTensor(m.tensor.to(DEV), m.scale, m.log_scale) for m in mxs]
        loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, states, data)
        assert all(g.dtype == dtype for g in grads)
        losses.append(float(loss))
        before = _lib.launch_count()
        opt.step(q, grads)
        launches.append(_lib.launch_count() - before)
        opt.iter += 1
    monkeypatch.undo()
    return losses, launches, opt.opt_state


@pytest.mark.parametrize("dtype,merged,rtol", [(torch.complex64, False, 1e-4), (torch.float64, True, 1e-10)],
                         ids=["complex64-mps", "float64-merged"])
def test_sgdg_training_end_to_end(built_lib, monkeypatch, dtype, merged, rtol):
    """Ten steps of tb.Optimizer(method="sgdg", momentum=0.9) through the public API (VM route): the losses track the
    same run on the torch route, every optimizer step is one launch of the table-free kernel."""
    got, launches, state = _train(dtype, merged, True, monkeypatch)
    want, launches_t, _ = _train(dtype, merged, False, monkeypatch)
    assert launches == [1] * len(got) and "_flat_offs" in state, launches
    assert launches_t == [0] * len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert abs(a - b) <= rtol * abs(b), (k, a, b)


ENTRY = [("c64", 64), ("f64", 64), ("c128", 48)]


@pytest.mark.parametrize("sfx,widest", ENTRY, ids=[e[0] for e in ENTRY])
def test_sgdg_bad_arguments_new_dtypes(built_lib, sfx, widest):
    """Null pointers and widths outside [1, max] fail with a message and launch nothing."""
    from tneq_b200 import _lib
    lib = _lib.load()
    p = torch.zeros(8, device=DEV).data_ptr()
    for flat in (False, True):
        name = f"tnq_sgdg_step{'_flat' if flat else ''}_{sfx}"
        fn = getattr(lib, name)
        ptrs = [p] * (6 if flat else 5)
        before = _lib.launch_count()
        assert fn(*([None] * len(ptrs)), 1, 4, 0.1, 0.0, None) != 0
        assert b"bad arguments" in lib.tnq_last_error() and name.encode() in lib.tnq_last_error()
        for i in range(len(ptrs)):
            assert fn(*(ptrs[:i] + [None] + ptrs[i + 1:]), 1, 4, 0.1, 0.0, None) != 0
            assert b"bad arguments" in lib.tnq_last_error()
        for width in (widest + 1, 0):
            assert fn(*ptrs, 1, width, 0.1, 0.0, None) != 0
            assert f"between 1 and {widest}".encode() in lib.tnq_last_error()
        assert _lib.launch_count() == before
