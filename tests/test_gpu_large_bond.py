"""The large-bond route (contractor/gemm_path.py) in float64 parity at the batch sizes where its GEMM variants fire.

Which kernels a plan launches depends on the batch size: the core-gradient GEMM that reads MN-major operands in place
(tnq_gemm_tf32x3_bk) only runs once batch x Kin > 256, and split-K (tnq_gemm.cu, launch_tma) only when a launch covers
at most 74 output tiles.  Each case below is a single-layer MPS (unitary cores, states e_{K-1}, measurements I + eps H)
whose values, loss and core gradients are compared with the complex128 / float64 yardstick helpers.mps_f64, on the route
that reads operands in place and on the transposing one (gemm_path.MN_IN_PLACE = False).  A route recorder asserts
that each case still reaches the variants it exists for (helpers.LARGE_BOND_CASES; the same expectations are checked
on meta tensors by tests/test_gemm_path_plan.py).  cfg4 itself (16 qubits, bond 64, B = 256) is too big for the
yardstick and is checked by known answers and by splitting its batch."""
import pytest
import torch

import tneq_b200
from helpers import LARGE_BOND_CASES, elem_rel_err, mps_f64, mps_f64_value, record_routes, rel_err
from tneq_b200.contractor import gemm_path
from tneq_b200.contractor.gemm_path import GemmPathRunner

pytestmark = pytest.mark.gpu
H = tneq_b200.QCTNHelper


@pytest.fixture
def routes(monkeypatch):
    """Counter of the GEMM-path kernel variants launched (keys: helpers.record_routes)."""
    return record_routes(monkeypatch, GemmPathRunner)


def _network(dtype, chi, n, seed):
    """Engine + network with unitary (complex, QR in complex128) or orthogonal (real, QR in float64) cores that
    require gradients, and the states e_{K-1}."""
    td = getattr(torch, dtype)
    graph = H.generate_example_graph(n=n, graph_type="mps", dim_char=str(chi))
    be = tneq_b200.BackendFactory.create_backend("b200", device="cuda:0", dtype=dtype)
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=chi)
    q = tneq_b200.QCTN(graph)
    torch.manual_seed(seed)
    for c in q.cores:
        m = torch.randn(chi * chi, chi * chi, dtype=torch.complex128 if td.is_complex else torch.float64, device="cuda")
        qm, _ = torch.linalg.qr(m)
        q.cores_weights[c] = qm.reshape(chi, chi, chi, chi).to(td).requires_grad_(True)
        del m, qm
    st = [torch.zeros(chi, dtype=td, device="cuda") for _ in range(n)]
    for s in st:
        s[-1] = 1.0
    return eng, q, st


def _measurements(dtype, chi, n, B, seed, eps=0.1):
    """I + eps H per qubit and sample (H Hermitian, unit scale): keeps the value O(1), where a random unitary's
    overlap alone would be ~K^-n."""
    td = getattr(torch, dtype)
    torch.manual_seed(seed)
    mx = []
    for _ in range(n):
        h = torch.randn(B, chi, chi, dtype=td, device="cuda") / (2.0 * chi ** 0.5)
        mx.append(torch.eye(chi, dtype=td, device="cuda") + eps * (h + h.transpose(1, 2).conj()))
    return mx


def _yardstick(q, st, mx):
    """values, loss -mean(log clamp(value, 1e-10)) and core gradients in complex128 / float64 (torch.autograd)."""
    td64 = torch.complex128 if st[0].is_complex() else torch.float64
    leaves = [q.cores_weights[c].detach().to(td64).requires_grad_(True) for c in q.cores]
    val = mps_f64_value(mps_f64(leaves, [s.to(td64) for s in st], [m.to(td64) for m in mx]))
    loss = -torch.log(torch.clamp(val, min=1e-10)).mean()
    grads = torch.autograd.grad(loss, leaves)
    return val.detach(), loss.detach(), [g.detach() for g in grads]


def _engine(eng, q, st, mx, fused=True):
    val = eng.contract_with_compiled_strategy(q, st, mx)
    loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, st, mx, fused=fused)
    torch.cuda.synchronize()
    return val.detach(), loss.detach(), [g.detach() for g in grads]


def _loss_err(got, want):
    # loss = -mean(log value): its ABSOLUTE error is the relative error of the values
    return abs(float(got) - float(want)) / max(abs(float(want)), 1.0)


def _errors(got, want):
    """(value, loss, worst gradient) error of one engine run against another result (float64 or float32)"""
    val, loss, grads = got
    wval, wloss, wgrads = want
    assert val.shape == wval.shape and len(grads) == len(wgrads)
    for g, w in zip(grads, wgrads):
        assert g.shape == w.shape
    return (rel_err(val.to(wval.dtype), wval), _loss_err(loss, wloss),
            max(rel_err(g.to(w.dtype), w) for g, w in zip(grads, wgrads)))


@pytest.mark.parametrize("dtype,chi,n,B,want_mn,want_tr", LARGE_BOND_CASES,
                         ids=[f"{c[0]}-chi{c[1]}-n{c[2]}-B{c[3]}" for c in LARGE_BOND_CASES])
def test_large_bond_vs_float64_on_both_routes(dtype, chi, n, B, want_mn, want_tr, routes, monkeypatch, built_lib):
    """Values (1e-5 relative, 2e-5 for |amp|^2), loss (1e-5) and every core gradient (1e-5 of its largest entry)
    against float64 on the in-place route and on the transposing route, which must also agree with each other to
    1e-5; at the smallest batch that reaches the in-place GEMM also through the autograd route (fused=False)."""
    eng, q, st = _network(dtype, chi, n, seed=3)
    mx = _measurements(dtype, chi, n, B, seed=4)
    truth = _yardstick(q, st, mx)
    assert 1e-3 < truth[0].min().item() and truth[0].max().item() < 1e3
    tol_v = 2e-5 if getattr(torch, dtype).is_complex else 1e-5        # |amplitude|^2: the amplitude's 1e-5 doubles
    fused_modes = (True, False) if (chi, n, B) == (64, 4, 5) else (True,)
    runs = {}
    for mn, want in ((True, want_mn), (False, want_tr)):
        monkeypatch.setattr(gemm_path, "MN_IN_PLACE", mn)
        for fused in fused_modes:
            routes.clear()
            runs[mn, fused] = got = _engine(eng, q, st, mx, fused=fused)
            assert want <= set(routes), (mn, fused, sorted(want - set(routes)))
            if not mn:
                assert not [k for k in routes if k[0] == "bk"]
            ev, el, eg = _errors(got, truth)
            print(f"[{dtype} chi={chi} n={n} B={B} mn_in_place={mn} fused={fused}] vs float64: value {ev:.2e} "
                  f"loss {el:.2e} grad {eg:.2e}")
            assert ev < tol_v and el <= 1e-5 and eg < 1e-5, (mn, fused, ev, el, eg)
    for fused in fused_modes:
        ev, el, eg = _errors(runs[True, fused], runs[False, fused])
        assert ev < 1e-5 and el <= 1e-5 and eg < 1e-5, ("routes disagree", fused, ev, el, eg)


def _degree_identity(q, grads, complex_):
    """Each core enters the value as a homogeneous function of degree 4 (|amp|^2, complex) or 2 (amp, real): scaling
    it by t adds -4 log t (-2 log t) to the loss, so sum Re(conj(grad) * core) = -4 (-2) for every core, whatever the
    measurements.  Returns the worst relative deviation."""
    want = -4.0 if complex_ else -2.0
    worst = 0.0
    for c, g in zip(q.cores, grads):
        s = (g.to(torch.complex128 if complex_ else torch.float64).conj() *
             q.cores_weights[c].detach().to(torch.complex128 if complex_ else torch.float64)).real.sum().item()
        worst = max(worst, abs(s - want) / abs(want))
    return worst


def test_cfg4_full_shape(routes, monkeypatch, built_lib):
    """cfg4 (16 qubits, bond 64, complex64, B = 256) at full shape, where no float64 reference fits:
    (1) KAT-1: unitary cores + identity measurements give value 1 (2e-5: |amplitude|^2) and loss 0 for every sample;
    (2) the degree identity of the core gradients (_degree_identity), with identity and with I + eps H measurements,
        to 2e-5: the identity compares the gradient with the value, so it carries the value's error;
    (3) the batch split 100 + 156: the halves take other GEMM variants (the forward view GEMM splits K at B = 100, not at
        156 or 256), yet the sample-weighted loss and gradients match the full batch to 1e-5 of the largest entry, and
        the values match per sample to 2e-5."""
    chi, n, B = 64, 16, 256
    monkeypatch.setattr(gemm_path, "MN_IN_PLACE", True)
    eng, q, st = _network("complex64", chi, n, seed=11)
    eye = torch.eye(chi, dtype=torch.complex64, device="cuda").expand(B, chi, chi).contiguous()
    val, loss, grads = _engine(eng, q, st, [eye] * n)
    cfg4 = LARGE_BOND_CASES[0]
    assert cfg4[:4] == ("complex64", 64, 5, 256)
    assert cfg4[4] <= set(routes), sorted(cfg4[4] - set(routes))
    assert routes[("bk", 1, 0, True)] + routes[("bk", 0, 1, True)] == 27 and routes[("bk", 1, 1, True)] == 1
    e_val = elem_rel_err(val.double(), torch.ones(B, dtype=torch.float64))
    e_id = _degree_identity(q, grads, True)
    print(f"[cfg4 KAT-1] value {e_val:.2e} loss {abs(loss.item()):.2e} degree identity {e_id:.2e}")
    assert val.shape == (B,) and e_val < 2e-5 and abs(loss.item()) < 2e-5 and e_id < 2e-5

    mx = _measurements("complex64", chi, n, B, seed=12)
    val, loss, grads = _engine(eng, q, st, mx)
    assert 1e-3 < val.min().item() and val.max().item() < 1e3
    e_id = _degree_identity(q, grads, True)
    halves = []
    for lo, hi, view_split in ((0, 100, True), (100, 256, False)):
        routes.clear()
        halves.append(_engine(eng, q, st, [m[lo:hi].contiguous() for m in mx]))
        assert routes[("view", view_split)] > 0 and routes[("view", not view_split)] == 0, dict(routes)
        assert routes[("bk", 1, 0, True)] > 0 and routes[("bk", 0, 1, True)] > 0
    (v1, l1, g1), (v2, l2, g2) = halves
    w1, w2 = 100 / B, 156 / B
    e_val = elem_rel_err(torch.cat([v1, v2]).double(), val.double())
    e_loss = _loss_err(w1 * l1.double() + w2 * l2.double(), loss.double())
    e_grad = max(rel_err(w1 * a.to(torch.complex128) + w2 * b.to(torch.complex128), g.to(torch.complex128))
                 for a, b, g in zip(g1, g2, grads))
    print(f"[cfg4 I + eps H] degree identity {e_id:.2e}; batch 100 + 156 vs 256: value {e_val:.2e} loss {e_loss:.2e} "
          f"grad {e_grad:.2e}")
    assert e_id < 2e-5 and e_val < 2e-5 and e_loss <= 1e-5 and e_grad < 1e-5, (e_id, e_val, e_loss, e_grad)
