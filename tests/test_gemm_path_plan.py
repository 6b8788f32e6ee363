"""Host logic of the large-bond route, checked WITHOUT a GPU: the GEMM-path runner walks the bond-64 plan on meta
tensors (tools/gemm_path_dryrun.py) and every launch it would make is logged.  Guards the data-movement decisions of
contractor/gemm_path.py: operands read in place through strided tensor-map views, fused circuit-state folding, row
order that keeps (index, re/im) pairs adjacent -- a regression here shows up as gigabytes of extra transpositions."""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import gemm_path_dryrun as dr  # noqa: E402
import pytest  # noqa: E402
import tneq_b200  # noqa: E402
from helpers import LARGE_BOND_CASES, record_routes  # noqa: E402
from tneq_b200.contractor import gemm_path  # noqa: E402
from tneq_b200.contractor.plan import ContractionPlan, signature_of  # noqa: E402


def _walk(n, chi, B, fired=None, dtype="complex64"):
    graph = tneq_b200.QCTNHelper.generate_example_graph(n=n, graph_type="mps", dim_char=str(chi))
    q = tneq_b200.QCTN(graph)
    td = getattr(torch, dtype)
    states = [torch.empty(chi, dtype=td, device="meta") for _ in range(n)]
    mxs = [torch.empty(B, chi, chi, dtype=td, device="meta") for _ in range(n)]
    sd, mi = signature_of(q.nqubits, states, mxs)
    plan = ContractionPlan(q.adjacency_table, q.nqubits, {c: q.core_shape(c) for c in q.cores}, sd, mi, dtype)
    g = plan.graph("bwd")
    r = dr.DryRunner(g)
    inputs = {}
    for key, ids in g.inputs.items():
        node = g.nodes[ids[0]]
        size = g.size(node.idx)
        inputs[key] = torch.empty((B, size) if node.batched else (size,), dtype=torch.float32, device="meta")
    seed = torch.empty(B * g.size(g.nodes[g.result].idx), dtype=torch.float32, device="meta")
    hook = (lambda key, t: fired.append((key, len(r.log)))) if fired is not None else None
    r.run(inputs, B, 1, with_adjoint=True, seed=seed, on_grad_ready=hook)
    return g, r


def test_bond64_plan_data_movement():
    g, r = _walk(5, 64, 256)
    kinds = [e[0] for e in r.log]
    views = [e for e in r.log if e[0] == "gemm" and isinstance(e[6], tuple) and e[6] and e[6][0] == "view"]
    # per middle qubit: one forward and one reverse contraction of the B*chi^3 intermediate read in place
    assert len(views) == 6
    for e in views:
        R1, R0, sR1, sR0, K1, K0, sK1 = e[6][1:]
        assert (R1, R0, K1, K0) == (256, 64, 64, 128) and sR0 == K0 and sK1 == R0 * K0 and sR1 == K1 * sK1
    # core gradients: the big operand is consumed MN-major in place, the batch joins the contraction index
    bks = [e for e in r.log if e[0] == "gemm" and isinstance(e[6], tuple) and e[6] and e[6][0] == "bk"]
    assert len(bks) == 6 and all(e[4] == 256 * 64 and (e[6][1] or e[6][2]) for e in bks)
    # circuit-state folding and its adjoint are the fused one-pass kernels, never a GEMM with two columns / K = 2
    assert kinds.count("foldvec") >= 2 * 4 and kinds.count("outeracc") >= 2 * 4
    assert not [e for e in r.log if e[0] == "gemm" and (e[3] == 2 or e[4] == 2) and e[2] >= 1 << 16]
    # no strided scalar transposition of a 537 MB tensor: every big permute has a long input-contiguous run after
    # merging neighbours (what tnq_permute_f32's canonicalisation needs for its tiled paths)
    moved = sum(e[1] for e in r.log if e[0] != "gemm")
    assert 2 * moved < 12e9, 2 * moved / 1e9            # 40.3 GB before this round's changes, 9.1 GB now
    for e in r.log:
        if e[0] == "permute" and e[1] > 500e6:
            dims, strides = e[2], e[3]
            # merge (as the C side does) and find the input-contiguous dimension
            md, ms = [dims[0]], [strides[0]]
            for d_, s_ in zip(dims[1:], strides[1:]):
                if ms[-1] == s_ * d_:
                    md[-1], ms[-1] = md[-1] * d_, s_
                else:
                    md.append(d_), ms.append(s_)
            assert 1 in ms and md[ms.index(1)] >= 64, (dims, strides)
    assert abs(r.flops - 0.829e12) < 0.01e12            # the arithmetic is unchanged: 3 GEMM-shaped contractions per qubit x 3


def test_grad_ready_hook_fires_once_per_core_in_reverse_use_order():
    fired = []
    g, r = _walk(5, 16, 8, fired)
    keys = [k for k, _ in fired]
    assert sorted(keys) == sorted(g.grads) and len(set(keys)) == len(keys)
    # the last core of the chain is final first, the first core last, and launches keep coming after the early ones
    order = {k: i for i, (k, _) in enumerate(fired)}
    names = sorted(g.grads, key=lambda k: str(k))
    assert order[names[-1]] < order[names[0]]
    assert fired[0][1] < len(r.log)


@pytest.mark.parametrize("dtype,chi,n,B,want_mn,want_tr", LARGE_BOND_CASES,
                         ids=[f"{c[0]}-chi{c[1]}-n{c[2]}-B{c[3]}" for c in LARGE_BOND_CASES])
@pytest.mark.parametrize("mn_in_place", [True, False])
def test_large_bond_case_plans_reach_their_variants(dtype, chi, n, B, want_mn, want_tr, mn_in_place, monkeypatch):
    """The GEMM variants each float64-parity case of tests/test_gpu_large_bond.py exists to reach (the same recorder,
    here around the dry runner): a routing change that drops a case's coverage fails here without a GPU."""
    monkeypatch.setattr(gemm_path, "MN_IN_PLACE", mn_in_place)
    seen = record_routes(monkeypatch, dr.DryRunner)
    _walk(n, chi, B, dtype=dtype)
    want = want_mn if mn_in_place else want_tr
    assert want <= set(seen), sorted(want - set(seen))
    if not mn_in_place:
        assert not [k for k in seen if k[0] == "bk"]
