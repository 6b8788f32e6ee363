"""The float64 yardstick of the large-bond tests (helpers.mps_f64) against the oracle, on the CPU.

At bond 32-128 the oracle's greedy einsum builds K^6 intermediates, so tests/test_gpu_large_bond.py and
tests/test_gpu_gemm_path.py compare the CUDA route with helpers.mps_f64 instead: the same single-layer MPS sweep
restated pairwise (3 K^4 per qubit and sample).  Here that restatement is pinned to the oracle where both fit:
values, and the autograd gradients of the engine's loss -mean(log clamp(value, 1e-10)) against
oc.loss_and_grads, in float64 and complex128."""
import pytest
import torch

import tneq_b200
from oracle import qctn_oracle as oc
from helpers import mps_f64, mps_f64_value, rel_err


def _case(n, K, B, td, seed):
    graph = tneq_b200.QCTNHelper.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))
    names, table, nq = oc.parse_graph(graph)
    torch.manual_seed(seed)
    cores = oc.random_cores(table, td)
    states = oc.unit_states(nq, K, td)
    # the measurement matrices of the GPU cases (I + eps H) plus the oracle's own (rank-one Hermite outer products),
    # so that both well-conditioned and strongly varying values are covered
    h = torch.randn(B, K, K, dtype=td) / (2.0 * K ** 0.5)
    mh = [torch.eye(K, dtype=td) + 0.1 * (h + h.transpose(1, 2).conj()) for _ in range(nq)]
    mg, _ = oc.generate_data(torch.randn(B, nq), K, td, "tensor")
    mxs = [torch.cat([a, b]) for a, b in zip(mh, mg)]
    return graph, names, cores, states, mxs


@pytest.mark.parametrize("dtype", ["float64", "complex128"])
@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_mps_f64_matches_oracle(n, K, dtype):
    td = getattr(torch, dtype)
    graph, names, cores, states, mxs = _case(n, K, 6, td, seed=100 * n + K)
    want = oc.forward(graph, cores, states, [m.clone() for m in mxs])
    leaves = [cores[c].clone().requires_grad_(True) for c in names]
    amp = mps_f64(leaves, states, mxs)
    assert amp.dtype == td and amp.shape == want.shape
    val = mps_f64_value(amp)
    assert rel_err(val, want) < 1e-12, rel_err(val, want)
    loss = -torch.log(torch.clamp(val, min=1e-10)).mean()
    grads = torch.autograd.grad(loss, leaves)
    wl, wg = oc.loss_and_grads(graph, cores, states, [m.clone() for m in mxs])
    assert abs(loss.item() - wl.item()) <= 1e-12 * max(abs(wl.item()), 1.0)
    assert len(grads) == len(wg)
    for g, w in zip(grads, wg):
        assert g.shape == w.shape and g.dtype == w.dtype
        assert rel_err(g, w) < 1e-12, rel_err(g, w)
