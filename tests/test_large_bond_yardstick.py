"""The float64 yardstick of the large-bond tests (helpers.mps_f64) against the oracle, on the CPU.

At bond 32-128 the oracle's greedy einsum builds K^6 intermediates, so tests/test_gpu_large_bond.py and
tests/test_gpu_gemm_path.py compare the CUDA route with helpers.mps_f64 instead: the same single-layer MPS sweep
restated pairwise (3 K^4 per qubit and sample).  Here that restatement is pinned to the oracle where both fit:
values, and the autograd gradients of the engine's loss -mean(log clamp(value, 1e-10)) against
oc.loss_and_grads, in float64 and complex128."""
import math

import pytest
import torch

import tneq_b200
from oracle import qctn_oracle as oc
from helpers import ladder_f64, ladder_layers, mps_f64, mps_f64_value, rel_err


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


def _merged_case(n, K, B, seed):
    q = tneq_b200.QCTN(tneq_b200.QCTNHelper.generate_example_graph(n=n, graph_type="mps", dim_char=str(K)))
    graph = tneq_b200.QCTN.merge(q, q).graph
    names, table, nq = oc.parse_graph(graph)
    torch.manual_seed(seed)
    cores = oc.random_cores(table, torch.float64)
    states = oc.unit_states(nq, K, torch.float64)
    h = torch.randn(B, K, K, dtype=torch.float64) / (2.0 * K ** 0.5)
    mh = [torch.eye(K, dtype=torch.float64) + 0.1 * (h + h.transpose(1, 2)) for _ in range(nq)]
    mg, _ = oc.generate_data(torch.randn(B, nq), K, torch.float64, "tensor")
    mxs = [torch.cat([a, b]) for a, b in zip(mh, mg)]
    return graph, cores, states, mxs


@pytest.mark.parametrize("tnt", [False, True])
@pytest.mark.parametrize("K", [2, 3])
@pytest.mark.parametrize("n", [3, 4, 5, 6])
def test_ladder_f64_matches_oracle(n, K, tnt):
    """helpers.ladder_f64 (the yardstick of tests/test_gpu_register_kernels.py for the two-layer kernels) against the
    oracle in float64: values, the engine's loss -mean(log clamp(value, 1e-10) + log_scale) and its autograd
    gradients, with the layer assignment the ladder route uses (plan.mps_ladder())."""
    graph, cores, states, mxs = _merged_case(n, K, 5, seed=10 * n + K)
    names, table, nq = oc.parse_graph(graph)
    layer1, layer2 = ladder_layers(graph, K)
    assert len(layer1) == len(layer2) == n - 1 and set(layer1 + layer2) == set(names)
    if tnt:
        wrapped = [oc.TNT(m.clone()) for m in mxs]
        for w in wrapped:
            w.auto_scale()
        mx_in, raw = wrapped, [w.tensor for w in wrapped]
        log_scale = sum(w.log_scale for w in wrapped)
    else:
        mx_in, raw, log_scale = [m.clone() for m in mxs], mxs, 0.0
    want = oc.forward(graph, cores, states, [oc.TNT(m.tensor.clone(), m.scale, m.log_scale) if tnt else m.clone()
                                             for m in mx_in])
    leaves = {k: cores[k].clone().requires_grad_(True) for k in names}
    val = ladder_f64([leaves[k] for k in layer1], [leaves[k] for k in layer2], states, raw)
    assert val.dtype == torch.float64 and val.shape == want.shape
    scale = math.exp(log_scale)
    assert rel_err(val * scale, want) < 1e-12, rel_err(val * scale, want)
    loss = -(torch.log(torch.clamp(val, min=1e-10)) + log_scale).mean()
    grads = torch.autograd.grad(loss, [leaves[k] for k in names])
    wl, wg = oc.loss_and_grads(graph, cores, states, [oc.TNT(m.tensor.clone(), m.scale, m.log_scale) if tnt
                                                       else m.clone() for m in mx_in])
    assert abs(loss.item() - wl.item()) <= 1e-12 * max(abs(wl.item()), 1.0)
    for g, w in zip(grads, wg):
        assert g.shape == w.shape
        assert rel_err(g, w) < 1e-12, rel_err(g, w)
