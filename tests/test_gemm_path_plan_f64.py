"""float64 / complex128 networks with big cores take the large-bond route in float64, checked WITHOUT a GPU: the
strategy routes them to the GEMM path, and the GEMM-path runner walks a bond-64 plan on meta tensors calling only the
_f64 kernels, on float64 buffers."""
import pytest
import torch

import tneq_b200
from tneq_b200.contractor import gemm_path
from tneq_b200.contractor.b200_strategy import _Bound
from tneq_b200.contractor.plan import ContractionPlan, signature_of


def _plan(n, chi, B, dtype):
    graph = tneq_b200.QCTNHelper.generate_example_graph(n=n, graph_type="mps", dim_char=str(chi))
    q = tneq_b200.QCTN(graph)
    td = getattr(torch, dtype)
    states = [torch.empty(chi, dtype=td, device="meta") for _ in range(n)]
    mxs = [torch.empty(B, chi, chi, dtype=td, device="meta") for _ in range(n)]
    sd, mi = signature_of(q.nqubits, states, mxs)
    return ContractionPlan(q.adjacency_table, q.nqubits, {c: q.core_shape(c) for c in q.cores}, sd, mi, dtype)


@pytest.mark.parametrize("dtype,chi,gemm", [("float64", 9, True), ("complex128", 7, True),
                                            ("float64", 8, False), ("complex128", 6, False)])
def test_big_float64_cores_take_the_gemm_path(dtype, chi, gemm, monkeypatch):
    """Cores above 4096 real elements (float64 bond 9: 6561; complex128 bond 7: 4802) go to the GEMM path in float64;
    one bond smaller stays on the shared-memory VM."""
    monkeypatch.delenv("TNQ_FORCE_GEMM_PATH", raising=False)
    b = _Bound(_plan(4, chi, 3, dtype), torch.device("cuda"))
    assert b.use_gemm_path == gemm and b.real_dtype == torch.float64
    assert not b.chain_rank and not b.ladder


@pytest.mark.parametrize("dtype", ["float64", "complex128"])
def test_forced_gemm_path_in_float64(dtype, monkeypatch):
    monkeypatch.setenv("TNQ_FORCE_GEMM_PATH", "1")
    b = _Bound(_plan(4, 3, 5, dtype), torch.device("cuda"))
    assert b.use_gemm_path and b.real_dtype == torch.float64


class _RecordingLib:
    """Stands in for the CUDA library: records the name of every entry point called, returns success."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("tnq_"):
            raise AttributeError(name)

        def entry(*args):
            self.calls.append(name)
            return 0
        return entry


class _MetaRunner(gemm_path.GemmPathRunner):
    """The real runner (its own _permute / _gemm / fold / expand calls) on meta tensors."""

    def __init__(self, graph, dtype):
        self.g, self.device, self.flops = graph, torch.device("meta"), 0.0
        self._set_dtype(dtype)
        self.lib = _RecordingLib()

    def _stream(self):
        return None


def _walk(dtype, n=5, chi=64, B=256):
    plan = _plan(n, chi, B, dtype)
    real = torch.float64 if plan.real_dtype == "f64" else torch.float32
    g = plan.graph("bwd")
    r = _MetaRunner(g, real)
    inputs = {}
    for key, ids in g.inputs.items():
        node = g.nodes[ids[0]]
        size = g.size(node.idx)
        inputs[key] = torch.empty((B, size) if node.batched else (size,), dtype=real, device="meta")
    seed = torch.empty(B, g.size(g.nodes[g.result].idx), dtype=real, device="meta")
    val, _ = r.run(inputs, B, 1, with_adjoint=True, seed=seed)
    return r, val


@pytest.mark.parametrize("mn_in_place", [True, False])
@pytest.mark.parametrize("dtype", ["float64", "complex128"])
def test_bond64_float64_plan_calls_only_f64_kernels(dtype, mn_in_place, monkeypatch):
    """Every launch of a bond-64 float64 / complex128 plan is an _f64 entry point (no tf32x3 GEMM, view or in-place
    variant, whatever gemm_path.MN_IN_PLACE says), and every buffer the runner produces is float64."""
    monkeypatch.setattr(gemm_path, "MN_IN_PLACE", mn_in_place)
    r, val = _walk(dtype)
    calls = set(r.lib.calls)
    assert calls and all(c.endswith("_f64") for c in calls), sorted(calls)
    assert not [c for c in calls if "tf32x3" in c]
    want = {"tnq_gemm_f64", "tnq_permute_f64"}
    if dtype == "complex128":
        want |= {"tnq_fold_vec_f64", "tnq_outer_acc_f64", "tnq_cplx_expand_f64"}
    assert want <= calls, sorted(want - calls)
    assert {v.dtype for v in val.values()} == {torch.float64}
    assert abs(r.flops - 0.829e12) < 0.02e12 if dtype == "complex128" else r.flops > 0


def test_bond64_complex64_plan_is_unchanged():
    """The float32 route of the same plan keeps its kernels: tf32x3 GEMMs incl. the in-place variants, _f32 layout
    kernels, no _f64 entry point."""
    r, val = _walk("complex64")
    calls = set(r.lib.calls)
    assert not [c for c in calls if c.endswith("_f64")]
    assert {"tnq_gemm_tf32x3", "tnq_gemm_tf32x3_view", "tnq_gemm_tf32x3_bk", "tnq_fold_vec_f32"} <= calls, sorted(calls)
    assert {v.dtype for v in val.values()} == {torch.float32}
