"""float64 parity of the register-resident kernels -- the single-layer MPS chain (csrc/tnq_chain.cu) and the two-layer
ladder (csrc/tnq_ladder.cu, and with TNQ_LADDER_V2=1 csrc/tnq_ladder2.cu) -- across the launch variants the host picks.

Which kernel runs depends on the batch stride of every measurement matrix (contiguous, a view of one (B,n,K,K) tensor
as EngineSiamese.generate_data returns them, stride 0 for a broadcast matrix), on the mode (values, fused loss, seeded
reverse sweep) and on K; every kernel walks the batch in passes whose number depends on B and the SM count.  Each case
here states the kernels it exists to reach (recorded with torch.profiler, helpers.KernelRecorder) and, for the
multi-pass cases, B is derived from the launch geometry so that the last pass is ragged.

Yardsticks, in float64 on the GPU on the same float32 inputs: helpers.mps_f64 (chain) and helpers.ladder_f64 (ladder),
both pinned to the oracle by tests/test_large_bond_yardstick.py.  Loss and gradients come from torch.autograd with the
engine's loss -mean(log(clamp(v, 1e-10)) + log_scale); mode 2 is torch.autograd.grad(values, cores, seed).
Bounds (DESIGN 5): values 1e-5 elementwise; loss and gradients max(1e-5, NOISE_FACTOR x the float32 oracle's own
error) on well-conditioned data, 1e-5 on near-identity data (multi-pass batches, 40 and 64 qubits), gradients relative
to each tensor's largest entry; signed seeds relative to the largest entry of sum_b |seed_b| |dv_b/dG|.
"""
import ctypes
import os
import time

import pytest
import torch

import tneq_b200
from oracle import qctn_oracle as oc
from helpers import (NOISE_FACTOR, KernelRecorder, elem_rel_err, ladder_f64, ladder_layers, mps_f64, rel_err,
                     well_conditioned_case)

pytestmark = pytest.mark.gpu
H = tneq_b200.QCTNHelper
DEV = "cuda:0"
CHAIN_THREADS = 128                   # csrc/tnq_chain.cu
CLAMP = 1e-10


@pytest.fixture(scope="module", autouse=True)
def _budget():
    """Wall time and peak device memory of this file (printed; run with -s to see them)."""
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    print(f"\n[register kernels] {time.time() - t0:.1f} s, peak device memory "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


@pytest.fixture(params=["warp-level", "second-generation"])
def generation(request):
    """Edge rank 3 of the ladder has two kernels: csrc/tnq_ladder.cu and, with TNQ_LADDER_V2=1, csrc/tnq_ladder2.cu."""
    old = os.environ.get("TNQ_LADDER_V2")
    if request.param == "second-generation":
        os.environ["TNQ_LADDER_V2"] = "1"
    else:
        os.environ.pop("TNQ_LADDER_V2", None)
    try:
        yield request.param
    finally:
        if old is None:
            os.environ.pop("TNQ_LADDER_V2", None)
        else:
            os.environ["TNQ_LADDER_V2"] = old


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- launch geometry (mirrors of the host rules) ---------------------------------------------------------------------
def chain_per_pass(kind, sms):
    """Samples one launch covers before its warps start a second pass over the batch (csrc/tnq_chain.cu)."""
    return {"fwd2": 2 * CHAIN_THREADS * 4 * sms,          # two samples per thread, grid <= 4 SMs' worth of CTAs
            "train2": 2 * CHAIN_THREADS * 4 * sms,
            "chain0": CHAIN_THREADS * 8 * sms,            # one sample per thread, grid <= 8 (mode 0) / 4 CTAs per SM
            "chain12": CHAIN_THREADS * 4 * sms,
            "sample": CHAIN_THREADS * 2 * sms,
            "chainx": 2 * CHAIN_THREADS * 4 * sms}[kind]


def ladder_dims(K, n):
    """Dims<K> of csrc/tnq_ladder_core.cuh: (samples per warp, constant-pool floats, per-warp floats fwd / train,
    gradient-slice floats, checkpoint floats)."""
    K2, K3, K4 = K * K, K ** 3, K ** 4
    r4 = lambda v: (v + 3) // 4 * 4
    spw = 32 // K2
    sst = 765 if K == 3 else 67
    usz = max(K3 * 4, K2 * r4(K2))
    off_bs = r4(K4) + K2 * r4(K2)
    off_bt = r4(off_bs + K2 * 4)
    cstep = r4(off_bt + K * r4(K2))
    e_sz, t2_sz = r4(spw * sst), r4(spw * K4)
    w_fwd = e_sz + spw * usz + t2_sz + r4(spw * K2) + 64
    w_train = w_fwd + e_sz + t2_sz
    cst = r4((n - 1) * cstep + K2)
    grad = r4((n - 1) * K4 + (n - 1) * K3 + K2)
    return spw, cst, w_fwd, w_train, grad, (n - 2) * (e_sz + t2_sz)


def ladder_geometry(K, n, B, mode):
    """geometry() of csrc/tnq_ladder.cu -> (samples per warp, warps per CTA, grid, passes)."""
    sms = _sms()
    spw, cst, w_fwd, w_train, _, _ = ladder_dims(K, n)
    ngroups = -(-B // spw)
    per_warp = 4 * (w_fwd if mode == 0 else w_train)
    fit = (torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 4 * cst) // per_warp
    wmax = min(16 if mode == 0 else 8, max(1, fit))
    wpc = min(max(1, -(-ngroups // sms)), wmax)
    grid = min(sms, -(-ngroups // wpc))
    return spw, wpc, grid, -(-ngroups // (grid * wpc))


def ladder_workspace(K, n, B):
    """workspace_bytes() of csrc/tnq_ladder.cu in training: checks the geometry mirror against the library."""
    _, wpc, grid, _ = ladder_geometry(K, n, B, 1)
    _, _, _, _, grad, ckpt = ladder_dims(K, n)
    return 4 * grid * wpc * (grad + 32 + ckpt) + 256


def ladder2_geometry(n, B, mode):
    """tnq_mps_ladder2_geometry -> (samples per tile, tiles, grid)."""
    out = (ctypes.c_int64 * 6)()
    assert tneq_b200._lib.load().tnq_mps_ladder2_geometry(n, B, mode, out) == 0
    return int(out[1]), int(out[2]), int(out[3])


# ---- networks and data ----------------------------------------------------------------------------------------------
def mps_graph(n, K):
    return H.generate_example_graph(n=n, graph_type="mps", dim_char=str(K))


def merged_graph(n, K):
    q = tneq_b200.QCTN(mps_graph(n, K))
    return tneq_b200.QCTN.merge(q, q).graph


def _engine(graph, K, cores):
    be = tneq_b200.BackendFactory.create_backend("b200", device=DEV, dtype="float32")
    eng = tneq_b200.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
    q = tneq_b200.QCTN(graph, backend=be)
    for k, v in cores.items():
        q.cores_weights[k] = v.to(DEV).contiguous().requires_grad_(True)
    return eng, q


def near_identity(B, n, K, seed):
    """eye + 0.05 noise: values stay O(1) along any chain length, so float32 keeps its digits without a selection."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.eye(K, device=DEV) + 0.05 * torch.randn(B, K, K, device=DEV, generator=g) for _ in range(n)]


def layout(ms, kind):
    """The measurement list as the kernels will see it.  ms: n device tensors (B,K,K).
    contig: as they are; strided: views of one (B,n,K,K) tensor (batch stride n K^2, what generate_data returns);
    bcast: stride 0 on the first qubit (the identity, expand) and, when n > 2, on the last ((1,K,K): sample 0's
    matrix), so that qubit 1 still varies per sample;
    mixed: per qubit strided / contiguous / identity broadcast in turn."""
    n, B, K = len(ms), ms[0].shape[0], ms[0].shape[-1]
    eye = torch.eye(K, device=DEV).expand(B, K, K)
    if kind == "contig":
        return [m.contiguous() for m in ms]
    stack = torch.stack(ms, 1)
    if kind == "strided":
        return [stack[:, q] for q in range(n)]
    if kind == "bcast":
        return [eye if q == 0 else ms[q][:1].clone() if q == n - 1 > 1 else ms[q].contiguous() for q in range(n)]
    assert kind == "mixed"
    return [stack[:, q] if q % 3 == 0 else ms[q].contiguous() if q % 3 == 1 else eye for q in range(n)]


def per_sample_qubit(kind, n):
    """A qubit whose matrix differs per sample in this layout (where the clamp's negation goes)."""
    return 1 if kind == "bcast" else 0


def negate_some(ms, q, B):
    """Samples 3, 10, 17, ... (every 7th) get qubit q's matrix negated: their value changes sign, so the loss clamps
    them (gradient zero, -log(1e-10) added to the loss); nothing lands near 1e-10 itself."""
    idx = torch.arange(3, B, 7, device=DEV)
    if len(idx):
        ms[q] = ms[q].clone()
        ms[q][idx] = -ms[q][idx]
    return idx


def _expand64(mx, B):
    return [m.double().expand(B, *m.shape[1:]) for m in mx]


def _f64_loss(val, log_scale=0.0):
    return -(torch.log(torch.clamp(val, min=CLAMP)) + log_scale).mean()


def _seeds(B, kind, tail):
    g = torch.Generator(device=DEV).manual_seed(B + 17)
    s = 0.5 + torch.rand(B, device=DEV, generator=g)
    if kind == "signed":
        s = s * torch.where(torch.rand(B, device=DEV, generator=g) < 0.5, -1.0, 1.0)
        s[2::5] = 0.0
    if tail:
        s[B - tail:] = 0.0
    return s


class _Ref:
    """float64 yardstick of one network on the float32 inputs: values, loss, gradients, seeded gradients.  Loss and
    gradients are sums over samples, so they are accumulated over slices of `chunk` samples: the autograd tape of the
    two-layer sweep holds ~K^7 doubles per sample and qubit."""

    def __init__(self, fn, names, cores, chunk):
        self.fn, self.names, self.chunk = fn, names, chunk
        self.leaves = {k: cores[k].detach().to(DEV, torch.float64).requires_grad_(True) for k in names}

    def values(self, mx):
        with torch.no_grad():
            return self.fn(self.leaves, mx)

    def _sum_grads(self, mx, part_of):
        B = mx[0].shape[0]
        total, grads = 0.0, None
        for b0 in range(0, B, self.chunk):
            val = self.fn(self.leaves, [m[b0:b0 + self.chunk] for m in mx])
            part = part_of(val, b0)
            g = torch.autograd.grad(part, [self.leaves[k] for k in self.names])
            total = total + part.detach()
            grads = list(g) if grads is None else [a + b for a, b in zip(grads, g)]
        return total, grads

    def loss_grads(self, mx, log_scale=0.0):
        B = mx[0].shape[0]
        return self._sum_grads(mx, lambda val, b0: _f64_loss(val, log_scale) * (val.shape[0] / B))

    def seeded(self, mx, seed):
        s64 = seed.double()
        return self._sum_grads(mx, lambda val, b0: (val * s64[b0:b0 + val.shape[0]]).sum())[1]

    def abs_seeded_max(self, mx, seed):
        """max entry per core of sum_b |seed_b| |dv_b/dG| (per-sample Jacobian; small batches only)."""
        val = self.fn(self.leaves, mx)
        B = val.shape[0]
        jac = torch.autograd.grad(val, [self.leaves[k] for k in self.names],
                                  grad_outputs=torch.eye(B, dtype=torch.float64, device=DEV), is_grads_batched=True)
        w = seed.double().abs().view(B, *([1] * 4))
        return [(w * j.abs()).sum(0).max().item() for j in jac]


def chain_ref(graph, names, cores, states):
    st64 = [s.to(DEV, torch.float64) for s in states]
    return _Ref(lambda lv, mx: mps_f64([lv[k] for k in names], st64, mx), names, cores, chunk=1 << 16)


def ladder_ref(graph, names, cores, states, K):
    l1, l2 = ladder_layers(graph, K)
    st64 = [s.to(DEV, torch.float64) for s in states]
    return _Ref(lambda lv, mx: ladder_f64([lv[k] for k in l1], [lv[k] for k in l2], st64, mx), names, cores,
                chunk=1024)


def _oracle_err(graph, cores, states, mx_cpu, truth_loss, truth_grads):
    """The float32 oracle's own error against the float64 yardstick (loss relative; per tensor, relative to its
    largest entry)."""
    wl, wg = oc.loss_and_grads(graph, cores, states, mx_cpu)
    lerr = abs(wl.item() - truth_loss.item())
    return lerr, [rel_err(w.double(), t.cpu()) for w, t in zip(wg, truth_grads)]


# ---- the shared driver -----------------------------------------------------------------------------------------------
def run_case(family, graph, K, cores, states, ms, kind, expected, oracle=True, tnt_scales=None, neg=True, tail=0,
             signed=True, modes=(0, 1, 2)):
    """All modes of one (network, measurements, layout) case through the engine API, each against float64, each with
    the kernels it must launch.  ms: n device float32 tensors (B,K,K) before the layout is applied.
    expected: mode -> list of kernel names.  tnt_scales: per-qubit (scale, log_scale) to pass TNTensors in mode 1."""
    names = list(cores)
    n, B = len(ms), ms[0].shape[0]
    ms = list(ms)
    if neg and B > 3:
        negate_some(ms, per_sample_qubit(kind, n), B)
    mx = layout(ms, kind)
    mx64 = _expand64(mx, B)
    ref = chain_ref(graph, names, cores, states) if family == "chain" else ladder_ref(graph, names, cores, states, K)
    eng, q = _engine(graph, K, cores)
    st = [s.to(DEV) for s in states]
    errs = {}
    # mode 0: values
    if 0 in modes:
        with torch.no_grad(), KernelRecorder() as rec:
            got = eng.contract_with_compiled_strategy(q, st, mx)
        rec.check(expected[0])
        want = ref.values(mx64)
        errs["values"] = elem_rel_err(got.double(), want)
        vbound = 1e-5
        if oracle:
            w32 = oc.forward(graph, cores, [s.cpu() for s in states], [m.expand(B, K, K).cpu().clone() for m in mx])
            vbound = max(vbound, NOISE_FACTOR * elem_rel_err(w32.double(), want))
        errs["values_bound"] = vbound
        assert got.shape == (B,) and errs["values"] < vbound, (errs, vbound)
    # mode 1: fused loss + gradients (TNTensor measurements: the loss carries their log_scale)
    if 1 in modes:
        log_scale = 0.0
        mx_in = mx
        if tnt_scales is not None:
            mx_in = [tneq_b200.TNTensor(m, s, ls) for m, (s, ls) in zip(mx, tnt_scales)]
            log_scale = sum(ls for _, ls in tnt_scales)
        with KernelRecorder() as rec:
            loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, st, mx_in)
        rec.check(expected[1])
        tl, tg = ref.loss_grads(mx64, log_scale)
        lbound, gbounds = 1e-5 * abs(tl.item()), [1e-5] * len(tg)
        if oracle:
            mx_cpu = [oc.TNT(m.expand(B, K, K).cpu().clone(), s, ls) for m, (s, ls) in zip(mx, tnt_scales)] \
                if tnt_scales is not None else [m.expand(B, K, K).cpu().clone() for m in mx]
            lerr, gerr = _oracle_err(graph, cores, [s.cpu() for s in states], mx_cpu, tl, tg)
            lbound = max(lbound, NOISE_FACTOR * lerr)
            gbounds = [max(b, NOISE_FACTOR * e) for b, e in zip(gbounds, gerr)]
        errs["loss"] = abs(loss.item() - tl.item()) / abs(tl.item())
        errs["loss_bound"] = lbound / abs(tl.item())
        assert abs(loss.item() - tl.item()) <= lbound, (loss.item(), tl.item(), lbound)
        errs["grads"] = 0.0
        for g, t, b in zip(grads, tg, gbounds):
            e = rel_err(g.double(), t)
            errs["grads"] = max(errs["grads"], e)
            errs["grads_vs_bound"] = max(errs.get("grads_vs_bound", 0.0), e / b)
            assert e < b, (e, b)
    # mode 2: torch.autograd.grad(values, cores, seed) -- forward kernel, then the seeded reverse sweep
    if 2 in modes:
        leaves = [q.cores_weights[k] for k in names]
        kinds = ("positive", "signed") if signed else ("positive",)
        errs["seeded"] = 0.0
        for sk in kinds:
            seed = _seeds(B, sk, tail)
            with KernelRecorder() as rec:
                vals = eng.contract_with_compiled_strategy(q, st, mx)
                grads = torch.autograd.grad(vals, leaves, grad_outputs=seed)
            rec.check(expected[2])
            tg = ref.seeded(mx64, seed)
            scale = ref.abs_seeded_max(mx64, seed) if sk == "signed" else [t.abs().max().item() for t in tg]
            for g, t, s in zip(grads, tg, scale):
                if s == 0.0:                                    # every seed zero: the gradient is exactly zero
                    assert (g == 0).all()
                    continue
                e = (g.double() - t).abs().max().item() / s
                errs["seeded"] = max(errs["seeded"], e)
                assert e < 1e-5, (sk, e)
    print(f"[{family} K={K} n={n} B={B} {kind}] " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    return errs


def chain_expected(K, kind, B):
    """Kernels of launch_chain (csrc/tnq_chain.cu) per mode for this layout."""
    packed = kind == "contig"
    fwd = f"tnq_chain_fwd2_kernel<{K}>" if packed else f"tnq_chain_kernel<{K}, 0>"
    fin = f"tnq_chain_finalize_kernel<{K}>"
    tr = (lambda m: f"tnq_chain_train2_kernel<{K}, {m}>") if (packed and K <= 3) else \
        (lambda m: f"tnq_chain_kernel<{K}, {m}>")
    return {0: [fwd], 1: [tr(1), fin], 2: [fwd, tr(2), fin]}


def ladder_expected(K, generation):
    if generation == "second-generation":      # template <R, NW, MODE>: R and NW follow from the batch
        l2, fin = ["tnq_l2_prep_kernel", "tnq_ladder2_kernel"], "tnq_l2_finalize_kernel"
        return {0: l2, 1: l2 + [fin], 2: l2 + [fin]}
    fin = f"tnq_ladder_finalize_kernel<{K}>"
    return {0: [f"tnq_ladder_kernel<{K}, 0>"], 1: [f"tnq_ladder_kernel<{K}, 1>", fin],
            2: [f"tnq_ladder_kernel<{K}, 0>", f"tnq_ladder_kernel<{K}, 2>", fin]}


# ---- chain: small batches, well-conditioned data, every layout ------------------------------------------------------
CHAIN_SMALL = [(K, kind, n, B) for K in (2, 3, 4) for kind, n, B in
               (("contig", 17, 127), ("strided", 3, 33), ("strided", 17, 65), ("strided", 2, 1), ("bcast", 3, 31),
                ("bcast", 2, 63), ("mixed", 17, 63), ("mixed", 3, 2))]


@pytest.mark.parametrize("K,kind,n,B", CHAIN_SMALL)
def test_chain_small_batches(K, kind, n, B, built_lib):
    graph = mps_graph(n, K)
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, B, "float32", seed=7 * n + K + B)
    ms = [m.tensor.to(DEV) for m in mxs]
    tnt = [(m.scale, m.log_scale) for m in mxs] if kind == "contig" else None
    run_case("chain", graph, K, cores, states, ms, kind, chain_expected(K, kind, B), tnt_scales=tnt)


# ---- chain: 2-3 passes plus a ragged tail for every kernel, near-identity data -------------------------------------
def _chain_multipass_cases():
    out = []
    for K in (2, 3, 4):
        # contiguous: fwd2 (mode 0), train2 (K <= 3) or the one-sample kernel's packed branch (K = 4)
        out.append((K, "contig", "fwd2", (0,)))
        out.append((K, "contig", "train2" if K <= 3 else "chain12", (1, 2)))
        # strided: the one-sample kernel's load_m branch in every mode
        out.append((K, "strided", "chain0", (0,)))
        out.append((K, "strided", "chain12", (1, 2)))
    return out


@pytest.mark.parametrize("K,kind,per,modes", _chain_multipass_cases())
def test_chain_multipass(K, kind, per, modes, built_lib):
    n = 3
    P = chain_per_pass(per, _sms())
    tile = 64 if per in ("fwd2", "train2") else 32
    B = 2 * P + 77                                      # two full passes and a ragged third
    assert B % tile and 2 < B / P <= 3
    graph = mps_graph(n, K)
    torch.manual_seed(40 + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    ms = near_identity(B, n, K, seed=K)
    run_case("chain", graph, K, cores, states, ms, kind, chain_expected(K, kind, B), oracle=False, modes=modes,
             tail=B % tile, signed=False)


@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("kind", ["contig", "strided"])
def test_chain_64_qubits(K, kind, built_lib):
    """The longest chain the kernels take (TNQ_CHAIN_MAX_QUBITS): the full 64-entry tape and, for K = 4, more than
    48 KB of shared memory."""
    n, B = 64, 300
    graph = mps_graph(n, K)
    torch.manual_seed(64 + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    ms = near_identity(B, n, K, seed=100 + K)
    run_case("chain", graph, K, cores, states, ms, kind, chain_expected(K, kind, B), oracle=False)


@pytest.mark.parametrize("K,kind", [(2, "contig"), (3, "strided"), (4, "contig")])
def test_chain_training_is_deterministic(K, kind, built_lib):
    """Mode 1 twice on the same inputs: bit-identical loss and gradients (fixed-order reductions), at 2+ passes."""
    n, B = 4, 2 * chain_per_pass("chain12", _sms()) + 45
    graph = mps_graph(n, K)
    torch.manual_seed(3)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    eng, q = _engine(graph, K, cores)
    st = [s.to(DEV) for s in oc.unit_states(nq, K)]
    mx = layout(near_identity(B, n, K, seed=9), kind)
    l1, g1 = eng.contract_with_compiled_strategy_for_gradient(q, st, mx)
    l2, g2 = eng.contract_with_compiled_strategy_for_gradient(q, st, mx)
    assert l1.item() == l2.item() and all(torch.equal(a, b) for a, b in zip(g1, g2))


# ---- ladder ---------------------------------------------------------------------------------------------------------
LADDER_SMALL = [(K, kind, n, B) for K in (2, 3) for kind, n, B in
                (("contig", 4, 65), ("strided", 3, 127), ("strided", 4, 1), ("bcast", 3, 31), ("mixed", 4, 31),
                 ("mixed", 3, 2), ("contig", 3, 33), ("bcast", 4, 2))]


@pytest.mark.parametrize("K,kind,n,B", LADDER_SMALL)
def test_ladder_small_batches(K, kind, n, B, built_lib, generation):
    if generation == "second-generation" and K != 3:
        pytest.skip("the second-generation kernel covers edge rank 3")
    graph = merged_graph(n, K)
    names, table, nq, cores, states, mxs = well_conditioned_case(graph, K, B, "float32", seed=11 * n + K + B)
    ms = [m.tensor.to(DEV) for m in mxs]
    tnt = [(m.scale, m.log_scale) for m in mxs] if kind == "contig" else None
    run_case("ladder", graph, K, cores, states, ms, kind, ladder_expected(K, generation), tnt_scales=tnt)


def _ladder_multipass_B(K, n, mode, generation):
    """The smallest B of the form (2 passes) + tail that gives 2-3 passes with a ragged last group / tile."""
    if generation == "second-generation":
        for B in range(1000, 400000, 997):
            spt, ntiles, grid = ladder2_geometry(n, B, mode)
            if B % spt and 2 < ntiles / grid <= 3:
                return B
        raise AssertionError("no multi-pass batch found")
    spw, wpc, grid, _ = ladder_geometry(K, n, 10 ** 7, mode)
    B = 2 * spw * wpc * grid + spw // 2 + 1
    assert ladder_geometry(K, n, B, mode)[3] == 3 and B % spw
    return B


@pytest.mark.parametrize("K,kind", [(2, "contig"), (2, "strided"), (3, "contig"), (3, "mixed")])
@pytest.mark.parametrize("train", [False, True])
def test_ladder_multipass(K, kind, train, built_lib, generation):
    """2 full passes of the persistent grid and a ragged third: LaneState (prefetched matrix, loss) and the per-warp
    gradient slice carried across groups, against float64 -- a bias shared by every pass is visible here."""
    if generation == "second-generation" and K != 3:
        pytest.skip("the second-generation kernel covers edge rank 3")
    n = 4
    B = _ladder_multipass_B(K, n, 1 if train else 0, generation)
    if train and generation == "warp-level":
        lib = tneq_b200._lib.load()
        assert lib.tnq_mps_ladder_workspace_bytes(K, n, B, 1) == ladder_workspace(K, n, B)
    graph = merged_graph(n, K)
    torch.manual_seed(50 + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    ms = near_identity(B, n, K, seed=20 + K)
    spw = 32 // (K * K)
    run_case("ladder", graph, K, cores, states, ms, kind, ladder_expected(K, generation), oracle=False,
             modes=(1, 2) if train else (0,), tail=B % spw, signed=False)


@pytest.mark.parametrize("K,n,B", [(2, 40, 200), (3, 40, 100), (2, 64, None), (3, 64, 64)])
def test_ladder_long_chains(K, n, B, built_lib, generation):
    """40 and 64 qubits (the constant pool leaves room for fewer warps) against float64; at K = 2, n = 64 with 2 full
    training passes and a ragged third (B = None)."""
    if generation == "second-generation" and K != 3:
        pytest.skip("the second-generation kernel covers edge rank 3")
    if B is None:
        B = _ladder_multipass_B(K, n, 1, generation)
    graph = merged_graph(n, K)
    torch.manual_seed(n + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    ms = near_identity(B, n, K, seed=n)
    run_case("ladder", graph, K, cores, states, ms, "strided", ladder_expected(K, generation), oracle=False,
             signed=B <= 128)


@pytest.mark.parametrize("train", [False, True])
def test_ladder_64_qubits_reduced_warps(train, built_lib, generation):
    """K = 3 at 64 qubits: the constant pool and the per-warp buffers no longer fit the full warp count (geometry() in
    csrc/tnq_ladder.cu lowers it), so the persistent grid is smaller; 2 full passes of that grid and a ragged third,
    against float64."""
    if generation == "second-generation":
        pytest.skip("the reduced warp count is the warp-level kernel's launch rule")
    K, n = 3, 64
    mode = 1 if train else 0
    full = 8 if train else 16
    spw, wpc, grid, _ = ladder_geometry(K, n, 10 ** 7, mode)
    assert wpc < full, (wpc, full)
    B = _ladder_multipass_B(K, n, mode, generation)
    assert ladder_geometry(K, n, B, mode)[1:] == (wpc, grid, 3)
    if train:
        assert tneq_b200._lib.load().tnq_mps_ladder_workspace_bytes(K, n, B, 1) == ladder_workspace(K, n, B)
    graph = merged_graph(n, K)
    torch.manual_seed(n + K + 1)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    ms = near_identity(B, n, K, seed=n + 1)
    print(f"[ladder K={K} n={n} mode {mode}] {wpc} of {full} warps per CTA, grid {grid}, B={B}")
    run_case("ladder", graph, K, cores, states, ms, "strided", ladder_expected(K, generation), oracle=False,
             modes=(1, 2) if train else (0,), tail=B % spw, signed=False)


# ---- contract_from_x, sample(method="prefix") -----------------------------------------------------------------------
@pytest.mark.parametrize("K", [2, 3, 4])
def test_contract_from_x_transposed_two_passes(K, built_lib):
    """x as a transposed view (xs_b = 1, xs_q = B) at two passes of tnq_chain_fwd2x_kernel: values and per-qubit
    scales against generate_data + mps_f64 in float64."""
    n = 5
    B = chain_per_pass("chainx", _sms()) + 1001
    graph = mps_graph(n, K)
    torch.manual_seed(70 + K)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    states = oc.unit_states(nq, K)
    eng, q = _engine(graph, K, cores)
    st = [s.to(DEV) for s in states]
    x = torch.randn(n, B, device=DEV).t()
    assert x.stride() == (1, B)
    probe = [torch.empty((B, K, K), device="meta")] * n
    fn = eng._compiled(q, st, probe, True, "symmetric")
    w = [float(v) for v in eng._mx_weights_np[:K].astype("float32")]
    with torch.no_grad(), KernelRecorder() as rec:
        vals, scale = fn.forward_from_x({k: q.cores_weights[k] for k in names}, st, x, w)
        got = eng.contract_from_x(q, st, x, K=K)
    rec.check([f"tnq_hermite_scale_kernel<{K}>", f"tnq_chain_fwd2x_kernel<{K}>"])
    mats, _ = oc.generate_data(x.double().cpu(), K, torch.float64, "TNTensor")
    want_scale = torch.tensor([m.scale for m in mats], dtype=torch.float64)
    assert rel_err(scale.double().cpu(), want_scale) < 1e-5
    c64 = [cores[k].to(DEV, torch.float64) for k in names]
    truth = mps_f64(c64, [s.double() for s in st], [m.tensor.to(DEV) for m in mats])    # scaled, as the kernel
    # the matrices are formed from x in float32 (Hermite recurrence, exp, weights): the reference's own float32
    # generate_data + forward carries the same input rounding, so the bound is DESIGN 5's
    m32, _ = oc.generate_data(x.cpu(), K, torch.float32, "TNTensor")
    want = oc.forward(graph, cores, states, m32).to(DEV).double()
    truth_abs = truth * want_scale.prod().item()
    ok = truth.abs() >= 0.05 * truth.abs().median()
    e_vals = elem_rel_err(vals.double()[ok], truth[ok])
    e_ref = elem_rel_err(want[ok], truth_abs[ok])
    print(f"[from_x K={K} B={B}] values {e_vals:.2e} (float32 oracle {e_ref:.2e})")
    assert e_vals < max(1e-5, NOISE_FACTOR * e_ref)
    assert rel_err(vals.double(), truth) < max(1e-5, NOISE_FACTOR * rel_err(want, truth_abs))
    assert rel_err(got.double(), truth_abs) < max(1e-5, NOISE_FACTOR * rel_err(want, truth_abs))


def test_sample_prefix_grid_in_global_memory(built_lib):
    """sample(method='prefix') with a grid too large for shared memory (the kernel reads it from global memory) and
    more than two passes of samples, against method='linear' from the same random numbers."""
    n, K, G = 3, 4, 2600
    assert 4 * (2 * (n - 1) * K ** 3 + K * K + G * K * K) > 160 * 1024         # host rule: in_smem = 0
    S = 2 * chain_per_pass("sample", _sms()) + 77
    graph = mps_graph(n, K)
    torch.manual_seed(90)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, torch.float32)
    eng, q = _engine(graph, K, cores)
    for k in names:
        q.cores_weights[k] = q.cores_weights[k].detach()
    st = [s.to(DEV) for s in oc.unit_states(nq, K)]
    out = {}
    for method in ("prefix", "linear"):
        torch.manual_seed(77)
        torch.cuda.manual_seed(77)
        if method == "prefix":
            with KernelRecorder() as rec:
                out[method] = eng.sample(q, st, num_samples=S, K=K, bounds=[-5, 5], grid_size=G, method=method)
            rec.check([f"tnq_chain_sample_kernel<{K}>"])
        else:
            out[method] = eng.sample(q, st, num_samples=S, K=K, bounds=[-5, 5], grid_size=G, method=method)
    torch.manual_seed(77)                               # the uniform numbers both methods drew (sample())
    torch.cuda.manual_seed(77)
    u = torch.cat([eng.backend.rand((S, 1), dtype=torch.float32) for _ in range(n)], dim=1)
    cell = 10.0 / (G - 1)
    diff = (out["prefix"] - out["linear"]).abs()
    far = torch.nonzero(diff >= 0.05 * cell).tolist()
    print(f"[sample G={G} S={S}] median {diff.median().item():.2e} max {diff.max().item() / cell:.2e} cells, "
          f"{len(far)} of {diff.numel()} draws beyond 0.05 cell")
    assert diff.median().item() < 1e-5
    # Every draw that differs by more than 0.05 cell must be a flipped comparison, and each method's value must be what
    # the reference's formula gives for the flipped or the unflipped count.  With idx = #(cdf < u) (clamped to G - 2),
    # y = x[idx] + (u - cdf[idx]) / (cdf[idx+1] - cdf[idx] + 1e-10) dx extrapolates from the first CDF value NOT below
    # u, so when one comparison cdf[j] < u flips, idx moves by one and y jumps by dx (1 - d[j+1] / d[j+2]) -- many cells
    # where the density changes fast.  A comparison can flip only where u lies within the float32 error of cdf[j]: the
    # running sum of G positive densities is within G 2^-24 relative of the exact one, doubled here for the rounding
    # of the densities themselves and of the normalisation.  So, in float64 and for each method on its OWN earlier
    # draws (a flip on an earlier qubit changes the densities of this one): J = the indices j with |cdf[j] - u| <= tol;
    # the method's value equals the formula's at the float64 count, or at a count from min(J) to max(J) + 1, to
    # 0.05 cell, plus what the CDF's own rounding moves the formula by: with r = (u - c0) /
    # (c1 - c0), an error e in c0 and c1 moves r by e (1 + 2|r|) / (c1 - c0).  For e the typical error of the
    # sequential running sum is taken, 3 sqrt(G) 2^-24 (a random walk of G roundings, with a 3x margin): it matters
    # only in cells that carry almost no probability, where the formula divides round-off-sized numbers.  Where the
    # two methods' earlier draws of the sample agree (to 1e-5), J is not empty: the difference must come from a flip
    # on this qubit.
    tol = 2 * G * 2.0 ** -24
    e_typ = 3 * G ** 0.5 * 2.0 ** -24
    grid_x = torch.linspace(-5, 5, G, dtype=torch.float64, device=DEV)
    mg, _ = oc.generate_data(grid_x.cpu().unsqueeze(1), K, torch.float64, "tensor")
    c64 = [cores[k].to(DEV, torch.float64) for k in names]
    s64 = [s.double() for s in st]
    eye64 = torch.eye(K, dtype=torch.float64, device=DEV).expand(G, K, K)

    def formula(cdf, uu, idx):
        """(y, allowance) of the reference's interpolation at count idx."""
        idx = min(idx, G - 2)
        c0, c1 = cdf[idx].item(), cdf[idx + 1].item()
        r = (uu - c0) / (c1 - c0 + 1e-10)
        return grid_x[idx].item() + r * cell, 0.05 * cell + cell * e_typ * (1 + 2 * abs(r)) / (c1 - c0 + 1e-10)

    for s_, qb in far:
        uu = u[s_, qb].item()
        for method in ("prefix", "linear"):
            prev, _ = oc.generate_data(out[method][s_:s_ + 1, :qb].double().cpu(), K, torch.float64, "tensor")
            mx = [p.to(DEV).expand(G, K, K) for p in prev] + [mg[0].to(DEV)] + [eye64] * (n - qb - 1)
            dens = mps_f64(c64, s64, mx).clamp_min(0)
            cdf = dens.cumsum(0) / (dens.sum() + 1e-10)
            near = torch.nonzero((cdf - uu).abs() <= tol).flatten().tolist()
            if qb == 0 or diff[s_, :qb].max().item() < 1e-5:
                assert near, (s_, qb, method, "no CDF value within the float32 error of u")
            counts = {int((cdf < uu).sum().item())}
            if near:
                counts |= set(range(min(near), max(near) + 2))
            y = out[method][s_, qb].item()
            fits = [(abs(y - yc), allow) for yc, allow in (formula(cdf, uu, c) for c in counts)]
            assert any(d < allow for d, allow in fits), (s_, qb, method, y, min(fits))


# ---- refusals -------------------------------------------------------------------------------------------------------
def _ptrs(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def test_chain_workspace_one_byte_short(built_lib):
    lib = tneq_b200._lib.load()
    K, n, B = 3, 5, 5000
    sms = _sms()
    torch.manual_seed(1)
    cores = [torch.randn(K, K, K, K, device=DEV) for _ in range(n - 1)]
    states = [torch.ones(K, device=DEV) for _ in range(n)]
    mx = [torch.randn(B, K, K, device=DEV) for _ in range(n)]
    grid = min(-(-B // CHAIN_THREADS), 4 * sms)
    need = 4 * grid * ((n - 1) * K ** 3 + 1)
    ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
    for mode in (1, 2):
        values = torch.full((B,), 12345.0, device=DEV)
        loss = torch.full((1,), 12345.0, device=DEV)
        grads = [torch.full_like(c, 12345.0) for c in cores]
        seed = torch.ones(B, device=DEV)
        args = lambda nbytes: (K, n, _ptrs(cores), _ptrs(states), _ptrs(mx), (ctypes.c_int64 * n)(*[K * K] * n), B,
                               mode, seed.data_ptr(), values.data_ptr(), loss.data_ptr(), _ptrs(grads), 0.0,
                               ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        l0 = tneq_b200._lib.launch_count()
        assert lib.tnq_mps_chain(*args(need - 1)) != 0
        assert b"workspace too small" in lib.tnq_last_error()
        assert tneq_b200._lib.launch_count() == l0
        torch.cuda.synchronize()
        assert (values == 12345.0).all() and (loss == 12345.0).all() and all((g == 12345.0).all() for g in grads)
        assert lib.tnq_mps_chain(*args(need)) == 0                        # the exact size is enough
        torch.cuda.synchronize()
        assert not (grads[0] == 12345.0).all()


def test_ladder_workspace_one_byte_short(built_lib):
    lib = tneq_b200._lib.load()
    K, n, B = 3, 5, 5000
    torch.manual_seed(2)
    ca = [torch.randn(K, K, K, K, device=DEV) for _ in range(n - 1)]
    cx = [torch.randn(K, K, K, K, device=DEV) for _ in range(n - 1)]
    states = [torch.ones(K, device=DEV) for _ in range(n)]
    mx = [torch.randn(B, K, K, device=DEV) for _ in range(n)]
    old = os.environ.pop("TNQ_LADDER_V2", None)
    try:
        for mode in (1, 2):
            need = int(lib.tnq_mps_ladder_workspace_bytes(K, n, B, mode))
            assert need == ladder_workspace(K, n, B)
            ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
            values = torch.full((B,), 12345.0, device=DEV)
            loss = torch.full((1,), 12345.0, device=DEV)
            ga = [torch.full_like(c, 12345.0) for c in ca]
            gx = [torch.full_like(c, 12345.0) for c in cx]
            seed = torch.ones(B, device=DEV)
            args = lambda nbytes: (K, n, _ptrs(ca), _ptrs(cx), _ptrs(states), _ptrs(mx),
                                   (ctypes.c_int64 * n)(*[K * K] * n), B, mode, seed.data_ptr(), values.data_ptr(),
                                   loss.data_ptr(), _ptrs(ga), _ptrs(gx), 0.0, ws.data_ptr(), nbytes,
                                   torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            l0 = tneq_b200._lib.launch_count()
            assert lib.tnq_mps_ladder(*args(need - 1)) != 0
            assert b"workspace too small" in lib.tnq_last_error()
            assert tneq_b200._lib.launch_count() == l0
            torch.cuda.synchronize()
            assert (values == 12345.0).all() and (loss == 12345.0).all()
            assert all((g == 12345.0).all() for g in ga + gx)
            assert lib.tnq_mps_ladder(*args(need)) == 0
            torch.cuda.synchronize()
            assert not (gx[0] == 12345.0).all()
    finally:
        if old is not None:
            os.environ["TNQ_LADDER_V2"] = old
