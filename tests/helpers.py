"""Shared helpers for the tests (oracle-side data + comparisons)."""
import numpy as np
import torch

from oracle import qctn_oracle as oc


# Two float32 implementations that sum in different orders carry INDEPENDENT rounding noise; where a
# batch amplifies it (1/p weights of samples that partly cancel) the ratio of their errors against
# float64 fluctuates by several x in either direction (measured 0.2 .. 5.3 on seeded batches, see
# DESIGN.md "Parity").  The CUDA path is therefore required to be within 1e-5, or within NOISE_FACTOR x
# the reference's own float32 error on the same batch, whichever is larger.
NOISE_FACTOR = 8


def make_case(graph, K, B, dtype, tnt=True, mode="a", seed=0, identity_q=()):
    """Seeded CPU inputs for one contraction: cores, unit states, measurement matrices."""
    torch.manual_seed(seed)
    td = getattr(torch, dtype)
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, td)
    x = torch.randn(B, nq)
    mxs, _ = oc.generate_data(x, K, td, "TNTensor" if tnt else "tensor")
    if identity_q:
        eye = torch.eye(K, dtype=td).expand(B, K, K)
        mxs = [eye if q in identity_q else m for q, m in enumerate(mxs)]
    if mode == "ab":
        eye = torch.eye(K, dtype=td).expand(B, K, K)
        mxs = [torch.stack([oc._raw(m), eye], dim=1) for m in mxs]
    states = oc.unit_states(nq, K, td)
    return names, table, nq, cores, states, mxs


def clone_mx(mxs):
    out = []
    for m in mxs:
        if isinstance(m, oc.TNT):
            out.append(oc.TNT(m.tensor.clone(), m.scale, m.log_scale))
        else:
            out.append(m.clone())
    return out


def rel_err(got, want):
    got, want = torch.as_tensor(got).detach().cpu(), torch.as_tensor(want).detach().cpu()
    return ((got - want).abs().max() / want.abs().max().clamp_min(1e-300)).item()


def elem_rel_err(got, want, floor=0.0):
    got, want = torch.as_tensor(got).detach().cpu(), torch.as_tensor(want).detach().cpu()
    return ((got - want).abs() / want.abs().clamp_min(floor if floor > 0 else 1e-300)).max().item()


def well_conditioned_case(graph, K, B, dtype, seed=0, keep=0.05, mode="a"):
    """Like make_case, but only keeps samples whose float64 value is at least `keep` x the
    median of 6B candidates, and of those a RANDOM B (seeded), not the B most probable ones.
    Samples whose amplitude almost cancels lose every digit in float32 in ANY implementation (the
    reference included) and, because d log p = dp / p, they dominate the gradient error; parity to
    1e-5 is only meaningful away from them (DESIGN.md, "Parity").  What happens on an unfiltered
    batch is bounded separately (tests/test_gpu_unfiltered.py)."""
    torch.manual_seed(seed)
    td = getattr(torch, dtype)
    td64 = torch.complex128 if td.is_complex else torch.float64
    names, table, nq = oc.parse_graph(graph)
    cores = oc.random_cores(table, td)
    states = oc.unit_states(nq, K, td)
    x = torch.randn(6 * B, nq)
    mx64, _ = oc.generate_data(x, K, td64, "tensor")
    p = oc.forward(graph, {k: v.to(td64) for k, v in cores.items()}, [s.to(td64) for s in states], mx64)
    survivors = torch.nonzero(p >= keep * p.median()).flatten()
    assert len(survivors) >= B, "not enough well-conditioned samples"
    gen = torch.Generator().manual_seed(1000 + seed)
    order = survivors[torch.randperm(len(survivors), generator=gen)]
    good = order[:B].sort().values
    for _ in range(4):
        # the loss clamps the SCALED value at 1e-10 (engine_siamese.py:490-530): a sample within 5 % of
        # the clamp flips between "gradient dp/p" and "gradient 0" on the last float32 bit -- swap those
        # for other survivors (the TNTensor scales depend on the selected batch, hence the loop)
        mxs, _ = oc.generate_data(x[good], K, td, "TNTensor")
        scale = 1.0
        for m in mxs:
            scale *= m.scale
        ps = p[good] / (scale ** 2 if td.is_complex else scale)
        near = (ps / 1e-10).log().abs() < 0.05
        if not near.any():
            break
        pool = [int(i) for i in order if int(i) not in set(good.tolist())]
        keepers = good[~near].tolist()
        good = torch.tensor(sorted(keepers + pool[:B - len(keepers)]))
    mxs, _ = oc.generate_data(x[good], K, td, "TNTensor")
    if mode == "ab":
        eye = torch.eye(K, dtype=td).expand(B, K, K)
        mxs = [torch.stack([oc._raw(m), eye], dim=1) for m in mxs]
    return names, table, nq, cores, states, mxs


def upcast(x, td):
    if isinstance(x, oc.TNT):
        return oc.TNT(x.tensor.to(td), x.scale, x.log_scale)
    return x.to(td)


def mps_f64(cores, states, mxs):
    """The single-layer MPS sweep (einsum strings 'cdef,c,aeg,higj,h,d,i->ajf', 'cdef,aeg,higj,ahc,d,i->ajf',
    'acd,adc->a') pairwise in the plan compiler's own order (3 K^4 per qubit and sample), on whatever device and
    dtype the inputs have: in float64 / complex128 on the GPU, the yardstick of the large-bond route where the CPU
    oracle's K^6 intermediates are out of reach.  Returns the amplitude (the engine reports |amp|^2 for complex
    networks, amp for real ones).  Pinned to the oracle by tests/test_large_bond_yardstick.py."""
    n = len(states)
    a0, ac = cores[0], cores[0].conj()
    v = torch.einsum("cdef,c,d->ef", a0, states[0], states[1])
    w = torch.einsum("higj,h,i->gj", ac, states[0], states[1])
    env = torch.einsum("ef,aeg,gj->ajf", v, mxs[0], w)
    for qd in range(1, n - 1):
        a = cores[qd]
        v = torch.einsum("cdef,d->cef", a, states[qd + 1])
        w = torch.einsum("higj,i->hgj", a.conj(), states[qd + 1])
        t1 = torch.einsum("ahc,cef->ahef", env, v)
        t2 = torch.einsum("ahef,aeg->ahgf", t1, mxs[qd])
        env = torch.einsum("ahgf,hgj->ajf", t2, w)
    return torch.einsum("acd,adc->a", env, mxs[n - 1])


def mps_f64_value(amp):
    """The value the engine reports for an amplitude: |amp|^2 for complex networks (reference quirk D10), amp for
    real ones."""
    return amp.real ** 2 + amp.imag ** 2 if amp.is_complex() else amp


def ladder_layers(graph, K):
    """(layer1, layer2): the core names of the two layers of a merged MPS network, as the ladder route reads them
    off the plan (plan.mps_ladder(), used by b200_strategy._ladder)."""
    import tneq_b200
    from tneq_b200.contractor.plan import ContractionPlan
    q = tneq_b200.QCTN(graph)
    n = q.nqubits
    plan = ContractionPlan(q.adjacency_table, n, {c: (K,) * 4 for c in q.cores}, {i: K for i in range(n)},
                           {i: ("a", K, K) for i in range(n)}, "float32")
    lad = plan.mps_ladder()
    assert lad is not None and lad[0] == K
    return lad[1], lad[2]


def ladder_f64(cores_a, cores_x, states, mxs):
    """The two-layer merged MPS sweep (QCTN.merge(mps_n, mps_n); greedy groups
    'cdef,eghi,c,ahj,klmn,mojp,k,d,l->agnpfio', 'cdef,ghij,aik,lmno,pqkr,aelpcgn,d,m->ahorfjq',
    'cdef,gfhi,ahj,klmn,onjp,aekocgm,d,l->api', 'acd,adc->a') restated pairwise in the order of DESIGN 3d, on whatever
    device and dtype the inputs have: the float64 yardstick of the ladder kernels, where the oracle's left-to-right
    einsum of a middle group builds B K^12 intermediates.  cores_a / cores_x: the n-1 cores of the first / second
    layer (plan.mps_ladder() order), A_q and X_q acting on wires (q, q+1).  Per qubit and sample the largest
    intermediate has K^7 entries.  Real networks only (what the ladder kernels take).  Returns the values (B,).
    Pinned to the oracle by tests/test_large_bond_yardstick.py."""
    n = len(states)
    a0, x0 = cores_a[0], cores_x[0]
    # first group: env[a,g,n,p,f,i,o] (ket: A_0 out on wire 1 = f, X_0 in / out on wire 1 = g / i; bra: n, o, p)
    v = torch.einsum("cdef,c,d->ef", a0, states[0], states[1])
    t = torch.einsum("ef,eghi->fghi", v, x0)
    u = torch.einsum("ahj,mojp->ahmop", mxs[0], x0)
    u = torch.einsum("mn,ahmop->ahnop", v, u)
    env = torch.einsum("fghi,ahnop->agnpfio", t, u)
    for q in range(1, n - 2):
        a, x = cores_a[q], cores_x[q]
        bs = torch.einsum("cdef,d->cef", a, states[q + 1])
        # A: T2[f,o,g,p] = sum_{c,e,l,n} Bs[c,e,f] Bs[l,n,o] E[c,l,n,p,e,g]
        t1 = torch.einsum("aelpcgn,cef->alnpgf", env, bs)
        t2 = torch.einsum("alnpgf,lno->afogp", t1, bs)
        # B: U[i,p,q,r] = sum_k M[i,k] X[p,q,k,r]
        u = torch.einsum("aik,pqkr->aipqr", mxs[q], x)
        # C: E'[f,o,q,r,h,j] = sum_{g,i,p} T2[f,o,g,p] U[i,p,q,r] X[g,h,i,j]
        w = torch.einsum("afogp,aipqr->afogiqr", t2, u)
        env = torch.einsum("afogiqr,ghij->ahorfjq", w, x)
    a, x = cores_a[n - 2], cores_x[n - 2]
    bs = torch.einsum("cdef,d->cef", a, states[n - 1])
    t1 = torch.einsum("aekocgm,cef->akogmf", env, bs)
    t2 = torch.einsum("akogmf,kmn->aogfn", t1, bs)
    u = torch.einsum("ahj,onjp->ahonp", mxs[n - 2], x)
    w = torch.einsum("aogfn,ahonp->agfhp", t2, u)
    out = torch.einsum("agfhp,gfhi->api", w, x)
    return torch.einsum("acd,adc->a", out, mxs[n - 1])


# ---- which GEMM variant a large-bond launch takes --------------------------------------------------------------------
GEMM_TILE = 128          # BM = BN of csrc/tnq_gemm.cu
GEMM_BK = 32             # BK of csrc/tnq_gemm.cu


def gemm_splitk(M, N, K, batch=1, accumulate=False):
    """Mirror of launch_tma's split-K rule (csrc/tnq_gemm.cu): a TMA-fed, non-small-K launch (K > 256) is split in
    two along K when batch == 1, the tile is written (not accumulated), it covers at most 74 output tiles of
    128 x 128 and K >= 32 k-blocks of 32."""
    tiles = -(-M // GEMM_TILE) * -(-N // GEMM_TILE)
    return batch == 1 and not accumulate and K > 256 and tiles <= 74 and K >= 32 * GEMM_BK


def record_routes(monkeypatch, cls):
    """Wrap the launch sites of a GemmPathRunner class (contractor/gemm_path.py) so that every kernel variant that
    ran is counted.  Keys of the returned Counter:
        ("view", split_k)              tnq_gemm_tf32x3_view (A permuted by the TMA unit)
        ("bk", a_mn, b_mn, split_k)    tnq_gemm_tf32x3_bk (batch into K; x_mn: operand read MN-major in place)
        ("gemm", split_k)              tnq_gemm_tf32x3 with batch 1 and K > 256 (the TMA-fed kernel)
        ("fold_vec",) ("outer_acc",)   tnq_fold_vec_f32 / tnq_outer_acc_f32
    Only launches that happened are counted (a refused view or bk falls back and is not)."""
    from collections import Counter
    from tneq_b200.contractor import gemm_path as gp
    seen = Counter()
    gemm, view, reduce_, fold, outer = cls._gemm, cls._gemm_view, cls._reduce_in_place, cls._fold_vec, cls._outer_acc

    def _gemm(self, A, B, C, M, N, K, lda, ldb, ldc, batch=1, sA=0, sB=0, sC=0, accumulate=False):
        gemm(self, A, B, C, M, N, K, lda, ldb, ldc, batch, sA, sB, sC, accumulate)
        if batch == 1 and K > 256 and not (lda % 4 or ldb % 4):
            seen[("gemm", gemm_splitk(M, N, K, batch, accumulate))] += 1

    def _gemm_view(self, A, v, Bm, C, N, ldb, ldc):
        ok = view(self, A, v, Bm, C, N, ldb, ldc)
        if ok:
            R1, R0, _, _, K1, K0, _ = v
            seen[("view", gemm_splitk(R1 * R0, N, K1 * K0))] += 1
        return ok

    def _reduce_in_place(self, tp, Lp, pf, tq, Lq, qf, shared, NS):
        out = reduce_(self, tp, Lp, pf, tq, Lq, qf, shared, NS)
        if out is not None:
            k = shared[0]
            a_mn = self._mn_in_place(Lp, pf, k, NS) is not None
            b_mn = self._mn_in_place(Lq, qf, k, NS) is not None
            split = gemm_splitk(self._size(pf, NS), self._size(qf, NS), NS * self._extent(k, NS))
            seen[("bk", int(a_mn), int(b_mn), split)] += 1
        return out

    def _fold_vec(self, n, val, lay):
        out = fold(self, n, val, lay)
        if out is not None:
            seen[("fold_vec",)] += 1
        return out

    def _outer_acc(self, n, val, lay):
        ok = outer(self, n, val, lay)
        if ok:
            seen[("outer_acc",)] += 1
        return ok

    for name, fn in (("_gemm", _gemm), ("_gemm_view", _gemm_view), ("_reduce_in_place", _reduce_in_place),
                     ("_fold_vec", _fold_vec), ("_outer_acc", _outer_acc)):
        monkeypatch.setattr(cls, name, fn)
    assert gp.GemmPathRunner in cls.__mro__
    return seen


# The float64-parity cases of tests/test_gpu_large_bond.py, each with the kernel variants it exists to reach (keys of
# record_routes) on the route that reads MN-major operands in place (gemm_path.MN_IN_PLACE) and on the transposing
# route.  tests/test_gemm_path_plan.py checks the same expectations on meta tensors without a GPU.
def _bk(split, pairs=((0, 1), (1, 0), (1, 1))):
    return {("bk", a, b, split) for a, b in pairs}


_FOLD = {("fold_vec",), ("outer_acc",)}
LARGE_BOND_CASES = [
    # dtype, chi, n, B, variants (MN in place), variants (transposing)
    ("complex64", 64, 5, 256, _bk(True) | {("view", False), ("gemm", True)} | _FOLD,       # cfg4's per-qubit variants
     {("view", False), ("gemm", True)} | _FOLD),
    ("complex64", 64, 4, 5, _bk(False) | {("view", True)} | _FOLD,                        # smallest batch with bk
     {("view", True)} | _FOLD),
    ("complex64", 64, 6, 32, _bk(True) | {("view", True), ("gemm", True)} | _FOLD,
     {("view", True), ("gemm", True)} | _FOLD),
    ("complex64", 32, 5, 256, {("view", True), ("gemm", True)} | _FOLD,
     {("view", True), ("gemm", True)} | _FOLD),
    ("float32", 64, 5, 256, {("view", False), ("gemm", True)},
     {("view", False), ("gemm", True)}),
    ("float32", 128, 4, 8, _bk(False) | {("view", True), ("gemm", True)},
     {("view", True), ("gemm", True), ("gemm", False)}),
    ("complex64", 128, 3, 2, {("view", True)} | _FOLD,
     {("view", True)} | _FOLD),
]


# ---- which register-resident kernels a call launches ----------------------------------------------------------------
class KernelRecorder:
    """Names of this library's CUDA kernels launched inside the `with` block, recorded with torch.profiler (CUDA
    activity).  The profiler reports demangled template instances, e.g.
    'void (anonymous namespace)::tnq_chain_kernel<3, 1>(...)'; `names` keeps the instance ('tnq_chain_kernel<3, 1>').
    A block that launches no tnq_ kernel at all fails: a profiler that cannot see kernel names must not turn a
    coverage assertion into no assertion."""

    def __enter__(self):
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        self._prof = profile(activities=[ProfilerActivity.CUDA])
        self._prof.__enter__()
        return self

    def __exit__(self, *exc):
        import re
        torch.cuda.synchronize()
        self._prof.__exit__(*exc)
        if exc[0] is not None:
            return False
        found = set()
        for ev in self._prof.events():
            m = re.search(r"tnq_\w+(<[^<>()]*>)?", ev.name)
            if m:
                found.add(m.group(0))
        assert found, "the profiler saw no tnq_ kernel"
        self.names = found
        return False

    def check(self, expected):
        """Every expected name (a template instance, or a prefix for non-template kernels) was launched, and nothing
        else of this library was."""
        for e in expected:
            assert any(n.startswith(e) for n in self.names), (e, sorted(self.names))
        for n in self.names:
            assert any(n.startswith(e) for e in expected), (n, sorted(expected))
