"""Large-bond-dimension execution of a contraction graph: permute -> tensor-core GEMM.

The shared-memory VM (vm_program.py / csrc/tnq_vm.cu) keeps every prepared core in shared
memory, which stops working once cores have 64^4 elements.  In that regime every pairwise
contraction of the sweep is a real GEMM, so the same contraction graph (cgraph.py) is executed
node by node on global-memory tensors (here a float32 / complex64 plan):

    contract   ->  [tnq_permute_f32 to put the contracted indices innermost, only if needed]
                   tnq_gemm_tf32x3   (tcgen05, fp32-faithful 3xTF32, TMEM accumulators)
    lin        ->  tnq_permute_f32 (permute / conj), tnq_cplx_expand_f32, tnq_cplx_fold_f32
    reduce over the batch (core gradients) -> the batch is folded into the GEMM's K dimension

float64 / complex128 plans run the same graph on the _f64 sibling of every kernel: tnq_gemm_f64 (FP64
tensor cores, mma.sync f64), tnq_permute_f64, tnq_fold_vec_f64, tnq_outer_acc_f64, tnq_cplx_expand_f64 and
tnq_cplx_fold_f64.  The two in-place GEMM variants (the TMA-permuted view, the MN-major core-gradient GEMM)
are float32 only; in float64 their operands are transposed explicitly instead.

Complex contractions are real GEMMs of the operand against the 2x2-real expansion of the other (see
cgraph.py).  PyTorch provides the buffers and the stream; all arithmetic on tensors is done by the kernels
named above.
"""
from __future__ import annotations

import ctypes
from ctypes import c_int64, c_void_p
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from .. import _lib
from .cgraph import CGraph, Node

BATCH = -1   # pseudo index id of the sample dimension in layouts
# core-gradient GEMMs with MN-major operands read in place (tnq_gemm_tf32x3_bk); TNQ_GEMM_MN=0 transposes instead
MN_IN_PLACE = __import__("os").environ.get("TNQ_GEMM_MN", "1") == "1"


class GemmPathRunner:
    dtype, f64, _sfx = torch.float32, False, "f32"

    def __init__(self, graph: CGraph, device: torch.device, dtype: torch.dtype = torch.float32):
        """dtype: the plan's real dtype, torch.float32 (float32 / complex64 plans) or torch.float64."""
        if device.type != "cuda":
            raise RuntimeError("the GEMM path runs on CUDA devices only (no CPU fallback)")
        self.g, self.device = graph, device
        self._set_dtype(dtype)
        self.lib = _lib.load()
        with torch.cuda.device(device):
            _lib.check(self.lib.tnq_device_check())
        self.flops = 0.0

    def _set_dtype(self, dtype: torch.dtype):
        if dtype not in (torch.float32, torch.float64):
            raise ValueError(f"the GEMM path computes in float32 or float64, not {dtype}")
        self.dtype = dtype
        self.f64 = dtype == torch.float64
        self._sfx = "f64" if self.f64 else "f32"

    def _entry(self, name: str):
        """The library entry point tnq_<name>_f32 or tnq_<name>_f64 of this runner's dtype."""
        return getattr(self.lib, f"tnq_{name}_{self._sfx}")

    # ---- raw kernel calls ------------------------------------------------------------
    def _stream(self):
        return c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _permute(self, src: torch.Tensor, src_strides: Sequence[int], out_dims: Sequence[int], vec: int, conj: bool):
        out = torch.empty(tuple(out_dims), dtype=self.dtype, device=self.device)
        n = len(out_dims)
        _lib.check(self._entry("permute")(c_void_p(src.data_ptr()), c_void_p(out.data_ptr()), n,
                                          (c_int64 * n)(*out_dims), (c_int64 * n)(*src_strides), vec, int(conj),
                                          self._stream()))
        return out

    def _gemm(self, A, B, C, M, N, K, lda, ldb, ldc, batch=1, sA=0, sB=0, sC=0, accumulate=False):
        gemm = self.lib.tnq_gemm_f64 if self.f64 else self.lib.tnq_gemm_tf32x3
        _lib.check(gemm(c_void_p(A.data_ptr()), c_void_p(B.data_ptr()), c_void_p(C.data_ptr()),
                        M, N, K, lda, ldb, ldc, batch, sA, sB, sC, int(accumulate), self._stream()))
        self.flops += 2.0 * M * N * K * batch

    def _gemm_view(self, A, view, Bm, C, N, ldb, ldc):
        """C = A_view x Bm^T with the permutation of A done by the TMA unit (tnq_gemm_tf32x3_view).  False: the
        view is not expressible as a tensor map, or the runner computes in float64 (float32 only); nothing was
        launched."""
        if self.f64:
            return False
        R1, R0, sR1, sR0, K1, K0, sK1 = view
        rc = self.lib.tnq_gemm_tf32x3_view(c_void_p(A.data_ptr()), R1, R0, sR1, sR0, K1, K0, sK1, c_void_p(Bm.data_ptr()),
                                           ldb, c_void_p(C.data_ptr()), ldc, N, self._stream())
        if rc == -2:
            return False
        _lib.check(rc)
        self.flops += 2.0 * R1 * R0 * N * K1 * K0
        return True

    # ---- big tensor x tiny tensor over one index (+ complex component): the circuit-state operands ----------------
    def _small_partner(self, n: Node, val, lay):
        """(big, small) operand nodes of `n` when one operand is a tiny non-batched rank-3 tensor [d, ri, ro] in its
        own memory order (the 2x2-real expansion of a complex vector) and the other a non-batched tensor whose
        innermost index is a complex component; else None."""
        g = self.g
        if n.reduce_batch:
            return None
        for big, small in ((g.nodes[n.p], g.nodes[n.q]), (g.nodes[n.q], g.nodes[n.p])):
            if big.batched or small.batched or len(small.idx) != 3 or len(big.idx) < 2:
                continue
            if lay[small.id] != list(small.idx) or g.dims[small.idx[1]] != 2 or g.dims[small.idx[2]] != 2:
                continue
            if g.dims[lay[big.id][-1]] != 2 or not val[small.id].is_contiguous() or not val[big.id].is_contiguous():
                continue
            return big, small
        return None

    def _fold_vec(self, n: Node, val, lay):
        """out[.., ro] = sum_{d, ri} big[.., d, .., ri] small[d, ri, ro] in one pass over `big` (tnq_fold_vec_f32)."""
        pair = self._small_partner(n, val, lay)
        if pair is None or n.acc_into >= 0:
            return None
        big, small = pair
        g, L = self.g, lay[big.id]
        d, ri, ro = small.idx
        shared = set(big.idx) & set(small.idx)
        if shared != {d, ri} or L[-1] != ri or d not in L[:-1]:
            return None
        j = L.index(d)
        A, D, C = self._size(L[:j], 1), g.dims[d], self._size(L[j + 1:-1], 1)
        out_layout = L[:j] + L[j + 1:-1] + [ro]
        out = torch.empty([g.dims[i] for i in out_layout], dtype=self.dtype, device=self.device)
        _lib.check(self._entry("fold_vec")(c_void_p(val[big.id].data_ptr()), c_void_p(val[small.id].data_ptr()),
                                           c_void_p(out.data_ptr()), A, D, C, self._stream()))
        self.flops += 2.0 * A * D * C * 4
        return out, out_layout

    def _outer_acc(self, n: Node, val, lay) -> bool:
        """target[.., d, .., ri] += sum_ro big[.., ro] small[d, ri, ro], accumulated in place in the target's memory
        order (tnq_outer_acc_f32): the adjoint of _fold_vec, instead of GEMM (K = 2) + transposition + add."""
        pair = self._small_partner(n, val, lay)
        if pair is None or n.acc_into < 0:
            return False
        big, small = pair
        g, L = self.g, lay[big.id]
        d, ri, ro = small.idx
        if set(big.idx) & set(small.idx) != {ro} or L[-1] != ro:
            return False
        T = list(n.idx)                              # the target's memory order
        if T[-1] != ri or d not in T[:-1]:
            return False
        j = T.index(d)
        if T[:j] + T[j + 1:-1] != L[:-1]:
            return False
        tgt = val[n.acc_into]
        if not tgt.is_contiguous():
            return False
        A, D, C = self._size(T[:j], 1), g.dims[d], self._size(T[j + 1:-1], 1)
        _lib.check(self._entry("outer_acc")(c_void_p(val[big.id].data_ptr()), c_void_p(val[small.id].data_ptr()),
                                            c_void_p(tgt.data_ptr()), A, D, C, self._stream()))
        self.flops += 2.0 * A * D * C * 4
        return True

    def _mn_in_place(self, layout: List[int], free: List[int], k: int, B: int):
        """`layout` == [BATCH, hi..., k, lo...] with the lo indices spanning exactly one 128-row tile: the operand can be
        consumed MN-major in place (tnq_gemm_tf32x3_bk).  Returns (row tiles, row order) or None."""
        if not layout or layout[0] != BATCH or k not in layout:
            return None
        j = layout.index(k)
        hi, lo = layout[1:j], layout[j + 1:]
        if sorted(hi + lo) != sorted(free) or self._size(lo, B) != 128 or self._extent(k, B) % 32:
            return None
        return self._size(hi, B), hi + lo

    def _reduce_in_place(self, tp, Lp, pf, tq, Lq, qf, shared, NS):
        """C[pf, qf] = sum over (batch, k) with at least one operand read in place, MN-major (the 537 MB intermediates of
        the bond-64 sweep are [batch][rows][k][128 rows]); the other operand is transposed explicitly when it is not of
        that form (it is the small one).  None: not expressible, or float64 (float32 only): the caller transposes
        both."""
        if len(shared) != 1 or not MN_IN_PLACE or self.f64:
            return None
        k = shared[0]
        a, b = self._mn_in_place(Lp, pf, k, NS), self._mn_in_place(Lq, qf, k, NS)
        if a is None and b is None:
            return None
        Kin = self._extent(k, NS)
        if NS * Kin <= 256:
            return None
        if a is None:
            A, rows_a = self._arrange(tp, Lp, pf, [BATCH, k], NS)
            a_tiles = 0
        else:
            A, (a_tiles, rows_a) = tp, a
        if b is None:
            Bm, rows_b = self._arrange(tq, Lq, qf, [BATCH, k], NS)
            b_tiles = 0
        else:
            Bm, (b_tiles, rows_b) = tq, b
        M, N = self._size(pf, NS), self._size(qf, NS)
        C = torch.empty((M, N), dtype=self.dtype, device=self.device)
        rc = self.lib.tnq_gemm_tf32x3_bk(c_void_p(A.data_ptr()), int(a is not None), a_tiles, c_void_p(Bm.data_ptr()),
                                         int(b is not None), b_tiles, c_void_p(C.data_ptr()), M, N, NS, Kin, self._stream())
        if rc == -2:
            return None
        _lib.check(rc)
        self.flops += 2.0 * M * N * NS * Kin
        out_layout = rows_a + rows_b
        return C.reshape([self.g.dims[i] for i in out_layout] or [1]), out_layout

    def _strided_view(self, layout: List[int], rows: List[int], cols: List[int], B: int):
        """`layout` read as rows x cols WITHOUT a copy, when memory order alternates as [rows][cols][rows][cols]
        (outer to inner; leading groups may be missing): (R1, R0, sR1, sR0, K1, K0, sK1) and the row order, or
        None.  cols must already be in memory order (they are: _tail_order)."""
        rs, cs = set(rows), set(cols)
        if [i for i in layout if i in cs] != list(cols) or len(rs) + len(cs) != len(layout):
            return None
        segs = []                                    # [(is_col, [indices])] outer -> inner
        for i in layout:
            c = i in cs
            if segs and segs[-1][0] == c:
                segs[-1][1].append(i)
            else:
                segs.append((c, [i]))
        if not segs or not segs[-1][0] or len(segs) not in (3, 4):
            return None                              # 1-2 groups: no transposition needed; 5+: not a 4-level view
        strides, s = {}, 1
        for i in reversed(layout):
            strides[i] = s
            s *= self._extent(i, B)
        size = lambda idx: self._size(idx, B)
        k0, r0 = segs[-1][1], segs[-2][1]
        k1 = segs[-3][1]
        r1 = segs[-4][1] if len(segs) == 4 else []
        view = (size(r1), size(r0), strides[r1[-1]] if r1 else 0, strides[r0[-1]], size(k1), size(k0), strides[k1[-1]])
        R1, R0, sR1, sR0, K1, K0, sK1 = view
        # what tnq_gemm_tf32x3_view can describe to the TMA unit (it re-checks, plus the pointer alignment)
        if K0 % 32 or not (R0 % 128 == 0 or 128 % R0 == 0) or K1 * K0 <= 256 or sR1 % 4 or sR0 % 4 or sK1 % 4:
            return None
        return view, r1 + r0

    # ---- layouts --------------------------------------------------------------------------
    def _extent(self, i, B):
        return B if i == BATCH else self.g.dims[i]

    def _size(self, idx, B):
        n = 1
        for i in idx:
            n *= self._extent(i, B)
        return n

    def _arrange(self, t: torch.Tensor, layout: List[int], rows: List[int], cols: List[int], B: int,
                 exact: bool = False):
        """Bring `t` (index order `layout`) into the form [rows..., cols...]: `cols` in exactly the
        given order, `rows` in any order (their current order is kept when no copy is needed)
        unless exact.  Returns (tensor, order of the row indices).  At most one permute kernel."""
        k = len(cols)
        if not exact:
            # rows in the order they have in memory: indices that are neighbours in the input stay neighbours in
            # the output, so tnq_permute_f32 can merge them into one contiguous run (a (index, re/im) pair split
            # by another row index forced the strided scalar path: 2.1 ms instead of 0.5 ms per 537 MB tensor)
            rs = set(rows)
            rows = [i for i in layout if i in rs]
        head, tail = layout[: len(layout) - k], layout[len(layout) - k:]
        if tail == list(cols) and (head == list(rows) if exact else sorted(head) == sorted(rows)):
            return t, head
        new_layout = list(rows) + list(cols)
        strides, s = {}, 1
        for i in reversed(layout):
            strides[i] = s
            s *= self._extent(i, B)
        dims = [self._extent(i, B) for i in new_layout]
        st = [strides[i] for i in new_layout]
        if not dims:
            return t, []
        # complex pairs travel together when (re, im) is innermost on both sides
        vec = 2 if (dims[-1] == 2 and st[-1] == 1 and len(dims) > 1 and all(x % 2 == 0 for x in st[:-1])) else 1
        return self._permute(t, st, dims, vec, False), list(rows)

    # ---- node execution ----------------------------------------------------------------------
    def run(self, inputs: Dict[Tuple[str, object], torch.Tensor], B: int, nb: int, with_adjoint: bool,
            seed=None, on_grad_ready=None):
        """inputs: real-view tensors of the runner's dtype per input key (batched ones with the sample dimension
        first, nsamples = B * nb).  Returns (values dict, layouts dict).
        on_grad_ready(core key, flat real-view gradient): called as soon as a core's gradient is FINAL (all its
        contributions accumulated), in reverse-use order of the cores -- data-parallel training starts that core's
        all-reduce on a side stream there, under the rest of the reverse sweep (the reference reduces every core
        after the backward pass, tneq_qc/distributed/comm/comm_torch.py:292-318, 510-522)."""
        g = self.g
        NS = B * nb
        fire = {}
        if on_grad_ready is not None and with_adjoint:
            final_at = {}
            for pos, m in enumerate(g.nodes):
                final_at[m.id] = max(final_at.get(m.id, -1), pos)
                if m.acc_into >= 0:
                    final_at[m.acc_into] = max(final_at.get(m.acc_into, -1), pos)
            for key, nid in g.grads.items():
                fire.setdefault(final_at[nid], []).append((key, nid))
        val: Dict[int, torch.Tensor] = {}
        lay: Dict[int, List[int]] = {}
        # look-ahead: the indices a node's consumer will contract (so the producer can emit them
        # innermost and the consumer needs no permute of the big tensor)
        self._knext = {}
        for m in g.nodes:
            if m.kind == "contract" and (with_adjoint or m.role != "adj"):
                p_, q_ = g.nodes[m.p], g.nodes[m.q]
                sh = set(p_.idx) & set(q_.idx)
                self._knext.setdefault(p_.id, sh)
                self._knext.setdefault(q_.id, sh)

        for pos, n in enumerate(g.nodes):
            self._run_node(n, val, lay, inputs, NS, with_adjoint, seed)
            for key, nid in fire.get(pos, ()):
                on_grad_ready(key, val[nid])
        return val, lay

    def _run_node(self, n: Node, val, lay, inputs, NS, with_adjoint, seed):
        """Execute one node of the graph (values and layouts are recorded in val / lay)."""
        g = self.g
        if n.role == "adj" and not with_adjoint:
            return
        if n.kind == "input":
            key = (n.operand.kind, n.operand.key)
            if key[0] == "gradseed":     # d loss / d result: a tensor, or a callable of the forward result
                t = seed(val[g.result], lay[g.result]) if callable(seed) else seed
            else:
                t = inputs[key]
            val[n.id] = t
            lay[n.id] = ([BATCH] if n.batched else []) + list(n.idx)
            return
        if n.is_accum:
            val[n.id] = torch.zeros(tuple(g.dims[i] for i in n.idx) or (1,), dtype=self.dtype, device=self.device)
            lay[n.id] = list(n.idx)
            return
        if n.kind == "seed":
            raise NotImplementedError("fused loss is not part of the GEMM path (autograd route only)")
        if n.kind == "lin":
            out, out_layout = self._lin(n, val, lay, NS)
        else:
            if self._outer_acc(n, val, lay):
                return
            fused = self._fold_vec(n, val, lay)
            out, out_layout = fused if fused is not None else self._contract(n, val, lay, NS)
        if n.acc_into >= 0:
            # a contribution is declared in the target's memory order (its own labels: a core's
            # L and R occurrences carry different index ids over the same buffer)
            tgt = val[n.acc_into]
            if out_layout != list(n.idx):
                out, _ = self._arrange(out, out_layout, list(n.idx), [], NS, exact=True)
            tgt.add_(out.reshape(tgt.shape))
        else:
            val[n.id], lay[n.id] = out, out_layout

    def _lin(self, n: Node, val, lay, NS):
        g = self.g
        src = g.nodes[n.p]
        t, L = val[src.id], lay[src.id]
        lead = [BATCH] if n.batched else []
        strides, s = {}, 1
        for i in reversed(L):
            strides[i] = s
            s *= self._extent(i, NS)
        if n.lin_kind in ("permute", "conj"):
            target = lead + list(n.idx)
            dims = [self._extent(i, NS) for i in target]
            st = [strides[i] for i in target]
            conj = n.lin_kind == "conj"
            if conj and not (L and L[-1] == src.idx[-1] and target[-1] == n.idx[-1]):
                raise NotImplementedError("conjugation expects (re, im) innermost")
            vec = 2 if (dims[-1] == 2 and st[-1] == 1 and len(dims) > 1) else 1
            if conj and vec != 2:
                raise NotImplementedError("conjugation expects interleaved complex data")
            return self._permute(t, st, dims, vec, conj), target
        if n.lin_kind == "expand":
            ri, ro = n.idx[-2], n.idx[-1]
            if strides[src.idx[-1]] != 1:      # (re, im) must be adjacent in the source
                t, _ = self._arrange(t, L, [i for i in L if i != src.idx[-1]], [src.idx[-1]], NS)
                L = [i for i in L if i != src.idx[-1]] + [src.idx[-1]]
                strides, s = {}, 1
                for i in reversed(L):
                    strides[i] = s
                    s *= self._extent(i, NS)
            target = lead + list(n.idx)
            dims = [self._extent(i, NS) for i in target]
            st = [0 if i in (ri, ro) else strides[i] for i in target]
            out = torch.empty(tuple(dims), dtype=self.dtype, device=self.device)
            k = len(dims)
            _lib.check(self._entry("cplx_expand")(c_void_p(t.data_ptr()), c_void_p(out.data_ptr()), k,
                                                  (c_int64 * k)(*dims), (c_int64 * k)(*st), k - 2, k - 1, 0,
                                                  self._stream()))
            return out, target
        if n.lin_kind == "fold":
            # source: gradient of the expanded tensor, layout contains ri, ro somewhere
            ri, ro = src.idx[-2], src.idx[-1]
            target = lead + list(n.idx)
            dims = [self._extent(i, NS) for i in target]
            st = [strides[i] for i in target[:-1]] + [0]
            out = torch.empty(tuple(dims), dtype=self.dtype, device=self.device)
            k = len(dims)
            _lib.check(self._entry("cplx_fold")(c_void_p(t.data_ptr()), c_void_p(out.data_ptr()), k,
                                                (c_int64 * k)(*dims), (c_int64 * k)(*st), strides[ri], strides[ro],
                                                0, 0, self._stream()))
            return out, target
        raise NotImplementedError(f"lin kind {n.lin_kind!r} in the GEMM path")

    def _contract(self, n: Node, val, lay, NS):
        g = self.g
        p, q = g.nodes[n.p], g.nodes[n.q]
        tp, Lp = val[p.id], lay[p.id]
        tq, Lq = val[q.id], lay[q.id]
        shared = [i for i in p.idx if i in q.idx]
        pf = [i for i in p.idx if i not in shared]
        qf = [i for i in q.idx if i not in shared]
        if n.reduce_batch:
            # gradient of a shared tensor: the sample index joins the contracted indices (GEMM K)
            fused = self._reduce_in_place(tp, Lp, pf, tq, Lq, qf, shared, NS)
            if fused is not None:
                return fused
            korder = self._tail_order(Lp, [BATCH] + shared)
            A, rows_a = self._arrange(tp, Lp, pf, korder, NS)
            Bm, rows_b = self._arrange(tq, Lq, qf, korder, NS)
            M, N, K = self._size(pf, NS), self._size(qf, NS), self._size(korder, NS)
            C = torch.empty((M, N), dtype=self.dtype, device=self.device)
            self._gemm(A, Bm, C, M, N, K, K, K, N)
            out_layout = rows_a + rows_b
            return C.reshape([g.dims[i] for i in out_layout] or [1]), out_layout
        if q.batched and not p.batched:   # the batched operand provides the GEMM rows
            p, q, tp, Lp, tq, Lq, pf, qf = q, p, tq, Lq, tp, Lp, qf, pf
        lead = [BATCH] if p.batched else []
        korder = self._tail_order(Lp, shared)
        K = self._size(shared, NS)
        if not q.batched and not self.f64:
            # the A operand read in place through a 4-D tensor map when its memory order is [rows][k][rows][k]
            sv = self._strided_view(Lp, lead + pf, korder, NS)
            if sv is not None:
                view, rows_a = sv
                kn = self._knext.get(n.id, set())
                want_b = [i for i in qf if i not in kn] + [i for i in qf if i in kn]
                cur_b = [i for i in Lq if i in set(qf)]
                Bm, rows_b = self._arrange(tq, Lq, want_b, korder, NS, exact=(want_b != cur_b))
                M, N = self._size(rows_a, NS), self._size(rows_b, NS)
                C = torch.empty((M, N), dtype=self.dtype, device=self.device)
                if self._gemm_view(tp, view, Bm, C, N, K, N):
                    out_layout = rows_a + rows_b
                    return C.reshape([self._extent(i, NS) for i in out_layout] or [1]), out_layout
        A, rows_a = self._arrange(tp, Lp, lead + pf, korder, NS)
        if q.batched:
            # both per-sample: one GEMM per sample (batch in grid.z)
            Bm, rows_b = self._arrange(tq, Lq, [BATCH] + qf, korder, NS)
            assert rows_a[0] == BATCH and rows_b[0] == BATCH
            M, N = self._size(rows_a[1:], NS), self._size(rows_b[1:], NS)
            C = torch.empty((NS, M, N), dtype=self.dtype, device=self.device)
            for b0 in range(0, NS, 32768):
                nb_ = min(32768, NS - b0)
                self._gemm(A[b0:] if b0 else A, Bm[b0:] if b0 else Bm, C[b0:] if b0 else C, M, N, K, K, K, N,
                           batch=nb_, sA=M * K, sB=N * K, sC=M * N)
            out_layout = [BATCH] + rows_a[1:] + rows_b[1:]
        else:
            # order B's kept indices so that what the consumer contracts next ends up innermost in C
            kn = self._knext.get(n.id, set())
            want_b = [i for i in qf if i not in kn] + [i for i in qf if i in kn]
            cur_b = [i for i in Lq if i in set(qf)]
            Bm, rows_b = self._arrange(tq, Lq, want_b, korder, NS, exact=(want_b != cur_b))
            M, N = self._size(rows_a, NS), self._size(rows_b, NS)
            C = torch.empty((M, N), dtype=self.dtype, device=self.device)
            self._gemm(A, Bm, C, M, N, K, K, K, N)
            out_layout = rows_a + rows_b
        return C.reshape([self._extent(i, NS) for i in out_layout] or [1]), out_layout

    @staticmethod
    def _tail_order(layout, kset):
        """The contracted indices in the order they already have in `layout`."""
        ks = set(kset)
        return [i for i in layout if i in ks]
