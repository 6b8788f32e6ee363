"""B200Strategy: the contraction strategy whose compute function runs the whole
qubit sweep as hand-written sm_100a CUDA (libtneq_b200.so).

Plug-in contract (reference: tneq_qc/contractor/base.py:12-62, used by
tneq_qc/contractor/compiler.py:66-126 and tneq_qc/core/engine_siamese.py:261-554):

    strategy.get_compute_function(qctn, shapes_info, backend, right_qctn="symmetric")
        -> compute_fn(cores_dict, circuit_states, measure_matrices, right_cores_dict=None)

compute_fn has the semantics of GreedyStrategy.compute_fn
(tneq_qc/contractor/greedy_strategy.py:45-598):
  * cores / states / measurements may be torch tensors or TNTensors; if any
    operand is a TNTensor the result is TNTensor(raw, scale=prod scales,
    log_scale=sum log_scales) (greedy_strategy.py:913-952), the host floats being
    combined in exactly the reference's operand order;
  * measurements are (B,K,K) or (B,2,K,K); None leaves that qubit's edges open;
  * the result is differentiable w.r.t. the core tensors (torch.autograd);
  * errors are Python exceptions (ValueError / RuntimeError).
Extra, used by this repository's own engine: compute_fn.loss_and_grads(...) runs
forward + loss + reverse sweep as one fused device program.
"""
from __future__ import annotations

import math
import os
from typing import Any, Callable, Dict, List, Optional, Tuple

import torch

from .. import _lib as _lib_mod
from ..core.tn_tensor import TNTensor
from .base import ContractionStrategy
from .device_plan import DeviceProgram
from .plan import ContractionPlan, signature_of

_DTYPE_NAME = {torch.float32: "float32", torch.float64: "float64",
               torch.complex64: "complex64", torch.complex128: "complex128"}


# process-wide switch for CUDA-graph replay of the fused training step (see loss_and_grads below);
# also set by the environment variable TNQ_CUDA_GRAPHS=1
_GRAPHS = {"enabled": False}


def set_cuda_graphs(flag: bool = True) -> None:
    _GRAPHS["enabled"] = bool(flag)


def _is_tnt(x) -> bool:
    # duck-typed: the reference's own TNTensor class is accepted too (reference_plugin.py)
    return (not isinstance(x, torch.Tensor)) and hasattr(x, "tensor") and hasattr(x, "scale") and hasattr(x, "log_scale")


def _raw(x):
    return x.tensor if _is_tnt(x) else x


def _items(container, n):
    """qubit -> entry for the containers the reference accepts (None, dict, list, tuple)."""
    if container is None:
        return {}
    if isinstance(container, dict):
        return {q: container[q] for q in range(n) if q in container}
    return {q: container[q] for q in range(min(n, len(container)))}


class _capture:
    """`with torch.cuda.graph(g)` without its torch.cuda.empty_cache() / gc.collect() (9 ms per capture on B200 with a
    warm allocator -- a quarter of the host time of a 50-step candidate in the population benchmark): side stream,
    capture_begin / capture_end, a private memory pool per graph."""
    _streams: Dict[torch.device, torch.cuda.Stream] = {}

    def __init__(self, graph: torch.cuda.CUDAGraph, device: torch.device):
        self.graph, self.device = graph, device

    def __enter__(self):
        dev = self.device
        torch.cuda.synchronize(dev)
        st = _capture._streams.get(dev)
        if st is None:
            st = _capture._streams[dev] = torch.cuda.Stream(dev)
        st.wait_stream(torch.cuda.current_stream(dev))
        self._ctx = torch.cuda.stream(st)
        self._ctx.__enter__()
        try:
            self.graph.capture_begin(capture_error_mode="global")
        except BaseException:
            self._ctx.__exit__(None, None, None)
            raise
        return self

    def __exit__(self, *exc):
        try:
            self.graph.capture_end()
        finally:
            self._ctx.__exit__(*exc)
        return False


def _real_view(t: torch.Tensor) -> torch.Tensor:
    return torch.view_as_real(t) if t.is_complex() else t


# Cores bigger than this (real elements) do not fit the shared-memory VM: the sweep is then
# executed contraction by contraction on the tensor-core GEMM path (gemm_path.py), in the plan's dtype.
VM_MAX_CORE_ELEMS = 4096


class _Bound:
    """One plan bound to one device: lowered programs are created lazily."""

    def __init__(self, plan: ContractionPlan, device: torch.device):
        import os
        self.plan, self.device = plan, device
        self._dev: Dict[str, DeviceProgram] = {}
        self._gemm: Dict[str, object] = {}
        biggest = max(int(torch.tensor(s).prod()) for s in plan.core_shapes.values()) * (2 if plan.complex_mode else 1)
        self.use_gemm_path = biggest > VM_MAX_CORE_ELEMS or os.environ.get("TNQ_FORCE_GEMM_PATH") == "1"
        self.chain_rank = 0 if (self.use_gemm_path or os.environ.get("TNQ_NO_CHAIN") == "1") else plan.mps_chain_rank()
        self._chain_ws = None
        self._scale_prog = None
        # two-layer merged MPS: warp-level ladder kernel (csrc/tnq_ladder.cu)
        self.ladder, self._ladder_order, self._ladder_ws_bytes = None, None, {}
        if not (self.use_gemm_path or self.chain_rank or os.environ.get("TNQ_NO_CHAIN") == "1"):
            self.ladder = plan.mps_ladder()
        # float32 / complex64 plans compute in float32, float64 / complex128 plans in float64
        self.real_dtype = torch.float64 if plan.real_dtype == "f64" else torch.float32

    def scale_program(self):
        """[(tmp id produced, [(is_tmp, operand key)])] per greedy step, operands in einsum order."""
        if self._scale_prog is None:
            prog = []
            for step in self.plan.schedule.steps:
                ops = []
                for op in step.operands:
                    if op.kind == "tmp":
                        ops.append((True, op.key))
                    else:
                        ops.append((False, ("core", op.key) if op.kind == "core_conj" else (op.kind, op.key)))
                prog.append((step.out, ops))
            self._scale_prog = prog
        return self._scale_prog

    def ones(self, elems: int, real_dtype) -> torch.Tensor:
        """A vector of ones in the plan's real representation (complex: interleaved (1, 0) pairs): the
        partner of an edge that einsum sums over on its own (cgraph.build_forward)."""
        dt = {"f32": torch.float32, "f64": torch.float64}.get(real_dtype, real_dtype)
        key = (int(elems), dt)
        cache = self.__dict__.setdefault("_ones", {})
        if key not in cache:
            if self.plan.complex_mode:
                t = torch.zeros(elems // 2, 2, dtype=dt, device=self.device)
                t[:, 0] = 1.0
                cache[key] = t.reshape(-1)
            else:
                cache[key] = torch.ones(elems, dtype=dt, device=self.device)
        return cache[key]

    def gemm_runner(self, mode: str):
        from .gemm_path import GemmPathRunner
        if mode not in self._gemm:
            self._gemm[mode] = GemmPathRunner(self.plan.graph(mode), self.device, self.real_dtype)
        return self._gemm[mode]

    def program(self, mode: str) -> DeviceProgram:
        if mode not in self._dev:
            self._dev[mode] = DeviceProgram(self.plan.program(mode), self.device)
        return self._dev[mode]


class _SweepFn(torch.autograd.Function):
    """forward: 'fwd' program; backward: 'bwd' program (forward recomputation + reverse sweep
    in one launch, nothing but the inputs is kept alive between the two)."""

    @staticmethod
    def forward(ctx, call, *cores):
        ctx.call = call
        ctx.save_for_backward(*cores)
        return call.forward(cores)

    @staticmethod
    def backward(ctx, grad_out):
        grads = ctx.call.backward(ctx.saved_tensors, grad_out)
        return (None,) + tuple(g if need else None for g, need in zip(grads, ctx.needs_input_grad[1:]))


class _Call:
    """Everything about one invocation except the core tensors."""

    def __init__(self, bound: _Bound, core_keys, states, mxs, B, dtype):
        self.bound, self.core_keys, self.states, self.mxs, self.B, self.dtype = bound, core_keys, states, mxs, B, dtype
        self.nb = bound.plan.nb
        self.nsamples = B * self.nb

    def _inputs(self, prog: DeviceProgram, cores, seed=None):
        out = []
        by_key = dict(zip(self.core_keys, cores))
        for slot in prog.prog.inputs:
            kind, key = slot.key
            if kind in ("core", "rcore"):
                t = _real_view(by_key[(kind, key)].detach().contiguous())
                out.append((t, 0, 0))
            elif kind == "state":
                out.append((_real_view(self.states[key].detach().contiguous()), 0, 0))
            elif kind == "ones":                 # partner of an edge that einsum sums over on its own
                out.append((self.bound.ones(slot.elems, prog.real_dtype), 0, 0))
            elif kind == "mx":
                m = self.mxs[key].detach()
                inner = m.shape[-2] * m.shape[-1]
                if m.stride(-1) != 1 or m.stride(-2) != m.shape[-1]:
                    m = m.contiguous()
                mul = 2 if m.is_complex() else 1
                if m.dim() == 4:
                    hi, lo = m.stride(0) * mul, m.stride(1) * mul
                else:
                    hi, lo = m.stride(0) * mul, 0
                if m.shape[0] == 1 and self.B != 1:
                    hi = 0
                out.append((_real_view(m), hi, lo))
                assert slot.elems == inner * mul
            elif kind == "gradseed":
                out.append((seed, slot.elems * self.nb, slot.elems))
            else:
                raise RuntimeError(f"unknown input slot {slot.key}")
        return out

    def _shape_result(self, flat: torch.Tensor) -> torch.Tensor:
        g = self.bound.plan.graph("fwd")
        res = g.nodes[g.result]
        body = [g.dims[i] for i in (res.idx[:-1] if res.cplx else res.idx)]
        lead = [self.B] + ([2] if self.nb == 2 else [])
        if res.cplx:
            return torch.view_as_complex(flat.reshape(lead + body + [2]))
        return flat.reshape(lead + body)

    # ---- single-layer MPS route: register-resident chain kernel (csrc/tnq_chain.cu) -----------
    def _chain(self, cores, mode, seed=None, log_scale=0.0, private_ws=False):
        import ctypes
        from ctypes import c_void_p, c_int64
        from .. import _lib
        lib = _lib.load()
        K, n, dev = self.bound.chain_rank, self.bound.plan.nqubits, self.bound.device
        by_key = dict(zip(self.core_keys, cores))
        order = [k for k in self.bound.plan.core_shapes]                   # ('core', name) in qctn.cores order
        cs = [c if c.is_contiguous() else c.contiguous() for c in (by_key[k] for k in order)]
        sts = [t if t.is_contiguous() else t.contiguous() for t in (self.states[q] for q in range(n))]
        ms, strides = [], []
        for q in range(n):
            m = self.mxs[q]
            st = m.stride()
            if st[-1] != 1 or st[-2] != K:
                m = m.contiguous()
                st = m.stride()
            ms.append(m)
            strides.append(0 if (m.shape[0] == 1 and self.B != 1) else st[0])
        ws_bytes = int(lib.tnq_mps_chain_workspace_bytes(K, n, self.B))
        if private_ws:                  # captured into a CUDA graph: the graph owns its scratch
            ws = self._keep = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        else:
            if self.bound._chain_ws is None or self.bound._chain_ws.numel() < ws_bytes:
                self.bound._chain_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            ws = self.bound._chain_ws
        values = torch.empty(self.B, dtype=torch.float32, device=dev) if mode != 2 else None
        loss = torch.empty(1, dtype=torch.float32, device=dev) if mode == 1 else None
        grads = [torch.empty_like(c) for c in cs] if mode != 0 else []
        arr = lambda ts: (c_void_p * max(1, len(ts)))(*[t.data_ptr() for t in ts])
        with torch.cuda.device(dev):
            _lib.check(lib.tnq_mps_chain(K, n, arr(cs), arr(sts), arr(ms), (c_int64 * n)(*strides), self.B, mode,
                                         c_void_p(seed.data_ptr()) if seed is not None else None,
                                         c_void_p(values.data_ptr()) if values is not None else None,
                                         c_void_p(loss.data_ptr()) if loss is not None else None,
                                         arr(grads) if grads else None, float(log_scale),
                                         c_void_p(ws.data_ptr()), ws.numel(),
                                         c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        gmap = dict(zip(order, grads))
        return values, (loss[0] if loss is not None else None), [gmap[k] for k in self.core_keys] if grads else []

    # ---- two-layer merged MPS route: warp-level ladder kernel (csrc/tnq_ladder.cu) -------------
    def _ladder(self, cores, mode, seed=None, log_scale=0.0, private_ws=False):
        from ctypes import c_void_p, c_int64
        from .. import _lib
        lib = _lib.load()
        bound = self.bound
        K, layer1, layer2 = bound.ladder
        n, dev, B = bound.plan.nqubits, bound.device, self.B
        order = bound._ladder_order
        if order is None or order[0] != self.core_keys:
            pos = {k: i for i, k in enumerate(self.core_keys)}
            order = bound._ladder_order = (list(self.core_keys), [pos[("core", k)] for k in layer1],
                                           [pos[("core", k)] for k in layer2])
        _, ia, ix = order
        cores = [c if c.is_contiguous() else c.contiguous() for c in cores]
        sts = [self.states[q] for q in range(n)]
        sts = [t if t.is_contiguous() else t.contiguous() for t in sts]
        ms, strides = [], []
        for q in range(n):
            m = self.mxs[q]
            st = m.stride()
            if st[2] != 1 or st[1] != K:
                m = m.contiguous()
                st = m.stride()
            ms.append(m)
            strides.append(0 if (m.shape[0] == 1 and B != 1) else st[0])
        key = (B, mode)
        ws_bytes = bound._ladder_ws_bytes.get(key)
        if ws_bytes is None:
            ws_bytes = bound._ladder_ws_bytes[key] = int(lib.tnq_mps_ladder_workspace_bytes(K, n, B, mode))
        if private_ws:                  # captured into a CUDA graph: the graph owns its scratch
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        else:
            if bound._chain_ws is None or bound._chain_ws.numel() < ws_bytes:
                bound._chain_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            ws = bound._chain_ws
        values = torch.empty(B, dtype=torch.float32, device=dev) if mode != 2 else None
        loss = torch.empty(1, dtype=torch.float32, device=dev) if mode == 1 else None
        ptr = [c.data_ptr() for c in cores]
        nc, K4 = len(cores), K ** 4
        if mode != 0:
            # one allocation for all core gradients, handed out as views in the caller's core order
            flat = torch.empty(nc * K4, dtype=torch.float32, device=dev)
            g0 = flat.data_ptr()
            ga = (c_void_p * (n - 1))(*[g0 + 4 * K4 * i for i in ia])
            gx = (c_void_p * (n - 1))(*[g0 + 4 * K4 * i for i in ix])
        else:
            flat = ga = gx = None
        ca = (c_void_p * (n - 1))(*[ptr[i] for i in ia])
        cx = (c_void_p * (n - 1))(*[ptr[i] for i in ix])
        with torch.cuda.device(dev):
            _lib.check(lib.tnq_mps_ladder(K, n, ca, cx, (c_void_p * n)(*[t.data_ptr() for t in sts]),
                                          (c_void_p * n)(*[t.data_ptr() for t in ms]), (c_int64 * n)(*strides), B, mode,
                                          seed.data_ptr() if seed is not None else None,
                                          values.data_ptr() if values is not None else None,
                                          loss.data_ptr() if loss is not None else None, ga, gx, float(log_scale),
                                          ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
        grads = list(flat.view(nc, K, K, K, K).unbind(0)) if flat is not None else []
        if private_ws:
            self._keep = ws
        return values, (loss[0] if loss is not None else None), grads

    # ---- large-bond route: node-by-node on the tcgen05 GEMM path ------------------------------
    def _gemm_inputs(self, cores):
        out = {}
        for key, c in zip(self.core_keys, cores):
            out[key] = _real_view(c.detach().contiguous())
        for q, s_ in self.states.items():
            out[("state", q)] = _real_view(s_.detach().contiguous())
        g = self.bound.gemm_runner("fwd").g
        for key, ids in g.inputs.items():
            if key[0] == "ones":
                out[key] = self.bound.ones(g.size(g.nodes[ids[0]].idx), self.bound.real_dtype)
        for q, m in self.mxs.items():
            m = m.detach()
            if m.shape[0] == 1 and self.B != 1:
                m = m.expand(self.B, *m.shape[1:])
            if self.nb == 2 and m.dim() == 3:
                m = m.unsqueeze(1).expand(-1, 2, -1, -1)
            out[("mx", q)] = _real_view(m.contiguous()).reshape(self.nsamples, -1)
        return out

    def _gemm_forward(self, cores):
        r = self.bound.gemm_runner("fwd")
        val, lay = r.run(self._gemm_inputs(cores), self.B, self.nb, with_adjoint=False)
        return self._shape_result(val[r.g.result].reshape(self.nsamples, -1))

    def _gemm_backward(self, cores, seed):
        r = self.bound.gemm_runner("bwd")
        hook = getattr(self.bound, "grad_hook", None)
        ready = None
        if hook is not None:
            names = {key: key[1] for key in self.core_keys}
            ready = lambda key, flat: hook(names.get(key, key), flat)
        val, lay = r.run(self._gemm_inputs(cores), self.B, self.nb, with_adjoint=True, seed=seed, on_grad_ready=ready)
        grads = []
        for key, c in zip(self.core_keys, cores):
            gflat = val[r.g.grads[key]]
            grads.append(torch.view_as_complex(gflat.reshape(tuple(c.shape) + (2,))) if c.is_complex()
                         else gflat.reshape(c.shape))
        return grads, val[r.g.result]

    def forward(self, cores, private_ws: bool = False):
        if self.bound.chain_rank:
            return self._chain(cores, 0, private_ws=private_ws)[0]
        if self.bound.ladder:
            return self._ladder(cores, 0, private_ws=private_ws)[0]
        if self.bound.use_gemm_path:
            return self._gemm_forward(cores)
        prog = self.bound.program("fwd")
        (flat,) = prog.run(self.nsamples, self._inputs(prog, cores))
        return self._shape_result(flat)

    def backward(self, cores, grad_out):
        if self.bound.chain_rank:
            return self._chain(cores, 2, seed=grad_out.reshape(-1).to(torch.float32).contiguous())[2]
        if self.bound.ladder:
            return self._ladder(cores, 2, seed=grad_out.reshape(-1).to(torch.float32).contiguous())[2]
        if self.bound.use_gemm_path:
            seed = _real_view(grad_out.contiguous()).reshape(self.nsamples, -1).to(self.bound.real_dtype).contiguous()
            return self._gemm_backward(cores, seed)[0]
        prog = self.bound.program("bwd")
        seed = _real_view(grad_out.contiguous()).reshape(self.nsamples, -1).to(prog.real_dtype).contiguous()
        outs = prog.run(self.nsamples, self._inputs(prog, cores, seed=seed))
        return self._grads(prog, outs, cores)

    def _grads(self, prog, outs, cores):
        grads = []
        for key, c in zip(self.core_keys, cores):
            gflat = outs[prog.prog.output_index(("grad",) + key)]
            if c.is_complex():
                grads.append(torch.view_as_complex(gflat.reshape(tuple(c.shape) + (2,))))
            else:
                grads.append(gflat.reshape(c.shape))
        return grads

    def graphable(self) -> bool:
        """Routes whose forward / training step is a fixed set of launches on caller-owned pointers."""
        return bool(self.bound.ladder) or bool(self.bound.chain_rank)

    def train(self, cores, log_scale: float, private_ws: bool = False):
        """Fused forward + loss + reverse sweep.  Returns (loss, grads, values)."""
        if self.bound.chain_rank:
            values, loss, grads = self._chain(cores, 1, log_scale=log_scale, private_ws=private_ws)
            return loss, grads, values
        if self.bound.ladder:
            values, loss, grads = self._ladder(cores, 1, log_scale=log_scale, private_ws=private_ws)
            return loss, grads, values
        if self.bound.use_gemm_path:
            # forward nodes, then the loss seed from the forward result (element-wise, torch), then the
            # adjoint nodes -- one walk over the graph
            box = {}
            inv = 1.0 / self.nsamples

            def seed_fn(res, layout):
                # in the plan's real dtype (the forward result's): float64 plans seed the reverse sweep in float64
                flat = res.reshape(self.nsamples, -1)
                if flat.shape[1] == 2 and self.bound.plan.complex_mode:
                    val = flat[:, 0] * flat[:, 0] + flat[:, 1] * flat[:, 1]
                else:
                    val = flat[:, 0]
                clamped = torch.clamp(val, min=1e-10)
                box["loss"] = -(torch.log(clamped) + log_scale).sum() * inv
                dval = torch.where(val >= 1e-10, -inv / clamped, torch.zeros_like(val))
                if flat.shape[1] == 2 and self.bound.plan.complex_mode:
                    return (flat * (2.0 * dval)[:, None]).contiguous()
                return dval[:, None].contiguous()

            grads, res = self._gemm_backward(cores, seed_fn)
            return box["loss"], grads, self._shape_result(res.reshape(self.nsamples, -1))
        prog = self.bound.program("train")
        outs = prog.run(self.nsamples, self._inputs(prog, cores), scalars=(log_scale, 1.0 / self.nsamples),
                        one_buffer=True)
        loss = outs[prog.prog.output_index(("loss", 0))][0]
        values = self._shape_result(outs[prog.prog.output_index(("result", 0))])
        return loss, self._grads(prog, outs, cores), values


class B200Strategy(ContractionStrategy):
    """Whole-sweep CUDA contraction; registered for modes 'balanced' and 'full'."""

    # class of the TNTensor results; reference_plugin.register() substitutes the reference's own
    # class so that the isinstance checks of its EngineSiamese (engine_siamese.py:332,476) hold
    tntensor_cls = TNTensor

    def check_compatibility(self, qctn, shapes_info: Dict[str, Any]) -> bool:
        # Inside the reference (reference_plugin.register) this strategy shares the registry with
        # GreedyStrategy: a network that lives on another backend (the reference's own 'pytorch' CPU
        # backend) stays with the reference's strategies -- there is no CPU path here.
        name = getattr(getattr(qctn, "backend", None), "get_backend_name", None)
        return name is None or name() == "b200"

    def estimate_cost(self, qctn, shapes_info: Dict[str, Any]) -> float:
        # below GreedyStrategy's fixed 5e5 (greedy_strategy.py:602-608) so that
        # StrategyCompiler.compile (compiler.py:123) picks this strategy
        return 1e5

    @property
    def name(self) -> str:
        return "b200"

    def get_compute_function(self, qctn, shapes_info: Dict[str, Any], backend, right_qctn="symmetric") -> Callable:
        plans: Dict[Any, _Bound] = {}
        hooks = {"grad_ready": None}          # set_grad_ready_hook
        tnt_cls = self.tntensor_cls
        nq = qctn.nqubits
        table = qctn.adjacency_table
        core_names = list(qctn.cores)
        if right_qctn is None or (isinstance(right_qctn, str) and right_qctn == "symmetric"):
            right_mode, right_table, right_names = right_qctn, None, []
        elif hasattr(right_qctn, "adjacency_table"):
            right_mode, right_table, right_names = "qctn", right_qctn.adjacency_table, list(right_qctn.cores)
        else:
            raise ValueError("Invalid right_qctn parameter.")

        core_keys = [("core", k) for k in core_names] + [("rcore", k) for k in right_names]

        def prepare(cores_dict, circuit_states, measure_matrices, right_cores_dict):
            """-> (call, raw core tensors, per-operand scale bookkeeping).  This runs on every call:
            one pass over the operands, everything else is cached per operand signature."""
            T = torch.Tensor
            tnt: Dict[Any, Any] = {}              # operands that arrived as TNTensors
            cores = []
            for k in core_names:
                v = cores_dict[k]
                if not isinstance(v, T):
                    if _is_tnt(v):
                        tnt[("core", k)] = v
                        v = v.tensor
                cores.append(v)
            if right_mode == "qctn":
                for k in right_names:
                    v = right_cores_dict[k]
                    if not isinstance(v, T):
                        if _is_tnt(v):
                            tnt[("rcore", k)] = v
                            v = v.tensor
                    cores.append(v)
            if not cores:
                raise RuntimeError("No tensor left after contraction")
            states_w, mxs_w = _items(circuit_states, nq), _items(measure_matrices, nq)
            states, mxs = {}, {}
            for q, v in states_w.items():
                if not isinstance(v, T):
                    if _is_tnt(v):
                        tnt[("state", q)] = v
                        v = v.tensor
                states[q] = v
            for q, v in mxs_w.items():
                if v is None:
                    continue
                if not isinstance(v, T):
                    if _is_tnt(v):
                        tnt[("mx", q)] = v
                        v = v.tensor
                mxs[q] = v
            dtypes = {t.dtype for t in cores}
            dtypes.update(t.dtype for t in states.values())
            dtypes.update(t.dtype for t in mxs.values())
            dtype = cores[0].dtype
            if len(dtypes) > 1:
                for t in list(states.values()) + list(mxs.values()) + cores[1:]:
                    dtype = torch.promote_types(dtype, t.dtype)
            if dtype not in _DTYPE_NAME:
                raise ValueError(f"unsupported dtype {dtype}")
            device = cores[0].device
            if device.type != "cuda":
                raise RuntimeError("B200Strategy needs CUDA tensors: tneq_b200 has no CPU fallback")
            if len(dtypes) > 1 or any(t.device != device for t in cores) or \
                    any(t.device != device for t in states.values()) or any(t.device != device for t in mxs.values()):
                conv = lambda t: t if (t.device == device and t.dtype == dtype) else t.to(device=device, dtype=dtype)
                cores = [conv(t) for t in cores]
                states = {q: conv(t) for q, t in states.items()}
                mxs = {q: conv(t) for q, t in mxs.items()}
            for q, s_ in states.items():
                if s_.dim() != 1:
                    raise ValueError(f"circuit state of qubit {q} must be 1-D (got shape {tuple(s_.shape)}); "
                                     "batched circuit states are not supported by the greedy contraction")
            B = None
            mx_sig = []
            for q, m in mxs.items():
                nd, shp = m.dim(), m.shape
                if nd not in (3, 4) or (nd == 4 and shp[1] != 2):
                    raise ValueError(f"measurement of qubit {q} must be (B,K,K) or (B,2,K,K), got {tuple(shp)}")
                if shp[0] != 1:
                    if B is not None and B != shp[0]:
                        raise ValueError("measurement matrices disagree on the batch size")
                    B = shp[0]
                mx_sig.append((q, nd, shp[-2], shp[-1]))
            if B is None:
                B = 1
            key = (tuple((q, t.shape[0]) for q, t in states.items()), tuple(mx_sig), dtype, device)
            bound = plans.get(key)
            if bound is None:
                state_dims, mx_info = signature_of(nq, states_w, {q: mxs_w.get(q) for q in range(nq)})
                shapes = {k: tuple(t.shape) for k, t in zip(core_names, cores)}
                rshapes = {k: tuple(t.shape) for k, t in zip(right_names, cores[len(core_names):])}
                plan = ContractionPlan(table, nq, shapes, state_dims, mx_info, _DTYPE_NAME[dtype], right=right_mode,
                                       right_table=right_table, right_core_shapes=rshapes)
                bound = plans[key] = _Bound(plan, device)
            bound.grad_hook = hooks["grad_ready"]
            call = _Call(bound, core_keys, states, mxs, B, dtype)
            return call, cores, _scale_of(bound, tnt)

        def compute_fn(cores_dict, circuit_states, measure_matrices, right_cores_dict=None):
            if (graphs["enabled"] or _GRAPHS["enabled"]) and right_mode != "qctn" and not torch.is_grad_enabled():
                hit = _forward_graph(cores_dict, circuit_states, measure_matrices)
                if hit is not None:
                    res, scale = hit
                    return tnt_cls(res, scale=scale[0], log_scale=scale[1]) if scale is not None else res
            call, cores, scale = prepare(cores_dict, circuit_states, measure_matrices, right_cores_dict)
            if torch.is_grad_enabled() and any(c.requires_grad for c in cores):
                res = _SweepFn.apply(call, *cores)
            else:
                res = call.forward(cores)
            if scale is not None:
                return tnt_cls(res, scale=scale[0], log_scale=scale[1])
            return res

        def _forward_graph(cores_dict, circuit_states, measure_matrices):
            """Replay (or, for operands seen before, capture) the forward launches of this operand set.
            Returns (values, scale) or None (not graphable / first sighting): the caller then launches
            directly.  The returned tensor is the graph's output buffer (same contract as the training
            step below)."""
            key, tnts = _raw_ptrs(cores_dict, circuit_states, measure_matrices)
            key = ("fwd",) + key
            ent = graphs["entries"].get(key)
            if ent is not None:
                bound, graph, values, _call, nk = ent
                graph.replay()
                graphs["replays"] += 1
                _lib_mod.add_graph_launches(nk)
                return values, _scale_of(bound, dict(tnts))
            if not graphs["seen"].get(key) or graphs["captures"] >= graphs["max_captures"]:
                if len(graphs["seen"]) > 64:
                    graphs["seen"].clear()
                graphs["seen"][key] = True
                return None
            call, cores, scale = prepare(cores_dict, circuit_states, measure_matrices, None)
            if not (call.graphable() and _captures_callers_buffers(key[1:], call, cores)):
                return None
            dev = cores[0].device
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            n0 = _lib_mod.launch_count()
            with _capture(graph, dev):
                values = call.forward(cores, private_ws=True)
            nk = _lib_mod.launch_count() - n0
            graphs["captures"] += 1
            graph.replay()
            if len(graphs["entries"]) >= graphs["max"]:
                graphs["entries"].pop(next(iter(graphs["entries"])))
            graphs["entries"][key] = (call.bound, graph, values, call, nk)
            return values, scale

        # ---- CUDA-graph replay of the fused training step (opt-in) ---------------------------------
        # A training loop calls loss_and_grads with the SAME device buffers step after step (cores are
        # updated in place, batches are copied into static input buffers).  With graphs enabled, the
        # second call that presents the same pointers captures the step's launches into a CUDA graph
        # and later calls replay it: one cudaGraphLaunch instead of ~0.5 ms of per-call Python.
        # Contract: the returned loss / gradient / value tensors of a replayed step are the graph's
        # own output buffers -- they are overwritten by the next replay with the same operands.
        # Capturing costs milliseconds, so it is rationed: a key must have been seen before, and a
        # compute function captures at most `max_captures` graphs in its life (callers that allocate
        # fresh input tensors every step present ever-changing pointers and simply stay on the direct
        # path).
        graphs = {"enabled": os.environ.get("TNQ_CUDA_GRAPHS") == "1", "seen": {}, "entries": {}, "max": 4,
                  "replays": 0, "captures": 0, "max_captures": 8, "epilogue": None, "last_extra": None, "memo": {}}

        def _raw_ptrs(cores_dict, circuit_states, measure_matrices):
            """Identity of the operand buffers: address, dtype, shape and strides of every operand
            (a graph bakes all of them in).  A training / serving loop presents the SAME tensor objects step
            after step (possibly inside fresh containers and fresh TNTensor wrappers): the raw tensors are
            collected (one pass), looked up by their object ids, and if every one `is` the tensor seen last time
            the stored key is reused -- ~100 identity checks instead of ~100 data_ptr() / stride() calls.
            Contract (as for graph replay in general): tensors are updated in place, not re-pointed with
            `.data =` / `set_()`."""
            T = torch.Tensor
            raws, tnts = [], []
            for k in core_names:
                v = cores_dict[k]
                if not isinstance(v, T):
                    tnts.append((("core", k), v))
                    v = v.tensor
                raws.append(v)
            for q, v in _items(circuit_states, nq).items():
                if not isinstance(v, T):
                    tnts.append((("state", q), v))
                    v = v.tensor
                raws.append(v)
            for q, v in _items(measure_matrices, nq).items():
                if v is not None and not isinstance(v, T):
                    tnts.append((("mx", q), v))
                    v = v.tensor
                raws.append(v)
            ids = tuple(map(id, raws))
            memo = graphs["memo"].get(ids)
            if memo is not None and all(a is b for a, b in zip(raws, memo[0])):
                return memo[1], tnts
            key = tuple(0 if v is None else (v.data_ptr(), v.dtype, v.shape, v.stride()) for v in raws)
            if len(graphs["memo"]) > 16:
                graphs["memo"].clear()
            graphs["memo"][ids] = (raws, key)
            return key, tnts

        def _captures_callers_buffers(key, call, cores):
            """True when the launches would read exactly the caller's buffers: prepare() converted
            nothing (device, dtype) and the route will not make contiguous copies.  Otherwise the
            graph would bake in the addresses of temporaries that are freed after the capture."""
            seen = {e[0] for e in key if e != 0}
            for t in list(cores) + list(call.states.values()) + list(call.mxs.values()):
                if t.data_ptr() not in seen:
                    return False
            if any(not c.is_contiguous() for c in cores) or any(not t.is_contiguous() for t in call.states.values()):
                return False
            for m in call.mxs.values():
                st = m.stride()
                if st[-1] != 1 or st[-2] != m.shape[-1]:
                    return False
            return True

        def _scale_of(bound, tnt):
            if not tnt:
                return None
            tmp = {}
            for out, ops in bound.scale_program():
                sc = ls = None
                for is_tmp, okey in ops:
                    if is_tmp:
                        pair = tmp[okey]
                        if pair is None:
                            continue
                        s0, l0 = pair
                    else:
                        w = tnt.get(okey)
                        if w is None:
                            continue
                        s0, l0 = w.scale, w.log_scale
                    sc = s0 if sc is None else sc * s0
                    ls = l0 if ls is None else ls + l0
                tmp[out] = None if sc is None else (sc, ls)
            return tmp[bound.plan.schedule.result.key]

        def loss_and_grads(cores_dict, circuit_states, measure_matrices, right_cores_dict=None):
            """Fused -mean(log(clamp(value,1e-10)) + log_scale) and its core gradients
            (engine_siamese.py:441-554), one device program."""
            if (graphs["enabled"] or _GRAPHS["enabled"]) and right_mode != "qctn":
                key, tnts = _raw_ptrs(cores_dict, circuit_states, measure_matrices)
                ent = graphs["entries"].get(key)
                graphs["last_extra"] = None
                if ent is not None:
                    bound, graph, loss0, grads, values, _call, nk, extra = ent
                    scale = _scale_of(bound, dict(tnts))
                    graph.replay()
                    graphs["replays"] += 1
                    graphs["last_extra"] = extra
                    _lib_mod.add_graph_launches(nk)
                    # the captured kernel runs with log_scale = 0: the loss is affine in it
                    loss = loss0 - float(scale[1]) if scale is not None else loss0
                    return loss, grads, values, scale
                if graphs["seen"].get(key) and graphs["captures"] < graphs["max_captures"]:
                    call, cores, scale = prepare(cores_dict, circuit_states, measure_matrices, right_cores_dict)
                    if call.graphable() and all(not c.requires_grad or c.is_leaf for c in cores) \
                            and _captures_callers_buffers(key, call, cores):
                        dev = cores[0].device
                        torch.cuda.synchronize(dev)
                        graph = torch.cuda.CUDAGraph()
                        n0 = _lib_mod.launch_count()
                        with _capture(graph, dev):
                            loss0, grads, values = call.train(cores, 0.0, private_ws=True)
                            # e.g. the gradient exchange of data-parallel training (set_graph_epilogue below):
                            # recorded into the same graph, so that a step is ONE graph launch
                            extra = graphs["epilogue"](loss0, grads) if graphs["epilogue"] is not None else None
                        nk = _lib_mod.launch_count() - n0      # kernels recorded into the graph
                        graphs["captures"] += 1
                        graph.replay()
                        graphs["last_extra"] = extra
                        if len(graphs["entries"]) >= graphs["max"]:
                            graphs["entries"].pop(next(iter(graphs["entries"])))
                        graphs["entries"][key] = (call.bound, graph, loss0, grads, values, call, nk, extra)
                        loss = loss0 - float(scale[1]) if scale is not None else loss0
                        return loss, grads, values, scale
                else:
                    if len(graphs["seen"]) > 64:
                        graphs["seen"].clear()
                    graphs["seen"][key] = True
            call, cores, scale = prepare(cores_dict, circuit_states, measure_matrices, right_cores_dict)
            loss, grads, values = call.train(cores, 0.0 if scale is None else float(scale[1]))
            return loss, grads, values, scale

        def enable_cuda_graphs(flag: bool = True):
            graphs["enabled"] = bool(flag)
            if not flag:
                graphs["entries"].clear()
                graphs["seen"].clear()

        def set_grad_ready_hook(fn_or_none):
            """fn(core name, flat real view of that core's gradient in the plan's real dtype -- float32, or float64 for
            float64 / complex128 networks), called DURING the reverse sweep of the
            large-bond route as soon as the gradient of a core is final (reverse-use order): data-parallel training
            starts the core's all-reduce on a side stream there, so that the exchange of the GB-sized gradients runs
            under the rest of the sweep (bench.py --workload cfg4 --gpus N).  The fused small-bond kernels produce all
            gradients at once (one 15 KB exchange, set_graph_epilogue); None removes the hook."""
            hooks["grad_ready"] = fn_or_none
            for b in plans.values():
                b.grad_hook = fn_or_none

        def set_graph_epilogue(fn_or_none):
            """fn(loss0, grads) -> anything, called INSIDE the capture of the fused training step, right after
            its launches (data-parallel training records its gradient exchange there).  After every call of
            loss_and_grads, graph_stats['last_extra'] holds what fn returned if that call ran the graph
            (capture or replay) and None if it launched directly -- the caller then runs the exchange itself.
            The captured loss is the kernel's (log_scale = 0): fn sees that one."""
            graphs["epilogue"] = fn_or_none
            graphs["entries"] = {k: v for k, v in graphs["entries"].items() if k and k[0] == "fwd"}
            graphs["last_extra"] = None

        def forward_from_x(cores_dict, circuit_states, x, weights):
            """Opt-in fusion of EngineSiamese.generate_data into the sweep (SURVEY 8f2): per-sample values for
            measurement matrices phi(x) phi(x)^T generated in registers (tnq_mps_chain_x).  x: (B, n) float32 on
            the device, weights: the K Hermite weights.  Returns (values, scale[n]) with the TNTensor convention of
            generate_data(ret_type='TNTensor') -- true value = values * prod(scale) -- or None when this network /
            these operands are not on the single-layer MPS route (the caller then materialises the matrices)."""
            from ctypes import c_void_p, c_float
            K = len(weights)
            if right_mode == "qctn" or x.dim() != 2 or x.shape[1] != nq or x.dtype != torch.float32 or not x.is_cuda:
                return None
            states_w = _items(circuit_states, nq)
            cores = [cores_dict[k] for k in core_names]
            cores = [c.tensor if _is_tnt(c) else c for c in cores]
            states = {q: (v.tensor if _is_tnt(v) else v) for q, v in states_w.items()}
            if len(states) != nq or any(t.dtype != torch.float32 or t.device != x.device for t in cores) or \
                    any(t.dtype != torch.float32 or t.device != x.device or t.dim() != 1 for t in states.values()):
                return None
            B = x.shape[0]
            device = x.device
            key = (tuple((q, t.shape[0]) for q, t in states.items()), tuple((q, 3, K, K) for q in range(nq)),
                   torch.float32, device)
            bound = plans.get(key)
            if bound is None:
                state_dims = {q: int(t.shape[0]) for q, t in states.items()}
                mx_info = {q: ("a", K, K) for q in range(nq)}
                shapes = {k: tuple(t.shape) for k, t in zip(core_names, cores)}
                plan = ContractionPlan(table, nq, shapes, state_dims, mx_info, "float32", right=right_mode)
                bound = plans[key] = _Bound(plan, device)
            if bound.chain_rank != K:
                return None
            lib = _lib_mod.load()
            order = [k[1] for k in bound.plan.core_shapes]
            by_name = dict(zip(core_names, cores))
            cs = [by_name[k].contiguous() for k in order]
            sts = [states[q].contiguous() for q in range(nq)]
            values = torch.empty(B, dtype=torch.float32, device=device)
            scale = torch.empty(nq, dtype=torch.float32, device=device)
            arr = lambda ts: (c_void_p * len(ts))(*[t.data_ptr() for t in ts])
            with torch.cuda.device(device):
                _lib_mod.check(lib.tnq_mps_chain_x(K, nq, arr(cs), arr(sts), c_void_p(x.data_ptr()), x.stride(0), x.stride(1),
                                                   (c_float * K)(*[float(w) for w in weights]), B,
                                                   c_void_p(scale.data_ptr()), c_void_p(values.data_ptr()),
                                                   c_void_p(torch.cuda.current_stream(device).cuda_stream)))
            return values, scale

        def sample_prefix(cores_dict, circuit_states, grid_x, mx_grid, u, weights):
            """sample() with prefix environments (SURVEY 8f3, tnq_mps_chain_sample): grid_x (G,), mx_grid (G,K,K) =
            generate_data(grid_x), u (S, n) uniform numbers in the reference's draw order, weights: the K Hermite
            weights.  Returns samples (S, n), or None when this network / these operands are not on the single-layer
            MPS route (the caller then takes the contraction-based procedure)."""
            from ctypes import c_void_p, c_float
            K = len(weights)
            if right_mode == "qctn" or u.dim() != 2 or u.shape[1] != nq or u.dtype != torch.float32 or not u.is_cuda:
                return None
            if mx_grid.dtype != torch.float32 or tuple(mx_grid.shape[1:]) != (K, K) or grid_x.dtype != torch.float32:
                return None
            states_w = _items(circuit_states, nq)
            cores = [cores_dict[k] for k in core_names]
            cores = [c.tensor * c.scale if _is_tnt(c) else c for c in cores]
            states = {q: (v.tensor * v.scale if _is_tnt(v) else v) for q, v in states_w.items()}
            device = u.device
            if len(states) != nq or any(t.dtype != torch.float32 or t.device != device for t in cores) or \
                    any(t.dtype != torch.float32 or t.device != device or t.dim() != 1 for t in states.values()):
                return None
            key = (tuple((q, t.shape[0]) for q, t in states.items()), tuple((q, 3, K, K) for q in range(nq)),
                   torch.float32, device)
            bound = plans.get(key)
            if bound is None:
                state_dims = {q: int(t.shape[0]) for q, t in states.items()}
                mx_info = {q: ("a", K, K) for q in range(nq)}
                shapes = {k: tuple(t.shape) for k, t in zip(core_names, cores)}
                plan = ContractionPlan(table, nq, shapes, state_dims, mx_info, "float32", right=right_mode)
                bound = plans[key] = _Bound(plan, device)
            if bound.chain_rank != K:
                return None
            lib = _lib_mod.load()
            order = [k[1] for k in bound.plan.core_shapes]
            by_name = dict(zip(core_names, cores))
            cs = [by_name[k].detach().contiguous() for k in order]
            sts = [states[q].detach().contiguous() for q in range(nq)]
            S, G = int(u.shape[0]), int(grid_x.shape[0])
            gx, mg, uu = grid_x.to(device).contiguous(), mx_grid.to(device).contiguous(), u.contiguous()
            samples = torch.empty(S, nq, dtype=torch.float32, device=device)
            arr = lambda ts: (c_void_p * len(ts))(*[t.data_ptr() for t in ts])
            with torch.cuda.device(device):
                _lib_mod.check(lib.tnq_mps_chain_sample(K, nq, arr(cs), arr(sts), S, G, c_void_p(gx.data_ptr()),
                                                        c_void_p(mg.data_ptr()), c_void_p(uu.data_ptr()),
                                                        (c_float * K)(*[float(w) for w in weights]),
                                                        c_void_p(samples.data_ptr()),
                                                        c_void_p(torch.cuda.current_stream(device).cuda_stream)))
            return samples

        def equations(circuit_states, measure_matrices):
            """The per-qubit einsum strings of this signature (index bookkeeping parity)."""
            sd, mi = signature_of(nq, circuit_states, measure_matrices)
            from .greedy_plan import build_schedule
            return build_schedule(table, nq, sd, mi, right=right_mode, right_table=right_table).equations

        compute_fn.loss_and_grads = loss_and_grads
        compute_fn.enable_cuda_graphs = enable_cuda_graphs
        compute_fn.set_graph_epilogue = set_graph_epilogue
        compute_fn.set_grad_ready_hook = set_grad_ready_hook
        compute_fn.graph_stats = graphs
        compute_fn.equations = equations
        compute_fn.forward_from_x = forward_from_x
        compute_fn.sample_prefix = sample_prefix
        compute_fn.plans = plans
        return compute_fn
