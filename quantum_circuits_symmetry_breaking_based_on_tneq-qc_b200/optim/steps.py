"""Parameter updates (reference: tneq_qc/backends/backend_pytorch.py:200-468).

optimizer_update(params, grads, state, method, hyperparams) -> (new_params, state)
with methods adam | sgd | momentum | nesterov | rmsprop | sgdg.  state['rng'] (optional, a
random.Random) replaces the process-global `random` stream for SGDG's 1 % QR-retraction draws.  'sgdg' is the
Stiefel-manifold SGD with a Cayley retraction used by the examples
(examples/example_train_single_node.py:229-240).  Params may be TNTensors:
the update acts on tensor*scale with grad/scale and re-wraps (:205-266).

These are small dense per-core operations (K^2 x K^2 matrices).  'sgdg', the
method the examples use, runs for all float32, complex64, float64 and complex128
cores of a network as ONE launch of csrc/tnq_sgdg.cu (one CTA per core); the
other methods and cores wider than their dtype's TNQ_SGDG_MAX_COLS* go through
torch on the device.
"""
from __future__ import annotations

import functools
import math
import random
from typing import Any, Dict, List, Tuple

import numpy as np
import torch


def _is_tnt(p):
    return hasattr(p, "tensor") and hasattr(p, "scale") and hasattr(p, "auto_scale")


def optimizer_update(params: List[Any], grads: List[Any], state: Dict[str, Any], method: str,
                     hp: Dict[str, Any]) -> Tuple[List[Any], Dict[str, Any]]:
    fn = {"adam": _adam, "sgd": _sgd, "momentum": _momentum, "nesterov": _nesterov,
          "rmsprop": _rmsprop, "sgdg": _sgdg}.get(method)
    if fn is None:
        raise ValueError(f"Unknown optimization method: {method}")
    with torch.no_grad():
        raw, info = [], []
        for p in params:
            if _is_tnt(p):
                raw.append(p.tensor * p.scale)
                info.append((p.scale, type(p)))
            else:
                raw.append(p)
                info.append(None)
        g = [gi / inf[0] if inf is not None else gi for gi, inf in zip(grads, info)]
        new, state = fn(raw, g, state, hp)
        for i, inf in enumerate(info):
            if inf is not None:
                params[i] = inf[1](new[i] / inf[0], inf[0])
                params[i].tensor.requires_grad_(True)
            else:
                params[i] = new[i]
                params[i].requires_grad_(True)
    return params, state


def _adam(params, grads, state, hp):
    lr, b1, b2 = hp.get("learning_rate", 0.01), hp.get("beta1", 0.9), hp.get("beta2", 0.999)
    eps, it = hp.get("epsilon", 1e-8), hp.get("iter", 0)
    if "m" not in state:
        state["m"] = [torch.zeros_like(p) for p in params]
        state["v"] = [torch.zeros_like(p) for p in params]
    out = []
    for i, (p, g) in enumerate(zip(params, grads)):
        state["m"][i] = b1 * state["m"][i] + (1 - b1) * g
        state["v"][i] = b2 * state["v"][i] + (1 - b2) * (g ** 2)
        mh = state["m"][i] / (1 - b1 ** (it + 1))
        vh = state["v"][i] / (1 - b2 ** (it + 1))
        out.append(p - lr * mh / (torch.sqrt(vh) + eps))
    return out, state


def _sgd(params, grads, state, hp):
    lr = hp.get("learning_rate", 0.01)
    return [p - lr * g for p, g in zip(params, grads)], state


def _momentum(params, grads, state, hp):
    lr = hp.get("learning_rate", 0.01)
    if "momentum_buffer" not in state:
        state["momentum_buffer"] = [torch.zeros_like(p) for p in params]
    out = []
    for i, (p, g) in enumerate(zip(params, grads)):
        state["momentum_buffer"][i] = 0.9 * state["momentum_buffer"][i] + lr * g
        out.append(p - state["momentum_buffer"][i])
    return out, state


def _nesterov(params, grads, state, hp):
    lr = hp.get("learning_rate", 0.01)
    if "momentum_buffer" not in state:
        state["momentum_buffer"] = [torch.zeros_like(p) for p in params]
    out = []
    for i, (p, g) in enumerate(zip(params, grads)):
        state["momentum_buffer"][i] = 0.9 * state["momentum_buffer"][i] + lr * g
        out.append(p - (state["momentum_buffer"][i] + lr * g))
    return out, state


def _rmsprop(params, grads, state, hp):
    lr, eps = hp.get("learning_rate", 0.01), hp.get("epsilon", 1e-8)
    if "square_avg" not in state:
        state["square_avg"] = [torch.zeros_like(p) for p in params]
    out = []
    for i, (p, g) in enumerate(zip(params, grads)):
        state["square_avg"][i] = 0.9 * state["square_avg"][i] + 0.1 * (g ** 2)
        out.append(p - lr * g / (torch.sqrt(state["square_avg"][i]) + eps))
    return out, state


SGDG_MAX_COLS = 64          # TNQ_SGDG_MAX_COLS, include/tneq_b200.h
# per dtype: suffix of the tnq_sgdg_step entry points and the widest matrix they take (TNQ_SGDG_MAX_COLS*)
SGDG_KERNELS = {torch.float32: ("", SGDG_MAX_COLS), torch.complex64: ("_c64", 64), torch.float64: ("_f64", 64),
                torch.complex128: ("_c128", 48)}
# The kernel divides every row by its norm + 1e-8; the reference takes a retracted core's rows as they are.  Stored
# 2^27 times larger, a unit row comes out of that division as itself to within rounding in float64 as well
# (1e-8 / 2^27 < 1e-16).  float32 keeps the unscaled retraction: 1e-8 is below its rounding at 1.
_RETRACT_SCALE = {torch.float32: 1.0}


@functools.lru_cache(maxsize=4096)
def _matrix_shape(shp):
    """(rows, columns) of a core seen as the matrix the Cayley step works on (backend_pytorch.py:392-399); cached:
    one call per core and step sat at 10 % of a candidate's host time in the population benchmark."""
    if len(shp) > 2:
        rows = math.prod(int(x) for x in shp[: len(shp) // 2])
        return rows, math.prod(int(x) for x in shp) // max(rows, 1)
    return (int(shp[0]), int(shp[1])) if len(shp) == 2 else (0, 0)


def sgdg_kernel_eligible(dtype, shape, device_type) -> bool:
    """Whether the Cayley step of a core of this dtype and shape runs in csrc/tnq_sgdg.cu: a Stiefel core
    (rows <= cols as the step's matrix) on a CUDA device, no wider than the maximum of its dtype."""
    kernel = SGDG_KERNELS.get(dtype)
    if kernel is None or device_type != "cuda":
        return False
    r, c = _matrix_shape(tuple(shape))
    return 1 <= r <= c <= kernel[1]


def _qr_retract(unity):
    qm, rm = torch.linalg.qr(unity.T, mode="reduced")
    d = torch.diag(rm)
    return (qm * (torch.sgn(d) if torch.is_complex(d) else torch.sign(d)).unsqueeze(0)).T


def _sgdg_flat_step(params, grads, state, lr, mom, out):
    """All cores in one launch with NO per-step host-to-device traffic: parameters are packed into one
    fresh buffer (the reference returns new tensors), gradients already sit in one buffer (the fused
    contraction routes return them as views of it), the momentum buffers live in one persistent
    buffer, and the offset table is static per network (tnq_sgdg_step_flat*).  All cores have one dtype; complex
    gradients may be complex views of one real buffer (view_as_complex), offsets count elements of the cores'
    dtype.  Returns False when the gradients are not views of one buffer."""
    from .. import _lib
    dtype = params[0].dtype
    esize = params[0].element_size()
    base = getattr(grads[0], "_base", None)
    if (base is None or not base.is_cuda or base.dtype not in (dtype, dtype.to_real()) or not base.is_contiguous()
            or base.data_ptr() % esize):
        return False
    b0 = base.data_ptr()
    g_off = []
    for g in grads:
        if getattr(g, "_base", None) is not base or not g.is_contiguous() or (g.data_ptr() - b0) % esize:
            return False
        g_off.append((g.data_ptr() - b0) // esize)
    lib = _lib.load()
    dev = params[0].device
    shapes = [_matrix_shape(p.shape) for p in params]
    sizes = [r * c for r, c in shapes]
    key = (dtype, tuple(shapes), tuple(g_off))
    with torch.cuda.device(dev):
        if state.get("_flat_key") != key:          # first step (or a different network): build the static tables
            p_off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
            table = np.stack([p_off, np.asarray(g_off, dtype=np.int64), p_off])
            state["_flat_key"] = key
            state["_flat_offs"] = torch.from_numpy(table).to(dev)
            state["_flat_dims"] = torch.tensor([[r for r, _ in shapes], [c for _, c in shapes]], dtype=torch.int32, device=dev)
            vflat = torch.zeros(int(sum(sizes)), dtype=dtype, device=dev)
            for i, (off, n) in enumerate(zip(p_off, sizes)):
                old = state["momentum_buffer"][i]
                r, c = shapes[i]
                if old is not None:
                    vflat[off: off + n].copy_(old.reshape(-1))
                state["momentum_buffer"][i] = vflat[off: off + n].view(c, r)
            state["_flat_v"] = vflat
            state["_flat_poff"] = [int(x) for x in p_off]
        if state.get("pingpong"):
            # two persistent parameter buffers used alternately: the cores of step i+2 live where those of step i
            # lived, so a training loop presents only two sets of addresses (CUDA-graph replay, DataParallelTrainer.
            # enable_cuda_graphs); the tensors returned two steps ago are overwritten
            bufs = state.setdefault("_flat_p", [torch.empty(int(sum(sizes)), dtype=dtype, device=dev) for _ in range(2)])
            flat = bufs[state.get("_flat_turn", 0) & 1]
            state["_flat_turn"] = state.get("_flat_turn", 0) + 1
            torch.cat([p.reshape(-1) for p in params], out=flat)
        else:
            flat = torch.cat([p.reshape(-1) for p in params])
        p_off = state["_flat_poff"]
        rng = state.get("rng", random)
        for n in range(len(params)):
            # the reference draws one random number per Stiefel core (backend_pytorch.py:382)
            if rng.randint(1, 101) == 1:
                r, c = shapes[n]
                x = flat[p_off[n]: p_off[n] + sizes[n]].view(r, c)
                x.copy_(_RETRACT_SCALE.get(dtype, 2.0 ** 27) * _qr_retract(x / (torch.norm(x, p=2, dim=1, keepdim=True) + 1e-8)))
        dims, offs = state["_flat_dims"], state["_flat_offs"]
        step = getattr(lib, "tnq_sgdg_step_flat" + SGDG_KERNELS[dtype][0])
        _lib.check(step(flat.data_ptr(), b0, state["_flat_v"].data_ptr(), offs.data_ptr(), dims[0].data_ptr(),
                        dims[1].data_ptr(), len(params), max(c for _, c in shapes), float(lr), float(mom),
                        torch.cuda.current_stream().cuda_stream))
    for n, p in enumerate(params):
        out[n] = flat[p_off[n]: p_off[n] + sizes[n]].view(p.shape)
    return True


def _sgdg_kernel_step(idx, params, grads, state, lr, mom, out):
    """All eligible cores, of one dtype, in one launch of tnq_sgdg_step* (csrc/tnq_sgdg.cu)."""
    from .. import _lib
    lib = _lib.load()
    dev, dtype = params[idx[0]].device, params[idx[0]].dtype
    shapes = [_matrix_shape(params[i].shape) for i in idx]
    sizes = [r * c for r, c in shapes]
    with torch.cuda.device(dev):
        # the update is in place on the device, the reference returns fresh tensors: work on a packed copy
        flat = torch.cat([params[i].reshape(-1) for i in idx])
        gs = [grads[i].contiguous() for i in idx]
        rng = state.get("rng", random)
        for n, i in enumerate(idx):
            # the reference draws one random number per Stiefel core (backend_pytorch.py:382)
            if rng.randint(1, 101) == 1:
                r, c = shapes[n]
                off = sum(sizes[:n])
                x = flat[off: off + sizes[n]].view(r, c)
                x.copy_(_RETRACT_SCALE.get(dtype, 2.0 ** 27) * _qr_retract(x / (torch.norm(x, p=2, dim=1, keepdim=True) + 1e-8)))
            if state["momentum_buffer"][i] is None:
                r, c = shapes[n]
                state["momentum_buffer"][i] = torch.zeros(c, r, dtype=dtype, device=dev)
            elif not state["momentum_buffer"][i].is_contiguous():
                state["momentum_buffer"][i] = state["momentum_buffer"][i].contiguous()
        vs = [state["momentum_buffer"][i] for i in idx]
        offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]) * flat.element_size()
        table = np.empty((3, len(idx)), dtype=np.int64)
        table[0] = flat.data_ptr() + offs
        table[1] = [g.data_ptr() for g in gs]
        table[2] = [v.data_ptr() for v in vs]
        key = tuple(shapes)
        if state.get("_sgdg_dims_key") != key:
            state["_sgdg_dims_key"] = key
            state["_sgdg_dims"] = torch.tensor([[r for r, _ in shapes], [c for _, c in shapes]], dtype=torch.int32,
                                               device=dev)
        dims = state["_sgdg_dims"]
        tdev = torch.from_numpy(table).to(dev)
        step = getattr(lib, "tnq_sgdg_step" + SGDG_KERNELS[dtype][0])
        _lib.check(step(tdev[0].data_ptr(), tdev[1].data_ptr(), tdev[2].data_ptr(), dims[0].data_ptr(), dims[1].data_ptr(),
                        len(idx), max(c for _, c in shapes), float(lr), float(mom), torch.cuda.current_stream().cuda_stream))
    off = 0
    for n, i in enumerate(idx):
        out[i] = flat[off: off + sizes[n]].view(params[i].shape)
        off += sizes[n]


def _sgdg(params, grads, state, hp):
    """Cayley-transform SGD on the Stiefel manifold (backend_pytorch.py:349-468)."""
    lr, mom, stiefel = hp.get("learning_rate", 0.01), hp.get("momentum", 0.0), hp.get("stiefel", True)
    eps = 1e-8
    if "momentum_buffer" not in state:
        state["momentum_buffer"] = [None] * len(params)
    out = [None] * len(params)
    fast = {}                   # dtype -> indices of the cores the kernel of that dtype takes
    if stiefel and hp.get("device_kernel", True):
        for i, (p, g) in enumerate(zip(params, grads)):
            if g.dtype == p.dtype and sgdg_kernel_eligible(p.dtype, p.shape, p.device.type):
                fast.setdefault(p.dtype, []).append(i)
    if (len(fast) == 1 and len(next(iter(fast.values()))) == len(params)
            and _sgdg_flat_step(params, grads, state, lr, mom, out)):
        return out, state
    for idx in fast.values():
        _sgdg_kernel_step(idx, params, grads, state, lr, mom, out)
    for i, (p, g) in enumerate(zip(params, grads)):
        if out[i] is not None:
            continue
        shp = p.shape
        if len(shp) > 2:
            rows = int(np.prod(shp[: len(shp) // 2]))
            x, gx = p.reshape(rows, -1), g.reshape(rows, -1)
        else:
            x, gx = p, g
        cplx = torch.is_complex(x)
        unity = x / (torch.norm(x, p=2, dim=1, keepdim=True) + eps)
        if not (stiefel and unity.shape[0] <= unity.shape[1]):
            out[i] = p - lr * g
            continue
        if state.get("rng", random).randint(1, 101) == 1:  # occasional QR retraction, same RNG stream as the reference
            unity = _qr_retract(unity)
        if state["momentum_buffer"][i] is None:
            state["momentum_buffer"][i] = torch.zeros(gx.T.shape, dtype=gx.dtype, device=p.device)
        hconj = (lambda m: torch.conj(m).T) if cplx else (lambda m: m.T)
        v = mom * state["momentum_buffer"][i] - hconj(gx)
        mx = v @ unity
        w_hat = mx - 0.5 * (hconj(unity) @ (unity @ mx))
        w = w_hat - hconj(w_hat)
        t = 0.5 * 2 / (torch.abs(w).sum(dim=0).max() + eps)
        alpha = min(t, lr)
        eye = torch.eye(w.shape[0], dtype=w.dtype, device=w.device)
        y = torch.inverse(eye - (alpha / 2) * w) @ (eye + (alpha / 2) * w) @ hconj(unity)
        pn = hconj(y)
        out[i] = pn.reshape(shp) if len(shp) > 2 else pn
        new_v = w @ hconj(unity)
        old_v = state["momentum_buffer"][i]
        if old_v.shape == new_v.shape and old_v.dtype == new_v.dtype:
            old_v.copy_(new_v)        # keep the buffer (it may be a view of the flat momentum buffer of tnq_sgdg_step_flat)
        else:
            state["momentum_buffer"][i] = new_v
    return out, state
