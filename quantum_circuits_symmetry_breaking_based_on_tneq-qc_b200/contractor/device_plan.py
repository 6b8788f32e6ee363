"""DeviceProgram: a lowered VM program living on one GPU, callable with torch tensors.

Thin marshalling layer between torch (device memory, streams) and the C ABI
(include/tneq_b200.h): raw device pointers, element strides and the current
CUDA stream go down; nothing but an error code comes back.
"""
from __future__ import annotations

import ctypes
import math
from ctypes import byref, c_double, c_int64, c_void_p
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from .. import _lib
from .vm_program import VMProgram


class DeviceProgram:
    def __init__(self, prog: VMProgram, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("tneq_b200 programs run on CUDA devices only (no CPU fallback)")
        self.prog = prog
        self.device = device
        self.lib = _lib.load()
        self.real_dtype = torch.float32 if prog.dtype == "f32" else torch.float64
        blob = np.ascontiguousarray(prog.to_blob(), dtype=np.int64)
        handle = c_void_p()
        with torch.cuda.device(device):
            _lib.check(self.lib.tnq_device_check())
            _lib.check(self.lib.tnq_plan_create(blob.ctypes.data_as(ctypes.POINTER(c_int64)), blob.size, byref(handle)))
        self.handle = handle
        self._ws = None
        self._info: Dict[int, _lib.RunInfo] = {}
        self.n_in, self.n_out = len(prog.inputs), len(prog.outputs)
        self._in_ptrs = (c_void_p * max(1, self.n_in))()
        self._hi = (c_int64 * max(1, self.n_in))()
        self._lo = (c_int64 * max(1, self.n_in))()
        self._out_ptrs = (c_void_p * max(1, self.n_out))()
        self._scalars = (c_double * 2)()

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.tnq_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def info(self, nsamples: int) -> _lib.RunInfo:
        if nsamples not in self._info:
            ri = _lib.RunInfo()
            _lib.check(self.lib.tnq_plan_query(self.handle, nsamples, byref(ri)))
            self._info[nsamples] = ri
        return self._info[nsamples]

    def run(self, nsamples: int, inputs: Sequence[Tuple[torch.Tensor, int, int]], scalars=(0.0, 1.0),
            one_buffer: bool = False):
        """inputs[i] = (tensor whose data_ptr is the slot's base, stride_hi, stride_lo) in
        program order; strides in real elements.  Returns the list of output tensors
        (batched: [nsamples, elems]; shared: [elems]) of the program's real dtype; with one_buffer they are
        views of ONE allocation, every slot starting on a 256-byte boundary (the optimizer's table-free SGDG
        launch takes gradients that way, optim/steps.py)."""
        ri = self.info(nsamples)
        if self._ws is None or self._ws.numel() < ri.workspace_bytes:
            self._ws = torch.empty(int(ri.workspace_bytes), dtype=torch.uint8, device=self.device)
        keep = []
        for i, (t, hi, lo) in enumerate(inputs):
            if t.device != self.device:
                raise RuntimeError(f"input slot {i} lives on {t.device}, the plan on {self.device}")
            keep.append(t)
            self._in_ptrs[i] = t.data_ptr()
            self._hi[i], self._lo[i] = int(hi), int(lo)
        outs = []
        shapes = [(nsamples, s.elems) if s.batched else (s.elems,) for s in self.prog.outputs]
        if one_buffer:
            align = 256 * 8 // torch.finfo(self.real_dtype).bits        # elements per 256 bytes
            starts = [0]
            for shp in shapes:
                starts.append(starts[-1] + -(-math.prod(shp) // align) * align)
            buf = torch.empty(starts[-1], dtype=self.real_dtype, device=self.device)
        for j, shp in enumerate(shapes):
            if one_buffer:
                o = buf[starts[j]: starts[j] + math.prod(shp)].view(shp)
            else:
                o = torch.empty(shp, dtype=self.real_dtype, device=self.device)
            outs.append(o)
            self._out_ptrs[j] = o.data_ptr()
        self._scalars[0], self._scalars[1] = float(scalars[0]), float(scalars[1])
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.tnq_plan_run(self.handle, nsamples, self._in_ptrs, self._hi, self._lo, self._out_ptrs,
                                             self._scalars, c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                             c_void_p(stream)))
        return outs
