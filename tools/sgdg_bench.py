#!/usr/bin/env python
"""Time of the SGDG optimizer step ('sgdg', the reference's default method) on the torch route against
csrc/tnq_sgdg.cu, for complex64, float64 and complex128 cores:

  * the step alone: 46 and 15 cores of (3,3,3,3) -- the 24-qubit two-layer network and cfg3's 16-qubit one --
    with gradients as separate tensors (pointer-table launch) and as views of one buffer (table-free launch);
  * a full training step of examples/train_single_node.py's flow (16-qubit MPS, K = 3, B = 512, momentum 0.9) with
    the optimizer on each route, and the example script itself;
  * one torch-route step on cfg4-shaped cores (15 x (64,64,64,64) complex64: 4096 x 4096 matrices), which are
    wider than any kernel takes.

    python tools/sgdg_bench.py [--steps 200] [--out results.json]

Times are host wall clock over many steps that end in a device synchronisation.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.build()
import tneq_b200 as tb  # noqa: E402
from tneq_b200 import _lib  # noqa: E402
from tneq_b200.optim import steps  # noqa: E402
from oracle import qctn_oracle as oc  # noqa: E402

DEV = torch.device("cuda:0")


def _torch_route(on):
    """Send every core to the torch route (the only route complex64 / float64 / complex128 had before)."""
    steps.sgdg_kernel_eligible = (lambda *a: False) if on else _ELIGIBLE


_ELIGIBLE = steps.sgdg_kernel_eligible


def time_step(dtype, ncores, route, n):
    torch.manual_seed(0)
    shape = (3, 3, 3, 3)
    params = [oc.init_random_core([9, 9], dtype).reshape(shape).to(DEV) for _ in range(ncores)]
    real = 0.3 * torch.randn(ncores * 81 * (2 if dtype.is_complex else 1), dtype=dtype.to_real(), device=DEV)
    flat = torch.view_as_complex(real.view(-1, 2)) if dtype.is_complex else real
    grads = list(flat.view(ncores, *shape).unbind(0))
    if route != "flat":
        grads = [g.clone() for g in grads]
    _torch_route(route == "torch")
    state, hp = {}, dict(learning_rate=0.01, momentum=0.9, stiefel=True)
    random.seed(1)
    try:
        for k in range(n + 10):
            if k == 10:
                torch.cuda.synchronize()
                t0, l0 = time.perf_counter(), _lib.launch_count()
            params, state = steps.optimizer_update(params, grads, state, "sgdg", hp)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        _torch_route(False)
    return 1e3 * dt / n, (_lib.launch_count() - l0) / n, "_flat_offs" in state


def time_training(dtype, route, n, nq=16, K=3, B=512):
    """examples/train_single_node.py's loop (same network, data, optimizer settings and warm-up)."""
    _torch_route(route == "torch")
    try:
        torch.manual_seed(42)
        random.seed(0)
        be = tb.BackendFactory.create_backend("b200", device="cuda:0", dtype=str(dtype)[6:])
        eng = tb.EngineSiamese(backend=be, strategy_mode="balanced", mx_K=K)
        q = tb.QCTN(tb.QCTNHelper.generate_example_graph(n=nq, graph_type="mps", dim_char=str(K)), backend=be)
        for name in q.cores:
            q.cores_weights[name].requires_grad_(True)
        states = [torch.zeros(K, device=DEV, dtype=dtype) for _ in range(nq)]
        for s in states:
            s[-1] = 1.0
        data = [eng.generate_data(torch.randn(B, nq, device=DEV), K=K, ret_type="TNTensor")[0] for _ in range(20)]
        opt = tb.Optimizer(method="sgdg", learning_rate=1e-2, max_iter=n, engine=eng, momentum=0.9, stiefel=True,
                           verbose=False)
        t_opt = 0.0
        for step in range(n + 10):
            if step == 10:
                torch.cuda.synchronize()
                t0, t_opt = time.perf_counter(), 0.0
            loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, states, data[step % len(data)])
            opt.step(q, grads)
            opt.iter += 1
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return 1e3 * dt / n, float(loss), "_flat_offs" in opt.opt_state
    finally:
        _torch_route(False)


def time_cfg4_torch_step():
    torch.manual_seed(0)
    ncores, shape = 15, (64, 64, 64, 64)
    params = [torch.randn(shape, dtype=torch.complex64, device=DEV) * 2 ** -6 for _ in range(ncores)]
    grads = [torch.randn(shape, dtype=torch.complex64, device=DEV) * 1e-3 for _ in range(ncores)]
    assert not any(steps.sgdg_kernel_eligible(p.dtype, p.shape, "cuda") for p in params)
    state, hp = {}, dict(learning_rate=0.01, momentum=0.9, stiefel=True)
    random.seed(1)
    out = []
    for k in range(3):                     # the first step allocates the momentum buffers and warms cuBLAS / cuSOLVER
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        params, state = steps.optimizer_update(params, grads, state, "sgdg", hp)
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return 1e3 * min(out[1:]), 1e3 * out[0]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=None, help="write the results as JSON")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else torch.cuda.get_device_name(0), "torch": torch.__version__, "step": [], "train": []}
    print(f"# {res['gpu']}", flush=True)
    for dtype in (torch.complex64, torch.float64, torch.complex128):
        for ncores in (46, 15):
            row = {"dtype": str(dtype)[6:], "cores": ncores}
            for route in ("torch", "table", "flat"):
                ms, launches, flat = time_step(dtype, ncores, route, args.steps)
                row[route] = {"ms": round(ms, 4), "launches_per_step": launches, "flat": flat}
            row["speedup_flat"] = round(row["torch"]["ms"] / row["flat"]["ms"], 1)
            res["step"].append(row)
            print(f"optimizer step  {row['dtype']:>10} {ncores:2d} x (3,3,3,3): torch {row['torch']['ms']:.3f} ms, "
                  f"kernel {row['table']['ms']:.3f} ms (pointer table), {row['flat']['ms']:.3f} ms (table-free), "
                  f"x{row['speedup_flat']}", flush=True)
    for dtype in (torch.complex64, torch.float64):
        row = {"dtype": str(dtype)[6:]}
        for route in ("torch", "kernel"):
            ms, loss, flat = time_training(dtype, route, args.steps)
            row[route] = {"ms": round(ms, 4), "final_loss": loss, "flat": flat}
        res["train"].append(row)
        print(f"training step   {row['dtype']:>10} 16-qubit MPS K=3 B=512: optimizer on torch {row['torch']['ms']:.3f} "
              f"ms/step, on the kernel {row['kernel']['ms']:.3f} ms/step (final losses {row['torch']['final_loss']:.6f} / "
              f"{row['kernel']['final_loss']:.6f})", flush=True)
        ex = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_single_node.py"), "--dtype",
                             str(dtype)[6:], "--num-step", str(args.steps)], capture_output=True, text=True)
        row["example_last_line"] = (ex.stdout.strip().splitlines() or [ex.stderr[-500:]])[-1]
        print(f"  examples/train_single_node.py --dtype {row['dtype']}: {row['example_last_line']}", flush=True)
    best, first = time_cfg4_torch_step()
    res["cfg4_torch_step_ms"] = {"steady": round(best, 1), "first": round(first, 1)}
    print(f"torch-route step on 15 x (64,64,64,64) complex64 (4096 x 4096 matrices): {best:.1f} ms "
          f"(first step {first:.1f} ms)", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
