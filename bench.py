#!/usr/bin/env python
"""bench.py -- throughput of the QCTN contraction hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Metric (BASELINE.json): samples/sec for the QCTN
forward+backward contraction.  Workloads (SURVEY.md 8(d)):

  cfg3 (default)  training step (forward + loss + reverse sweep: the warp-level ladder kernel,
                  replayed from a CUDA graph; + one gradient/loss exchange when N > 1: this
                  repository's one-shot NVLink all-reduce kernel) of the 24-qubit two-layer merged
                  MPS network, K=3, float32, GLOBAL batch 16384 split over the N GPUs (strong scaling)
  cfg2            forward probabilities, 16-qubit MPS, K=3, batch 4096
  cfg2-large      the same with batch 2^20 (bandwidth/compute visible above launch latency)

A "step" is one pass of the hot path over one batch of synthetic measurements
(x ~ N(0,1), torch.manual_seed(42); cores QR-orthogonal, torch.manual_seed(1234); states
e_{K-1}; Mx = TNTensor-normalised Hermite-function outer products).

`value`  : device-resident inputs, CUDA-event timed per step on the launching stream, L2
           flushed between timed steps, max over ranks.
`e2e`    : the same step through the public engine API with the batch's measurement
           matrices in PINNED HOST memory: every timed step contains the host->device copy of one
           batch (issued on a copy stream one step ahead, awaited inside the step) and the
           device->host read of the loss.
`--impl reference`: the reference's own CPU algorithm (oracle port of GreedyStrategy +
           torch.autograd, bit-identical to /root/reference on CPU, see oracle/) on the box's host
           cores, on a bounded sample of the same workload.
`--dump-outputs DIR`: after the timed steps, what the last timed step returned (loss, per-sample values,
           core gradients) as DIR/<name>.npy (see dump_outputs).  The inputs are seeded, so dumps of two
           builds taken with the same arguments compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg3": dict(kind="merged", n=24, K=3, batch=16384, mode="train", dtype="float32",
                 name="cfg3: 24-qubit 2-layer merged MPS QCTN, K=3, fwd+loss+bwd, global batch 16384"),
    "cfg3-fwd": dict(kind="merged", n=24, K=3, batch=16384, mode="fwd", dtype="float32",
                     name="24-qubit 2-layer merged MPS QCTN, K=3, forward only, batch 16384"),
    "cfg4": dict(kind="mps", n=16, K=64, batch=256, mode="train", dtype="complex64", weak=True, near_identity=True,
                 name="cfg4: 16-qubit MPS QCTN, bond 64, complex64, fwd+loss+bwd, batch 256 per GPU (tcgen05 GEMM path)"),
    "cfg4-128": dict(kind="mps", n=16, K=128, batch=8, mode="train", dtype="complex64", weak=True, near_identity=True,
                     name="cfg4: 16-qubit MPS QCTN, bond 128, complex64, fwd+loss+bwd, batch 8 per GPU (tcgen05 GEMM path; 32 per GPU does not fit 180 GB with the cores' 64 GB)"),
    "cfg4-32": dict(kind="mps", n=16, K=32, batch=256, mode="train", dtype="complex64", weak=True, near_identity=True,
                    name="16-qubit MPS QCTN, bond 32, complex64, fwd+loss+bwd, batch 256 per GPU (tcgen05 GEMM path)"),
    "cfg2": dict(kind="mps", n=16, K=3, batch=4096, mode="fwd", dtype="float32",
                 name="cfg2: 16-qubit MPS QCTN, K=3, forward probabilities, batch 4096"),
    "cfg2-large": dict(kind="mps", n=16, K=3, batch=1 << 20, mode="fwd", dtype="float32",
                       name="cfg2-large: 16-qubit MPS QCTN, K=3, forward probabilities, batch 2^20"),
    "cfg2-large-x": dict(kind="mps", n=16, K=3, batch=1 << 20, mode="fwdx", dtype="float32",
                         name="cfg2-large with generate_data fused into the sweep (EngineSiamese.contract_from_x): "
                              "16-qubit MPS QCTN, K=3, forward probabilities from x, batch 2^20"),
    "cfg2-train": dict(kind="mps", n=16, K=3, batch=1 << 18, mode="train", dtype="float32",
                       name="16-qubit MPS QCTN, K=3, fwd+loss+bwd, batch 2^18"),
}


def build_graph(tb, kind, n, K):
    g = tb.QCTNHelper.generate_example_graph(n=n, graph_type="mps" if kind == "merged" else kind, dim_char=str(K))
    if kind == "merged":
        q = tb.QCTN(g)
        return tb.QCTN.merge(q, q).graph
    return g


def synth_inputs(graph, K, B, dtype):
    """CPU tensors, seeded as SURVEY 8(d) prescribes (oracle helpers: test infrastructure only)."""
    import torch
    from oracle import qctn_oracle as oc
    names, table, nq = oc.parse_graph(graph)
    torch.manual_seed(1234)
    cores = oc.random_cores(table, getattr(torch, dtype))
    torch.manual_seed(42)
    x = torch.randn(B, nq)
    return names, table, nq, cores, x


DUMP_BYTES = 60 << 20          # data of all dumped arrays together; with the .npy headers under 64 MB


def dump_outputs(outdir, arrays):
    """Write each named array (tensor or float) as outdir/<name>.npy: float64 data as float64, everything else as
    float32, complex data with a trailing (real, imag) axis of 2.  When the arrays together exceed DUMP_BYTES, each
    array larger than an equal share of it is replaced by that many of its elements (flattened, in index order),
    chosen by a seeded permutation: the same elements on every run, so that dumps of two builds compare element for
    element."""
    import numpy as np
    import torch
    os.makedirs(outdir, exist_ok=True)
    wide = (torch.float64, torch.complex128)
    arrays = {k: torch.as_tensor(v).detach() for k, v in arrays.items()}
    esz = {k: (2 if t.is_complex() else 1) * (8 if t.dtype in wide else 4) for k, t in arrays.items()}
    sample = sum(t.numel() * esz[k] for k, t in arrays.items()) > DUMP_BYTES
    share = DUMP_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        if sample and t.numel() * esz[name] > share:
            gen = torch.Generator().manual_seed(0)
            idx = torch.randperm(t.numel(), generator=gen)[:share // esz[name]].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        if t.is_complex():
            t = torch.view_as_real(t.to(torch.complex128 if t.dtype in wide else torch.complex64))
        else:
            t = t.to(torch.float64 if t.dtype in wide else torch.float32)
        np.save(os.path.join(outdir, name + ".npy"), t.cpu().numpy())


class ClockSampler:
    """nvidia-smi sampling while the timed region runs (B200_PROFILING.md, clocks line)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def time_reference(args, wl):
    """--impl reference / cpu_baseline: the oracle (reference algorithm) on host cores."""
    import torch
    import tneq_b200 as tb
    from oracle import qctn_oracle as oc
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    wl = dict(wl)
    note = ""
    if wl["K"] > 8:
        # left-to-right einsum keeps B*K^6 intermediates: infeasible on a CPU at bond 64; the largest
        # bond that runs in bounded time is used and said so (SURVEY 8(d))
        note = f" [bond reduced from {wl['K']} to 8: the reference's B*K^6 intermediates do not fit at bond {wl['K']}]"
        wl["K"] = 8
    graph = build_graph(tb, wl["kind"], wl["n"], wl["K"])
    names, table, nq, cores, x_all = synth_inputs(graph, wl["K"], 4096, wl["dtype"])
    states = oc.unit_states(nq, wl["K"], getattr(torch, wl["dtype"]))
    n_steps = args.steps if args.impl == "reference" else 3
    n_warm = max(1, args.warmup) if args.impl == "reference" else 1

    # The REAL reference (unmodified tneq_qc: /root/reference in the build container, the copy staged by
    # build() under baseline/_ref/ on the GPU box) through its own EngineSiamese + 'pytorch' CPU backend
    # + GreedyStrategy; the oracle port only where no copy of the reference exists.
    from oracle import ref_harness as rh
    kind = "port"
    ref_eng = ref_q = None
    if rh.available() and not os.environ.get("TNQ_BENCH_REFERENCE_PORT"):
        try:
            ns = rh.load()
            with rh.quiet():
                ref_be, ref_eng = rh.make_engine(wl["dtype"], wl["K"])
                ref_q = ns.QCTN(graph, backend=ref_be)
                for k, v in cores.items():
                    ref_q.cores_weights[k] = v.detach().clone().requires_grad_(True)
            kind = "reference"
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] reference import failed ({type(exc).__name__}: {exc}); timing the oracle port", file=sys.stderr)
            ref_eng = None

    def run_once(xb):
        if ref_eng is not None:
            with rh.quiet():
                t0 = time.perf_counter()                 # (fwdx: generating the matrices is part of the step)
                mx, _ = ref_eng.generate_data(xb, K=wl["K"], ret_type="TNTensor")
                if wl["mode"] != "fwdx":
                    t0 = time.perf_counter()
                if wl["mode"] == "train":
                    ref_eng.contract_with_compiled_strategy_for_gradient(ref_q, states, mx)
                else:
                    with torch.no_grad():
                        ref_eng.contract_with_compiled_strategy(ref_q, states, mx)
                return time.perf_counter() - t0
        mx, _ = oc.generate_data(xb, wl["K"], getattr(torch, wl["dtype"]), "TNTensor")  # fresh: auto_scale is in place
        t0 = time.perf_counter()
        if wl["mode"] == "train":
            oc.loss_and_grads(graph, cores, states, mx)
        else:
            with torch.no_grad():
                oc.forward(graph, cores, states, mx)
        return time.perf_counter() - t0

    if args.ref_batch:
        sample_b = args.ref_batch
    else:
        # bounded sample: probe the cost at a tiny batch, then size the batch so that the whole
        # warmup + steps run takes about `budget` seconds (left-to-right einsum intermediates make
        # the two-layer network cost ~1 s per sample on 8 cores)
        budget = 90.0 if args.impl == "reference" else 20.0
        t2 = run_once(x_all[:2])
        t2 = min(t2, run_once(x_all[:2]))
        per_sample = max(t2 / 2, 1e-6)
        sample_b = int(max(1, min(4096, budget / ((n_steps + n_warm) * per_sample))))
    x = x_all[:sample_b]
    def step():
        return run_once(x)

    for _ in range(n_warm):
        step()
    times = [step() for _ in range(n_steps)]
    total = sum(times)
    val = sample_b * len(times) / total
    what = ("the unmodified reference (tneq_qc EngineSiamese + 'pytorch' CPU backend + GreedyStrategy, torch.einsum left to right)"
            if kind == "reference" else "oracle port of the reference CPU path (bit-identical to /root/reference on CPU)")
    return dict(value=val, unit="samples/s", cores=threads, kind=kind,
                sample=f"{len(times)} steps of batch {sample_b} of the same network ({wl['mode']}), " + what + note,
                ms_per_step=1e3 * total / len(times), batch=sample_b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="override the workload's global batch")
    ap.add_argument("--ref-batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="do not replay the training step from a CUDA graph")
    ap.add_argument("--profile-step", action="store_true",
                    help="after the warm-up, run ONE step between cudaProfilerStart/Stop and exit (ncu --profile-from-start off: "
                         "the launch list of exactly one steady-state step)")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="average gradients with NCCL instead of the one-shot NVLink kernel (tnq_allreduce_oneshot)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        ref = time_reference(args, wl)
        line = {"impl": "reference", "metric": "samples/sec for QCTN fwd+bwd contraction", "value": ref["value"],
                "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ref["ms_per_step"], "higher_is_better": True,
                "scaling": "weak" if wl.get("weak") else "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["name"], "reference_sample_batch": ref["batch"]},
                "cpu_baseline": {k: ref[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": ref["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    import torch
    import __graft_entry__ as ge
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        dist = None
    if rank == 0:
        ge.build()                             # no-op when the in-tree library is current
    if dist is not None:
        dist.barrier()
    import tneq_b200 as tb
    from tneq_b200 import _lib
    _lib.load()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)

    K, n = wl["K"], wl["n"]
    esz = 8 if "complex" in wl["dtype"] else 4
    graph = build_graph(tb, wl["kind"], n, K)
    weak = bool(wl.get("weak"))
    B_global = wl["batch"] * world if weak else wl["batch"]
    B = B_global // world                      # strong scaling: global batch fixed; weak: per-GPU batch fixed
    big = K >= 16
    if big:                                    # 64^4 cores: QR-orthogonal init on the device (seeded)
        from oracle import qctn_oracle as oc
        names, table, nq = oc.parse_graph(graph)
        torch.manual_seed(1234)
        tdt = getattr(torch, wl["dtype"])
        cores_cpu = {}
        for c in names:
            m = torch.randn(K * K, K * K, dtype=tdt, device=f"cuda:{local_rank}")
            qm, rm = torch.linalg.qr(m)
            d = torch.diagonal(rm)
            cores_cpu[c] = (qm * (d / d.abs()).conj().unsqueeze(0)).reshape(K, K, K, K)
        torch.manual_seed(42)
        x_cpu = torch.randn(B_global, nq)
    else:
        names, table, nq, cores_cpu, x_cpu = synth_inputs(graph, K, B_global, wl["dtype"])
    x_local = x_cpu[rank * B:(rank + 1) * B]

    backend = tb.BackendFactory.create_backend("b200", device=str(dev), dtype=wl["dtype"])
    engine = tb.EngineSiamese(backend=backend, strategy_mode="balanced", mx_K=K)
    engine.enable_cuda_graphs(not args.no_graphs)      # opt-in product feature (EngineSiamese.enable_cuda_graphs)
    qctn = tb.QCTN(graph, backend=backend)
    for c in names:
        w = cores_cpu[c].to(dev).clone(memory_format=torch.contiguous_format)
        if dist is not None:                   # the reference forgets this (SURVEY 3.3)
            dist.broadcast(torch.view_as_real(w) if w.is_complex() else w, src=0)
        qctn.cores_weights[c] = w.requires_grad_(True)
    tdt = getattr(torch, wl["dtype"])
    states = [torch.zeros(K, device=dev, dtype=tdt) for _ in range(nq)]
    for s in states:
        s[-1] = 1.0
    if wl.get("near_identity"):
        # large bond: a random unitary's overlap with a product state is ~K^-n, far below the loss's
        # 1e-10 clamp (SURVEY D11) for ANY projector data; measurement matrices I + 0.1 H (H random
        # Hermitian, unit spectral scale) keep the value O(1) so that loss and gradients are live
        torch.manual_seed(42 + rank)
        mx_dev = []
        for _ in range(nq):
            h = torch.randn(B, K, K, dtype=tdt, device=dev) / (2.0 * K ** 0.5)
            m = torch.eye(K, dtype=tdt, device=dev) + 0.1 * (h + h.transpose(1, 2).conj())
            mx_dev.append(tb.TNTensor(m))
    else:
        mx_dev, _ = engine.generate_data(x_local.to(dev), K=K, ret_type="TNTensor")
    log_scale = sum(m.log_scale for m in mx_dev)
    mx_dev = [tb.TNTensor(m.tensor.contiguous(), m.scale, m.log_scale) for m in mx_dev]
    mx_host = [m.tensor.cpu().pin_memory() for m in mx_dev]
    mx_scales = [(m.scale, m.log_scale) for m in mx_dev]
    h2d_bytes = sum(m.numel() * m.element_size() for m in mx_host)
    if wl["mode"] == "fwdx":
        h2d_bytes = x_local.numel() * 4

    fn = engine._compiled(qctn, states, mx_dev, True, "symmetric")
    cores_dict = {c: qctn.cores_weights[c] for c in names}
    train = wl["mode"] == "train"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # gradient + loss averaging: ONE exchange per step.  Small messages (15 KB for cfg3) go through this
    # repository's one-shot NVLink kernel over symmetric memory; big ones (cfg4: GBs) through NCCL.
    oneshot = None
    n_grad = sum(v.numel() for v in cores_cpu.values())
    if dist is not None and train and esz == 4 and n_grad < (1 << 18) and not args.nccl_allreduce:
        from tneq_b200.distributed.oneshot import OneShotAllReduce
        oneshot = OneShotAllReduce.create(n_grad + 16, dev)

    checked = {"oneshot": False}

    def average(loss, grads):
        base = grads[0]._base if len(grads) else None
        if oneshot is not None and base is not None and base.numel() == n_grad and base.is_contiguous():
            out = oneshot.mean(base, loss.reshape(1))
            if not checked["oneshot"]:
                # first (warm-up) exchange on the ranks that are about to be timed: the one-shot kernel must
                # agree with NCCL's all-reduce of the same buffers, and be bit-identical on every rank
                checked["oneshot"] = True
                want = torch.cat([base.detach().reshape(-1), loss.detach().reshape(1)]).clone()
                dist.all_reduce(want)
                want /= world
                err = (out - want).abs().max().item()
                ref_mag = want.abs().max().item()
                assert err <= 2e-6 * max(ref_mag, 1e-30), f"one-shot all-reduce disagrees with NCCL: {err} vs {ref_mag}"
                every = [torch.empty_like(out) for _ in range(world)]
                dist.all_gather(every, out)
                assert all(torch.equal(e, every[0]) for e in every), "one-shot all-reduce differs between ranks"
                checked["err_vs_nccl"] = err / max(ref_mag, 1e-30)
            return out
        flat = torch.cat([g.reshape(-1) for g in grads] + [loss.reshape(1)])
        dist.all_reduce(flat)
        flat /= world
        return flat

    # GB-sized gradients (cfg4: 15 cores x 134 MB): every core's all-reduce starts on a side stream as soon as that
    # core's gradient is final (the reverse sweep finishes the cores in reverse-use order) and runs under the rest
    # of the sweep; the step then only waits for the last one (reference: one blocking collective per core AFTER the
    # backward pass, comm_torch.py:292-318, 510-522)
    overlap = {"on": False, "checked": False}
    if dist is not None and train and oneshot is None and hasattr(fn, "set_grad_ready_hook") and not args.nccl_allreduce:
        comm_stream = torch.cuda.Stream(device=dev)
        overlap["on"] = True

        def grad_ready(name, flat):
            comm_stream.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(comm_stream):
                dist.all_reduce(flat)
                flat.div_(world)

        def average_overlapped(loss, grads):
            """all core gradients are already being reduced in place; only the loss is left"""
            l = loss.detach().reshape(1).clone()
            dist.all_reduce(l)
            l /= world
            torch.cuda.current_stream(dev).wait_stream(comm_stream)
            return l

    if dist is not None and train and oneshot is not None and not args.no_graphs:
        # the exchange is recorded into the training step's CUDA graph: a step is one graph launch
        fn.set_graph_epilogue(lambda loss0, grads: average(loss0, grads))

    last = {}                                  # what the latest step_device() returned (--dump-outputs)

    def step_device():
        if train:
            last["out"] = fn.loss_and_grads(cores_dict, states, mx_dev)
            loss, grads, _vals, _sc = last["out"]
            if dist is not None:
                if overlap["on"]:
                    average_overlapped(loss, grads)
                elif fn.graph_stats["last_extra"] is None:
                    average(loss, grads)
            return loss
        with torch.no_grad():
            if wl["mode"] == "fwdx":
                last["out"] = engine.contract_from_x(qctn, states, x_dev, K=K)
            else:
                last["out"] = fn(cores_dict, states, mx_dev)
            return last["out"]

    def outputs_of(out):
        """step_device()'s result as named arrays: loss, per-sample values, each core's gradient in qctn.cores
        order (grad_000, ...: two core names can differ only in case), and the values' (scale, log_scale)."""
        if not train:
            if isinstance(out, torch.Tensor):
                return {"values": out}
            return {"values": out.tensor, "scale": torch.tensor([float(out.scale), float(out.log_scale)], dtype=torch.float64)}
        loss, grads, vals, sc = out
        arrays = {"loss": loss, "values": vals}
        arrays.update((f"grad_{i:03d}", g) for i, g in enumerate(grads))
        if sc is not None:
            arrays["scale"] = torch.tensor([float(s) for s in sc], dtype=torch.float64)
        return arrays

    if overlap["on"]:
        # once, on the ranks that are about to be timed: the overlapped per-core exchange must give what ONE packed NCCL
        # all-reduce after the step gives (the cores are not updated in between)
        real = lambda g: torch.view_as_real(g).reshape(-1) if g.is_complex() else g.reshape(-1)
        loss_a, grads_a, _v, _s = fn.loss_and_grads(cores_dict, states, mx_dev)
        want = average(loss_a, grads_a)
        want = torch.cat([real(want[:-1]), want[-1:].real.reshape(1)]) if want.is_complex() else want
        del grads_a
        fn.set_grad_ready_hook(grad_ready)
        loss_b, grads_b, _v, _s = fn.loss_and_grads(cores_dict, states, mx_dev)
        l_b = average_overlapped(loss_b, grads_b)
        got = torch.cat([real(g) for g in grads_b] + [l_b.reshape(1).float()])
        err = (got - want.float()).abs().max().item() / max(want.abs().max().item(), 1e-30)
        assert err <= 1e-5, f"overlapped per-core all-reduce disagrees with the packed one: {err}"
        overlap["checked"], overlap["err"] = True, err
        del want, got, grads_b

    x_dev = x_local.to(dev).contiguous()
    use_graphs = train and not args.no_graphs
    # e2e input pipeline: two sets of STATIC device buffers (the CUDA-graph contract of
    # EngineSiamese.enable_cuda_graphs) filled from pinned host memory on a copy stream; the copy of
    # batch i+1 is issued before the contraction of batch i and awaited before the step ends, so
    # every timed step contains one full H2D of a batch (overlapped with compute) and the D2H of the loss
    # (the batch lives in ONE pinned (n, B, K, K) host tensor and one device tensor per slot, so a
    # step's input is a single cudaMemcpyAsync; the engine gets the per-qubit views it expects)
    host_all = torch.stack(mx_host, 0).pin_memory()
    dev_all = [torch.empty_like(host_all, device=dev) for _ in range(2)]
    mx_static = [[d[q] for q in range(nq)] for d in dev_all]
    copy_stream = torch.cuda.Stream(device=dev)
    pipe = {"i": 0, "ready": None}

    def issue_copy(slot):
        copy_stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(copy_stream):
            dev_all[slot].copy_(host_all, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    x_host = x_local.contiguous().pin_memory()
    x_static = [torch.empty_like(x_host, device=dev) for _ in range(2)]
    # the step's result travels back every step as an asynchronous D2H copy into pinned memory and is READ on the host one
    # step later (an event per copy): the host prepares step i+1 while step i runs instead of idling the GPU behind a
    # blocking .item() -- what a training loop that logs its loss does
    res_pin = torch.zeros(2, dtype=torch.float32).pin_memory()
    res = {"pending": None, "last": float("nan"), "reads": 0}

    def read_back(scalar):
        """queue the D2H copy of this step's result; return the previous step's value (read on the host now)"""
        slot = pipe["i"] % 2
        prev = res["pending"]
        if prev is not None:                       # the copy issued one step ago: wait for it, read it
            prev[0].synchronize()
            res["last"] = float(res_pin[prev[1]])
            res["reads"] += 1
        res_pin[slot:slot + 1].copy_(scalar.detach().reshape(1).float(), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        res["pending"] = (ev, slot)
        return res["last"]

    def step_e2e_x():
        """fwdx: the step's input is x itself (B x n floats from pinned host memory)."""
        cur = pipe["i"] % 2
        x_static[cur].copy_(x_host, non_blocking=True)
        with torch.no_grad():
            out = engine.contract_from_x(qctn, states, x_static[cur], K=K)
        val = read_back(out.sum())
        pipe["i"] += 1
        return val

    def step_e2e():
        if wl["mode"] == "fwdx":
            return step_e2e_x()
        cur = pipe["i"] % 2
        if pipe["ready"] is None:
            pipe["ready"] = issue_copy(cur)
        torch.cuda.current_stream(dev).wait_event(pipe["ready"])
        nxt_ready = issue_copy(1 - cur)
        mxs = [tb.TNTensor(d, sc, ls) for d, (sc, ls) in zip(mx_static[cur], mx_scales)]
        if train:
            loss, grads = engine.contract_with_compiled_strategy_for_gradient(qctn, states, mxs)
            if dist is not None:
                avg = fn.graph_stats["last_extra"]          # the exchange ran inside the step's graph ...
                if overlap["on"]:
                    avg = average_overlapped(loss, grads)   # ... or core by core under the reverse sweep (cfg4) ...
                elif avg is None:
                    avg = average(loss, grads)              # ... or the step was launched directly
                val = read_back(avg[-1])
            else:
                val = read_back(loss)
        else:
            with torch.no_grad():
                out = engine.contract_with_compiled_strategy(qctn, states, mxs)
            val = read_back(out.sum())
        torch.cuda.current_stream(dev).wait_event(nxt_ready)     # the next batch's H2D is part of this step
        pipe["ready"], pipe["i"] = nxt_ready, pipe["i"] + 1
        return val

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(step, steps, warmup):
        for _ in range(warmup):
            step()
        barrier()
        launches0 = _lib.launch_count()
        evs = []
        with ClockSampler(local_rank) as cs:
            for _ in range(steps):
                flush.fill_(1)                                 # evict L2 between timed steps (not timed)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step()
                e1.record()
                evs.append((e0, e1))
            barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        launches = _lib.launch_count() - launches0
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, cs.summary()

    if args.profile_step:
        for _ in range(args.warmup):
            step_device()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        step_device()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled": "one step", "workload": wl["name"]}), flush=True)
        return
    ms_total, launches, clocks = timed(step_device, args.steps, args.warmup)
    ms_step = ms_total / args.steps
    value = B_global / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # now: the e2e steps below replay the same CUDA graph, whose output buffers they overwrite
        dump_outputs(args.dump_outputs, outputs_of(last["out"]))

    e2e = None
    if not args.no_e2e:
        def step_e2e_timed():
            return step_e2e()
        # wall-clock inside CUDA events is not enough here (host work is part of e2e): use events
        # bracketing the whole call including the .item() read
        ms_e2e, _, _ = timed(step_e2e_timed, args.steps, 6)
        ms_e2e_step = ms_e2e / args.steps
        e2e = {"value": B_global / (ms_e2e_step * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e_step,
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
               "api": "EngineSiamese.contract_with_compiled_strategy" + ("_for_gradient" if train else ""),
               "pipeline": "H2D of batch i+1 (pinned host -> static device buffers, copy stream) overlaps step i; "
                           "awaited inside the timed step; the step's result is copied to pinned host memory every step "
                           "(asynchronous D2H) and read on the host one step later",
               "host_reads_of_result": res["reads"], "last_result_on_host": res["last"]}
        if not (res["reads"] > 0 and res["last"] == res["last"]):
            raise RuntimeError("e2e: the step results never reached the host")

    # roofline of the dominant kernel (tnq_body_kernel): measured alone with CUDA events
    bound = next(iter(fn.plans.values()))
    gemm_path = bound.use_gemm_path
    if gemm_path:
        runner = bound.gemm_runner("bwd" if train else "fwd")
        f0 = runner.flops
        step_device()
        torch.cuda.synchronize(dev)
        flops_launch = runner.flops - f0           # real fp32-equivalent flops of all GEMMs of one step
        info = None
    elif bound.chain_rank or bound.ladder:
        info = None
        # algorithmic flops: the plan compiler's pairwise count (= SURVEY 8(d) closed form for forward)
        flops_launch = bound.plan.program("train" if train else "fwd").flops_per_sample * B
    else:
        prog = bound.program("train" if train else "fwd")
        info = prog.info(B * bound.plan.nb)
        flops_launch = prog.prog.flops_per_sample * B * bound.plan.nb
    mx_bytes = B * nq * (1 if wl["mode"] == "fwdx" else K * K) * esz
    core_bytes = sum(v.numel() * esz for v in cores_cpu.values())
    alg_bytes = mx_bytes + B * 4 + core_bytes * (2 if train else 1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # measured fp32 FMA peak of this GPU (SURVEY 8(d): not in MEASURED_PEAKS.json; torch.matmul, TF32 off)
    torch.backends.cuda.matmul.allow_tf32 = False
    a = torch.randn(8192, 8192, device=dev)
    b = torch.randn(8192, 8192, device=dev)
    for _ in range(2):
        a @ b
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        a @ b
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, e0.elapsed_time(e1))
    fp32_peak = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    del a, b
    kernel_ms = ms_step  # the sweep kernel is >95% of the step (profiles/ ncu launch list)
    # DRAM bytes per launch of the dominant kernel (dram__bytes_read.sum + dram__bytes_write.sum of one
    # `ncu --set full` capture): cannot be measured live, so it is looked up in profiles/traffic.json under
    # the content hash of the kernel sources it was captured from -- a stale capture reads as null
    traffic = None
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = table.get(f"{args.workload}:{B}")
        if ent and world == 1 and ent.get("csrc_sha256") == ge.csrc_digest(ent.get("files")):
            traffic = ent["dram_bytes_per_launch"]
    except Exception:
        traffic = None
    achieved_tf = flops_launch / (kernel_ms * 1e-3) / 1e12
    hbm = {"algorithmic_bytes": alg_bytes, "achieved_gbs": alg_bytes / (kernel_ms * 1e-3) / 1e9,
           "peak_gbs": peaks.get("hbm_gbs"), "source": "MEASURED_PEAKS.json (measured)" if peaks else None}
    if gemm_path:
        # tensor-core roofline: fp32-equivalent flops; 3xTF32 issues 3 TF32 MMAs per product and dense TF32
        # runs at half the bf16 rate, so the fp32-equivalent peak is bf16_measured / 2 / 3
        bf16 = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0
        tc_peak = bf16 / 2.0 / 3.0
        roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": tc_peak, "unit": "TFLOP/s",
                    "frac": achieved_tf / tc_peak, "traffic": None,
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (measured)" if peaks else "fallback 1590")
                                   + " / 2 (TF32 rate) / 3 (3xTF32 passes); whole step incl. permutes",
                    "kernel": "tnq_gemm_tf32x3_kernel", "flops_per_launch": flops_launch,
                    "issued_tf32_tflops": 3 * achieved_tf, "fp32_simt_peak_measured": fp32_peak, "hbm": hbm}
    else:
        roofline = {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": achieved_tf / fp32_peak, "traffic": traffic if (bound.ladder or bound.chain_rank) else None,
                    "peak_source": "measured here: torch.matmul 8192^3 fp32 (TF32 off), best of 5",
                    "kernel": "tnq_chain_kernel" if bound.chain_rank else ("tnq_ladder_kernel" if bound.ladder else "tnq_body_kernel"),
                    "flops_per_launch": flops_launch, "hbm": hbm}
        if info is not None:
            roofline.update({"tile_samples": info.tile_samples, "grid": info.grid,
                             "frame_in_smem": bool(info.frame_in_smem), "smem_bytes": info.smem_bytes})
        if bound.chain_rank and hbm["peak_gbs"]:
            # the chain kernel streams Mx once: report the tighter of the two bounds as the headline
            hfrac = hbm["achieved_gbs"] / hbm["peak_gbs"]
            if hfrac > roofline["frac"]:
                roofline.update({"bound": "hbm", "achieved": hbm["achieved_gbs"], "peak": hbm["peak_gbs"], "unit": "GB/s",
                                 "frac": hfrac, "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)",
                                 "fp32": {"achieved_tflops": achieved_tf, "peak_tflops": fp32_peak}})

    line = {"metric": "samples/sec for QCTN fwd+bwd contraction" if train else "samples/sec for QCTN forward contraction",
            "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak" if weak else "strong",
            "vs_baseline": None,
            "dtype": "f32" if esz == 4 else "c64 (real fp32 arithmetic: 3xTF32 on tcgen05)", "data": "synthetic",
            "config": {"workload": wl["name"], "global_batch": B_global, "per_gpu_batch": B, "qubits": nq, "K": K,
                       "cores": len(names), "l2": "flushed between timed steps (256 MiB write)",
                       "cuda_graphs": bool(not args.no_graphs and (bound.ladder or bound.chain_rank) and wl["mode"] != "fwdx"),
                       "parallelism": f"batch sharded over {world} GPU(s); cores replicated; "
                                      + (("one one-shot NVLink all-reduce (tnq_allreduce_oneshot, symmetric memory) of grads+loss per step"
                                          if oneshot is not None else
                                          ("NCCL all-reduce per core, started when the core's gradient is final and overlapped with "
                                           "the rest of the reverse sweep" if overlap["on"] else
                                           "one packed NCCL all-reduce of grads+loss per step"))
                                         if world > 1 else "no collective"),
                       "oneshot_vs_nccl_rel_err": checked.get("err_vs_nccl"),
                       "overlapped_vs_packed_rel_err": overlap.get("err")},
            "clocks": clocks, "gpu_launches": launches, "roofline": roofline}
    if wl["mode"] == "fwdx":
        # the same job without the fusion: x -> generate_data (torch, device) -> contraction, timed the same way
        def step_unfused():
            with torch.no_grad():
                mats, _ = engine.generate_data(x_dev, K=K, ret_type="TNTensor")
                return engine.contract_with_compiled_strategy(qctn, states, mats)
        ms_unf, _, _ = timed(step_unfused, args.steps, 3)
        line["config"]["unfused_from_x_ms_per_step"] = ms_unf / args.steps
    if e2e is not None:
        line["e2e"] = e2e
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = time_reference(args, wl)
        line["cpu_baseline"] = {k: ref[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
