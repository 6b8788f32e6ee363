"""tnq_gemm_f64 on the GEMM shapes of one cfg4 step in complex128 (16 qubits, bond 64, B = 256), against
torch.matmul in float64 (cuBLAS DGEMM) on the same shapes: ms per call (CUDA events, 10 calls after 3 warm-up
calls), TFLOP/s, and the largest difference between the two relative to the largest entry.
    python tools/gemm_f64_only.py"""
import ctypes
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import tneq_b200  # noqa: F401
from tneq_b200 import _lib

# (M, N, K, batch, calls per cfg4 step): the forward contractions and the core-gradient GEMMs (split-K)
SHAPES = [(16384, 8192, 128, 1, 28), (4096, 128, 128, 256, 28), (16384, 128, 8192, 1, 28),
          (128, 8192, 16384, 1, 14), (8192, 128, 16384, 1, 14)]


def timed(fn, iters=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    lib = _lib.load()
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"device: {torch.cuda.get_device_name(dev)} ({q})")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    total_ours = total_cublas = 0.0
    for M, N, K, nb, per_step in SHAPES:
        torch.manual_seed(0)
        A = torch.randn(nb, M, K, dtype=torch.float64, device=dev)
        B = torch.randn(nb, N, K, dtype=torch.float64, device=dev)
        C = torch.empty(nb, M, N, dtype=torch.float64, device=dev)

        def ours():
            _lib.check(lib.tnq_gemm_f64(ctypes.c_void_p(A.data_ptr()), ctypes.c_void_p(B.data_ptr()),
                                        ctypes.c_void_p(C.data_ptr()), M, N, K, K, K, N, nb, M * K, N * K, M * N, 0, st))

        Bt = B.transpose(1, 2)
        ref = torch.empty_like(C)

        def cublas():
            torch.matmul(A, Bt, out=ref)

        ms_o, ms_c = timed(ours), timed(cublas)
        err = ((C - ref).abs().max() / ref.abs().max()).item()
        fl = 2.0 * M * N * K * nb
        total_ours += per_step * ms_o
        total_cublas += per_step * ms_c
        print(f"M {M:6d} N {N:5d} K {K:6d} batch {nb:4d}: tnq_gemm_f64 {ms_o:8.3f} ms {fl / ms_o / 1e9:6.2f} TFLOP/s | "
              f"cuBLAS DGEMM {ms_c:8.3f} ms {fl / ms_c / 1e9:6.2f} TFLOP/s | max diff {err:.1e} of the largest entry",
              flush=True)
        del A, B, C, ref, Bt
        torch.cuda.empty_cache()
    print(f"GEMMs of one cfg4 complex128 step: tnq_gemm_f64 {total_ours:.1f} ms, cuBLAS DGEMM {total_cublas:.1f} ms")


if __name__ == "__main__":
    main()
