"""tcgen05 3xTF32 GEMM (tnq_gemm_tf32x3) against a float64 torch reference.

Tolerance: 3xTF32 keeps ~21 mantissa bits per product; with fp32 accumulation the result must
be within 1e-5 of the float64 product relative to the largest entry (north_star's bound), and in
practice lands near plain fp32 (few 1e-7)."""
import ctypes

import pytest
import torch

from helpers import gemm_splitk

pytestmark = pytest.mark.gpu


def _gemm(A, B, C=None, accumulate=False):
    """A: [b, M, K] (or [M, K]) row-major, B: [b, N, K]; returns C [b, M, N] = A @ B^T."""
    from tneq_b200 import _lib
    lib = _lib.load()
    A3 = A if A.dim() == 3 else A[None]
    B3 = B if B.dim() == 3 else B[None]
    nb = max(A3.shape[0], B3.shape[0])
    M, K = A3.shape[-2:]
    N = B3.shape[-2]
    if C is None:
        C = torch.empty(nb, M, N, device=A.device, dtype=torch.float32)
    sA = A3.stride(0) if A3.shape[0] > 1 else 0
    sB = B3.stride(0) if B3.shape[0] > 1 else 0
    rc = lib.tnq_gemm_tf32x3(ctypes.c_void_p(A3.data_ptr()), ctypes.c_void_p(B3.data_ptr()), ctypes.c_void_p(C.data_ptr()),
                             M, N, K, A3.stride(-2), B3.stride(-2), C.stride(-2), nb, sA, sB, C.stride(0),
                             1 if accumulate else 0, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc)
    return C


@pytest.mark.parametrize("M,N,K,nb", [(128, 128, 32, 1), (128, 128, 128, 1), (256, 384, 96, 1), (100, 72, 36, 1),
                                      (1, 8, 4, 1), (300, 130, 260, 3), (4096, 128, 128, 2), (64, 8192, 128, 1),
                                      # long k-loop over few tiles: split-K by two (atomic adds into a zeroed tile)
                                      (128, 384, 4096, 1), (100, 130, 1500, 1)])
def test_gemm_matches_float64(M, N, K, nb, built_lib):
    torch.manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(nb, M, K, device="cuda")
    B = torch.randn(nb, N, K, device="cuda")
    C = _gemm(A, B)
    torch.cuda.synchronize()
    ref = A.double() @ B.double().transpose(-1, -2)
    err = ((C.double() - ref).abs().max() / ref.abs().max()).item()
    assert err < 1e-5, err
    torch.backends.cuda.matmul.allow_tf32 = False
    fp32 = ((A @ B.transpose(-1, -2)).double() - ref).abs().max() / ref.abs().max()
    assert err < 20 * fp32.item() + 1e-7        # fp32-faithful, not TF32-grade (1e-3)


def test_gemm_shared_operand_strides_and_accumulate(built_lib):
    torch.manual_seed(5)
    nb, M, N, K = 5, 96, 40, 64
    Abig = torch.randn(nb, M, K + 12, device="cuda")
    A = Abig[:, :, :K]                                   # lda > K
    B = torch.randn(N, K, device="cuda")                 # shared across the batch (stride 0)
    C0 = torch.randn(nb, M, N, device="cuda")
    C = _gemm(A, B, C0.clone(), accumulate=True)
    torch.cuda.synchronize()
    ref = C0.double() + A.double() @ B.double().T
    assert ((C.double() - ref).abs().max() / ref.abs().max()).item() < 1e-5


def test_gemm_unaligned_shapes(built_lib):
    """Odd K / leading dimensions (outer products, K = 1) go through the guarded scalar loader."""
    torch.manual_seed(9)
    for M, N, K in [(8, 6, 6), (1, 16, 1), (50, 3, 7), (130, 129, 33)]:
        A = torch.randn(2, M, K, device="cuda")
        B = torch.randn(2, N, K, device="cuda")
        C = _gemm(A, B)
        torch.cuda.synchronize()
        ref = A.double() @ B.double().transpose(-1, -2)
        assert ((C.double() - ref).abs().max() / ref.abs().max()).item() < 1e-5


@pytest.mark.parametrize("R1,R0,K1,K0,N", [(3, 64, 5, 64, 128), (2, 256, 3, 128, 72), (5, 32, 9, 32, 40), (1, 128, 4, 96, 130),
                                           (256, 64, 4, 128, 128),
                                           # split-K (K >= 1024, at most 74 tiles): the (k1, k0) k-blocks are divided
                                           # between two CTAs; K1 odd puts the split inside a k1 group
                                           (2, 64, 16, 64, 128), (4, 128, 8, 128, 256), (1, 128, 33, 32, 72),
                                           # cfg4's forward view: 128 row tiles, K = 8192, no split-K
                                           (256, 64, 64, 128, 128)])
def test_gemm_strided_view_operand(R1, R0, K1, K0, N, built_lib):
    """tnq_gemm_tf32x3_view: the A operand is read in place through a 4-D tensor map -- memory order
    [r1][k1][r0][k0], rows (r1, r0), contraction index (k1, k0) -- i.e. the transposition is done by the TMA
    unit; against float64 of the explicitly permuted operand (tile tails in M through zero fill)."""
    from tneq_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(R1 * 100 + K1)
    X = torch.randn(R1, K1, R0, K0, device="cuda")
    B = torch.randn(N, K1 * K0, device="cuda")
    M, K = R1 * R0, K1 * K0
    C = torch.empty(M, N, device="cuda")
    rc = lib.tnq_gemm_tf32x3_view(ctypes.c_void_p(X.data_ptr()), R1, R0, X.stride(0), X.stride(2), K1, K0, X.stride(1),
                                  ctypes.c_void_p(B.data_ptr()), K, ctypes.c_void_p(C.data_ptr()), N, N,
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc)
    torch.cuda.synchronize()
    ref = X.permute(0, 2, 1, 3).reshape(M, K).double() @ B.double().T
    err = ((C.double() - ref).abs().max() / ref.abs().max()).item()
    assert err < 1e-5, (err, gemm_splitk(M, N, K))
    # not expressible (K0 not a multiple of 32): refused without a launch, the caller transposes
    assert lib.tnq_gemm_tf32x3_view(ctypes.c_void_p(X.data_ptr()), R1, R0, X.stride(0), X.stride(2), K1, K0 - 4, X.stride(1),
                                    ctypes.c_void_p(B.data_ptr()), K, ctypes.c_void_p(C.data_ptr()), N, N,
                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)) == -2


@pytest.mark.parametrize("a_mn,b_mn,ta,tb,batch,Kin", [(1, 1, 1, 3, 5, 64), (1, 0, 2, 1, 9, 32), (0, 1, 1, 2, 4, 96), (1, 1, 1, 64, 256, 64),
                                                       # one operand MN-major with split-K (64 tiles, K = 2048 and 16 384:
                                                       # the core gradients of cfg4) ...
                                                       (1, 0, 1, 64, 32, 64), (0, 1, 64, 1, 32, 64), (1, 0, 64, 1, 256, 64),
                                                       (0, 1, 1, 64, 256, 64),
                                                       # ... and without it (more than 74 output tiles)
                                                       (1, 0, 1, 80, 16, 64), (0, 1, 80, 1, 16, 64), (1, 1, 5, 16, 8, 128)])
def test_gemm_batch_into_k_mn_major_in_place(a_mn, b_mn, ta, tb, batch, Kin, built_lib):
    """tnq_gemm_tf32x3_bk: C[m, n] = sum_{b, k} A_b[m, k] B_b[n, k] with operands stored [batch][row tile][k][128 rows]
    consumed IN PLACE (5-D tensor map with the 32-byte-atom swizzle, MN-major UMMA descriptors of layout type
    SWIZZLE_128B_BASE32B) -- the core-gradient contraction of the large-bond
    sweep without the transposition -- against float64."""
    from tneq_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(a_mn * 10 + b_mn + batch)
    M, N = ta * 128, tb * 128

    def operand(mn, tiles):
        if mn:
            x = torch.randn(batch, tiles, Kin, 128, device="cuda")                  # in place
            ref = x.permute(1, 3, 0, 2).reshape(tiles * 128, batch * Kin)           # rows (tile, r), K (b, k)
        else:
            x = torch.randn(tiles * 128, batch * Kin, device="cuda")
            ref = x
        return x, ref.double()

    A, Ar = operand(a_mn, ta)
    B, Br = operand(b_mn, tb)
    C = torch.empty(M, N, device="cuda")
    rc = lib.tnq_gemm_tf32x3_bk(ctypes.c_void_p(A.data_ptr()), a_mn, ta, ctypes.c_void_p(B.data_ptr()), b_mn, tb,
                                ctypes.c_void_p(C.data_ptr()), M, N, batch, Kin,
                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc)
    torch.cuda.synchronize()
    ref = Ar @ Br.T
    err = ((C.double() - ref).abs().max() / ref.abs().max()).item()
    assert err < 1e-5, err


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def test_gemm_refusals_launch_nothing(built_lib):
    """What tnq_gemm_tf32x3_bk and tnq_gemm_tf32x3_view cannot express returns -2 with nothing launched (the caller
    then transposes explicitly), and C is left untouched."""
    from tneq_b200 import _lib
    lib = _lib.load()
    X = torch.randn(1 << 20, device="cuda")
    C = torch.full((1 << 16,), 7.0, device="cuda")
    n0 = _lib.launch_count()
    # bk: Kin not a multiple of 32; M != 128 a_tiles (A MN-major); N != 128 b_tiles; K = batch * Kin <= 256
    assert lib.tnq_gemm_tf32x3_bk(_p(X), 1, 1, _p(X), 0, 0, _p(C), 128, 128, 16, 48, _stream()) == -2
    assert lib.tnq_gemm_tf32x3_bk(_p(X), 1, 2, _p(X), 0, 0, _p(C), 128, 128, 16, 64, _stream()) == -2
    assert lib.tnq_gemm_tf32x3_bk(_p(X), 0, 0, _p(X), 1, 1, _p(C), 128, 256, 16, 64, _stream()) == -2
    assert lib.tnq_gemm_tf32x3_bk(_p(X), 1, 1, _p(X), 1, 1, _p(C), 128, 128, 8, 32, _stream()) == -2
    assert lib.tnq_gemm_tf32x3_bk(_p(X), 1, 1, _p(X), 1, 1, _p(C), 128, 128, 4, 64, _stream()) == -2
    # view: K = K1 * K0 <= 256
    assert lib.tnq_gemm_tf32x3_view(_p(X), 2, 64, 2 * 128 * 64, 128, 2, 128, 64 * 128, _p(X), 256, _p(C), 128, 128,
                                    _stream()) == -2
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0
    assert bool((C == 7.0).all())


def _row_err(C, ref):
    """max over output rows of |C - ref| relative to that row's own largest |ref|"""
    C, ref = C.double(), ref.double()
    return ((C - ref).abs().amax(-1) / ref.abs().amax(-1)).max().item()


@pytest.mark.parametrize("variant", ["plain", "plain_splitk", "view", "view_splitk", "bk_a_mn", "bk_b_mn_splitk"])
def test_gemm_rows_of_very_different_magnitude(variant, built_lib):
    """Rows of A scaled by 2^e, e in [-40, 40] (a sweep's rows are samples whose values differ by orders of magnitude):
    every output row must be right relative to ITS OWN largest entry -- a bound relative to the global maximum cannot
    see a row that lost its digits."""
    from tneq_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(len(variant))
    N, K = {"plain": (1280, 512), "plain_splitk": (256, 2048), "view": (256, 512), "view_splitk": (128, 1024),
            "bk_a_mn": (128 * 80, 1024), "bk_b_mn_splitk": (128, 2048)}[variant]
    M = 256
    e = torch.randint(-40, 41, (M,), device="cuda").double()
    scale = torch.pow(2.0, e).float()
    if variant.startswith("plain"):
        A = torch.randn(M, K, device="cuda") * scale[:, None]
        B = torch.randn(N, K, device="cuda")
        C = _gemm(A, B)[0]
        ref = A.double() @ B.double().T
    elif variant.startswith("view"):
        R0, K0 = 64, 128                              # memory [r1][k1][r0][k0], rows (r1, r0)
        R1, K1 = M // R0, K // K0
        X = torch.randn(R1, K1, R0, K0, device="cuda") * scale.reshape(R1, 1, R0, 1)
        B = torch.randn(N, K, device="cuda")
        C = torch.empty(M, N, device="cuda")
        _lib.check(lib.tnq_gemm_tf32x3_view(_p(X), R1, R0, X.stride(0), X.stride(2), K1, K0, X.stride(1), _p(B), K, _p(C),
                                            N, N, _stream()))
        ref = X.permute(0, 2, 1, 3).reshape(M, K).double() @ B.double().T
    else:
        Kin = 64
        batch = K // Kin
        if variant == "bk_a_mn":                      # A in place [batch][tiles][Kin][128], B K-major
            X = torch.randn(batch, M // 128, Kin, 128, device="cuda") * scale.reshape(1, M // 128, 1, 128)
            Bm = torch.randn(N, K, device="cuda")
            C = torch.empty(M, N, device="cuda")
            _lib.check(lib.tnq_gemm_tf32x3_bk(_p(X), 1, M // 128, _p(Bm), 0, 0, _p(C), M, N, batch, Kin, _stream()))
            ref = X.permute(1, 3, 0, 2).reshape(M, K).double() @ Bm.double().T
        else:                                         # A K-major with scaled rows, B in place
            A = torch.randn(M, K, device="cuda") * scale[:, None]
            Y = torch.randn(batch, N // 128, Kin, 128, device="cuda")
            C = torch.empty(M, N, device="cuda")
            _lib.check(lib.tnq_gemm_tf32x3_bk(_p(A), 0, 0, _p(Y), 1, N // 128, _p(C), M, N, batch, Kin, _stream()))
            ref = A.double() @ Y.permute(1, 3, 0, 2).reshape(N, K).double().T
    torch.cuda.synchronize()
    assert gemm_splitk(M, N, K) == variant.endswith("splitk")
    err = _row_err(C, ref)
    assert err < 1e-5, err
