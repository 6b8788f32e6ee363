"""Which cores the SGDG step sends to csrc/tnq_sgdg.cu (optim/steps.py::sgdg_kernel_eligible); no GPU needed."""
import os
import re

import pytest
import torch

from tneq_b200.optim import steps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDEST = {torch.float32: 64, torch.complex64: 64, torch.float64: 64, torch.complex128: 48}


def test_widths_match_the_header():
    """The Python table and the C header agree on every dtype's widest matrix."""
    text = open(os.path.join(ROOT, "include", "tneq_b200.h")).read()
    macros = dict(re.findall(r"#define (TNQ_SGDG_MAX_COLS\w*) (\d+)", text))
    names = {torch.float32: "TNQ_SGDG_MAX_COLS", torch.complex64: "TNQ_SGDG_MAX_COLS_C64",
             torch.float64: "TNQ_SGDG_MAX_COLS_F64", torch.complex128: "TNQ_SGDG_MAX_COLS_C128"}
    assert set(steps.SGDG_KERNELS) == set(names)
    for dtype, name in names.items():
        assert steps.SGDG_KERNELS[dtype][1] == int(macros[name]) == WIDEST[dtype]


@pytest.mark.parametrize("dtype", list(WIDEST), ids=[str(d)[6:] for d in WIDEST])
def test_stiefel_cores_up_to_the_widest_take_the_kernel(dtype):
    w = WIDEST[dtype]
    for shape in [(2, 2, 2, 2), (3, 3, 3, 3), (4, 4, 4, 4), (3, 3, 3), (3, 9), (8, 8), (4, 16), (1, w), (w, w)]:
        assert steps.sgdg_kernel_eligible(dtype, shape, "cuda"), shape
        assert steps.sgdg_kernel_eligible(dtype, torch.Size(shape), "cuda"), shape
    for shape in [(w + 1, w + 1), (1, w + 1), (9, 3), (4, 2, 1), (5,), ()]:
        # wider than the dtype's maximum, more rows than columns (not a Stiefel core), or no matrix at all
        assert not steps.sgdg_kernel_eligible(dtype, shape, "cuda"), shape
    assert not steps.sgdg_kernel_eligible(dtype, (3, 3, 3, 3), "cpu")


def test_per_dtype_limits():
    assert steps.sgdg_kernel_eligible(torch.complex64, (8, 8, 8, 8), "cuda")
    assert steps.sgdg_kernel_eligible(torch.float64, (8, 8, 8, 8), "cuda")
    assert not steps.sgdg_kernel_eligible(torch.complex128, (8, 8, 8, 8), "cuda")
    assert not steps.sgdg_kernel_eligible(torch.complex128, (7, 7, 7, 7), "cuda")
    assert steps.sgdg_kernel_eligible(torch.complex128, (6, 8, 6, 8), "cuda")
    for dtype in (torch.float16, torch.bfloat16, torch.int32):
        assert not steps.sgdg_kernel_eligible(dtype, (3, 3, 3, 3), "cuda")
