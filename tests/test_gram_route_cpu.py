"""GramCache's route decision on plain integers (no GPU, no library build): which library call takes an activation of
each precision, shape, alignment and dtype, and which routes may wait for the grouped launch of flush()."""
import pytest
import torch

from vl_merging_b200.gram import _DEFERRED_ROUTES, _GramLaunch, _gram_route

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
A = 1 << 20     # a 16-byte aligned activation address
TEXT = 40 * 64  # rows of a VLMo-base text Gram at batch 64


# (precision, use_simt, dtype, rows, d, ptr, ldx, seg_stride) -> route
CASES = [
    # int8x4: the integer tensor cores from 2^20 elements, d % 128 == 0 and 16-byte / 4-element alignment; fp64 otherwise
    (("int8x4", False, F32, 2048, 512, A, 512, 0), "i8x4"),               # rows * d == 2^20
    (("int8x4", False, F32, 2047, 512, A, 512, 0), "f64"),                # one row short of 2^20 elements
    (("int8x4", False, F32, TEXT, 768, A, 768, 0), "i8x4"),
    (("int8x4", False, F32, 36928, 3072, A, 3072, 0), "i8x4"),
    (("int8x4", False, BF16, 36928, 768, A, 768, 0), "i8x4"),
    (("int8x4", False, F16, 36928, 768, A, 768, 0), "i8x4"),
    (("int8x4", False, F32, 36928, 192, A, 192, 0), "f64"),               # d % 128 != 0
    (("int8x4", False, F32, 36928, 800, A, 800, 0), "f64"),
    (("int8x4", False, F32, 36928, 768, A + 8, 768, 0), "f64"),           # ptr % 16 != 0
    (("int8x4", False, F32, 36928, 768, A, 770, 0), "f64"),               # ldx % 4 != 0
    (("int8x4", False, F32, 64 * 577, 768, A, 768, 617 * 768), "i8x4"),   # row slice h[:, 40:] of (64, 617, 768)
    (("int8x4", False, F32, 64 * 577, 768, A, 768, 617 * 768 + 2), "f64"),  # seg_stride % 4 != 0
    (("int8x4", True, F32, 36928, 768, A, 768, 0), "i8x4"),               # use_simt leaves fp64 Grams alone
    (("int8x4", True, F32, 1000, 768, A, 768, 0), "f64"),
    # fp64: always the fp64 pipe
    (("fp64", False, F32, 36928, 768, A, 768, 0), "f64"),
    (("fp64", False, BF16, 100, 200, A + 2, 201, 0), "f64"),
    (("fp64", True, F32, 36928, 3072, A, 3072, 0), "f64"),
    # tf32x3: fp32 activations split when d % 32 == 0, ptr 16-byte aligned, ldx and seg_stride multiples of 4
    (("tf32x3", False, F32, 36928, 768, A, 768, 0), "split"),
    (("tf32x3", False, F32, TEXT, 768, A, 768, 0), "split"),
    (("tf32x3", False, F32, 64 * 577, 768, A, 768, 617 * 768), "split"),
    (("tf32x3", False, F32, 1000, 200, A, 200, 0), "simt"),               # d % 32 != 0
    (("tf32x3", False, F32, 1000, 768, A + 4, 768, 0), "simt"),           # ptr % 16 != 0
    (("tf32x3", False, F32, 1000, 768, A, 770, 0), "simt"),               # ldx % 4 != 0
    (("tf32x3", False, F32, 64 * 577, 768, A, 768, 617 * 768 + 2), "simt"),  # seg_stride % 4 != 0
    (("tf32x3", False, BF16, 36928, 768, A, 768, 0), "library"),          # exact tensor-core operands already
    (("tf32x3", False, F16, 1000, 200, A + 2, 201, 0), "library"),
    (("tf32x3", True, F32, 36928, 768, A, 768, 0), "simt"),
    (("tf32x3", True, BF16, 36928, 768, A, 768, 0), "simt"),
    # tf32: the library picks the kernel, whatever the shape, unless use_simt
    (("tf32", False, F32, 36928, 3072, A, 3072, 0), "library"),
    (("tf32", False, F32, 1000, 200, A + 4, 201, 0), "library"),
    (("tf32", False, BF16, 64 * 577, 768, A, 768, 617 * 768), "library"),
    (("tf32", True, F32, 36928, 3072, A, 3072, 0), "simt"),
    (("tf32", True, F16, 1000, 768, A, 768, 0), "simt"),
]


@pytest.mark.parametrize("args,route", CASES, ids=[f"{a[0]}-{i}-{r}" for i, (a, r) in enumerate(CASES)])
def test_route(args, route):
    assert _gram_route(*args) == route


def test_every_route_is_taken():
    assert {r for _, r in CASES} == {"i8x4", "f64", "simt", "split", "library"}


@pytest.mark.parametrize("route,deferred", [("i8x4", False), ("f64", False), ("simt", False), ("split", True),
                                            ("library", True)])
def test_deferred_routes(route, deferred):
    """Only the routes vlm_syrk_accum_batch takes wait for flush(); fp64 Grams and the CUDA-core kernel launch at once."""
    assert (route in _DEFERRED_ROUTES) == deferred


def test_record_keeps_rows_and_d_at_4_and_5():
    """bench.py's TimedCache reads (rows, d) of a pending record as its fields 4 and 5."""
    assert _GramLaunch._fields[:9] == ("code", "keep", "g", "ptr", "rows", "d", "ldx", "seg_rows", "seg_stride")
