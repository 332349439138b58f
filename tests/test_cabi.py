"""The C-ABI library loads and exports every symbol include/vlmerge.h declares (no compute, no GPU)."""
import ctypes
import os
import re

import pytest

import vl_merging_b200 as vlm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "vlmerge.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vlm_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound():
    names = _declared_symbols()
    assert len(names) >= 14
    if not os.path.exists(vlm._lib.LIB_PATH):
        vlm.build()
    h = ctypes.CDLL(vlm._lib.LIB_PATH)
    for n in names:
        assert hasattr(h, n), f"{n} declared in include/vlmerge.h but not exported"
    assert sorted(vlm._lib.SIGNATURES) == names  # the ctypes shim binds exactly the header
    assert vlm._lib.lib().vlm_version() == 3
    assert vlm._lib.lib().vlm_last_error() is not None


def test_merge_seg_layout_matches_header():
    # dst(8) + src[4](32) + coef[4](16) + n(8) + n_src(4) + mode(4)
    assert ctypes.sizeof(vlm._lib.MergeSeg) == 72
    assert vlm._lib.MergeSeg.n.offset == 56 and vlm._lib.MergeSeg.mode.offset == 68


def test_argument_validation_happens_before_any_cuda_call():
    L = vlm._lib.lib()
    assert L.vlm_syrk_accum(None, 0, 16, 128, 128, None, 128, None) == -1       # g is NULL
    assert b"g is NULL" in L.vlm_last_error()
    assert L.vlm_syrk_accum(None, 7, 16, 128, 128, None, 128, None) == -1       # bad dtype
    assert L.vlm_sym_mirror_batch(None, 1, vlm._lib.VLM_F32, None) == -1
    assert L.vlm_merge_plan_run(None, None) == -1
    assert L.vlm_regmean_rhs(None, 1, 1, 1, None, 3, 1, 1.0, None, 1, 0, None) == -1
    # the integer-tensor-core Gram: dtype, width and alignment are checked up front
    buf = (ctypes.c_char * 4096)()
    a16 = (ctypes.addressof(buf) + 15) & ~15
    assert L.vlm_syrk_accum_i8x4(a16, 9, 32, 128, 128, 0, 0, a16, 1 << 20, a16, 128, None) == -1        # bad dtype
    assert L.vlm_syrk_accum_i8x4(a16, vlm._lib.VLM_F32, 32, 96, 96, 0, 0, a16, 1 << 20, a16, 96, None) != 0   # d % 128
    assert b"multiple of 128" in L.vlm_last_error()
    assert L.vlm_syrk_accum_i8x4(a16 + 4, vlm._lib.VLM_F16, 32, 128, 128, 0, 0, a16, 1 << 20, a16, 128, None) != 0  # x alignment
    assert L.vlm_syrk_accum_i8x4(a16, vlm._lib.VLM_F32, 32, 128, 128, 0, 0, a16, 16, a16, 128, None) == -1  # scratch too small
    assert L.vlm_syrk_i8x4_scratch_bytes(32, 128) >= 4 * 32 * 128 + 8 * 128
    seg = vlm._lib.MergeSeg()
    seg.n_src = 9
    plan = ctypes.c_void_p()
    assert L.vlm_merge_plan_create(ctypes.pointer(seg), 1, ctypes.byref(plan)) == -1
    with pytest.raises(vlm.VlmError):
        vlm._lib.check(-1)


def test_no_cpu_fallback_without_cuda():
    import torch

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        vlm.GramCache(device="cpu")
    with pytest.raises(RuntimeError, match="CUDA device only"):
        vlm.merge_weights({"a": torch.zeros(1)}, {})
