"""_lib.py — ctypes binding of libvlmerge.so (C ABI: include/vlmerge.h).

There is no fallback: if the library is missing, or a call fails, the caller gets an exception.
"""
import ctypes
import itertools
import os
import subprocess
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libvlmerge.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

VLM_F32, VLM_BF16, VLM_F16, VLM_F64, VLM_TF32X2 = 0, 1, 2, 3, 4
MERGE_WSUM, MERGE_SEQ_LERP, MERGE_MEAN = 0, 1, 2
MERGE_MAX_SRC = 4
ERR_NOT_SPD = -5


class MergeSeg(ctypes.Structure):
    """vlm_merge_seg"""
    _fields_ = [
        ("dst", c_void_p),
        ("src", c_void_p * MERGE_MAX_SRC),
        ("coef", c_float * MERGE_MAX_SRC),
        ("n", c_uint64),
        ("n_src", c_int32),
        ("mode", c_int32),
    ]


class SymItem(ctypes.Structure):
    """vlm_sym_item"""
    _fields_ = [("full", c_void_p), ("packed", c_void_p), ("d", c_int32), ("reserved", c_int32), ("ld", c_int64)]


def sym_items(grams, packed=None, offsets=None):
    """vlm_sym_item array for the square row-major tensors `grams`.  packed: the flat tensor of the packed upper
    triangles, Gram i's from element offsets[i] on (offsets None: back to back in list order); None for
    vlm_sym_mirror_batch, which reads no packed form."""
    items = (SymItem * len(grams))()
    if offsets is None:
        offsets = itertools.accumulate((g.shape[0] * (g.shape[0] + 1) // 2 for g in grams), initial=0)
    for it, g, off in zip(items, grams, offsets):
        it.full, it.d, it.ld = g.data_ptr(), g.shape[0], g.stride(0)
        if packed is not None:
            it.packed = packed.data_ptr() + packed.element_size() * off
    return items


class SymSpan(ctypes.Structure):
    """vlm_sym_span"""
    _fields_ = [("offset_bytes", ctypes.c_uint64), ("d", c_int32), ("reserved", c_int32), ("ld", c_int64)]


class SyrkProblem(ctypes.Structure):
    """vlm_syrk_problem"""
    _fields_ = [
        ("x", c_void_p),
        ("rows", c_int64),
        ("ldx", c_int64),
        ("g", c_void_p),
        ("ldg", c_int64),
        ("d", c_int32),
        ("reserved", c_int32),
        ("seg_rows", c_int64),
        ("seg_stride", c_int64),
    ]


class VlmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libvlmerge error {code}: {msg}")
        self.code = code


# every symbol include/vlmerge.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "vlm_version": (c_int, []),
    "vlm_last_error": (c_char_p, []),
    "vlm_launch_count": (c_uint64, []),
    "vlm_set_deterministic": (c_int, [c_int]),
    "vlm_get_deterministic": (c_int, []),
    "vlm_syrk_accum": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int64, c_void_p]),
    "vlm_tf32_split": (c_int, [c_void_p, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "vlm_syrk_accum_f64": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                   c_void_p]),
    "vlm_syrk_i8x4_scratch_bytes": (c_uint64, [c_int64, c_int]),
    "vlm_syrk_accum_i8x4": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_uint64,
                                    c_void_p, c_int64, c_void_p]),
    "vlm_syrk_accum_batch": (c_int, [POINTER(SyrkProblem), c_int, c_int, c_void_p]),
    "vlm_syrk_accum_strided": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                       c_void_p]),
    "vlm_syrk_accum_simt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int64, c_void_p]),
    "vlm_sym_pack_upper_batch": (c_int, [POINTER(SymItem), c_int, c_int, c_void_p]),
    "vlm_sym_unpack_batch": (c_int, [POINTER(SymItem), c_int, c_int, c_void_p]),
    "vlm_sym_allreduce_multimem": (c_int, [c_void_p, POINTER(SymSpan), c_int, c_int, c_int, c_int, c_void_p]),
    "vlm_sym_mirror_batch": (c_int, [POINTER(SymItem), c_int, c_int, c_void_p]),
    "vlm_syrk_pair_schedule_host": (c_int, [c_int64, c_int, c_int, c_int, POINTER(c_int32), c_int, POINTER(c_int32),
                                            c_int, POINTER(c_int)]),
    "vlm_merge_plan_create": (c_int, [POINTER(MergeSeg), c_int, POINTER(c_void_p)]),
    "vlm_merge_plan_run": (c_int, [c_void_p, c_void_p]),
    "vlm_merge_plan_destroy": (c_int, [c_void_p]),
    "vlm_merge_plan_bytes": (c_uint64, [c_void_p]),
    "vlm_copy_batch": (c_int, [c_void_p, POINTER(c_uint64), POINTER(c_void_p), POINTER(c_uint64), c_int, c_void_p]),
    "vlm_gram_scale_accum": (c_int, [c_void_p, c_int, c_int, c_int64, c_double, c_void_p, c_int64, c_int, c_void_p]),
    "vlm_regmean_rhs": (c_int, [c_void_p, c_int, c_int, c_int64, c_void_p, c_int, c_int64, c_double, c_void_p,
                                c_int64, c_int, c_void_p]),
    "vlm_regmean_rhs_diff": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p, c_int, c_int64, c_double,
                                     c_void_p, c_int64, c_int, c_void_p]),
    "vlm_widen_add": (c_int, [c_void_p, c_int, c_int, c_int64, c_void_p, c_int64, c_void_p]),
    "vlm_spd_solve_right": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p]),
    "vlm_sim_topk_splits": (c_int, [c_int64, c_int64]),
    "vlm_sim_topk": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int,
                             c_void_p]),
    "vlm_lu_solve_right": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p]),
    "vlm_spd_solve_right_async": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p, c_void_p]),
}

_lib = None


def build(verbose=False):
    """Compile libvlmerge.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", CSRC_DIR, f"-j{min(8, os.cpu_count() or 1)}", "all"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building libvlmerge.so failed (see output above)")
    return LIB_PATH


def lib():
    """The loaded library; raises if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C vl-merging_b200/csrc`.  There is no CPU fallback for the merge hot path.")
        h = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            if not hasattr(h, name):
                raise RuntimeError(f"{LIB_PATH} does not export {name}: rebuild it (make -C vl-merging_b200/csrc)")
            fn = getattr(h, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if h.vlm_version() != 3:
            raise RuntimeError(f"libvlmerge ABI version {h.vlm_version()} != 3: rebuild it (make -C vl-merging_b200/csrc)")
        _lib = h
    return _lib


def check(rc):
    if rc != 0:
        raise VlmError(rc, lib().vlm_last_error().decode(errors="replace"))


def launch_count():
    return int(lib().vlm_launch_count())


def syrk_pair_schedule(rows, d, elem_bytes=4, nsm=148):
    """Host-side view of the CTA-pair SYRK decomposition: (list of (super_row, super_col, k0, k1), offsets)."""
    cap = 1 << 16
    segs = (c_int32 * (4 * cap))()
    off = (c_int32 * (nsm + 2))()
    ncl = c_int(0)
    n = lib().vlm_syrk_pair_schedule_host(rows, d, elem_bytes, nsm, segs, cap, off, nsm + 2, ctypes.byref(ncl))
    if n < 0:
        check(n)
    return [tuple(segs[4 * i: 4 * i + 4]) for i in range(n)], list(off[: ncl.value + 1])
