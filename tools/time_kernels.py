"""Development helper: device time of the library's entry points at the shapes of VLMo-base calibration and merging.

    python tools/time_kernels.py [--full] [--only SUBSTR]

Every case calls the C ABI through `_lib` on torch buffers, warms its shape up, then times a run of launches on the
current stream between two CUDA events.  One JSON line per case: name, shape, ms per launch, and the rate:
rows * d * (d + 1) flops for a SYRK (the symmetric count), 2 * out * in * in for the RegMean right-hand side,
2 * m * n * d for the similarity, vlm_merge_plan_bytes for the merge.  The first line names the card, its power
limit and its top SM clock, read with nvidia-smi (read only: no setting is changed).  Nothing is checked for
correctness here: the pytest suite does that.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vl_merging_b200 import _lib  # noqa: E402

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
CODE = {F32: _lib.VLM_F32, BF16: _lib.VLM_BF16, F16: _lib.VLM_F16}
SHORT = {F32: "f32", BF16: "bf16", F16: "f16"}


def card():
    """name, power limit and top SM clock of cuda:0 as nvidia-smi reports them."""
    query = ["nvidia-smi", f"--id=GPU-{torch.cuda.get_device_properties(0).uuid}",
             "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        name, power, clock = (s.strip() for s in subprocess.run(query, capture_output=True, text=True,
                                                                 check=True).stdout.strip().split(","))
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, power, clock = torch.cuda.get_device_name(0), None, None
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


class Timer:
    def __init__(self, only):
        self.only = only
        self.lib = _lib.lib()
        self.stream = torch.cuda.current_stream().cuda_stream

    def wants(self, name):
        return self.only is None or self.only in name

    def run(self, name, shape, fn, iters=10, work=None, unit="TFLOP/s"):
        """fn() launches once and returns the library's status.  work: flops (or bytes for GB/s) of one launch."""
        for _ in range(3):
            _lib.check(fn())
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            _lib.check(fn())
        b.record()
        b.synchronize()
        self.report(name, shape, a.elapsed_time(b) / iters, work, unit)

    @staticmethod
    def report(name, shape, ms, work, unit):
        scale = 1e-9 if unit == "TFLOP/s" else 1e-6     # work / ms -> TFLOP/s or GB/s
        print(json.dumps({"case": name, "shape": shape, "ms": round(ms, 4), unit: round(work / ms * scale, 1)}), flush=True)


def syrk_flops(rows, d):
    return rows * d * (d + 1)


def time_syrk(t, full):
    shapes = [(F32, 2560, 768), (F32, 2560, 3072), (F32, 36928, 768), (F32, 36928, 3072), (BF16, 36928, 768),
              (BF16, 36928, 3072)]
    if full:
        shapes += [(F32, 36928, 1024), (F32, 36928, 4096), (F16, 36928, 4096)]
    for dtype, rows, d in shapes:
        name = f"syrk {SHORT[dtype]} {rows}x{d}"
        if t.wants(name):
            x = torch.randn(rows, d, device="cuda").to(dtype)
            g = torch.zeros(d, d, device="cuda")
            t.run(name, [rows, d], lambda: t.lib.vlm_syrk_accum(x.data_ptr(), CODE[dtype], rows, d, d, g.data_ptr(), d,
                                                                t.stream), work=syrk_flops(rows, d))


def time_strided(t):
    """The text and image row slices of a 64 x 617 x 768 activation, read in place, and the contiguous kernel on a
    packed copy of each."""
    h = None
    for part, lo, hi in (("image", 40, 617), ("text", 0, 40)):
        name = f"syrk strided f32 64x617x768 {part} slice"
        if not t.wants(name):
            continue
        if h is None:
            h = torch.randn(64, 617, 768, device="cuda")
        x, rows, d = h[:, lo:hi], 64 * (hi - lo), 768
        packed = x.contiguous()
        g = torch.zeros(d, d, device="cuda")
        t.run(name, [64, hi - lo, d], lambda: t.lib.vlm_syrk_accum_strided(
            x.data_ptr(), _lib.VLM_F32, rows, d, d, hi - lo, 617 * d, g.data_ptr(), d, t.stream), work=syrk_flops(rows, d))
        t.run(f"{name}, packed copy", [rows, d], lambda: t.lib.vlm_syrk_accum(
            packed.data_ptr(), _lib.VLM_F32, rows, d, d, g.data_ptr(), d, t.stream), work=syrk_flops(rows, d))


def time_split(t):
    for rows, d in ((2560, 3072), (36928, 768), (36928, 3072)):
        name = f"tf32x3 {rows}x{d}"
        if not t.wants(name):
            continue
        x = torch.randn(rows, d, device="cuda")
        planes = torch.empty(2, rows, d, device="cuda")
        g = torch.zeros(d, d, device="cuda")
        # reads x once, writes the two planes
        t.run(f"{name} split", [rows, d], lambda: t.lib.vlm_tf32_split(x.data_ptr(), rows, d, d, 0, 0, planes.data_ptr(),
                                                                       t.stream), work=12 * rows * d, unit="GB/s")
        t.run(f"{name} syrk", [rows, d], lambda: t.lib.vlm_syrk_accum(planes.data_ptr(), _lib.VLM_TF32X2, rows, d, d,
                                                                      g.data_ptr(), d, t.stream), work=syrk_flops(rows, d))


def time_exact(t):
    """The RegMean-grade Grams: fp64 DMMA, and int8 digit planes on the integer tensor cores (pre-pass included)."""
    for rows, d in ((2560, 768), (36928, 768), (36928, 3072)):
        name = f"syrk_f64 f32 {rows}x{d}"
        if t.wants(name):
            x = torch.randn(rows, d, device="cuda")
            g = torch.zeros(d, d, dtype=torch.float64, device="cuda")
            t.run(name, [rows, d], lambda: t.lib.vlm_syrk_accum_f64(x.data_ptr(), _lib.VLM_F32, rows, d, d, 0, 0,
                                                                    g.data_ptr(), d, t.stream),
                  iters=3 if d >= 3072 else 10, work=syrk_flops(rows, d))
    for rows, d in ((2560, 3072), (36928, 768), (36928, 3072)):
        name = f"syrk_i8x4 f32 {rows}x{d}"
        if t.wants(name):
            x = torch.randn(rows, d, device="cuda")
            g = torch.zeros(d, d, dtype=torch.float64, device="cuda")
            nbytes = t.lib.vlm_syrk_i8x4_scratch_bytes(rows, d)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            t.run(name, [rows, d], lambda: t.lib.vlm_syrk_accum_i8x4(x.data_ptr(), _lib.VLM_F32, rows, d, d, 0, 0,
                                                                     scratch.data_ptr(), nbytes, g.data_ptr(), d,
                                                                     t.stream), work=syrk_flops(rows, d))


def time_grouped(t):
    """What GramCache.flush issues: a slice of the image tower, and the 48 Grams of the text tower of one forward."""
    for groups in ([(9, 36928, 768)], [(36, 2560, 768), (12, 2560, 3072)]):
        name = "grouped " + "+".join(f"{n}x{rows}x{d}" for n, rows, d in groups)
        if not t.wants(name):
            continue
        shapes = [(rows, d) for n, rows, d in groups for _ in range(n)]
        xs = [torch.randn(rows, d, device="cuda") for rows, d in shapes]
        gs = [torch.zeros(d, d, device="cuda") for _, d in shapes]
        probs = (_lib.SyrkProblem * len(shapes))()
        for p, x, g, (rows, d) in zip(probs, xs, gs, shapes):
            p.x, p.rows, p.ldx, p.g, p.ldg, p.d = x.data_ptr(), rows, d, g.data_ptr(), d, d
        t.run(name, [list(grp) for grp in groups],
              lambda: t.lib.vlm_syrk_accum_batch(probs, len(shapes), _lib.VLM_F32, t.stream),
              work=sum(syrk_flops(rows, d) for rows, d in shapes))


def time_sim_topk(t):
    m, n, d = 5000, 25000, 768
    name = f"sim_topk f16 {m}x{n}x{d}"
    if not t.wants(name):
        return
    a = torch.randn(m, d, device="cuda").half()
    b = torch.randn(n, d, device="cuda").half()
    splits = t.lib.vlm_sim_topk_splits(m, n)
    val = torch.empty(m * splits * 10, device="cuda")
    idx = torch.empty(m * splits * 10, dtype=torch.int32, device="cuda")
    t.run(name, [m, n, d], lambda: t.lib.vlm_sim_topk(a.data_ptr(), m, d, b.data_ptr(), n, d, d, _lib.VLM_F16,
                                                      val.data_ptr(), idx.data_ptr(), splits, t.stream),
          work=2 * m * n * d)


def time_merge(t):
    """The VLMo-base interpolation (2 sources) and modality arithmetic (3) over all 85,045,248 merged elements."""
    n = 85_045_248
    for name, mode, coefs in (("merge wsum 2 sources", _lib.MERGE_WSUM, (0.5, 0.5)),
                              ("merge seq_lerp 3 sources", _lib.MERGE_SEQ_LERP, (1.0, 0.75, 0.75))):
        if not t.wants(name):
            continue
        srcs = [torch.randn(n, device="cuda") for _ in coefs]
        dst = torch.empty(n, device="cuda")
        seg = _lib.MergeSeg()
        seg.dst, seg.n, seg.n_src, seg.mode = dst.data_ptr(), n, len(coefs), mode
        for i, (s, c) in enumerate(zip(srcs, coefs)):
            seg.src[i], seg.coef[i] = s.data_ptr(), c
        plan = ctypes.c_void_p()
        _lib.check(t.lib.vlm_merge_plan_create(ctypes.byref(seg), 1, ctypes.byref(plan)))
        try:
            t.run(name, [n], lambda: t.lib.vlm_merge_plan_run(plan, t.stream), work=t.lib.vlm_merge_plan_bytes(plan),
                  unit="GB/s")
        finally:
            t.lib.vlm_merge_plan_destroy(plan)


def time_regmean(t):
    """The RegMean step of one linear: right-hand side W * Ghat and scale_G from an fp32 Gram, then the SPD solve."""
    for out_f, in_f in ((2304, 768), (768, 768), (3072, 768), (768, 3072)):
        shape = f"{out_f}x{in_f}"
        if not any(t.wants(f"{what} {shape}") for what in ("regmean_rhs", "gram_scale_accum", "spd_solve_right")):
            continue
        w = torch.randn(out_f, in_f, device="cuda")
        x = torch.randn(2 * in_f, in_f, device="cuda")
        g = x.T @ x
        acc = torch.randn(out_f, in_f, dtype=torch.float64, device="cuda")
        s = torch.empty(in_f, in_f, dtype=torch.float64, device="cuda")
        if t.wants(f"regmean_rhs {shape}"):
            t.run(f"regmean_rhs {shape}", [out_f, in_f], lambda: t.lib.vlm_regmean_rhs(
                w.data_ptr(), out_f, in_f, in_f, g.data_ptr(), _lib.VLM_F32, in_f, 0.9, acc.data_ptr(), in_f, 0,
                t.stream), work=2 * out_f * in_f * in_f)
        def scale():
            return t.lib.vlm_gram_scale_accum(g.data_ptr(), _lib.VLM_F32, in_f, in_f, 0.9, s.data_ptr(), in_f, 0,
                                              t.stream)

        _lib.check(scale())      # s = scale_G(g): the solve's operand
        if t.wants(f"gram_scale_accum {shape}"):
            # reads the fp32 Gram, writes the fp64 one
            t.run(f"gram_scale_accum {shape}", [in_f, in_f], scale, work=12 * in_f * in_f, unit="GB/s")
        if t.wants(f"spd_solve_right {shape}"):
            # the solve overwrites both operands: each launch gets fresh copies, made outside the timed events
            ms = 0.0
            s0, r0 = s.clone(), acc.clone()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for i in range(13):
                s.copy_(s0)
                acc.copy_(r0)
                a.record()
                _lib.check(t.lib.vlm_spd_solve_right(s.data_ptr(), in_f, in_f, acc.data_ptr(), out_f, in_f, t.stream))
                b.record()
                b.synchronize()
                ms += a.elapsed_time(b) if i >= 3 else 0.0
            # Cholesky in_f^3 / 3, then two triangular solves of out_f rows
            t.report(f"spd_solve_right {shape}", [out_f, in_f], ms / 10, in_f ** 3 / 3 + 2 * out_f * in_f ** 2,
                     "TFLOP/s")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--full", action="store_true", help="also the 1024- and 4096-wide SYRK shapes")
    ap.add_argument("--only", metavar="SUBSTR", help="only the cases whose name contains SUBSTR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_kernels.py: no CUDA device; these timings can only be taken on the GPU")
    print(json.dumps(card()), flush=True)
    t = Timer(args.only)
    time_syrk(t, args.full)
    time_strided(t)
    time_split(t)
    time_exact(t)
    time_grouped(t)
    time_sim_topk(t)
    time_merge(t)
    time_regmean(t)


if __name__ == "__main__":
    main()
