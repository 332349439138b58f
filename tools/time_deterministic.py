"""Cost of the deterministic Gram mode (vlm_set_deterministic / GramCache(deterministic=True)).

One JSON line per case: CUDA-event times of the default and the deterministic mode, alternated in one process (median
of --reps windows of --inner launches each), how many Gram entries differ between four default-mode runs of the same
launch (runs 1 and 3 overlap a matmul loop on another stream) and the same count for the deterministic mode, which
must be 0.  Then one VLMo-base calibration step (batch 64, fp32 forward, defer_bytes = 128 MB) in the tf32 and int8x4
precisions, both modes, in samples/s.  Every line carries the GPU's name and power limit, read in the same process.
--other-lib PATH: also time the default mode of another libvlmerge.so build (e.g. the previous commit's), alternated
with the two modes of this one.

    python tools/time_deterministic.py [--reps 15] [--inner 10] [--other-lib PATH] [--no-step]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vl_merging_b200 as vlm  # noqa: E402
from vl_merging_b200 import _lib  # noqa: E402

CODE = {torch.float32: _lib.VLM_F32, torch.bfloat16: _lib.VLM_BF16, torch.float16: _lib.VLM_F16}


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        power = out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return {"gpu": name, "power_limit": power}


def load_other(path):
    h = ctypes.CDLL(os.path.abspath(path))
    for name, (restype, argtypes) in _lib.SIGNATURES.items():
        if hasattr(h, name):
            getattr(h, name).restype, getattr(h, name).argtypes = restype, argtypes
    return h


def real(shape, dtype, seed, positive=True):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(*shape, generator=g, device="cuda")
    return (x.abs() if positive else x).to(dtype)


def cases():
    """name -> (make(L) -> (call(g), g0))"""
    out = {}
    for rows, d in [(36928, 3072), (36928, 768), (2560, 768), (2560, 3072)]:
        for dtype in (torch.float32, torch.bfloat16, torch.float16):
            def make(L, rows=rows, d=d, dtype=dtype):
                x = real((rows, d), dtype, rows + d)
                return (lambda g: L.vlm_syrk_accum(x.data_ptr(), CODE[dtype], rows, d, d, g.data_ptr(), d, None),
                        torch.zeros(d, d, device="cuda"))
            out[f"pair-{str(dtype)[6:]}-{rows}x{d}"] = make

    def rowslice(L):
        h = real((64, 617, 768), torch.float32, 3)
        x = h[:, 40:]
        return (lambda g: L.vlm_syrk_accum_strided(x.data_ptr(), _lib.VLM_F32, 64 * 577, 768, 768, 577, 617 * 768,
                                                   g.data_ptr(), 768, None), torch.zeros(768, 768, device="cuda"))
    out["strided-float32-64x577x768"] = rowslice

    def grouped(L):
        shapes = [(2560, 768)] * 36 + [(2560, 3072)] * 12
        xs = [real(s, torch.float32, i) for i, s in enumerate(shapes)]
        n = sum(d * d for _, d in shapes)

        def call(arena):
            probs = (_lib.SyrkProblem * len(shapes))()
            off = 0
            for q, x, (r, d) in zip(probs, xs, shapes):
                q.x, q.rows, q.ldx, q.d, q.g, q.ldg = x.data_ptr(), r, d, d, arena.data_ptr() + 4 * off, d
                off += d * d
            return L.vlm_syrk_accum_batch(probs, len(shapes), _lib.VLM_F32, None)
        return call, torch.zeros(n, device="cuda")
    out["batch-text-tower-36x2560x768+12x2560x3072"] = grouped

    for rows, d in [(36928, 768), (2560, 3072)]:
        def i8(L, rows=rows, d=d):
            x = real((rows, d), torch.float32, rows)
            s = torch.empty(L.vlm_syrk_i8x4_scratch_bytes(rows, d), dtype=torch.uint8, device="cuda")
            return (lambda g: L.vlm_syrk_accum_i8x4(x.data_ptr(), _lib.VLM_F32, rows, d, d, 0, 0, s.data_ptr(), s.numel(),
                                                    g.data_ptr(), d, None), torch.zeros(d, d, dtype=torch.float64, device="cuda"))
        out[f"i8x4-float32-{rows}x{d}"] = i8

    def f64(L):
        x = real((2560, 768), torch.float32, 5)
        return (lambda g: L.vlm_syrk_accum_f64(x.data_ptr(), _lib.VLM_F32, 2560, 768, 768, 0, 0, g.data_ptr(), 768, None),
                torch.zeros(768, 768, dtype=torch.float64, device="cuda"))
    out["f64-float32-2560x768"] = f64

    def simt(L):
        x = real((36928, 200), torch.float32, 6)
        return (lambda g: L.vlm_syrk_accum(x.data_ptr(), _lib.VLM_F32, 36928, 200, 200, g.data_ptr(), 200, None),
                torch.zeros(200, 200, device="cuda"))
    out["simt-float32-36928x200"] = simt
    return out


def differing(L, det, call, g0, runs=4):
    """Entries of G that differ from run 0, worst over runs 1..3 (runs 1 and 3 under a concurrent matmul loop)."""
    L.vlm_set_deterministic(int(det))
    other = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device="cuda", dtype=torch.bfloat16)
    gs = []
    for i in range(runs):
        g = g0.clone()
        torch.cuda.synchronize()
        if i % 2:
            with torch.cuda.stream(other):
                for _ in range(30):
                    a = (a @ a).clamp_(-1, 1)
        _lib.check(call(g))
        torch.cuda.synchronize()
        gs.append(g)
    L.vlm_set_deterministic(0)
    diff = [int((g != gs[0]).sum()) for g in gs[1:]]
    rel = max(((g - gs[0]).abs().max() / gs[0].abs().max()).item() for g in gs[1:])
    return max(diff), rel


def time_modes(arms, reps, inner):
    """arms: name -> (L, det, call, g).  Median ms per launch of each arm, windows alternated."""
    times = {k: [] for k in arms}
    for name, (L, det, call, g) in arms.items():      # warm-up (schedules, modules)
        if hasattr(L, "vlm_set_deterministic"):
            L.vlm_set_deterministic(int(det))
        for _ in range(3):
            rc = call(g)
            assert rc == 0, rc
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, (L, det, call, g) in arms.items():
            if hasattr(L, "vlm_set_deterministic"):
                L.vlm_set_deterministic(int(det))
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(inner):
                call(g)
            b.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(b) / inner)
    for L, _, _, _ in arms.values():
        if hasattr(L, "vlm_set_deterministic"):
            L.vlm_set_deterministic(0)
    return {k: round(statistics.median(v), 4) for k, v in times.items()}


def calibration_step(info, reps):
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    cfg = vlm.vlmo_config("base")
    with torch.device("cuda"):
        model = vlm.VLMo(cfg)
    vlm.init_synthetic_(model.eval(), seed=1)
    B = 64
    batch = vlm.synthetic_batch(B, cfg, seed=1234, device="cuda")
    for precision in ("tf32", "int8x4"):
        caches = {det: vlm.GramCache(defer_bytes=128 << 20, precision=precision, deterministic=det) for det in (False, True)}
        for c in caches.values():
            c.register(model, use_moe=True)
            c.enabled = False
        per = {False: [], True: []}
        for r in range(reps + 1):
            for det, c in caches.items():
                c.enabled = True
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                with torch.no_grad():
                    for _ in range(3):
                        model(batch)
                b.record()
                torch.cuda.synchronize()
                c.enabled = False
                if r:
                    per[det].append(a.elapsed_time(b) / 3)
        for c in caches.values():
            c.remove_hooks()
        ms = {det: statistics.median(v) for det, v in per.items()}
        print(json.dumps({"case": f"calibration-step-vlmo-base-{precision}", "batch": B,
                          "default_samples_per_s": round(B / (ms[False] * 1e-3), 1),
                          "deterministic_samples_per_s": round(B / (ms[True] * 1e-3), 1),
                          "default_ms": round(ms[False], 3), "deterministic_ms": round(ms[True], 3), **info}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--inner", type=int, default=10)
    ap.add_argument("--other-lib", default=None)
    ap.add_argument("--no-step", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_deterministic.py needs a CUDA device")
    L = _lib.lib()
    other = load_other(args.other_lib) if args.other_lib else None
    info = gpu_info()
    for name, make in cases().items():
        call, g0 = make(L)
        arms = {"default": (L, False, call, g0.clone()), "deterministic": (L, True, call, g0.clone())}
        if other is not None:
            ocall, og0 = make(other)
            arms["other_default"] = (other, False, ocall, og0)
        t = time_modes(arms, args.reps, args.inner)
        nd, rel = differing(L, False, call, g0)
        dd, _ = differing(L, True, call, g0)
        row = {"case": name, "default_ms": t["default"], "deterministic_ms": t["deterministic"],
               "ratio": round(t["deterministic"] / t["default"], 3),
               "default_entries_differing": nd, "default_max_rel_diff": float(f"{rel:.3g}"),
               "deterministic_entries_differing": dd, "numel": g0.numel(), **info}
        if other is not None:
            row["other_lib_default_ms"] = t["other_default"]
        print(json.dumps(row), flush=True)
        del call, arms
        torch.cuda.empty_cache()
    if not args.no_step:
        calibration_step(info, reps=3)


if __name__ == "__main__":
    main()
