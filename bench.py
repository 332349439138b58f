#!/usr/bin/env python
"""bench.py — headline benchmark of the merge hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one calibration batch of RegMean Gram caching for VLMo-base all_moe (configs[1] of
BASELINE.json): the frozen image and text towers (stock torch) run over B=64 synthetic 384-px images +
40-token texts per GPU, and every hooked module input goes through GramCache.hook_gram_input ->
vlm_syrk_accum (96 launches per step).  `value` = samples/s with the batch resident in HBM; `e2e` =
the same call with the batch in pinned host memory (H2D of images/text and D2H of the logits inside
the timed region).  N > 1: one process per GPU, batches are data-parallel (weak scaling), and the ONE
all-reduce of the Gram arena that ends a calibration run is inside the timed region.

Extra objects on the JSON line: `roofline` (the SYRK kernel, tensor-bound), `merge` (kernel (b):
interpolation of the same checkpoint, GB/s resident and end-to-end, with its own HBM roofline),
`cpu_baseline` (the reference's CPU path restated in oracle/, timed on this box's host cores).

--impl reference times the reference's CPU implementation of the path (stock forward on the host +
the reference hook, oracle.reference_hook_torch) on a bounded sample per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

BATCH_PER_GPU = 64
ROWS_PER_SAMPLE = 577 + 40
METRIC = "gram_cache_samples_per_sec"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [ln.split(", ") for t, ln in self.lines if t0 <= t <= t1 + 0.2] or [ln.split(", ") for _, ln in self.lines[-3:]]
        sm, reasons, smax, power = [], set(), None, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                power.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "power_w_max": max(power) if power else None, "samples": len(sm)}


def ncu_dram_traffic(name):
    """dram read + write bytes of one launch from a committed `ncu --set full` summary under profiles/ (or None)."""
    prof = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(prof):
        return None
    vals = {}
    for line in open(prof):
        parts = line.strip().split(",")
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            vals[parts[0]] = float(parts[2]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(parts[1], 1.0)
    return int(sum(vals.values())) if len(vals) == 2 else None


# ---------------------------------------------------------------------------------------------------
def syrk_flops(rows, d):
    return rows * d * (d + 1)  # symmetric count, SURVEY.md §8(d)


def make_timed_cache(vlm):
    class TimedCache(vlm.GramCache):
        """GramCache that brackets every vlm_syrk_accum launch with CUDA events on the launching stream."""
        events, timing = [], False

        def accumulate(self, name, x):
            rows = x.numel() // x.shape[-1]
            if not self.timing or 0 < x.numel() * x.element_size() <= self.defer_bytes:
                return super().accumulate(name, x)   # deferred activations are timed in flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            super().accumulate(name, x)
            b.record()
            self.events.append((a, b, syrk_flops(rows, x.shape[-1]), f"{rows}x{x.shape[-1]}:{str(x.dtype).replace('torch.', '')}", 1))

        def flush(self):
            if not self.timing or not self._pending:
                return super().flush()
            flops = sum(syrk_flops(p[4], p[5]) for p in self._pending)   # (rows, d) of each pending problem
            n = len(self._pending)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            super().flush()
            b.record()
            self.events.append((a, b, flops, "grouped launches (text Grams + 768-wide image Grams)", n))

    return TimedCache


DUMP_GRAM_SAMPLES = 1 << 15


def dump_outputs(path, logits, cache):
    """What the timed calibration run hands its caller, as DIR/<name>.npy: `logits.npy`, the similarity logits of the
    last timed step (float32), and one `gram.<module name>.npy` per Gram the run accumulated, in the cache's element
    type (float32, or float64 for the RegMean-grade precisions).  A Gram file holds the Gram's diagonal followed by its
    entries at DUMP_GRAM_SAMPLES upper-triangle positions drawn from a generator seeded with the Gram's width, so every
    run and every build samples the same positions (VLMo-base: 96 files, 13 MB in float32)."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "logits.npy"), logits.float().cpu().numpy())
    picks = {}
    for name in cache.live_names():
        g = cache.gram(name)
        d = g.shape[0]
        if d not in picks:
            ij = torch.randint(0, d, (2, DUMP_GRAM_SAMPLES), generator=torch.Generator().manual_seed(d))
            diag = torch.arange(d)
            picks[d] = (torch.cat([diag, ij.min(0).values]).to(g.device), torch.cat([diag, ij.max(0).values]).to(g.device))
        rows, cols = picks[d]
        np.save(os.path.join(path, f"gram.{name}.npy"), g[rows, cols].cpu().numpy())


def run_ours(args):
    import torch.distributed as dist

    import vl_merging_b200 as vlm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    torch.backends.cuda.matmul.allow_tf32 = True   # the frozen forward is stock torch; TF32 matmuls like the SYRK
    torch.backends.cudnn.allow_tf32 = True
    peaks = load_peaks()

    cfg = vlm.vlmo_config(args.model, attn_impl=args.attn)
    with torch.device(dev):
        model = vlm.VLMo(cfg)
    vlm.init_synthetic_(model.eval(), seed=1)
    amp = {"fp32": None, "bf16": torch.bfloat16, "fp16": torch.float16}[args.autocast]

    TimedCache = make_timed_cache(vlm)
    exact = args.gram_precision in ("int8x4", "fp64")      # RegMean-grade modes: fp64 Grams, launched from the hook
    cache = TimedCache(dev, defer_bytes=0 if exact else args.defer_mb << 20, max_pending_bytes=args.defer_cap_mb << 20,
                       precision=args.gram_precision, symmetric=bool(args.symmetric and world > 1))
    cache.register(model, use_moe=True)
    B = args.batch
    host_batches = [vlm.synthetic_batch(B, cfg, seed=1234 + rank * 16 + i) for i in range(2)]
    for hb in host_batches:
        hb["image"] = [hb["image"][0].pin_memory()]
        for k in ("text_ids", "text_masks", "text_labels"):
            hb[k] = hb[k].pin_memory()
    dev_batches = [{"image": [hb["image"][0].to(dev)], **{k: hb[k].to(dev) for k in ("text_ids", "text_masks", "text_labels")}}
                   for hb in host_batches]

    def step(batch, amp=amp):
        with torch.no_grad():
            if amp is None:
                return model(batch)
            with torch.autocast("cuda", dtype=amp):
                return model(batch)

    copy_stream = torch.cuda.Stream(device=dev)
    inflight = {}

    def h2d_async(i, hb):
        """Host -> device copy of step i's batch on a side stream (what a pin_memory DataLoader + prefetch does)."""
        with torch.cuda.stream(copy_stream):
            batch = {"image": [hb["image"][0].to(dev, non_blocking=True)],
                     **{k: hb[k].to(dev, non_blocking=True) for k in ("text_ids", "text_masks", "text_labels")}}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        inflight[i] = (batch, ev)

    def step_e2e(i, nsteps):
        """Step i end to end: its batch comes from pinned host memory (copy overlapped with step i-1's compute),
        its logits go back to the host (synchronising)."""
        if i not in inflight:
            h2d_async(i, host_batches[i % 2])
        batch, ev = inflight.pop(i)
        torch.cuda.current_stream(dev).wait_event(ev)
        if i + 1 < nsteps:
            h2d_async(i + 1, host_batches[(i + 1) % 2])
        out = step(batch)
        for t in [batch["image"][0], batch["text_ids"], batch["text_masks"], batch["text_labels"]]:
            t.record_stream(torch.cuda.current_stream(dev))
        return out.float().cpu()   # D2H of the step's result; synchronises

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, with_allreduce):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for i in range(steps):
            fn(i)
        ar_ms = 0.0
        if with_allreduce and world > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            cache.all_reduce(group)
            e1.record()
        b.record()
        barrier()
        t1 = time.perf_counter()
        ms = a.elapsed_time(b)
        if with_allreduce and world > 1:
            ar_ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, t0, t1, ar_ms

    if args.profile:
        # ncu --profile-from-start off: only the --steps calibration steps between cudaProfilerStart/Stop are captured
        for i in range(args.warmup):
            step(dev_batches[i % 2])
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        for i in range(args.steps):
            step(dev_batches[i % 2])
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return None

    # ---- warm-up, then the timed region (device-resident inputs) --------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early: nvidia-smi takes ~0.3 s to come up
    for i in range(max(args.warmup, 3)):
        step(dev_batches[i % 2])
    if world > 1:
        cache.all_reduce(group)   # warm-up of the collective too (NCCL connects its channels on first use)
    cache.reset()
    launches0 = vlm._lib.launch_count()
    cache.timing, cache.events = True, []
    last = {}
    ms, t0, t1, ar_ms = timed(lambda i: last.__setitem__("logits", step(dev_batches[i % 2])), args.steps, with_allreduce=True)
    cache.timing = False
    launches = vlm._lib.launch_count() - launches0
    n_live, reduce_bytes = len(cache.live_names()), getattr(cache, "last_reduce_bytes", 0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["logits"], cache)   # before the exchange below overwrites the Grams
    ar_alone_ms = None
    if world > 1:
        # the exchange step on its own, ranks aligned by a barrier first (the in-region figure also contains the wait
        # for the slowest rank's last step); the values are garbage afterwards, the cache is reset before its next use
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        cache.all_reduce(group)
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_alone_ms = round(t.item(), 3)
    clocks = sampler.stop(t0, t1) if sampler else None
    value = world * B * args.steps / (ms * 1e-3)

    # per-launch SYRK time, measured live on the launching stream inside the timed region
    tot_ms = tot_flops = 0.0
    by_shape = {}
    n_problems = 0
    for a, b, flops, key, nprob in cache.events:
        dms = a.elapsed_time(b)
        tot_ms += dms
        tot_flops += flops
        n_problems += nprob
        s = by_shape.setdefault(key, [0, 0.0, 0.0])
        s[0] += 1
        s[1] += dms
        s[2] += flops
    n_ev = max(len(cache.events), 1)
    # DRAM traffic per launch of the dominant shape (36928 x 3072 fp32) from the committed ncu --set full capture
    traffic = None
    traffic = ncu_dram_traffic("r02_syrk_2sm_f32_36928x3072.summary.csv") or ncu_dram_traffic("r01_syrk_tc2_f32_36928x3072.summary.csv")
    sixteen = amp is not None
    # TF32 runs at half the bf16 tensor rate; the MEASURED bf16 figure (sustained: kernel timed inside a long step)
    peak_tf = peaks["bf16_tflops_sustained"] * (1.0 if sixteen else 0.5)
    achieved_tf = tot_flops / (tot_ms * 1e-3) * 1e-12 if tot_ms > 0 else 0.0
    if args.gram_precision == "int8x4":
        # 13 int8 digit-plane products per Gram at twice the bf16 tensor rate: the effective peak on the 1x flop count
        peak_tf = peaks["bf16_tflops_sustained"] * 2.0 / 13.0
        traffic = ncu_dram_traffic("r02_syrk_i8x4_36928x3072.summary.csv")
    elif args.gram_precision == "fp64":
        peak_tf, traffic = 40.0, None                      # B200 fp64 tensor peak (nominal)
    elif args.gram_precision == "tf32x3":
        peak_tf, traffic = peak_tf / 3.0, ncu_dram_traffic("r02_syrk_2sm_split_36928x3072.summary.csv")
    roofline = {
        "kernel": {"int8x4": "syrk_i8x4_kernel (fp32 -> four int8 digit planes; 13 tcgen05.mma.cta_group::2 kind::i8 products, int32 TMEM accumulators, fp64 TMA reduce-add) incl. its digit pre-pass",
                   "fp64": "syrk_f64_kernel (DMMA m8n8k4, red.global.add.f64)",
                   "tf32x3": "syrk_2sm_kernel, split mode (hi'hi + hi'lo + lo'hi) incl. vlm_tf32_split"}.get(args.gram_precision) or
        ("syrk_2sm_kernel (CTA pairs, one tcgen05.mma.cta_group::2 kind::tf32 stream per pair, TMA loads, TMEM accumulators, TMA reduce-add)" if not sixteen
         else "syrk_2sm_kernel (mixed kind::tf32 / kind::f16 launches under autocast)"),
        "bound": "tensor", "achieved": round(achieved_tf, 2), "peak": round(peak_tf, 1), "unit": "TFLOP/s",
        "frac": round(achieved_tf / peak_tf, 4), "traffic": traffic,
        "traffic_note": "dram read+write bytes of ONE 36928x3072 fp32 launch (ncu --set full, profiles/); its algorithmic minimum is one read of X = 453.8 MB",
        "frac_of_nominal_1.1PF_tf32": round(achieved_tf / 1100.0, 4) if (not sixteen and args.gram_precision == "tf32") else None,
        "peak_source": {"int8x4": f"{peaks['source']}: bf16_tflops_sustained x 2 (int8) / 13 products, on the 1x (symmetric) flop count",
                        "fp64": "nominal B200 fp64 tensor peak", "tf32x3": f"{peaks['source']}: bf16_tflops_sustained / 2 / 3 products"}.get(
                            args.gram_precision, f"{peaks['source']}: bf16_tflops_sustained{' / 2 (TF32)' if not sixteen else ''}"),
        "flops_per_launch_avg": tot_flops / n_ev, "ms_per_launch_avg": tot_ms / n_ev, "launches_timed": len(cache.events), "grams_accumulated": n_problems,
        "syrk_share_of_step": round(tot_ms / (ms if ms > 0 else 1), 4),
        "by_shape": {k: {"launches": v[0], "ms_avg": round(v[1] / v[0], 4), "tflops": round(v[2] / (v[1] * 1e-3) * 1e-12, 1)}
                     for k, v in sorted(by_shape.items())},
    }

    # ---- end to end: host buffers in, logits out, every step --------------------------------------
    cache.reset()
    for i in range(2):
        step_e2e(i, 2)
    ms_e2e, _, _, _ = timed(lambda i: step_e2e(i, args.steps), args.steps, with_allreduce=True)
    h2d = sum(host_batches[0][k].numel() * host_batches[0][k].element_size() for k in ("text_ids", "text_masks", "text_labels"))
    h2d += host_batches[0]["image"][0].numel() * 4
    e2e = {"value": round(world * B * args.steps / (ms_e2e * 1e-3), 2), "unit": "samples/s",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * B * 4}

    # ---- Gram parity spot check on the bench's own activations (cheap; not timed) ------------------
    L = cfg["num_layers"]
    parity_names = ["transformer.blocks.0.attn.v", f"transformer.blocks.{L - 1}.mlp.v.fc2", f"transformer.blocks.{L // 2 - 1}.mlp.l.fc1"]

    def fp64_probes(names, store):
        """The reference hook's arithmetic (cache_gram_matrices.py:250-253) on the device, for a few modules."""
        mods = dict(model.named_modules())

        def probe(m, i, o):
            x = (i[0] if isinstance(i, tuple) else i).double()
            x = x.reshape(-1, x.shape[-1])
            store[m.module_name] = store.get(m.module_name, 0) + x.T @ x
        return [mods[n].register_forward_hook(probe) for n in names]

    def gram_parity(vamp=amp):
        cache.reset()
        probe = {}
        hs = fp64_probes(parity_names, probe)
        step(dev_batches[0], vamp)
        for h in hs:
            h.remove()
        out = {n: float(((cache.gram(n).double() - probe[n]).norm() / probe[n].norm()).item()) for n in parity_names}
        cache.reset()
        return out

    parity = gram_parity() if rank == 0 else None

    # ---- N > 1: the REDUCED Grams against the sum of per-rank fp64 reference-hook Grams (every rank checks) ----
    reduced_parity = None
    if world > 1:
        cache.reset()
        probe = {}
        hs = fp64_probes(parity_names, probe)
        step(dev_batches[0])                     # every rank its own shard of the calibration set
        for h in hs:
            h.remove()
        cache.all_reduce(group)
        errs = []
        for n in parity_names:
            ref = probe[n].clone()
            dist.all_reduce(ref)                 # fp64 sum over the ranks = the single-process reference Gram
            errs.append((cache.gram(n).double() - ref).norm() / ref.norm())
        worst = torch.stack(errs).max()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        reduced_parity = float(worst.item())
        cache.reset()

    # ---- informational: the same calibration with faster stock-torch forwards ----------------------
    variants = {}
    if not args.no_variants:
        attn_mods = [m for m in model.modules() if hasattr(m, "attn_impl")]
        for vname, impl, vamp in (("fp32_tf32_reference_attention" if args.attn == "sdpa" else "fp32_tf32_sdpa",
                                   "reference" if args.attn == "sdpa" else "sdpa", None),
                                  ("autocast_bf16_sdpa", "sdpa", torch.bfloat16)):
            for m in attn_mods:
                m.attn_impl = impl
            for i in range(3):
                step(dev_batches[i % 2], vamp)
            cache.reset()
            vms, _, _, _ = timed(lambda i: step(dev_batches[i % 2], vamp), args.steps, with_allreduce=True)
            variants[vname] = {"value": round(world * B * args.steps / (vms * 1e-3), 2), "unit": "samples/s",
                               "ms_per_step": round(vms / args.steps, 3)}
        for m in attn_mods:
            m.attn_impl = args.attn
        cache.reset()
        # Gram launches on a second stream, overlapping the rest of the forward (GramCache(side_stream=True))
        cache.set_side_stream(True)
        for i in range(3):
            step(dev_batches[i % 2])
        cache.reset()
        vms, _, _, _ = timed(lambda i: step(dev_batches[i % 2]), args.steps, with_allreduce=True)
        variants["fp32_tf32_" + args.attn + "_side_stream_grams"] = {
            "value": round(world * B * args.steps / (vms * 1e-3), 2), "unit": "samples/s", "ms_per_step": round(vms / args.steps, 3)}
        cache.set_side_stream(False)
        cache.reset()
        # the public default, GramCache(): every Gram launched from its hook (defer_bytes = 0)
        saved_defer, cache.defer_bytes = cache.defer_bytes, 0
        for i in range(3):
            step(dev_batches[i % 2])
        cache.reset()
        cache.timing, cache.events = True, []
        vms, _, _, _ = timed(lambda i: step(dev_batches[i % 2]), args.steps, with_allreduce=True)
        cache.timing = False
        sy_ms = sum(a.elapsed_time(b) for a, b, *_ in cache.events)
        sy_fl = sum(e[2] for e in cache.events)
        variants["default_api_one_launch_per_hook"] = {
            "value": round(world * B * args.steps / (vms * 1e-3), 2), "unit": "samples/s", "ms_per_step": round(vms / args.steps, 3),
            "syrk_tflops": round(sy_fl / (sy_ms * 1e-3) * 1e-12, 1) if sy_ms > 0 else None, "syrk_launches_timed": len(cache.events)}
        cache.defer_bytes = saved_defer
        cache.reset()
        # the reference's own calibration precision: PL precision=16 autocast (src/vilt/config.py:116) with the
        # reference's explicit attention — hook inputs are a mix of fp32 (LayerNorm outputs) and fp16 (attention /
        # GELU outputs), the latter on the kind::f16 tensor path
        for m in attn_mods:
            m.attn_impl = "reference"
        for i in range(3):
            step(dev_batches[i % 2], torch.float16)
        cache.reset()
        vms, _, _, _ = timed(lambda i: step(dev_batches[i % 2], torch.float16), args.steps, with_allreduce=True)
        variants["autocast_fp16_reference_attention"] = {
            "value": round(world * B * args.steps / (vms * 1e-3), 2), "unit": "samples/s", "ms_per_step": round(vms / args.steps, 3),
            "gram_parity_rel_fro": gram_parity(torch.float16) if rank == 0 else None,
            "note": "the reference's own precision (fp16 autocast, mixed fp32 / fp16 hook inputs); parity vs the fp64 hook on the same activations"}
        for m in attn_mods:
            m.attn_impl = args.attn
        cache.reset()

    # ---- kernel (b): interpolation merge of this checkpoint ---------------------------------------
    merge = bench_merge(vlm, model, cfg, dev, group, world, rank, peaks, args)

    # ---- config 3: full RegMean merge from the cached Grams (kernel (c) + cuSOLVER, timed separately) ----
    regmean = gram_file = None
    if not args.no_regmean:
        cache.reset()
        for i in range(2):  # 2 x 64 x 40 = 5120 text rows >= 3072: every summed Gram is full rank
            step(dev_batches[i % 2])
        if world > 1:
            cache.all_reduce(group)
        regmean = bench_regmean(vlm, model, cfg, cache, dev, group, world, args)
        if world == 1 and not args.no_gramfile and not exact:   # the packed container holds fp32 Grams
            gram_file = bench_gramfile(vlm, cache, dev)
        if world == 1 and args.model == "base":
            regmean.update(bench_regmean_chain(vlm, model, cfg, cache, dev, step, dev_batches, B))
        cache.reset()

    # ---- SURVEY §8f rank 3 (opt-in): Gram caching on the fused vision-language route (type_id 2) ----
    fused = None
    if args.fused:
        def fstep(i):
            with torch.no_grad():
                model.infer(dev_batches[i % 2])
            cache.flush()
        for i in range(3):
            fstep(i)
        cache.reset()
        l0 = vlm._lib.launch_count()
        cache.timing, cache.events = True, []
        fms, _, _, _ = timed(fstep, args.steps, with_allreduce=True)
        cache.timing = False
        l1 = vlm._lib.launch_count()
        sy_ms = sum(a.elapsed_time(b) for a, b, *_ in cache.events)
        sy_fl = sum(e[2] for e in cache.events)
        # parity of one ROW-SLICED Gram (image rows of the joint sequence into the `v` expert) on identical activations
        cache.reset()
        probe = {}
        mod = dict(model.named_modules())["transformer.blocks.3.mlp.v.fc1"]
        h = mod.register_forward_hook(lambda m, i, o: probe.__setitem__("x", (i[0].is_contiguous(), i[0].double().reshape(-1, i[0].shape[-1]))))
        fstep(0)
        h.remove()
        contiguous, x64 = probe["x"]
        want = x64.T @ x64
        err = float(((cache.gram("transformer.blocks.3.mlp.v.fc1").double() - want).norm() / want.norm()).item())
        fused = {"value": round(world * B * args.steps / (fms * 1e-3), 2), "unit": "samples/s",
                 "ms_per_step": round(fms / args.steps, 3), "gpu_launches": int(l1 - l0),
                 "syrk_tflops": round(sy_fl / (sy_ms * 1e-3) * 1e-12, 1) if sy_ms > 0 else None,
                 "syrk_share_of_step": round(sy_ms / fms, 4), "grams": len(cache.live_names()),
                 "sliced_input_was_contiguous": bool(contiguous), "sliced_gram_rel_fro": err,
                 "note": "model.infer: 40 text + 577 image tokens in one sequence; layers < vlffn_start feed row slices to "
                         "the l / v experts (read in place, 4-D TMA), layers >= vlffn_start run the vl experts"}
        cache.reset()

    irtr = bench_irtr(vlm, model, cfg, dev, group, world, args) if (args.irtr or (args.model == "base" and not args.no_irtr)) else None
    vitl = bench_vitl(vlm, dev, group, world, args) if (args.model == "base" and not args.no_vitl) else None

    # ---- the reference's own hook, unchanged, with the model on the B200 (the GPU-vs-GPU "before", SURVEY §8d) ----
    ref_gpu = None
    if world == 1 and not args.no_gpu_baseline:
        ref_gpu = bench_reference_hook_on_gpu(vlm, model, cache, dev_batches, B)

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": ({"int8x4": "int8x4 (exact digit-plane products, fp64 Grams)", "fp64": "f64", "tf32x3": "tf32x3"}.get(args.gram_precision, "tf32")
                      if not sixteen else f"{args.autocast}" + ("" if args.gram_precision == "tf32" else f" + {args.gram_precision} Grams")),
            "data": "synthetic (hash-seeded images U(-1,1) 384px + 40-token ids; random-init VLMo weights)",
            "config": {"workload": f"RegMean Gram caching, VLMo-{args.model} all_moe, {B} x (577 image + 40 text tokens) per GPU per step; "
                                   "96 Grams (72 x 768^2 + 24 x 3072^2)" if args.model == "base" else f"RegMean Gram caching, VLMo-{args.model} all_moe",
                       "global_batch": world * B, "parallelism": f"dp{world}", "forward": f"stock torch ({args.attn} attention), " + ("fp32 with TF32 matmuls" if not sixteen else f"autocast {args.autocast}"),
                       "l2": "inputs larger than L2 (each step streams >2 GB of weights and activations)",
                       "gram_hooks": (f"activations <= {args.defer_mb} MB are held by reference and issued as grouped launches "
                                      f"(flush at {args.defer_cap_mb} MB pending and after every forward); larger ones launch "
                                      "from the hook") if (args.defer_mb > 0 and not exact) else "one SYRK launch per hook call",
                       "gram_precision": args.gram_precision,
                       "allreduce_ms_in_timed_region": round(ar_ms, 3), "allreduce_ms_after_barrier": ar_alone_ms,
                       "allreduce": (f"ONE kernel over NVSwitch multicast memory (multimem.ld_reduce / multimem.st on the symmetric Gram arenas, "
                                     f"{reduce_bytes / 1e6:.0f} MB of upper triangles, no staging buffer, no NCCL call)") if (world > 1 and cache.symmetric) else
                                    (f"packed {'fp64' if exact else 'fp32'} upper triangles of the {n_live} live Grams in one NCCL all-reduce "
                                     f"({reduce_bytes / 1e6:.0f} MB)") if world > 1 else None},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "merge": merge, "reference_hook_on_gpu": ref_gpu, "regmean": regmean, "gram_file": gram_file, "fused_route": fused, "irtr": irtr, "vitl": vitl, "gram_parity_rel_fro": parity,
            "gram_parity_rel_fro_reduced": reduced_parity,
            "forward_variants": variants,
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_sample(args.model, budget_s=25.0)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def bench_merge(vlm, model, cfg, dev, group, world, rank, peaks, args):
    """Interpolation merge (alpha = 0.5, IRTR-used experts) of the bench checkpoint: kernel-only GB/s with
    everything resident (one vlm_merge_plan launch), and end to end from pinned host memory and back."""
    import ctypes

    import torch.distributed as dist

    from vl_merging_b200 import _lib
    from vl_merging_b200.plan import plan_merge_weights

    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], only_activate_used_experts=True, merge_ratio=0.5,
                loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    L = cfg["num_layers"]
    lib = _lib.lib()
    # resident: build the plan once, time the launch alone (CUDA events on the launching stream)
    ops = [op for op in plan_merge_weights(sd.keys(), mcfg, L) if not op.passthrough]
    total = sum(sd[op.srcs[0]].numel() for op in ops)
    out = torch.empty(total + 4 * len(ops), dtype=torch.float32, device=dev)
    segs = (_lib.MergeSeg * len(ops))()
    off = 0
    for s, op in enumerate(ops):
        n = sd[op.srcs[0]].numel()
        segs[s].dst = out.data_ptr() + off * 4
        for j, k in enumerate(op.srcs):
            segs[s].src[j] = sd[k].data_ptr()
            segs[s].coef[j] = op.coefs[j]
        segs[s].n, segs[s].n_src, segs[s].mode = n, len(op.srcs), op.mode
        off += (n + 3) // 4 * 4
    plan = ctypes.c_void_p()
    _lib.check(lib.vlm_merge_plan_create(segs, len(ops), ctypes.byref(plan)))
    nbytes = int(lib.vlm_merge_plan_bytes(plan))
    stream = torch.cuda.current_stream(dev).cuda_stream
    for _ in range(3):
        _lib.check(lib.vlm_merge_plan_run(plan, stream))
    reps = 20
    evs = []
    for _ in range(reps):  # bytes moved per launch (1.02 GB) exceed L2, no flush needed
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(lib.vlm_merge_plan_run(plan, stream))
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize(dev)
    ms = sum(a.elapsed_time(b) for a, b in evs) / reps
    lib.vlm_merge_plan_destroy(plan)
    gbs = nbytes / (ms * 1e-3) * 1e-9

    # end to end through the public API: pinned host state_dict in, merged host tensors out.  N > 1: every rank stages
    # and merges its shard, one all-gather leaves the result on every GPU, and the HOST copy is made once (rank 0) —
    # N simultaneous device->host copies of the same 340 MB into one host's memory were slower than one GPU
    # (profiles/r01_bench_n8.json: 28.9 vs 53.0 GB/s)
    host_sd = {k: (v.cpu().pin_memory() if "transformer.blocks" in k else v.cpu()) for k, v in sd.items()}
    out_dev = "cpu" if rank == 0 else "cuda"
    vlm.merge_weights(host_sd, mcfg, device=dev, num_layers=L, group=group, out_device=out_dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    stats = {}
    merged = vlm.merge_weights(host_sd, mcfg, device=dev, num_layers=L, group=group, stats=stats, out_device=out_dev)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = t.item()
    # N > 1: the tensor-sharded merge + all-gather against the same merge done locally on this rank, every tensor
    sharded_equal = None
    if world > 1:
        local = vlm.merge_weights(sd, mcfg, device=dev, num_layers=L)
        shard = vlm.merge_weights(sd, mcfg, device=dev, num_layers=L, group=group)
        eq = torch.tensor([int(all(torch.equal(local[op.dst], shard[op.dst]) for op in ops))], device=dev)
        dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        sharded_equal = bool(eq.item())
        del local, shard
    k0 = "transformer.blocks.0.mlp.fc1.weight"
    ok = torch.equal(merged[k0].cpu(), 0.5 * host_sd["transformer.blocks.0.mlp.v.fc1.weight"] + 0.5 * host_sd["transformer.blocks.0.mlp.l.fc1.weight"])
    return {
        "metric": "merge_GBps", "workload": f"linear interpolation alpha=0.5, VLMo-{args.model} all_moe -> ufo, IRTR-used experts "
                                            f"({len(ops)} tensors, {nbytes / 1e6:.1f} MB algorithmic: read 2 experts + write 1 per layer)",
        "value": round(gbs, 1), "unit": "GB/s", "ms_per_launch": round(ms, 4), "launches_per_merge": 1,
        "roofline": {"kernel": "merge_segments_kernel", "bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm_gbs"],
                     "unit": "GB/s", "frac": round(gbs / peaks["hbm_gbs"], 4),
                     "traffic": ncu_dram_traffic("r01_merge_wsum2_85M.summary.csv") if args.model == "base" else None,
                     "traffic_note": "dram read+write bytes of one launch of this workload (ncu --set full, profiles/r01_merge_wsum2_85M.summary.csv); algorithmic bytes = " + str(nbytes),
                     "peak_source": f"{peaks['source']}: hbm_gbs (burst copy)", "frac_of_nominal_8TBps": round(gbs / 8000.0, 4)},
        "e2e": {"value": round(nbytes / dt * 1e-9, 2), "unit": "GB/s", "seconds": round(dt, 4),
                "h2d_bytes": stats.get("h2d_bytes"), "d2h_bytes": stats.get("d2h_bytes"), "bit_exact_vs_torch": bool(ok),
                "host_copy": "rank 0 only; the other ranks keep the gathered result on their GPU" if world > 1 else "this rank"},
        "sharded_bit_equal_to_local": sharded_equal,
    }


def bench_irtr(vlm, model, cfg, dev, group, world, args, n_img=5000, per_img=5, bs=64):
    """Config 4: modality arithmetic (lambda = 0.75, centre = a second synthetic ufo checkpoint) -> ufo model ->
    IRTR forward over 5,000 synthetic images x 25,000 synthetic captions -> 5k x 25k similarity + recalls
    (objectives.py:572-710), batches sharded over the ranks."""
    import numpy as np

    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], only_activate_used_experts=True, sum_lambda=0.75,
                loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ufo_cfg = dict(cfg, use_moe=False)
    with torch.device(dev):
        central = vlm.init_synthetic_(vlm.VLMo(ufo_cfg).eval(), seed=2)
    t0 = time.perf_counter()
    merged = vlm.sum_task_vectors(sd, mcfg, device=dev, num_layers=cfg["num_layers"], group=group,
                                  central_weight=central.state_dict())
    central.load_state_dict(merged, strict=False)   # reuse the module as the merged ufo model
    torch.cuda.synchronize(dev)
    t_merge = time.perf_counter() - t0
    ufo = central
    # synthetic eval set: every item distinct (so that the score matrix has no exact ties), generated on the device
    # batch by batch from two hash-seeded base batches: image i = base + noise_i, caption ids re-drawn per batch
    ib = [vlm.synthetic_batch(bs, cfg, seed=900 + i, device=dev) for i in range(2)]
    tb = [vlm.synthetic_batch(bs, cfg, seed=950 + i, device=dev, pad=True) for i in range(2)]
    n_ib, n_tb = (n_img + bs - 1) // bs, (n_img * per_img + bs - 1) // bs

    class Lazy:
        def __init__(self, n, make):
            self.n, self.make = n, make

        def __len__(self):
            return self.n

        def __iter__(self):
            return (self.make(i) for i in range(self.n))

    def make_image(i):
        gen = torch.Generator(device=dev).manual_seed(7000 + i)
        return {**ib[i % 2], "image": [ib[i % 2]["image"][0] + 0.25 * torch.randn(ib[0]["image"][0].shape, device=dev, generator=gen)]}

    def make_text(i):
        gen = torch.Generator(device=dev).manual_seed(9000 + i)
        base = tb[i % 2]
        ids = torch.randint(999, cfg["vocab_size"] - 1, base["text_ids"].shape, device=dev, generator=gen) * base["text_masks"]
        ids[:, 0] = 101
        return {**base, "text_ids": ids}

    image_batches, text_batches = Lazy(n_ib, make_image), Lazy(n_tb, make_text)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    img, txt = vlm.irtr_features(ufo, image_batches, text_batches, autocast_dtype=torch.float16, group=group)
    img, txt = img[:n_img], txt[: n_img * per_img]
    torch.cuda.synchronize(dev)
    t_towers = time.perf_counter() - t0
    iids, tiids = np.arange(n_img), np.arange(n_img * per_img) // per_img

    def timed_ms(fn, reps=3):
        fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            out = fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps, out

    # objectives.py:684-710 two ways on the same features: the reference's form (materialised 5k x 25k scores + six
    # topk calls, stock torch) and the fused kernel (vlm_sim_topk twice, no score matrix)
    ms_plain, (scores, recalls) = timed_ms(lambda: vlm.irtr_recall(img.float(), txt.float(), iids, tiids))
    ms_fused, (recalls_f, (by_image, _)) = timed_ms(lambda: vlm.irtr_recall_fused(img, txt, iids, tiids))
    # random-init towers give nearly identical features (recalls at chance level, many near-ties), so the check is on
    # the scores of the chosen columns: every row's ten fused picks must score what the materialised matrix says
    top_f = torch.gather(scores, 1, by_image)
    top_t = scores.topk(10, dim=1).values
    pick_err = float((top_f - top_t).abs().max().item())
    dt = t_towers + ms_fused * 1e-3
    flops = 2 * 2.0 * n_img * n_img * per_img * img.shape[1]
    return {"merge_seconds": round(t_merge, 4), "eval_seconds": round(dt, 3), "towers_seconds": round(t_towers, 3),
            "images": n_img, "captions": n_img * per_img, "scores_shape": list(scores.shape),
            "forwards_per_sec": round((n_img + n_img * per_img) / t_towers, 1),
            "autocast": "fp16 (as objectives.py:657,669)", "recalls": [round(float(r), 5) for r in recalls_f],
            "similarity_topk": {"fused_ms": round(ms_fused, 3), "torch_scores_plus_6_topk_ms": round(ms_plain, 3),
                                "fused_tflops": round(flops / (ms_fused * 1e-3) * 1e-12, 1),
                                "recalls_torch_path": [round(float(r), 5) for r in recalls],
                                "top10_score_max_abs_diff_vs_torch": pick_err,
                                "note": "vlm_sim_topk (TMA + tcgen05 kind::f16, running top-10 in the accumulator epilogue), both "
                                        "directions, vs img @ txt.T (500 MB fp32) + topk x 6 in torch"}}


def bench_regmean(vlm, model, cfg, cache, dev, group, world, args):
    """RegMean of the bench checkpoint with the Grams just cached on the device (scaling_for_non_diag = 0.9):
    wall time of the whole merge with the linear problems spread over 8 streams (three repeats), and the W*Ghat
    GEMMs (kernel (c), fp64 DMMA) / SPD solves (cuSOLVER) split from a one-stream run, timed with CUDA events on
    that stream; one linear checked against torch fp64 on the same Grams."""
    import torch.distributed as dist

    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], scaling_for_non_diag=0.9,
                loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    L = cfg["num_layers"]

    def run(streams):
        stats = {}
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        out = vlm.regmean(sd, mcfg, device=dev, num_layers=L, group=group, gram_matrices=cache, stats=stats,
                          solve_streams=streams)
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t0, stats, out

    NS = 8
    run(NS)                     # warm-up: cuSOLVER handles + workspaces per stream, lazy module loading
    run(1)
    runs = [run(NS) for _ in range(3)]
    dt, _, merged = min(runs, key=lambda r: r[0])
    dt_seq, stats, merged_seq = min((run(1) for _ in range(2)), key=lambda r: r[0])
    same = all(torch.equal(merged[k], merged_seq[k]) for k in merged)
    # check: layer 0 attention projection, torch fp64 on the same device Grams
    a = 0.9
    num = den = 0
    for m in ("v", "l"):
        g = cache.gram(f"transformer.blocks.0.attn.{m}.proj").double()
        gh = a * g + (1 - a) * torch.diag(torch.diag(g))
        num = num + sd[f"transformer.blocks.0.attn.{m}.proj.weight"].double() @ gh
        den = den + gh
    want = torch.linalg.solve(den, num.T).T
    got = merged["transformer.blocks.0.attn.proj.weight"]
    err = ((got - want).norm() / want.norm()).item()
    d, h = cfg["hidden_size"], cfg["hidden_size"] * cfg["mlp_ratio"]
    # executed GEMMs: M - 1 = 1 per linear (difference form, W_base + ((W_v - W_base) Ghat_v) S^-1), not the M = 2 of the
    # formula as written: 260.9 GFLOP for VLMo-base instead of 521.8
    rhs_flops = L * 1 * 2 * (3 * d * d * d + d * d * d + h * d * d + d * h * h)
    secs = sorted(r[0] for r in runs)
    return {"seconds": round(dt, 4), "seconds_all_runs": [round(r[0], 4) for r in runs],
            "spread": round(secs[-1] / secs[0] - 1.0, 3), "solve_streams": NS,
            "seconds_sequential": round(dt_seq, 4), "concurrent_equals_sequential": bool(same),
            "rhs_seconds": round(stats.get("rhs_seconds", 0.0), 4),
            "solve_seconds": round(stats.get("solve_seconds", 0.0), 4),
            "rhs_fp64_tflops": round(rhs_flops / max(stats.get("rhs_seconds", 1e-9), 1e-9) * 1e-12 / world, 2),
            "linear_problems": 4 * L, "dtype": "f64", "check_rel_err_vs_torch_fp64": err,
            "rhs_gflop_executed": round(rhs_flops * 1e-9 / world, 1),
            "note": "RHS = fp64 DMMA kernel incl. scale_G and the sum of Grams, in the difference form (one GEMM per two-expert linear); solve = cuSOLVER potrf/potrs (off the hot path); "
                    "seconds = host wall clock of the whole merge, linear problems spread over 8 streams; rhs / solve seconds = "
                    "CUDA-event time of those launches in the one-stream run"}


def bench_regmean_chain(vlm, model, cfg, cache, dev, step, dev_batches, B):
    """Config 3 END TO END on identical activations: forward hooks -> device Grams -> regmean, against the reference
    formula (scale_G, sum, explicit inverse in fp64: vilt_module.py:388-392, :423-434) fed with the fp64 Grams of
    the reference hook (cache_gram_matrices.py:250-253) taken on the same activations.  Two calibration steps of
    64 samples: 5,120 text rows >= 3,072, every summed Gram is full rank.  Checked linears: all four of the first and
    the last layer (768- and 3072-wide).  Also the calibration throughput of the Gram precision modes."""
    L = cfg["num_layers"]
    layers = sorted({0, L - 1})
    c64 = vlm.GramCache(dev, precision="fp64")
    c64.register(model, use_moe=True)
    ci8 = vlm.GramCache(dev, precision="int8x4")
    ci8.register(model, use_moe=True)
    ref, mods = {}, dict(model.named_modules())
    names = [f"transformer.blocks.{i}.{t}" for i in layers for m in ("v", "l")
             for t in (f"attn.{m}", f"attn.{m}.proj", f"mlp.{m}.fc1", f"mlp.{m}.fc2")]

    def probe(m, i, o):
        x = (i[0] if isinstance(i, tuple) else i).double()
        x = x.reshape(-1, x.shape[-1])
        ref[m.module_name] = ref.get(m.module_name, 0) + x.T @ x

    cache.reset()
    hs = [mods[n].register_forward_hook(probe) for n in names]
    for i in range(2):
        step(dev_batches[i % 2])
    for h in hs:
        h.remove()
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    out = {}
    worst = {"fp64": 0.0, "int8x4": 0.0, "tf32": 0.0}
    detail = {}
    for alpha in (1.0, 0.9):
        mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], scaling_for_non_diag=alpha,
                    loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
        import warnings

        with warnings.catch_warnings():      # regmean warns about exactly the combination measured here (tf32 Grams, alpha = 1)
            warnings.simplefilter("ignore", RuntimeWarning)
            merged = {"fp64": vlm.regmean(sd, mcfg, device=dev, num_layers=L, gram_matrices=c64),
                      "int8x4": vlm.regmean(sd, mcfg, device=dev, num_layers=L, gram_matrices=ci8),
                      "tf32": vlm.regmean(sd, mcfg, device=dev, num_layers=L, gram_matrices=cache)}
        for i in layers:
            for tgt, wk, gk in ((f"transformer.blocks.{i}.attn.qkv.weight", "transformer.blocks.{i}.attn.{m}.qkv.weight", "transformer.blocks.{i}.attn.{m}"),
                                (f"transformer.blocks.{i}.attn.proj.weight", "transformer.blocks.{i}.attn.{m}.proj.weight", "transformer.blocks.{i}.attn.{m}.proj"),
                                (f"transformer.blocks.{i}.mlp.fc1.weight", "transformer.blocks.{i}.mlp.{m}.fc1.weight", "transformer.blocks.{i}.mlp.{m}.fc1"),
                                (f"transformer.blocks.{i}.mlp.fc2.weight", "transformer.blocks.{i}.mlp.{m}.fc2.weight", "transformer.blocks.{i}.mlp.{m}.fc2")):
                num = den = 0
                for m in ("v", "l"):
                    g = ref[gk.format(i=i, m=m)]
                    gh = alpha * g + (1 - alpha) * torch.diag_embed(torch.diagonal(g))      # scale_G
                    num = num + sd[wk.format(i=i, m=m)].double() @ gh
                    den = den + gh
                want = num @ torch.inverse(den)                                              # :432-434
                for mode in merged:
                    e = float(((merged[mode][tgt] - want).norm() / want.norm()).item())
                    worst[mode] = max(worst[mode], e)
                    detail[f"{mode} a={alpha} {tgt.split('blocks.')[1]}"] = float(f"{e:.3e}")
    out["e2e_rel_err_vs_fp64_grams"] = worst["fp64"]
    out["e2e_rel_err_vs_fp64_grams_int8x4"] = worst["int8x4"]
    out["e2e_rel_err_vs_fp64_grams_single_pass_tf32"] = worst["tf32"]
    out["e2e_detail"] = detail
    out["e2e_note"] = ("whole chain on identical activations: hooks -> device Grams -> regmean vs the reference formula on the "
                       "reference hook's fp64 Grams; worst of 8 linears (layers 0 and L-1) x scaling_for_non_diag in {1.0, 0.9}. "
                       "e2e_rel_err_vs_fp64_grams = GramCache(precision='fp64') (the RegMean-grade mode, BASELINE 1e-4); _int8x4 = the same "
                       "grade from the integer tensor cores (exact int8 digit-plane products); "
                       "single_pass_tf32 = the default fast mode (Gram tolerance 1e-3)")
    gram_err = max(float(((c64.gram(n) - g).norm() / g.norm()).item()) for n, g in ref.items())
    out["fp64_mode_gram_rel_fro"] = gram_err
    out["int8x4_mode_gram_rel_fro"] = max(float(((ci8.gram(n) - g).norm() / g.norm()).item()) for n, g in ref.items())

    # calibration throughput of the precision modes (same forward, same batches; CUDA events, 3 steps each)
    cache.enabled = False
    modes = {}
    c3 = vlm.GramCache(dev, precision="tf32x3", defer_bytes=cache.defer_bytes, max_pending_bytes=cache.max_pending_bytes)
    c3.register(model, use_moe=True)
    # (int8x4 also under the reference's own fp16 autocast, config.py:116: the fp16 inputs of proj / fc2 are widened exactly)
    for mode, c, mamp in (("fp64", c64, None), ("int8x4", ci8, None), ("int8x4_fp16_autocast", ci8, torch.float16),
                          ("tf32x3", c3, None)):
        for other in (c64, ci8, c3):
            other.enabled = other is c
        c.reset()
        for i in range(2):
            step(dev_batches[i], mamp)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(4):
            step(dev_batches[i % 2], mamp)
        b.record()
        torch.cuda.synchronize(dev)
        modes[mode] = {"value": round(4 * B / (a.elapsed_time(b) * 1e-3), 2), "unit": "samples/s",
                       "ms_per_step": round(a.elapsed_time(b) / 4, 2)}
    c64.remove_hooks()
    ci8.remove_hooks()
    c3.remove_hooks()
    del c64, ci8, c3
    cache.enabled = True
    cache.reset()
    out["gram_precision_modes"] = modes
    return out


def bench_vitl(vlm, dev, group, world, args, B=32, steps=4):
    """Config 5: ViT-L/16 multiway (24 layers, 1024 / 4096 wide, vl experts from layer 21): Gram caching at B = 32 per
    GPU (+ the one all-reduce at N > 1), one 4096-wide Gram checked against the fp64 hook, then the RegMean merge
    of the 96 linear problems (sharded over the ranks) from those Grams."""
    import torch.distributed as dist

    cfg = vlm.vlmo_config("large", attn_impl=args.attn)
    with torch.device(dev):
        model = vlm.VLMo(cfg)
    vlm.init_synthetic_(model.eval(), seed=1)
    rank = dist.get_rank(group) if group is not None else 0
    cache = make_timed_cache(vlm)(dev, defer_bytes=args.defer_mb << 20, max_pending_bytes=args.defer_cap_mb << 20)
    cache.register(model, use_moe=True)
    batches = [vlm.synthetic_batch(B, cfg, seed=4321 + rank * 16 + i, device=dev) for i in range(2)]

    def step(i):
        with torch.no_grad():
            model(batches[i % 2])

    for i in range(2):
        step(i)
    if world > 1:
        cache.all_reduce(group)
    cache.reset()
    # parity of one 4096-wide Gram on identical activations
    name = "transformer.blocks.23.mlp.v.fc2"
    probe = {}
    h = dict(model.named_modules())[name].register_forward_hook(
        lambda m, i, o: probe.__setitem__("g", (lambda x: x.T @ x)(i[0].double().reshape(-1, i[0].shape[-1]))))
    step(0)
    h.remove()
    err = float(((cache.gram(name).double() - probe["g"]).norm() / probe["g"].norm()).item())
    del probe
    cache.reset()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    cache.timing, cache.events = True, []
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        step(i)
    if world > 1:
        cache.all_reduce(group)
    b.record()
    torch.cuda.synchronize(dev)
    cache.timing = False
    ms = a.elapsed_time(b)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    sy_ms = sum(x.elapsed_time(y) for x, y, *_ in cache.events)
    sy_fl = sum(e[2] for e in cache.events)
    # RegMean from these Grams: text rows = steps x 32 x 40 x world >= 4096 -> every summed Gram is full rank
    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], scaling_for_non_diag=0.9,
                loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    rm = []
    for _ in range(2):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        merged = vlm.regmean(sd, mcfg, device=dev, num_layers=24, group=group, gram_matrices=cache)
        torch.cuda.synchronize(dev)
        rm.append(time.perf_counter() - t0)
    finite = bool(torch.isfinite(merged["transformer.blocks.23.mlp.fc2.weight"]).all().item())
    out = {"value": round(world * B * steps / (ms * 1e-3), 2), "unit": "samples/s", "ms_per_step": round(ms / steps, 2),
           "batch_per_gpu": B, "steps": steps, "grams": len(cache.live_names()),
           "syrk_tflops": round(sy_fl / (sy_ms * 1e-3) * 1e-12, 1) if sy_ms > 0 else None,
           "syrk_share_of_step": round(sy_ms / ms, 4), "gram_parity_rel_fro_4096": err,
           "regmean_seconds": round(min(rm), 4), "regmean_linear_problems": 96, "regmean_finite": finite,
           "workload": "VLMo-large all_moe (ViT-L/16 multiway, 24 layers, 51 experts), 192 Grams (144 x 1024^2 + 48 x 4096^2)"}
    cache.remove_hooks()
    del model, cache, sd, merged
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------
REF_BATCH = 4   # samples per reference-arm step (BASELINE.md §3), bounded so that --steps K --warmup W ends within minutes


def build_cpu_reference(model_name):
    """The reference's CPU implementation of the path.  Where the reference sources are present (the build
    container: /root/reference/src, or $VLM_REFERENCE_SRC) this is the UNMODIFIED reference — ViLTransformerSS
    built like src/run.py:165-185, its own hook registered by the loop of src/cache_gram_matrices.py:264-281 —
    imported through the stand-ins of oracle/ref_shims (kind "reference").  On the GPU box the sources are absent
    and the arm falls back to the port: the stock-torch mirror of the forward + the hook restated in oracle/
    (kind "port").  Returns (kind, cfg, step(batch_size, seed) -> samples, store)."""
    import oracle
    import vl_merging_b200 as vlm
    from vl_merging_b200.gram import select_hooked_modules

    torch.set_num_threads(os.cpu_count() or 1)
    cfg = vlm.vlmo_config(model_name)
    store = oracle.new_gram_store()
    kind = "port"
    model = None
    try:
        import ref_harness as rh
        if rh.reference_available() and model_name in ("base", "large") and not os.environ.get("VLM_BENCH_FORCE_PORT"):
            named = {"base": "task_finetune_irtr_coco_square_randaug_base_image384",
                     "large": "task_finetune_irtr_f30k_square_randaug_large_image384"}[model_name]
            ref_cfg = rh.make_config([named, "all_moe"], load_path="", random_initialization=True, per_gpu_batchsize=REF_BATCH)
            model = rh.build_model(ref_cfg)
            rh.ref_register_gram_hooks(model, store, use_moe=True)
            kind = "reference"
    except Exception as e:   # the stand-ins do not cover this environment: say so and time the port
        print(f"# reference import failed ({type(e).__name__}: {e}); timing the port", file=sys.stderr)
        model = None
        store = oracle.new_gram_store()
    if model is None:
        model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1)
        hook = oracle.reference_hook_torch(store)
        for name, module in select_hooked_modules(model, use_moe=True):
            module.module_name = name
            module.register_forward_hook(hook)

    def step(batch_size, seed):
        batch = vlm.synthetic_batch(batch_size, cfg, seed=seed)
        with torch.no_grad():
            if kind == "reference":   # the two towers compute_irtr runs per validation batch (objectives.py:372-470)
                model.infer_text_ft(batch)
                model.infer_image_ft(batch)
            else:
                model(batch)
        return batch_size

    return kind, cfg, step, store


def cpu_baseline_sample(model_name, budget_s=25.0):
    kind, cfg, step, store = build_cpu_reference(model_name)
    t0 = time.perf_counter()
    step(1, 0)  # warm-up (also sizes the sample)
    warm = time.perf_counter() - t0
    per = REF_BATCH if warm * REF_BATCH * 2 < budget_s else 1
    n = max(1, min(8, int(budget_s / max(warm * per, 1e-3)) - 1))
    t0 = time.perf_counter()
    done = 0
    for i in range(n):
        done += step(per, 100 + i)
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": round(done / dt, 4), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{done // per} calibration step(s) of {per} sample(s) (577+40 tokens each, {len(store)} fp64 Grams) of the same VLMo-{model_name} workload, "
                      f"stock forward + reference hook on the host, after 1 warm-up step",
            "cpu_model": cpu_model_name()}


def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    kind, cfg, step, store = build_cpu_reference(args.model)
    per_step = REF_BATCH if args.model != "large" else 1
    for i in range(args.warmup):
        step(per_step, i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(per_step, 1000 + i)
    dt = time.perf_counter() - t0
    v = per_step * args.steps / dt
    sample = (f"{per_step} samples per step (577 image + 40 text tokens each, {len(store)} fp64 Grams), VLMo-{args.model} all_moe, "
              f"host cores only; {'UNMODIFIED reference sources through oracle/ref_shims' if kind == 'reference' else 'port: stock-torch mirror of the forward + the reference hook restated in oracle/ (reference sources absent on this box)'}")
    out = {
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic (same generator as the GPU arm)",
        "config": {"workload": f"RegMean Gram caching, VLMo-{args.model} all_moe, reference CPU path (stock forward + hook_gram_input, "
                               "src/cache_gram_matrices.py:246-254), bounded sample", "global_batch": per_step,
                   "parallelism": "host threads"},
        "cpu_baseline": {"value": round(v, 4), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": sample, "cpu_model": cpu_model_name()},
        "e2e": {"value": round(v, 4), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return out


def bench_reference_hook_on_gpu(vlm, model, cache, dev_batches, B, steps=3):
    """What the reference does when its model sits on a GPU (src/cache_gram_matrices.py:246-254, restated here line
    for line): cast the activation to fp64, one fp64 matmul on the device, a synchronous .cpu() of the d x d result
    and the accumulation on the host — same stock-torch forward, same batches.  Our hooks are removed for good
    (this leg runs last)."""
    from collections import defaultdict

    from vl_merging_b200.gram import select_hooked_modules

    cache.remove_hooks()
    store = defaultdict(float)

    def hook_gram_input(module, input, output):
        if isinstance(input, tuple):
            input = input[0]
        flatten_input = input.reshape(-1, input.shape[-1]).to(torch.float64)
        gram = torch.matmul(flatten_input.T, flatten_input)
        store[module.module_name] += gram.detach().cpu()

    handles = []
    for name, module in select_hooked_modules(model, use_moe=True):
        module.module_name = name
        handles.append(module.register_forward_hook(hook_gram_input))
    try:
        with torch.no_grad():
            model(dev_batches[0])                      # warm-up (cuBLAS fp64 plans, host buffers)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(steps):
                model(dev_batches[(i + 1) % 2])
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
    finally:
        for h in handles:
            h.remove()
    return {"value": round(B * steps / dt, 2), "unit": "samples/s", "steps": steps, "ms_per_step": round(dt / steps * 1e3, 1),
            "grams": len(store),
            "note": "reference hook unchanged (fp64 cast + fp64 matmul on the GPU + .cpu() + host accumulate) on the same "
                    "stock-torch forward and batches; wall clock, one B200"}


def bench_gramfile(vlm, cache, dev):
    """SURVEY §8f rank 4: the Gram artefact on disk.  The reference's format (torch.save of full fp64 matrices,
    cache_gram_matrices.py:349 / vilt_module.py:386) against the packed fp32 upper-triangle container, both written
    from the same device cache and read back onto the device."""
    import shutil
    import tempfile

    tmp = tempfile.mkdtemp(prefix="vlm_gram_")
    ref, packed = os.path.join(tmp, "grams.pth"), os.path.join(tmp, "grams.vlmgram")
    try:
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        cache.save(ref)
        t_ref_save = time.perf_counter() - t
        t = time.perf_counter()
        nbytes = cache.save_packed(packed)
        t_packed_save = time.perf_counter() - t
        t = time.perf_counter()
        g_ref = {k: v.to(dev) for k, v in torch.load(ref, map_location="cpu", weights_only=False).items()}
        torch.cuda.synchronize(dev)
        t_ref_load = time.perf_counter() - t
        t = time.perf_counter()
        g_packed = vlm.gramfile.load_packed(packed, dev)
        torch.cuda.synchronize(dev)
        t_packed_load = time.perf_counter() - t
        same = all(torch.equal(g_packed[k].double(), g_ref[k]) for k in list(g_ref)[:8])
        return {"reference_format": {"bytes": os.path.getsize(ref), "save_seconds": round(t_ref_save, 3),
                                     "load_to_device_seconds": round(t_ref_load, 3)},
                "packed_fp32_upper": {"bytes": nbytes, "save_seconds": round(t_packed_save, 3),
                                      "load_to_device_seconds": round(t_packed_load, 3)},
                "identical_values": bool(same), "grams": len(g_ref)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="base", choices=["base", "large", "tiny"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU)
    ap.add_argument("--autocast", default="fp32", choices=["fp32", "bf16", "fp16"])
    ap.add_argument("--attn", default="sdpa", choices=["reference", "sdpa"],
                    help="attention of the stock-torch forward on the GPU: torch's fused F.scaled_dot_product_attention "
                         "(default; same math, agrees with the explicit form to 1e-7) or the reference's explicit "
                         "softmax(QK^T + bias)V chain, which is also reported under forward_variants")
    ap.add_argument("--no-variants", action="store_true", help="skip the extra (informational) forward variants")
    ap.add_argument("--defer-mb", type=int, default=128,
                    help="GramCache(defer_bytes=...): activations of at most this many MB (text tower, 768-wide image "
                         "activations) are grouped into shared launches; 0 = one launch per hook call")
    ap.add_argument("--defer-cap-mb", type=int, default=1024, help="flush grouped launches once this much is pending")
    ap.add_argument("--gram-precision", default="tf32", choices=["tf32", "tf32x3", "int8x4", "fp64"],
                    help="GramCache precision of the headline run (default: the single TF32 pass; int8x4 / fp64: RegMean-grade fp64 Grams)")
    ap.add_argument("--symmetric", action="store_true",
                    help="N > 1: Gram arenas in torch symmetric memory, exchange as one multimem kernel instead of NCCL")
    ap.add_argument("--no-regmean", action="store_true")
    ap.add_argument("--no-gramfile", action="store_true", help="skip timing the Gram file formats (writes ~2.7 GB to a temp dir)")
    ap.add_argument("--fused", action="store_true",
                    help="also time Gram caching on the fused vision-language route (model.infer, type_id 2: row-sliced activations)")
    ap.add_argument("--irtr", action="store_true",
                    help="also run config 4: modality-arithmetic merge + IRTR forward over 5k synthetic images x 25k captions")
    ap.add_argument("--no-vitl", action="store_true", help="skip the ViT-L leg (config 5) of the default line")
    ap.add_argument("--no-irtr", action="store_true", help="skip the modality-arithmetic + 5k x 25k IRTR leg (config 4) of the default line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip timing the reference's fp64 hook with the model on the GPU")
    ap.add_argument("--profile", action="store_true",
                    help="for ncu launch lists: run exactly --warmup + --steps calibration steps and exit (no JSON line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's logits and a fixed sample of every Gram as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.profile):
        ap.error("--dump-outputs writes the results of the timed GPU run: it needs --impl ours and no --profile")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
