"""Development helper: where the time of GramCache.all_reduce() goes (host wall clock per phase, GPU drained after each).
torchrun --nproc-per-node N tools/exchange_trace.py [--symmetric]
    the phases are the library's own steps: exchange_plan (the buffer-set agreement and the counter all-reduce;
    agree_on_buffers alone is timed too), the cache's multicast setup and its batched pack / unpack / mirror launches
torchrun --nproc-per-node N tools/exchange_trace.py --reduce-scatter
    whole-call host time of reduce_scatter() (by regmean_gram_owners) against all_reduce(), for fp32 and fp64 caches,
    NCCL and multimem (symmetric=True), after a barrier and ending in a device synchronise; VLMo-base's 96 Grams."""
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vl_merging_b200 as vlm  # noqa: E402
from vl_merging_b200 import gram as G  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
symmetric = "--symmetric" in sys.argv
cfg = vlm.vlmo_config("base")
with torch.device(dev):
    model = vlm.VLMo(cfg)
vlm.init_synthetic_(model.eval(), seed=1)
modules = dict(model.named_modules())


def fire(cache):
    """Pretend every registered Gram of the v / l experts fired (the 96 Grams of an irtr calibration)."""
    for n in cache.buffers:
        if ".vl" not in n and not isinstance(modules[n], torch.nn.ModuleDict):
            cache.calls[n], cache.rows[n] = 1, 617
            cache.buffers[n].fill_(1.0)
    cache._finalized = False


cache = vlm.GramCache(dev, symmetric=symmetric)
cache.register(model)
fire(cache)


def timed(label, fn):
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) * 1e3
    if rank == 0 and label is not None:
        print(f"{label:34s} {dt:8.3f} ms", flush=True)
    return out if label is not None else dt


def reduce_scatter_leg(iters=7):
    if rank == 0:
        limit = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip()
        print(f"card: {torch.cuda.get_device_name(dev)}, power limit {limit}, world {world}", flush=True)
    sd = model.state_dict()
    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], scaling_for_non_diag=1.0,
                loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0})
    for precision in ("tf32", "fp64"):
        for sym in (False, True):
            c = vlm.GramCache(dev, precision=precision, symmetric=sym)
            c.register(model)
            fire(c)
            owners = vlm.regmean_gram_owners(sd, mcfg, c.live_names(), world)
            what = f"{'fp64' if precision == 'fp64' else 'fp32'} {'multimem' if sym else 'NCCL'}"
            times = {"all_reduce": [], "reduce_scatter": []}
            try:
                for _ in range(iters):
                    times["all_reduce"].append(timed(None, c.all_reduce))
                    bytes_ar = c.last_reduce_bytes
                    c.reset()
                    fire(c)
                    times["reduce_scatter"].append(timed(None, lambda: c.reduce_scatter(owners)))
                    bytes_rs = c.last_reduce_bytes
                    c.reset()
                    fire(c)
            except RuntimeError as e:
                if "multicast" not in str(e):
                    raise
                if rank == 0:
                    print(f"{what:14s} skipped: {e}", flush=True)
                continue
            if rank == 0:
                for k, v in times.items():
                    v = v[1:]                     # the first call of each sets up the exchange buffers / communicators
                    print(f"{what:14s} {k:15s} median {statistics.median(v):7.3f} ms  min {min(v):7.3f} ms  "
                          f"max {max(v):7.3f} ms  ({len(v)} calls, last_reduce_bytes "
                          f"{bytes_ar if k == 'all_reduce' else bytes_rs})", flush=True)
            del c
            torch.cuda.empty_cache()


if "--reduce-scatter" in sys.argv:
    reduce_scatter_leg()
    dist.destroy_process_group()
    sys.exit(0)

L = vlm._lib.lib()
for it in range(3):
    if rank == 0:
        print(f"--- iteration {it} ({'multimem' if symmetric else 'NCCL'}, world {world})", flush=True)
    timed("whole all_reduce()", lambda: cache.all_reduce())
    timed("agree_on_buffers", lambda: G.agree_on_buffers(cache.buffers, None, None, device=dev))
    plan = timed("exchange_plan", lambda: G.exchange_plan(cache.buffers, cache.calls, cache.rows, None,
                                                          symmetric=symmetric, device=dev))
    x = torch.ones(134_544_384, device=dev)
    timed("NCCL all_reduce of 538 MB", lambda: dist.all_reduce(x))
    if symmetric:
        timed("handle.barrier()", lambda: cache._symm.barrier(channel=0))
        mc, spans = cache._multicast_spans(plan.names, plan.mine, dist.group.WORLD)
        st = torch.cuda.current_stream().cuda_stream
        timed("multimem kernel alone", lambda: vlm._lib.check(L.vlm_sym_allreduce_multimem(
            mc, spans, len(spans), cache._sym_code, rank, world, st)))
        timed("local mirror alone", lambda: cache._sym_launch(L.vlm_sym_mirror_batch, plan.mine))
    else:
        flat = torch.empty(len(plan.sections) * plan.width, device=dev)
        timed("pack (one launch)", lambda: cache._sym_launch(L.vlm_sym_pack_upper_batch, plan.names, flat, plan.offsets))
        timed("unpack (one launch)", lambda: cache._sym_launch(L.vlm_sym_unpack_batch, plan.mine, flat, plan.offsets))
dist.destroy_process_group()
