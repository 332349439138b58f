"""Development helper: where the time of GramCache.all_reduce() goes (host wall clock per phase, GPU drained after each).
torchrun --nproc-per-node N tools/exchange_trace.py [--symmetric]"""
import os
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
cache = vlm.GramCache(dev, symmetric=symmetric)
cache.register(model)
for n in cache.buffers:                       # pretend every registered Gram fired
    if ".vl" not in n and not isinstance(dict(model.named_modules())[n], torch.nn.ModuleDict):
        cache.calls[n], cache.rows[n] = 1, 617
        cache.buffers[n].fill_(1.0)
cache._finalized = False


def timed(label, fn):
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) * 1e3
    if rank == 0:
        print(f"{label:34s} {dt:8.3f} ms", flush=True)
    return out


for it in range(3):
    if rank == 0:
        print(f"--- iteration {it} ({'multimem' if symmetric else 'NCCL'}, world {world})", flush=True)
    timed("whole all_reduce()", lambda: cache.all_reduce())
    names = timed("agree_on_buffers", lambda: G.agree_on_buffers(cache.buffers, None, None, device=dev))
    timed("_reduce_counts", lambda: G._reduce_counts(cache.buffers, names, dict(cache.calls), dict(cache.rows), None))
    x = torch.ones(134_544_384, device=dev)
    timed("NCCL all_reduce of 538 MB", lambda: dist.all_reduce(x))
    if symmetric:
        timed("handle.barrier()", lambda: cache._symm.barrier(channel=0))
        from vl_merging_b200 import _lib
        live = cache.live_names()
        arena = cache._arenas[0]
        spans = (_lib.SymSpan * len(live))()
        for sp, n in zip(spans, live):
            g = cache.buffers[n]
            sp.offset_bytes, sp.d, sp.ld = g.data_ptr() - arena.data_ptr(), g.shape[0], g.stride(0)
        st = torch.cuda.current_stream().cuda_stream
        L = _lib.lib()
        mc = int(cache._symm.multicast_ptr)
        timed("multimem kernel alone", lambda: _lib.check(L.vlm_sym_allreduce_multimem(mc, spans, len(live), 0, rank, world, st)))
        items = _lib.sym_items([cache.buffers[n] for n in live])
        timed("local mirror alone", lambda: _lib.check(L.vlm_sym_mirror_batch(items, len(live), 0, st)))
    else:
        from vl_merging_b200 import _lib
        live = cache.live_names()
        grams = [cache.buffers[n] for n in live]
        flat = torch.empty(sum(g.shape[0] * (g.shape[0] + 1) // 2 for g in grams), device=dev)
        items = _lib.sym_items(grams, flat)
        st = torch.cuda.current_stream().cuda_stream
        L = _lib.lib()
        timed("pack (one launch)", lambda: _lib.check(L.vlm_sym_pack_upper_batch(items, len(live), 0, st)))
        timed("unpack (one launch)", lambda: _lib.check(L.vlm_sym_unpack_batch(items, len(live), 0, st)))
dist.destroy_process_group()
