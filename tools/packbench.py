"""Development helper: the batched pack / unpack / mirror launches over the 96 Grams of VLMo-base (one GPU)."""
import sys, os, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vl_merging_b200 import _lib

dims = [768] * 72 + [3072] * 24
dev = torch.device("cuda")
arena = torch.randn(sum(d * d for d in dims), device=dev)
sizes = [d * (d + 1) // 2 for d in dims]
flat = torch.empty(sum(sizes), device=dev)
grams, off = [], 0
for d in dims:
    grams.append(arena[off: off + d * d].view(d, d))
    off += d * d
items = _lib.sym_items(grams, flat)
L, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
fns = {"pack": lambda: L.vlm_sym_pack_upper_batch(items, len(dims), 0, st),
       "unpack": lambda: L.vlm_sym_unpack_batch(items, len(dims), 0, st),
       "mirror": lambda: L.vlm_sym_mirror_batch(items, len(dims), 0, st)}
for name, fn in fns.items():
    for _ in range(2):
        _lib.check(fn())
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        _lib.check(fn())
    b.record()
    torch.cuda.synchronize()
    print(f"{name:8s} {a.elapsed_time(b) / 10:7.3f} ms per launch (CUDA events)")
