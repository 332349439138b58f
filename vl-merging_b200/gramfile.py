"""gramfile.py — packed Gram container (SURVEY.md §8f rank 4).

The reference writes its Gram matrices with `torch.save(middle_representations, ...)`
(src/cache_gram_matrices.py:349) and reads them back with `torch.load` in regmean
(src/vilt/modules/vilt_module.py:386): a pickle of full symmetric fp64 matrices — 2.15 GB for VLMo-base,
7.65 GB for ViT-L — although the accumulators here are fp32 and symmetric.  This container stores the
row-major UPPER TRIANGLE in fp32 (a quarter of the bytes) as one flat blob:

    bytes 0..7     magic  b"VLMGRAM1"
    bytes 8..15    little-endian uint64: length H of the JSON header
    bytes 16..16+H header: {"version": 1, "dtype": "float32" | "float64", "layout": "upper_rowmajor",
                            "entries": [{"name", "d", "offset" (in elements), "rows", "calls"}, ...]}
    zero padding to a multiple of 4096
    data: for each entry d*(d+1)/2 values, row r = columns r..d-1

dtype float32 is what the default cache accumulates; float64 (half the reference file instead of a quarter) keeps the
Grams of the RegMean-grade caches (GramCache(precision="int8x4" / "fp64")) exactly.

`GramCache.save_packed` / `save_packed` write it (ONE pack launch on the device, ONE device->host copy),
`load_packed` reads it back as device matrices for `regmean` (ONE host->device copy + ONE unpack launch, in the
file's element type), and `export_reference` / `import_reference` convert to and from the reference's own file, so
either side can consume the other's artefact.  The kernels are vlm_sym_pack_upper_batch / vlm_sym_unpack_batch.
"""
import json
import os
import struct
from collections import defaultdict

import numpy as np
import torch

from . import _lib

MAGIC = b"VLMGRAM1"
_ALIGN = 4096


def is_packed_file(path):
    try:
        with open(path, "rb") as f:
            return f.read(len(MAGIC)) == MAGIC
    except (OSError, TypeError):
        return False


def _packed_len(d):
    return d * (d + 1) // 2


def _device_of(device):
    device = torch.device(device if device is not None else "cuda")
    if device.type != "cuda":
        raise RuntimeError("the packed Gram container is packed / unpacked on the GPU: there is no CPU fallback")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def save_packed(grams, path, rows=None, calls=None, device=None, dtype=None):
    """grams: {name: (d, d) tensor} (any float dtype / device; only the upper triangles are read) or a
    GramCache.  dtype: torch.float32 or torch.float64 of the stored values; None = float64 for a cache that
    accumulates fp64 Grams, float32 otherwise.  Returns the number of bytes written."""
    if hasattr(grams, "buffers") and hasattr(grams, "live_names"):
        if dtype is None:
            dtype = grams.dtype
        cache = grams
        cache.flush()
        device = cache.device
        rows, calls = cache.rows, cache.calls
        grams = {n: cache.buffers[n] for n in cache.live_names()}
    device = _device_of(device)
    dtype = dtype or torch.float32
    if dtype not in (torch.float32, torch.float64):
        raise ValueError("dtype must be torch.float32 or torch.float64")
    esz, code = (4, _lib.VLM_F32) if dtype == torch.float32 else (8, _lib.VLM_F64)
    lib = _lib.lib()
    names = list(grams.keys())
    entries, total = [], 0
    for n in names:
        d = int(grams[n].shape[0])
        if grams[n].dim() != 2 or grams[n].shape[1] != d:
            raise ValueError(f"{n}: Gram must be square, got {tuple(grams[n].shape)}")
        entries.append({"name": n, "d": d, "offset": total, "rows": int((rows or {}).get(n, 0)),
                        "calls": int((calls or {}).get(n, 0))})
        total += _packed_len(d)
    with torch.cuda.device(device):
        packed = torch.empty(total, dtype=dtype, device=device)
        stream = torch.cuda.current_stream(device).cuda_stream
        keep = []
        for n in names:
            g = grams[n].detach().to(device=device, dtype=dtype)
            keep.append(g if g.stride(1) == 1 else g.contiguous())
        items = _lib.sym_items(keep, packed, [e["offset"] for e in entries])
        _lib.check(lib.vlm_sym_pack_upper_batch(items, len(entries), code, stream))   # one launch for all Grams
        host = torch.empty(total, dtype=dtype, pin_memory=True)
        host.copy_(packed, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
    header = json.dumps({"version": 1, "dtype": "float32" if dtype == torch.float32 else "float64", "layout": "upper_rowmajor",
                         "entries": entries}).encode()
    pre = MAGIC + struct.pack("<Q", len(header)) + header
    pad = (-len(pre)) % _ALIGN
    tmp = f"{path}.tmp.{os.getpid()}"
    try:
        with open(tmp, "wb") as f:
            f.write(pre + b"\0" * pad)
            f.write(memoryview(host.numpy()).cast("B"))
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return len(pre) + pad + esz * total


def read_header(path, with_dtype=False):
    """(entries, data_offset_in_bytes) of a packed Gram file; with_dtype: (entries, offset, torch dtype of the values)."""
    with open(path, "rb") as f:
        if f.read(len(MAGIC)) != MAGIC:
            raise ValueError(f"{path} is not a packed Gram file (bad magic)")
        (hlen,) = struct.unpack("<Q", f.read(8))
        header = json.loads(f.read(hlen).decode())
    if header.get("version") != 1 or header.get("layout") != "upper_rowmajor" or header.get("dtype") not in ("float32", "float64"):
        raise ValueError(f"{path}: unsupported packed Gram header {header.get('version')}/{header.get('layout')}/{header.get('dtype')}")
    pre = len(MAGIC) + 8 + hlen
    off = pre + ((-pre) % _ALIGN)
    if with_dtype:
        return header["entries"], off, torch.float32 if header["dtype"] == "float32" else torch.float64
    return header["entries"], off


def load_packed(path, device=None, dtype=None):
    """{name: full symmetric (d, d) device tensor}: what regmean(gram_matrices=...) takes.  dtype: torch.float32 or
    torch.float64 of the returned matrices; None = the file's own.  One host->device copy of the blob, then one unpack
    launch for all Grams in the file's element type; another dtype is converted Gram by Gram after that."""
    device = _device_of(device)
    entries, off, fdtype = read_header(path, with_dtype=True)
    dtype = dtype or fdtype
    if dtype not in (torch.float32, torch.float64):
        raise ValueError("dtype must be torch.float32 or torch.float64")
    esz = 4 if fdtype == torch.float32 else 8
    total = sum(_packed_len(e["d"]) for e in entries)
    size = os.path.getsize(path)
    if size < off + esz * total:
        raise ValueError(f"{path}: truncated ({size} bytes, header promises {off + esz * total})")
    lib = _lib.lib()
    host = torch.empty(total, dtype=fdtype, pin_memory=True)
    view, got = memoryview(host.numpy()).cast("B"), 0
    with open(path, "rb", buffering=0) as f:
        f.seek(off)
        while got < esz * total:           # one read() moves at most 2 GB
            n = f.readinto(view[got:got + (1 << 30)])
            if not n:
                raise ValueError(f"{path}: short read")
            got += n
    with torch.cuda.device(device):
        packed = host.to(device, non_blocking=True)
        stream = torch.cuda.current_stream(device).cuda_stream
        grams = [torch.empty(e["d"], e["d"], dtype=fdtype, device=device) for e in entries]
        items = _lib.sym_items(grams, packed, [e["offset"] for e in entries])
        _lib.check(lib.vlm_sym_unpack_batch(items, len(grams), _lib.VLM_F32 if fdtype == torch.float32 else _lib.VLM_F64,
                                            stream))
        if dtype != fdtype:
            for i in range(len(grams)):      # one Gram at a time: each file-dtype matrix is released once converted
                grams[i] = grams[i].to(dtype)
        torch.cuda.current_stream(device).synchronize()   # `packed` and `host` may be released after this
    return {e["name"]: g for e, g in zip(entries, grams)}


def export_reference(packed_path, reference_path, device=None):
    """Packed container -> the reference's Gram file: torch.save of {name: fp64 CPU (d, d)} in a defaultdict
    (src/cache_gram_matrices.py:236,349), consumable by the unmodified reference regmean."""
    grams = load_packed(packed_path, device, dtype=torch.float64)
    out = defaultdict(float)
    for k, v in grams.items():
        out[k] = v.cpu()
    torch.save(out, reference_path)
    return reference_path


def import_reference(reference_path, packed_path, device=None, dtype=torch.float32):
    """The reference's Gram file -> packed container (the lower triangles are dropped; values rounded to fp32 unless
    dtype=torch.float64)."""
    grams = torch.load(reference_path, map_location="cpu", weights_only=False)
    return save_packed({k: v for k, v in grams.items() if torch.is_tensor(v)}, packed_path, device=device, dtype=dtype)


def packed_bytes(dims, dtype=torch.float32):
    """Size of the data section for Grams of the given widths; e.g. VLMo-base IRTR: 72 x 768 + 24 x 3072."""
    return (4 if dtype == torch.float32 else 8) * int(np.sum([_packed_len(int(d)) for d in dims]))
