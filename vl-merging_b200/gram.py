"""gram.py — RegMean Gram-matrix caching, the drop-in for the hook closure of
src/cache_gram_matrices.py:236-281 and the artefact written at :349.

Reference                                   here
------------------------------------------  ----------------------------------------------------------
middle_representations = defaultdict(float)  GramCache ([d,d] device buffers, one per hooked module: fp32, or fp64
                                             in the RegMean-grade modes precision="int8x4" / "fp64")
hook_gram_input(module, input, output)       GramCache.hook_gram_input — same signature, same use of
                                             module.module_name; one vlm_syrk_accum (/_i8x4 /_f64) launch on
                                             the current stream instead of fp64 cast + DGEMM + .cpu()
registration loop (:278-281)                 GramCache.register(model, use_moe)
torch.save(middle_representations, path)     GramCache.save(path): {name: fp64 CPU (d,d)} — the file
                                             regmean() loads (vilt_module.py:386)
(absent: every DDP rank writes its own sums) GramCache.all_reduce(): ONE NCCL all-reduce of the packed upper triangles;
                                             GramCache.reduce_scatter(owners): each Gram's sum on the rank whose
                                             regmean(..., group=g) solves it only (ONE NCCL reduce-scatter)
"""
import contextlib
from collections import defaultdict
from typing import NamedTuple

import torch
import torch.nn as nn

from . import _lib

# src/cache_gram_matrices.py:264-276 (the duplicate entry is the reference's)
ALL_KEYS_MOE = (
    "mlp.fc1", "mlp.fc1",
    "mlp.v.fc1", "mlp.l.fc1", "mlp.vl.fc1", "mlp.v.fc2", "mlp.l.fc2", "mlp.vl.fc2",
    "attn",
    "attn.v", "attn.l", "attn.vl",
    "attn.proj",
    "attn.v.proj", "attn.l.proj", "attn.vl.proj",
)
ALL_KEYS_UFO = ("mlp.fc1", "mlp.fc2", "attn.proj", "norm1", "norm2")

_DTYPES = {torch.float32: _lib.VLM_F32, torch.bfloat16: _lib.VLM_BF16, torch.float16: _lib.VLM_F16}


def _in_features(module):
    """Width of the activation a hooked module receives, if it can be known before the first call."""
    if isinstance(module, nn.Linear):
        return module.in_features
    if isinstance(module, nn.LayerNorm):
        return module.normalized_shape[-1]
    qkv = getattr(module, "qkv", None)  # Attention modules: their input is the qkv input
    if isinstance(qkv, nn.Linear):
        return qkv.in_features
    return None


def select_hooked_modules(model, use_moe=True, all_keys=None):
    """The reference's selection rule (src/cache_gram_matrices.py:278-279): every module whose qualified
    name ends with one of all_keys and does not contain '.bias'.  Returns [(name, module)]."""
    keys = all_keys if all_keys is not None else (ALL_KEYS_MOE if use_moe else ALL_KEYS_UFO)
    return [(name, module) for name, module in model.named_modules()
            if any(name.endswith(k) for k in keys) and ".bias" not in name]


def _same_everywhere(obj, group, device):
    """Whether every rank of `group` passed an object with the same repr: one 16-byte all-reduce of a 56-bit digest (the
    max of the digest and of its negation agree only if all digests are equal); the same answer on every rank."""
    import hashlib

    import torch.distributed as dist

    if dist.get_backend(group) == "nccl" and torch.device(device).type != "cuda":
        device = torch.device("cuda", torch.cuda.current_device())
    elif dist.get_backend(group) != "nccl":
        device = torch.device("cpu")
    digest = int.from_bytes(hashlib.sha256(repr(obj).encode()).digest()[:7], "little")      # 56 bits: exact in int64
    t = torch.tensor([digest, -digest], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    hi, neg_lo = t.tolist()
    return hi == -neg_lo


def agree_on_buffers(buffers, group=None, make=None, device=None):
    """Ranks may hold different sets of lazily created buffers (a module whose width was unknown at register() fires on
    some ranks only): agree on the union of (name, width) first and create zero buffers for the names missing
    locally, so every rank issues the same collectives on the same shapes.  Raises if two ranks disagree on a width.
    The common case — every rank holds the same set — costs one 16-byte all-reduce of a digest (max of the digest and
    of its complement agree only if all digests are equal); only a mismatch pays for the all_gather_object."""
    import torch.distributed as dist

    mine = sorted((n, int(g.shape[0])) for n, g in buffers.items())
    if device is None:
        device = next(iter(buffers.values())).device if buffers else torch.device("cpu")
    if _same_everywhere(mine, group, device):    # every rank takes part, with or without buffers
        return [n for n, _ in mine]
    everyone = [None] * dist.get_world_size(group)
    dist.all_gather_object(everyone, mine, group=group)
    union = {}
    for lst in everyone:
        for n, d in lst:
            if union.setdefault(n, d) != d:
                raise RuntimeError(f"Gram {n}: width {d} on one rank, {union[n]} on another")
    for n, d in sorted(union.items()):
        if n not in buffers:
            buffers[n] = make(d)
    return sorted(union)


class ExchangePlan(NamedTuple):
    """What one packed Gram exchange moves (exchange_plan)."""
    names: list      # the Grams that travel, in packed order
    offsets: list    # element offset of each one's packed upper triangle in the flat buffer
    sections: list   # elements per owner rank (all-reduce: one section, every live Gram)
    width: int       # elements per section in the flat buffer: the largest section
    mine: list       # the Grams whose sums this rank keeps, in packed order
    nbytes: int      # last_reduce_bytes
    calls: dict      # {agreed name: call count summed over the ranks}
    rows: dict       # {agreed name: row count summed over the ranks}
    owners: dict     # {name: rank} of the Grams that travel (None for an all-reduce)
    rank: int
    world: int


def exchange_plan(buffers, calls, rows, group=None, owners=None, symmetric=False, make=None, device=None):
    """The host side of a Gram exchange, the same for GramCache.all_reduce() and reduce_scatter(); any backend, no
    CUDA.  Collectives, in this order on every rank: the buffer-set digest (agree_on_buffers, which creates zero
    buffers with `make` for names missing here), one all-reduce of the call / row counters (none when no rank holds a
    buffer), and, with `owners`, one digest of the owner map.  The caller's `calls` and `rows` are never written: their
    sums come back in the plan, to be committed once every check has passed.  Raises ValueError on every rank alike
    when the ranks passed different owner maps, or the map names a Gram that is not live or a rank outside the group.
    owners None: every live Gram travels, back to back in live order, and every rank keeps all of them.  owners
    {name: rank}: the owned Grams travel sorted by owner (stable, so in live order inside each owner's section),
    section r at element r * width of a [world x width] buffer, and this rank keeps its own.
    nbytes: what the NCCL transport moves (the whole flat buffer, padding included), or with `symmetric` what the
    multimem one reduces for this rank (its own triangles)."""
    import torch.distributed as dist

    if device is None:
        device = next(iter(buffers.values())).device if buffers else torch.device("cpu")
    names = agree_on_buffers(buffers, group, make, device)
    summed = {}
    if names:
        counts = torch.tensor([[calls.get(n, 0), rows.get(n, 0)] for n in names], dtype=torch.int64,
                              device=buffers[names[0]].device)
        dist.all_reduce(counts, group=group)
        summed = dict(zip(names, counts.tolist()))
    live = [n for n in names if summed[n][0] > 0]
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if owners is None:
        order, where = live, dict.fromkeys(live, 0)
    else:
        if not _same_everywhere(sorted(owners.items()), group, device):
            raise ValueError("GramCache.reduce_scatter: the ranks passed different owner maps (build it on every rank "
                             "from the same state_dict, config and world, and the live names every rank holds)")
        for n, r in owners.items():
            if n not in live:
                raise ValueError(f"GramCache.reduce_scatter: owner map names {n!r}, which is not a live Gram of this cache "
                                 "(build the map from cache.live_names())")
            if not isinstance(r, int) or not 0 <= r < world:
                raise ValueError(f"GramCache.reduce_scatter: owner {r!r} of {n!r} is not a rank of a {world}-rank group")
        where = {n: owners[n] for n in live if n in owners}
        order = sorted(where, key=where.get)
    tri = {n: buffers[n].shape[0] * (buffers[n].shape[0] + 1) // 2 for n in order}
    sections, offsets = [0] * (1 if owners is None else world), []
    for n in order:
        offsets.append(sections[where[n]])
        sections[where[n]] += tri[n]
    width = max(sections)
    mine = [n for n in order if owners is None or where[n] == rank]
    esz = buffers[names[0]].element_size() if names else 0
    return ExchangePlan(
        names=order, offsets=[where[n] * width + off for n, off in zip(order, offsets)], sections=sections,
        width=width, mine=mine, nbytes=esz * (sum(tri[n] for n in mine) if symmetric else len(sections) * width),
        calls={n: c for n, (c, _) in summed.items()}, rows={n: r for n, (_, r) in summed.items()},
        owners=None if owners is None else where, rank=rank, world=world)


def reduce_gram_buffers(buffers, arenas, calls, rows, group=None):
    """Sum Gram buffers over the ranks of `group`: the per-name call / row counters (exchange_plan), then one
    all-reduce per flat arena (normally exactly one) plus one per buffer that lives outside the arenas, so every
    rank ends up with the same keys.  Works on any backend (NCCL on the GPUs, gloo in the CPU tests)."""
    import torch.distributed as dist

    ref = next(iter(buffers.values()), torch.zeros(0))
    plan = exchange_plan(buffers, calls, rows, group, make=lambda d: torch.zeros(d, d, dtype=ref.dtype, device=ref.device))
    for arena in arenas:
        dist.all_reduce(arena, op=dist.ReduceOp.SUM, group=group)
    spans = [(a.data_ptr(), a.data_ptr() + a.numel() * a.element_size()) for a in arenas]
    for name in plan.calls:     # every agreed name, live or not
        g = buffers[name]
        if not any(lo <= g.data_ptr() < hi for lo, hi in spans):
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
    calls.update(plan.calls)
    rows.update(plan.rows)


def _gram_route(precision, use_simt, dtype, rows, d, ptr, ldx, seg_stride):
    """Which library call takes a GramCache activation of rows x d `dtype` elements at byte address ptr, row pitch ldx
    and segment pitch seg_stride (0: plain rows) in elements: "i8x4", "f64" or "simt" (vlm_syrk_accum_i8x4 / _f64 /
    _simt; simt: exact fp32 products on CUDA cores), "split" (vlm_tf32_split, then the Gram of its {hi, lo} planes) or
    "library" (vlm_syrk_accum / _strided / _batch, which pick the CTA-pair or the CUDA-core kernel themselves)."""
    if precision in ("int8x4", "fp64"):
        aligned = ptr % 16 == 0 and ldx % 4 == 0 and seg_stride % 4 == 0
        return "i8x4" if precision == "int8x4" and d % 128 == 0 and rows * d >= 1 << 20 and aligned else "f64"
    if use_simt:
        return "simt"
    if precision == "tf32x3" and dtype == torch.float32:   # what vlm_tf32_split and the split kernel take
        return "simt" if d % 32 or ptr % 16 or ldx % 4 or seg_stride % 4 else "split"
    return "library"


_DEFERRED_ROUTES = ("split", "library")   # the routes vlm_syrk_accum_batch takes: no CUDA-core-only or fp64 form


class _GramLaunch(NamedTuple):
    """One hooked activation on its way to a Gram entry point (GramCache._launch); GramCache._pending holds the
    deferred ones.  bench.py's TimedCache reads fields 4 and 5 of a pending record as (rows, d): keep the order."""
    code: int             # _DTYPES code of the activation
    keep: torch.Tensor    # the tensor the activation is read from, referenced until its launch is issued
    g: torch.Tensor       # the Gram buffer
    ptr: int              # byte address of the first row
    rows: int
    d: int
    ldx: int              # row pitch, elements
    seg_rows: int         # row slice: rows per segment (0: plain rows)
    seg_stride: int       # row slice: elements between the first rows of consecutive segments
    name: str
    version: int          # keep._version at hook time
    route: str            # _gram_route


class GramCache:
    """Accumulates G[name] += X^T X for every hooked module call, on the GPU (fp32 Grams from one TF32 tensor-core pass by
    default; exact fp64 Grams from the integer tensor cores or the fp64 pipe on request: `precision`).

    All buffers of the modules known at register() time live in one flat arena, so the data-parallel
    reduction is a single all-reduce and the buffers never move.  Modules whose width is only known
    at their first call get individual buffers.
    """

    def __init__(self, device=None, use_simt=False, defer_bytes=0, max_pending=256, max_pending_bytes=1 << 30,
                 side_stream=False, precision="tf32", symmetric=False, deterministic=None):
        """precision: how fp32 activations reach the tensor cores.  "tf32" (default): one TF32 pass, operands rounded
        by TMA — Gram within ~3e-5 of the reference's fp64 Gram (cache_gram_matrices.py:251-252), inside the 1e-3
        tolerance, but its 2^-11 operand rounding noise is amplified by the inverse in regmean
        (vilt_module.py:432-434).  "tf32x3": RegMean-grade Grams — every fp32 activation is split into
        {hi, lo} TF32 planes (vlm_tf32_split) and the kernel forms hi'hi + hi'lo + lo'hi, ~3x the tensor work;
        bf16 / fp16 activations are exact on the tensor core either way.  Both tcgen05 modes accumulate in the
        tensor core's truncating fp32 accumulator (a ~2e-5 non-uniform shrink), which regmean still amplifies when
        the summed Gram has a small eigen-direction (LayerNorm outputs: measured 1.7e-2 on the B200).
        "fp64": the reference's own arithmetic — fp64 products, fp64 accumulation, fp64 Gram buffers
        (vlm_syrk_accum_f64, DMMA tensor cores); the mode that carries regmean to its 1e-4 tolerance.  Launches
        immediately (no grouping).
        "int8x4": the same RegMean-grade fp64 Grams from the INTEGER tensor cores — every column is scaled by a
        power of two and cut into four int8 digit planes, whose products accumulate exactly in int32
        (vlm_syrk_accum_i8x4; Gram error ~1e-9, regmean within 1e-4 like "fp64") at an eighth of the cost (fp32, fp16
        and bf16 activations alike); small problems and widths that are not multiples of 128 take the fp64 path.
        defer_bytes > 0: an activation of at most that many bytes is not launched on its own (the Gram of a
        40-token text batch is launch-bound: ~7 us of fixed cost for ~2 us of tensor-core work, and a 768-wide
        image Gram exposes its prologue and final epilogue); the hook keeps a REFERENCE to it (no copy) and
        flush() issues everything pending as one grouped launch (vlm_syrk_accum_batch), in which one problem's
        epilogue overlaps the next one's mainloop.  register() then also flushes after every forward of the
        registered model.
        Only valid when nothing modifies a hooked activation in place after the hooked module ran — true for the
        VLMo blocks (LayerNorm / attention / GELU outputs are fresh tensors); flush() checks the version counter of
        every held activation and raises if one was written to.  The default 0 keeps the reference's immediate
        semantics.  Deferred activations stay allocated until the flush; a flush is forced
        after max_pending activations or max_pending_bytes of them.
        symmetric=True (under an initialised torch.distributed NCCL group, one process per GPU of one NVSwitch domain):
        the Gram arena is allocated in torch symmetric memory, and all_reduce() then runs as ONE kernel over the
        NVSwitch multicast mapping (vlm_sym_allreduce_multimem: multimem.ld_reduce / multimem.st, no staging buffer,
        no NCCL call) instead of pack -> NCCL all-reduce -> unpack.
        side_stream=True: the SYRK launches go to a second CUDA stream (ordered after the producer of each
        activation by an event), so they overlap the rest of the forward — its LayerNorm / GELU / softmax
        phases leave the tensor pipes idle; flush() joins the two streams.  Like deferral it holds a reference to
        every hooked activation until the next flush() and assumes nothing modifies them in place; register()
        flushes after every forward of the registered model.  Not for precision="int8x4": its persistent 148-CTA kernels
        and the forward's GEMMs do not share SMs well (measured 649 vs 834 samples/s).
        deterministic: every Gram launch of this cache (immediate, deferred or grouped, side stream, every precision)
        runs in the library's deterministic mode (vlm_set_deterministic): the same activations give the same Gram bits
        in every run on the same GPU model and library build, at the cost of a slot workspace and one reduction launch
        per call.  None (default): torch.are_deterministic_algorithms_enabled() at construction.  The library's
        thread-local flag is set only around this cache's own calls."""
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("GramCache needs a CUDA device: the Gram hot path has no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = _lib.lib()
        if precision not in ("tf32", "tf32x3", "fp64", "int8x4"):
            raise ValueError(f"precision must be 'tf32', 'tf32x3', 'fp64' or 'int8x4' (got {precision!r})")
        self.precision = precision
        self.dtype = torch.float64 if precision in ("fp64", "int8x4") else torch.float32   # of the Gram buffers
        self._sym_code = _lib.VLM_F64 if self.dtype == torch.float64 else _lib.VLM_F32    # vlm_sym_* dtype of the buffers
        self._planes = None    # scratch for the {hi, lo} planes of the split mode (grown on demand, reused in stream order)
        self._use_simt = bool(use_simt)   # every fp32-Gram launch on the CUDA-core kernel (device-side oracle)
        self.buffers = {}       # name -> fp32 [d, d] (upper triangle authoritative until finalize())
        self._arenas = []      # flat fp32 arenas the registered buffers are views of
        self.calls = defaultdict(int)
        self.rows = defaultdict(int)
        self._handles = []
        self._finalized = True
        self.enabled = True    # False: the hooks stay registered but ignore their calls
        self.defer_bytes, self.max_pending, self.max_pending_bytes = int(defer_bytes), int(max_pending), int(max_pending_bytes)
        self._pending = []     # _GramLaunch records of the deferred activations
        self._pending_bytes = 0
        self.symmetric, self._symm = bool(symmetric), None   # symmetric-memory arena and its rendezvous handle
        self._side = torch.cuda.Stream(self.device) if side_stream else None
        self._side_keep = []   # activations a side-stream launch may still be reading
        self.deterministic = bool(torch.are_deterministic_algorithms_enabled() if deterministic is None else deterministic)
        self.owners = None     # after reduce_scatter(): {name: rank} of the exchanged Grams; this rank holds its own only
        self._rank = None      # this cache's rank in the reduce_scatter() group

    @contextlib.contextmanager
    def _mode(self):
        """The library's thread-local deterministic flag at this cache's mode for the cache's own launches, restored
        after them."""
        prev = self._lib.vlm_get_deterministic()
        if prev == self.deterministic:
            yield
            return
        self._lib.vlm_set_deterministic(int(self.deterministic))
        try:
            yield
        finally:
            self._lib.vlm_set_deterministic(prev)

    # ---- the hook -------------------------------------------------------------------------------
    def hook_gram_input(self, module, input, output):
        """Forward hook: same contract as the reference closure (cache_gram_matrices.py:246-254)."""
        if not self.enabled:
            return
        if isinstance(input, tuple):
            input = input[0]
        self.accumulate(module.module_name, input)

    __call__ = hook_gram_input

    def accumulate(self, name, x):
        self._require_whole("accumulate")
        with self._mode():
            self._accumulate(name, x)

    def _accumulate(self, name, x):
        d = x.shape[-1]
        if x.device != self.device:
            raise RuntimeError(f"activation for {name} is on {x.device}, GramCache is on {self.device}")
        x = x.detach()
        if x.dtype not in _DTYPES:
            x = x.float()
        elem = x.element_size()
        seg_rows = seg_stride = 0
        try:
            x2 = x.view(-1, d)          # the reference's input.reshape(-1, D) when it is a view
        except RuntimeError:
            x2 = None
        if x2 is None and x.dim() == 3 and x.stride(2) == 1 and x.stride(1) >= d and x.shape[0] > 1 \
                and (x.stride(0) * elem) % 16 == 0 and x.stride(0) > 0:
            # a row slice h[:, a:b] of a (B, N, D) activation (the fused vision-language route hands these to the
            # per-modality experts): read in place as B row segments, where the reference's reshape copies
            rows, ldx, seg_rows, seg_stride, keep = x.shape[0] * x.shape[1], x.stride(1), x.shape[1], x.stride(0), x
        else:
            if x2 is None:
                x2 = x.reshape(-1, d)
            if x2.stride(-1) != 1 or (x2.shape[0] > 1 and x2.stride(0) < d):
                x2 = x2.contiguous()
            rows, ldx, keep = x2.shape[0], (x2.stride(0) if x2.shape[0] > 1 else d), x2
        ptr = keep.data_ptr()
        route = _gram_route(self.precision, self._use_simt, keep.dtype, rows, d, ptr, ldx, seg_stride)
        if route == "simt" and seg_rows:
            keep = x.contiguous()        # the CUDA-core kernel takes plain rows only
            ptr, ldx, seg_rows, seg_stride = keep.data_ptr(), d, 0, 0
        g = self.buffers.get(name)
        if g is None:
            g = self.buffers[name] = torch.zeros(d, d, dtype=self.dtype, device=self.device)
        elif g.shape[0] != d:
            raise RuntimeError(f"{name}: activation width changed from {g.shape[0]} to {d}")
        self.calls[name] += 1
        self.rows[name] += rows
        self._finalized = False
        rec = _GramLaunch(_DTYPES[keep.dtype], keep, g, ptr, rows, d, ldx, seg_rows, seg_stride, name, keep._version, route)
        nbytes = rows * ldx * elem
        if route in _DEFERRED_ROUTES and 0 < nbytes <= self.defer_bytes:
            self._pending.append(rec)
            self._pending_bytes += nbytes
            if len(self._pending) >= self.max_pending or self._pending_bytes >= self.max_pending_bytes:
                self.flush()
            return
        self._launch([rec], self._launch_stream(keep), grouped=False)

    def _launch(self, recs, stream, grouped):
        """Issue the Gram launches of `recs` on `stream`: one record on its route's single-launch entry point, or
        (grouped) records of one dtype and route as ONE vlm_syrk_accum_batch, whose schedule is not the single launch's."""
        lib, route = self._lib, recs[0].route
        if route == "split":   # each record's {hi, lo} planes, back to back in the scratch, stand in for its activation
            planes = self._plane_scratch(sum(2 * r.rows * r.d for r in recs)).data_ptr()
            recs = list(recs)
            for i, r in enumerate(recs):
                _lib.check(lib.vlm_tf32_split(r.ptr, r.rows, r.d, r.ldx, r.seg_rows, r.seg_stride, planes, stream))
                recs[i] = r._replace(code=_lib.VLM_TF32X2, ptr=planes, ldx=r.d, seg_rows=0, seg_stride=0)
                planes += 8 * r.rows * r.d
        if grouped:
            probs = (_lib.SyrkProblem * len(recs))(*(_lib.SyrkProblem(x=r.ptr, rows=r.rows, ldx=r.ldx, g=r.g.data_ptr(),
                ldg=r.g.stride(0), d=r.d, seg_rows=r.seg_rows, seg_stride=r.seg_stride) for r in recs))
            return _lib.check(lib.vlm_syrk_accum_batch(probs, len(recs), recs[0].code, stream))
        (r,) = recs
        g, ldg = r.g.data_ptr(), r.g.stride(0)
        if route == "i8x4":
            nbytes = int(lib.vlm_syrk_i8x4_scratch_bytes(r.rows, r.d))
            scratch = self._plane_scratch((nbytes + 3) // 4).data_ptr()
            _lib.check(lib.vlm_syrk_accum_i8x4(r.ptr, r.code, r.rows, r.d, r.ldx, r.seg_rows, r.seg_stride, scratch, nbytes,
                                               g, ldg, stream))
        elif route == "f64" or r.seg_rows:
            fn = lib.vlm_syrk_accum_f64 if route == "f64" else lib.vlm_syrk_accum_strided
            _lib.check(fn(r.ptr, r.code, r.rows, r.d, r.ldx, r.seg_rows, r.seg_stride, g, ldg, stream))
        else:
            fn = lib.vlm_syrk_accum_simt if route == "simt" else lib.vlm_syrk_accum
            _lib.check(fn(r.ptr, r.code, r.rows, r.d, r.ldx, g, ldg, stream))

    def _plane_scratch(self, numel):
        """fp32 scratch of at least `numel` elements for the {hi, lo} planes.  One buffer, reused by every launch:
        all launches of a cache go to one stream (the current or the side stream), which orders the reuse."""
        if self._planes is None or self._planes.numel() < numel:
            if self._planes is not None and self._side is not None:
                self._planes.record_stream(self._side)
            self._planes = None
            self._planes = torch.empty(int(numel), dtype=torch.float32, device=self.device)
            if self._side is not None:
                self._planes.record_stream(self._side)
        return self._planes

    def _launch_stream(self, keep=None):
        """Raw handle of the stream a SYRK launch goes to.  Side-stream mode: the side stream, made to wait for
        everything queued so far on the current stream (the activation's producer); `keep` stays referenced until
        the join in flush()."""
        cur = torch.cuda.current_stream(self.device)
        if self._side is None:
            return cur.cuda_stream
        self._side.wait_stream(cur)
        if keep is not None:
            self._side_keep.append(keep)
        return self._side.cuda_stream

    def set_side_stream(self, enabled):
        """Switch side-stream mode on or off between forwards (joins first)."""
        self.flush()
        self._side = torch.cuda.Stream(self.device) if enabled else None

    def _join(self):
        if self._side is not None:
            torch.cuda.current_stream(self.device).wait_stream(self._side)
            self._side_keep = []

    def flush(self):
        """Issue every deferred activation (one grouped launch per dtype) and, in side-stream mode, make the
        current stream wait for the Gram launches."""
        with self._mode():
            self._flush()

    def _flush(self):
        if not self._pending:
            return self._join()
        pending, self._pending, self._pending_bytes = self._pending, [], 0
        for p in pending:   # an in-place write to a held activation bumps its version counter: refuse to use it
            if p.keep._version != p.version:
                raise RuntimeError(
                    f"GramCache: the activation hooked for {p.name} was modified in place before the deferred Gram launch "
                    "(its Gram would be taken of the modified values); use defer_bytes=0 for this model")
        stream = self._launch_stream()
        for key in sorted({(p.code, p.route) for p in pending}):   # a cache defers each dtype on one route only
            self._launch([p for p in pending if (p.code, p.route) == key], stream, grouped=True)
        self._join()
        # `pending` (and with it the activations) is released here: the launches are already ordered on the stream

    # ---- registration ---------------------------------------------------------------------------
    def register(self, model, use_moe=True, all_keys=None):
        """The reference's selection rule (cache_gram_matrices.py:278-281): every module whose
        qualified name ends with one of all_keys and does not contain '.bias'.  Sets
        module.module_name and registers the hook; returns the list of hooked names."""
        picked = []
        for name, module in select_hooked_modules(model, use_moe, all_keys):
            module.module_name = name
            self._handles.append(module.register_forward_hook(self.hook_gram_input))
            picked.append((name, _in_features(module)))
        self._allocate_arena([(n, d) for n, d in picked if d is not None and n not in self.buffers])
        if self.defer_bytes > 0 or self._side is not None:
            self._handles.append(model.register_forward_hook(lambda m, i, o: self.flush()))
        return [n for n, _ in picked]

    def _allocate_arena(self, named_dims):
        if not named_dims:
            return
        total = sum(d * d for _, d in named_dims)
        if self.symmetric:
            import torch.distributed._symmetric_memory as symm_mem

            if self._arenas:
                raise RuntimeError("GramCache(symmetric=True): register the model once (one symmetric arena)")
            with torch.cuda.device(self.device):
                arena = symm_mem.empty(total, dtype=self.dtype, device=self.device)
            arena.zero_()
        else:
            arena = torch.zeros(total, dtype=self.dtype, device=self.device)
        off = 0
        for name, d in named_dims:
            self.buffers[name] = arena[off: off + d * d].view(d, d)
            off += d * d
        self._arenas.append(arena)

    def remove_hooks(self):
        self.flush()
        for h in self._handles:
            h.remove()
        self._handles = []

    # ---- results --------------------------------------------------------------------------------
    def live_names(self):
        """Names whose hook fired at least once (ModuleDicts and unused experts never do)."""
        return [n for n in self.buffers if self.calls[n] > 0]

    def all_reduce(self, group=None, packed=True):
        """Data-parallel calibration: sum the per-rank Gram buffers over the ranks of `group` onto every rank (the
        reference has no such step: every DDP rank writes its own file, SURVEY.md §2.2).
        packed: only the upper triangles of the Grams that fired travel (VLMo-base: 0.54 GB instead of the 1.17 GB arena
        with its lower triangles and never-fired `vl` experts; twice that for the fp64 Grams of the int8x4 / fp64
        modes).  Plain caches: one vlm_sym_pack_upper_batch into one flat buffer, ONE NCCL all-reduce, one
        vlm_sym_unpack_batch back into the full symmetric buffers; symmetric caches: one vlm_sym_allreduce_multimem
        launch between two cross-rank barriers, then the local mirror.  Every check that can fail runs, with the same
        outcome on every rank, before the cache changes, so a refused call can be followed by all_reduce(packed=False):
        one all-reduce of each whole arena and of each buffer outside them."""
        self._require_whole("all_reduce")
        self.flush()
        if not packed:
            return reduce_gram_buffers(self.buffers, self._arenas, self.calls, self.rows, group)
        self._exchange(group)

    def reduce_scatter(self, owners, group=None):
        """Data-parallel calibration followed by a sharded regmean(..., group=group): sum each Gram over the ranks of
        `group` onto its owner only.  owners: {Gram name: rank in group}, normally
        regmean_gram_owners(state_dict, config, cache.live_names(), world, num_layers) with the arguments regmean will
        get; it must name live Grams only, and live Grams it leaves out (ones no regmean problem reads) are not summed.
        All ranks must pass the same map.
        Plain caches: the owned upper triangles are packed by owner into [world x width] (width: the largest owner's
        section; one vlm_sym_pack_upper_batch), ONE NCCL reduce-scatter, and this rank's section unpacked into its
        Grams (one vlm_sym_unpack_batch): each rank sends (world - 1) / world of the buffer instead of the all-reduce's
        2 (world - 1) / world, and unpacks only its own Grams.  Symmetric caches: one vlm_sym_reduce_multimem
        launch over this rank's Grams between two cross-rank barriers, then their local mirror.  Checks as in
        all_reduce(), the owner map's included, before the cache changes.
        Afterwards the cache is scattered: `owners` records the map, this rank's own Grams hold the full symmetric
        sums and gram() returns them; the other Grams, state_dict() / save() / save_packed(), all_reduce() and
        further accumulation raise until reset().  live_names() is still the full agreed list on every rank."""
        self._require_whole("reduce_scatter")
        self.flush()
        self._exchange(group, owners)

    def _exchange(self, group, owners=None):
        """Both packed exchanges: the plan (agreement, counters, owner-map checks), the multicast setup of a symmetric
        cache (its checks and rendezvous), then the commit and one transport."""
        import torch.distributed as dist

        group = group if group is not None else dist.group.WORLD
        plan = exchange_plan(self.buffers, self.calls, self.rows, group, owners, self.symmetric,
                             lambda d: torch.zeros(d, d, dtype=self.dtype, device=self.device), self.device)
        if owners is None and not plan.names:
            return                             # no Gram fired on any rank
        if self.symmetric:
            mc, spans = self._multicast_spans(plan.names, plan.mine, group)
        self.calls.update(plan.calls)
        self.rows.update(plan.rows)
        if owners is not None:
            self.owners, self._rank = plan.owners, plan.rank
        self._finalized = True
        self.last_reduce_bytes = plan.nbytes
        if not plan.names:
            return
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if self.symmetric:
            with torch.cuda.device(self.device):
                self._symm.barrier(channel=0)  # every rank's Gram launches have completed
                if owners is None:             # every sum stored into every rank's arena (multimem.st)
                    _lib.check(self._lib.vlm_sym_allreduce_multimem(mc, spans, len(spans), self._sym_code, plan.rank,
                                                                    plan.world, stream))
                else:                          # this rank's sums stored into its own arena only
                    _lib.check(self._lib.vlm_sym_reduce_multimem(mc, self._arenas[0].data_ptr(), spans, len(spans),
                                                                 self._sym_code, stream))
                self._symm.barrier(channel=0)  # every store has landed, and nobody reads a rank's arena any more
                self._sym_launch(self._lib.vlm_sym_mirror_batch, plan.mine)     # lower triangles, locally
            return
        flat = torch.empty(len(plan.sections) * plan.width, dtype=self.dtype, device=self.device)  # padding: never read
        self._sym_launch(self._lib.vlm_sym_pack_upper_batch, plan.names, flat, plan.offsets)
        if owners is None:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
            out, base = flat, 0
        else:
            out, base = torch.empty(plan.width, dtype=self.dtype, device=self.device), plan.rank * plan.width
            dist.reduce_scatter_tensor(out, flat, op=dist.ReduceOp.SUM, group=group)
        offset = dict(zip(plan.names, plan.offsets))
        self._sym_launch(self._lib.vlm_sym_unpack_batch, plan.mine, out, [offset[n] - base for n in plan.mine])

    def _require_whole(self, what, name=None):
        """Raise if this cache was reduce_scatter()ed (and `name`, when given, is not one of this rank's Grams)."""
        if self.owners is None or (name is not None and self.owners.get(name) == self._rank):
            return
        raise RuntimeError(f"GramCache.{what}: this cache was reduce_scatter()ed, so this rank holds the summed Grams it "
                           "owns only; pass the cache to regmean(..., gram_matrices=cache, group=...) with the same "
                           "arguments as the owner map, use all_reduce() instead of reduce_scatter() for Gram files and "
                           "state_dict(), or reset() it to calibrate again")

    def _multicast_spans(self, names, mine, group):
        """Checks of the multimem exchange and its spans: (multicast address, vlm_sym_span array of `mine`).  Every
        Gram of `names` must lie in the one symmetric arena and meet the kernel's alignment rules, so every rank
        raises or none does."""
        import torch.distributed._symmetric_memory as symm_mem

        if len(self._arenas) != 1:
            raise RuntimeError("GramCache(symmetric=True): no symmetric arena (register() the model before calibrating)")
        arena = self._arenas[0]
        lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel() * arena.element_size()
        for n in names:
            g = self.buffers[n]
            if not lo <= g.data_ptr() < hi:
                raise RuntimeError("GramCache(symmetric=True): a Gram buffer lives outside the symmetric arena (a module "
                                   "whose width was unknown at register()); use a plain cache (NCCL exchange) for this model")
            if (g.data_ptr() - lo) % 16 or (self.dtype == torch.float32 and (g.shape[0] % 4 or g.stride(0) % 4)):
                raise RuntimeError(f"GramCache(symmetric=True): Gram {n} of width {g.shape[0]} does not meet the multimem "
                                   "alignment rules (16-byte offset; fp32 widths a multiple of 4); use a plain cache")
        if self._symm is None:
            self._symm = symm_mem.rendezvous(arena, group)          # collective: every rank, same order
        mc = int(self._symm.multicast_ptr or 0)
        if mc == 0:
            raise RuntimeError("GramCache(symmetric=True): this system offers no multicast mapping (NVSwitch + driver "
                               "support needed); use a plain cache (NCCL exchange)")
        spans = (_lib.SymSpan * len(mine))()
        for sp, n in zip(spans, mine):
            g = self.buffers[n]
            sp.offset_bytes, sp.d, sp.ld = g.data_ptr() - lo, g.shape[0], g.stride(0)
        return mc, spans

    def finalize(self):
        """Mirror the upper triangles into the lower ones (after the last accumulate / all_reduce)."""
        self.flush()
        if self._finalized:
            return
        self._sym_launch(self._lib.vlm_sym_mirror_batch, self.live_names())
        self._finalized = True

    def _sym_launch(self, fn, names, packed=None, offsets=None):
        """One batched vlm_sym_* launch (pack_upper, unpack or mirror) over the named Grams, on the current stream;
        packed / offsets as in _lib.sym_items."""
        items = _lib.sym_items([self.buffers[n] for n in names], packed, offsets)
        _lib.check(fn(items, len(names), self._sym_code, torch.cuda.current_stream(self.device).cuda_stream))

    def gram(self, name):
        """Full symmetric fp32 Gram of one module, on the device (of a scattered cache: one this rank owns)."""
        self._require_whole(f"gram({name!r})", name)
        self.finalize()
        return self.buffers[name]

    def state_dict(self, dtype=torch.float64, device="cpu"):
        """{module_name: (d,d) tensor} for every module that fired — by default fp64 CPU tensors, the
        format of the reference's Gram file, in the reference's insertion order (first-call order
        there; registration order here, which is the same for a sequential forward)."""
        self._require_whole("state_dict")
        self.finalize()
        out = defaultdict(float)
        for name in self.live_names():
            # dtype first, on the device (a blocking .to(device, dtype) would convert on the host, after the copy);
            # an fp64 cache never hands out its own buffers, an fp32 one does for fp32 on its own device
            out[name] = self.buffers[name].to(dtype).to(device, copy=self.dtype == dtype == torch.float64)
        return out

    def save(self, path):
        """torch.save of the reference-format dict (src/cache_gram_matrices.py:349)."""
        self._require_whole("save")
        torch.save(self.state_dict(), path)

    def save_packed(self, path):
        """The packed upper-triangle container (gramfile.py) in the cache's own element type: fp32 (a quarter of the
        reference file's bytes) or, for the RegMean-grade caches, fp64 (half); regmean reads either, and the
        reference's own format.  Returns the number of bytes written."""
        from . import gramfile
        return gramfile.save_packed(self, path)

    def reset(self):
        self._pending, self._pending_bytes = [], 0
        self._join()
        for g in self.buffers.values():
            g.zero_()
        self.calls.clear()
        self.rows.clear()
        self._finalized = True
        self.owners = None


def hook_gram_input_factory(cache):
    """For code that wants a bare function like the reference's closure."""

    def hook_gram_input(module, input, output):
        cache.hook_gram_input(module, input, output)

    return hook_gram_input


def cache_gram_matrices(model, batches, path=None, use_moe=True, autocast_dtype=None, group=None, **cache_kwargs):
    """The calibration flow of src/cache_gram_matrices.py:236-349 as one call: register the hooks on `model`
    (already on its GPU, eval mode), run it over `batches` (an iterable of batch dicts; under torch.distributed
    each rank passes ITS shard), sum the ranks, optionally write the reference-format Gram file (rank 0 only —
    the reference lets every rank overwrite the same path).  Returns the GramCache."""
    import torch.distributed as dist

    device = next(model.parameters()).device
    cache = GramCache(device, **cache_kwargs)
    cache.register(model, use_moe=use_moe)
    try:
        with torch.no_grad():
            for batch in batches:
                if autocast_dtype is None:
                    model(batch)
                else:
                    with torch.autocast("cuda", dtype=autocast_dtype):
                        model(batch)
    finally:
        cache.remove_hooks()
    if group is not None or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        cache.all_reduce(group)
    if path is not None and (not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0):
        cache.save(path)
    return cache
