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
(absent: every DDP rank writes its own sums) GramCache.all_reduce(): ONE NCCL all-reduce of the packed upper triangles
"""
import contextlib
from collections import defaultdict

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


def agree_on_buffers(buffers, group=None, make=None, device=None):
    """Ranks may hold different sets of lazily created buffers (a module whose width was unknown at register() fires on
    some ranks only): agree on the union of (name, width) first and create zero buffers for the names missing
    locally, so every rank issues the same collectives on the same shapes.  Raises if two ranks disagree on a width.
    The common case — every rank holds the same set — costs one 16-byte all-reduce of a digest (max of the digest and
    of its complement agree only if all digests are equal); only a mismatch pays for the all_gather_object."""
    import hashlib

    import torch.distributed as dist

    mine = sorted((n, int(g.shape[0])) for n, g in buffers.items())
    if device is None:
        device = next(iter(buffers.values())).device if buffers else torch.device("cpu")
    if dist.get_backend(group) == "nccl" and torch.device(device).type != "cuda":
        device = torch.device("cuda", torch.cuda.current_device())
    elif dist.get_backend(group) != "nccl":
        device = torch.device("cpu")
    digest = int.from_bytes(hashlib.sha256(repr(mine).encode()).digest()[:7], "little")      # 56 bits: exact in int64
    t = torch.tensor([digest, -digest], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)    # every rank takes part, with or without buffers
    hi, neg_lo = t.tolist()
    if hi == -neg_lo:                                         # max == min: the same set everywhere (same test on every rank)
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


def reduce_gram_buffers(buffers, arenas, calls, rows, group=None):
    """Sum Gram buffers over the ranks of `group`: one all-reduce per flat arena (normally exactly one)
    plus one per buffer that lives outside the arenas, then the per-name call / row counters, so every
    rank ends up with the same keys.  Works on any backend (NCCL on the GPUs, gloo in the CPU tests)."""
    import torch.distributed as dist

    if buffers:
        ref = next(iter(buffers.values()))
        names = agree_on_buffers(buffers, group, lambda d: torch.zeros(d, d, dtype=ref.dtype, device=ref.device))
    else:
        names = agree_on_buffers(buffers, group, lambda d: torch.zeros(d, d))
    for arena in arenas:
        dist.all_reduce(arena, op=dist.ReduceOp.SUM, group=group)
    spans = [(a.data_ptr(), a.data_ptr() + a.numel() * a.element_size()) for a in arenas]
    for name in names:
        g = buffers[name]
        if not any(lo <= g.data_ptr() < hi for lo, hi in spans):
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
    _reduce_counts(buffers, names, calls, rows, group)


def _reduce_counts(buffers, names, calls, rows, group):
    import torch.distributed as dist

    if names:
        dev = buffers[names[0]].device
        counts = torch.tensor([[calls[n], rows[n]] for n in names], dtype=torch.int64, device=dev)
        dist.all_reduce(counts, group=group)
        for n, (c, r) in zip(names, counts.tolist()):
            calls[n], rows[n] = c, r


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
        self._pending = []     # (dtype code, keep-alive tensor, g, ptr, rows, d, ldx, seg_rows, seg_stride)
        self._pending_bytes = 0
        self.symmetric, self._symm = bool(symmetric), None   # symmetric-memory arena and its rendezvous handle
        self._side = torch.cuda.Stream(self.device) if side_stream else None
        self._side_keep = []   # activations a side-stream launch may still be reading
        self.deterministic = bool(torch.are_deterministic_algorithms_enabled() if deterministic is None else deterministic)

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
        # tf32x3 splits fp32 activations that vlm_tf32_split and the split kernel take (d % 32 == 0, 16-byte aligned x,
        # ldx and seg_stride multiples of 4); any other one goes to the CUDA-core kernel (exact fp32 products) at once:
        # it must not join a deferred group, which flush() issues as split planes
        split = self.precision == "tf32x3" and keep.dtype == torch.float32
        simt = self._use_simt or (split and bool(d % 32 or ptr % 16 or ldx % 4 or seg_stride % 4))
        split = split and not simt
        if simt and seg_rows:
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
        code = _DTYPES[keep.dtype]
        nbytes = rows * ldx * elem
        if self.precision == "int8x4" and d % 128 == 0 and rows * d >= (1 << 20) \
                and ptr % 16 == 0 and ldx % 4 == 0 and seg_stride % 4 == 0:
            nbytes = int(self._lib.vlm_syrk_i8x4_scratch_bytes(rows, d))
            scratch = self._plane_scratch((nbytes + 3) // 4)
            _lib.check(self._lib.vlm_syrk_accum_i8x4(ptr, code, rows, d, ldx, seg_rows, seg_stride, scratch.data_ptr(),
                                                     nbytes, g.data_ptr(), g.stride(0), self._launch_stream(keep)))
            return
        if self.dtype == torch.float64:
            _lib.check(self._lib.vlm_syrk_accum_f64(ptr, code, rows, d, ldx, seg_rows, seg_stride,
                                                    g.data_ptr(), g.stride(0), self._launch_stream(keep)))
            return
        if 0 < nbytes <= self.defer_bytes and not simt:
            self._pending.append((code, keep, g, ptr, rows, d, ldx, seg_rows, seg_stride, name, keep._version))
            self._pending_bytes += nbytes
            if len(self._pending) >= self.max_pending or self._pending_bytes >= self.max_pending_bytes:
                self.flush()
            return
        stream = self._launch_stream(keep)
        if split:
            planes = self._plane_scratch(2 * rows * d)
            _lib.check(self._lib.vlm_tf32_split(ptr, rows, d, ldx, seg_rows, seg_stride, planes.data_ptr(), stream))
            _lib.check(self._lib.vlm_syrk_accum(planes.data_ptr(), _lib.VLM_TF32X2, rows, d, d, g.data_ptr(),
                                                g.stride(0), stream))
        elif seg_rows:
            _lib.check(self._lib.vlm_syrk_accum_strided(ptr, code, rows, d, ldx, seg_rows, seg_stride, g.data_ptr(),
                                                        g.stride(0), stream))
        else:
            fn = self._lib.vlm_syrk_accum_simt if simt else self._lib.vlm_syrk_accum
            _lib.check(fn(ptr, code, rows, d, ldx, g.data_ptr(), g.stride(0), stream))

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
            if p[1]._version != p[10]:
                raise RuntimeError(
                    f"GramCache: the activation hooked for {p[9]} was modified in place before the deferred Gram launch "
                    "(its Gram would be taken of the modified values); use defer_bytes=0 for this model")
        pending = [p[:9] for p in pending]
        stream = self._launch_stream()
        for code in sorted({p[0] for p in pending}):
            group = [p for p in pending if p[0] == code]
            probs = (_lib.SyrkProblem * len(group))()
            # split mode: accumulate() defers only fp32 activations the split takes, so all of this group is split; the
            # planes of every problem, back to back in the scratch
            split = self.precision == "tf32x3" and code == _lib.VLM_F32
            if split:
                planes = self._plane_scratch(sum(2 * p[4] * p[5] for p in group))
                off = 0
            for q, (_, _keep, g, ptr, rows, d, ldx, seg_rows, seg_stride) in zip(probs, group):
                if split:
                    dst = planes.data_ptr() + off * 4
                    _lib.check(self._lib.vlm_tf32_split(ptr, rows, d, ldx, seg_rows, seg_stride, dst, stream))
                    off += 2 * rows * d
                    q.x, q.rows, q.ldx, q.g, q.ldg, q.d, q.seg_rows, q.seg_stride = dst, rows, d, g.data_ptr(), g.stride(0), d, 0, 0
                else:
                    q.x, q.rows, q.ldx, q.g, q.ldg, q.d = ptr, rows, ldx, g.data_ptr(), g.stride(0), d
                    q.seg_rows, q.seg_stride = seg_rows, seg_stride
            _lib.check(self._lib.vlm_syrk_accum_batch(probs, len(group), _lib.VLM_TF32X2 if split else code, stream))
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
        """Data-parallel calibration: sum the per-rank Gram buffers (ONE NCCL all-reduce over NVLink).
        The reference has no such step (every DDP rank writes its own file, SURVEY.md §2.2).
        packed: only the upper triangles of the Grams that fired travel — vlm_sym_pack_upper_batch (one launch) into one flat
        buffer, one all-reduce of it (VLMo-base: 0.54 GB instead of the 1.17 GB arena with its lower triangles
        and never-fired `vl` experts; twice that for the fp64 Grams of the int8x4 / fp64 modes), vlm_sym_unpack_batch
        back into the full symmetric buffers (which leaves the cache finalized).  packed=False: one all-reduce of the
        whole arena."""
        import torch.distributed as dist

        self.flush()
        if self.symmetric and packed:
            return self._all_reduce_multimem(group)
        if not packed:
            return reduce_gram_buffers(self.buffers, self._arenas, self.calls, self.rows, group)
        live = self._agree_on_live(group)
        if not live:
            return
        grams = [self.buffers[n] for n in live]
        flat = torch.empty(sum(g.shape[0] * (g.shape[0] + 1) // 2 for g in grams), dtype=self.dtype, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        items = _lib.sym_items(grams, flat)
        _lib.check(self._lib.vlm_sym_pack_upper_batch(items, len(live), self._sym_code, stream))   # one launch for all Grams
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        _lib.check(self._lib.vlm_sym_unpack_batch(items, len(live), self._sym_code, stream))
        self._finalized = True
        self.last_reduce_bytes = flat.numel() * flat.element_size()

    def _agree_on_live(self, group):
        """The first step of both exchanges: every rank agrees on the buffer set (creating zero buffers for names it
        lacks) and sums the call / row counters; returns the names that fired on some rank, the same list everywhere."""
        names = agree_on_buffers(self.buffers, group,
                                 lambda d: torch.zeros(d, d, dtype=self.dtype, device=self.device), device=self.device)
        _reduce_counts(self.buffers, names, self.calls, self.rows, group)
        return [n for n in names if self.calls[n] > 0]

    def _all_reduce_multimem(self, group=None):
        """all_reduce() of a symmetric cache: one kernel over the NVSwitch multicast mapping of the arena, bracketed by
        two cross-rank barriers on the current stream.  Every rank ends with bit-identical, fully symmetric Grams."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem

        group = group if group is not None else dist.group.WORLD
        live = self._agree_on_live(group)
        if not live:
            return
        if len(self._arenas) != 1:
            raise RuntimeError("GramCache(symmetric=True): no symmetric arena (register() the model before calibrating)")
        arena = self._arenas[0]
        lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel() * arena.element_size()
        if any(not (lo <= self.buffers[n].data_ptr() < hi) for n in live):
            raise RuntimeError("GramCache(symmetric=True): a Gram buffer lives outside the symmetric arena (a module whose "
                               "width was unknown at register()); use a plain cache (NCCL exchange) for this model")
        if self._symm is None:
            self._symm = symm_mem.rendezvous(arena, group)          # collective: every rank, same order
        h = self._symm
        mc = int(h.multicast_ptr or 0)
        if mc == 0:
            raise RuntimeError("GramCache(symmetric=True): this system offers no multicast mapping (NVSwitch + driver "
                               "support needed); use a plain cache (NCCL exchange)")
        spans = (_lib.SymSpan * len(live))()
        for sp, n in zip(spans, live):
            g = self.buffers[n]
            sp.offset_bytes, sp.d, sp.ld = g.data_ptr() - lo, g.shape[0], g.stride(0)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            h.barrier(channel=0)               # every rank's Gram launches have completed
            _lib.check(self._lib.vlm_sym_allreduce_multimem(mc, spans, len(live), self._sym_code, dist.get_rank(group),
                                                            dist.get_world_size(group), stream))
            h.barrier(channel=0)               # every rank's stores have landed everywhere
            self._mirror(live, stream)         # lower triangles, locally
        self._finalized = True
        esz = 8 if self.dtype == torch.float64 else 4
        self.last_reduce_bytes = sum(self.buffers[n].shape[0] * (self.buffers[n].shape[0] + 1) // 2 for n in live) * esz

    def finalize(self):
        """Mirror the upper triangles into the lower ones (after the last accumulate / all_reduce)."""
        self.flush()
        if self._finalized:
            return
        self._mirror(self.live_names(), torch.cuda.current_stream(self.device).cuda_stream)
        self._finalized = True

    def _mirror(self, names, stream):
        """The lower triangles of the named Grams from their upper ones, in place: one launch."""
        items = _lib.sym_items([self.buffers[n] for n in names])
        _lib.check(self._lib.vlm_sym_mirror_batch(items, len(names), self._sym_code, stream))

    def gram(self, name):
        """Full symmetric fp32 Gram of one module, on the device."""
        self.finalize()
        return self.buffers[name]

    def state_dict(self, dtype=torch.float64, device="cpu"):
        """{module_name: (d,d) tensor} for every module that fired — by default fp64 CPU tensors, the
        format of the reference's Gram file, in the reference's insertion order (first-call order
        there; registration order here, which is the same for a sequential forward)."""
        self.finalize()
        out = defaultdict(float)
        for name in self.live_names():
            # dtype first, on the device (a blocking .to(device, dtype) would convert on the host, after the copy);
            # an fp64 cache never hands out its own buffers, an fp32 one does for fp32 on its own device
            out[name] = self.buffers[name].to(dtype).to(device, copy=self.dtype == dtype == torch.float64)
        return out

    def save(self, path):
        """torch.save of the reference-format dict (src/cache_gram_matrices.py:349)."""
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
