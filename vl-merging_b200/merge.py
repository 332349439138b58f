"""merge.py — the three merge methods of ViLTransformerSS as state_dict -> state_dict functions on the
B200: merge_weights (src/vilt/modules/vilt_module.py:533-638), sum_task_vectors (:640-746) and
regmean (:366-531).  Same names, same config keys, same key layout of the result, same dtypes
(fp32, and fp64 for RegMean's linear weights); the arithmetic runs in libvlmerge:

  * every elementwise target of a call goes through ONE vlm_merge_plan launch (kernel (b));
  * RegMean's W*Ghat / sum Ghat / solve run per linear through vlm_regmean_rhs(_diff),
    vlm_gram_scale_accum and vlm_spd_solve_right (kernel (c) + cuSOLVER).

Inputs may live on the CPU (the reference's case: torch.load(map_location="cpu")) or already on the
GPU.  CPU inputs are staged into one device arena and the result comes back in one pinned buffer;
GPU inputs are used in place and the result stays on the GPU.  With a process group, targets are
sharded by tensor over the ranks and the merged tensors are all-gathered at the end.
"""
import ctypes
from types import SimpleNamespace

import torch

from . import _lib, gramfile
from .plan import MEAN, SEQ_LERP, WSUM, is_passthrough_key, plan_merge_weights, plan_regmean, plan_sum_task_vectors

_ALIGN = 4  # elements: keeps every arena segment 16-byte aligned for the 128-bit path


def _round_up(n, a=_ALIGN):
    return (n + a - 1) // a * a


def _load(path):
    """torch.load for the reference's pickled artefacts (PL checkpoints, defaultdict Gram files)."""
    return torch.load(path, map_location="cpu", weights_only=False)


def _resolve_device(state_dict, device):
    if device is not None:
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        return device
    for v in state_dict.values():
        if torch.is_tensor(v) and v.is_cuda:
            return v.device
    if not torch.cuda.is_available():
        raise RuntimeError("the merge hot path runs on a CUDA device only (no CPU fallback)")
    # host checkpoint and no device given.  Under a one-process-per-GPU launcher (torchrun / Lightning DDP) the
    # merges are called from the model constructor, BEFORE the trainer calls set_device: follow LOCAL_RANK there,
    # so that N ranks do not all stage their arenas on cuda:0.
    import os

    local = os.environ.get("LOCAL_RANK")
    if local is not None and local.isdigit() and int(local) < torch.cuda.device_count():
        return torch.device("cuda", int(local))
    return torch.device("cuda", torch.cuda.current_device())


def _shard(ops, cost, world):
    """Greedy size-balanced assignment of ops to ranks (largest first); deterministic on every rank."""
    owner = {}
    load = [0] * world
    for idx in sorted(range(len(ops)), key=lambda i: (-cost(ops[i]), i)):
        r = min(range(world), key=lambda k: (load[k], k))
        owner[idx] = r
        load[r] += cost(ops[idx])
    return owner


class ShardLayout:
    """Tensor-sharded placement of merge targets over `world` ranks and the flat layout of the
    all-gathered result.  Pure Python: every rank derives the same layout from (sizes, world), so the
    only thing that travels is one all_gather_into_tensor of equal-width shards."""

    def __init__(self, sizes, world, cost=None, align=_ALIGN):
        self.sizes, self.world = list(sizes), world
        idx = list(range(len(self.sizes)))
        cost = cost or (lambda i: self.sizes[i])
        self.owner = _shard(idx, cost, world) if world > 1 else {i: 0 for i in idx}
        self.offset, self.shard_size = {}, [0] * world
        for i in idx:
            r = self.owner[i]
            self.offset[i] = self.shard_size[r]
            self.shard_size[r] += _round_up(self.sizes[i], align)
        self.width = max(self.shard_size + [1])

    def mine(self, rank):
        return [i for i in range(len(self.sizes)) if self.owner[i] == rank]

    def gather(self, local, rank, group):
        """local: flat tensor holding this rank's shard (>= shard_size[rank] elements).  Returns the
        flat tensor [world * width] with every rank's shard."""
        import torch.distributed as dist

        if self.world == 1:
            return local
        padded = torch.zeros(self.width, dtype=local.dtype, device=local.device)
        padded[: self.shard_size[rank]].copy_(local[: self.shard_size[rank]])
        out = torch.empty(self.world * self.width, dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(out, padded, group=group)
        return out

    def view(self, full, i, shape):
        base = (self.owner[i] * self.width if self.world > 1 else 0) + self.offset[i]
        return full[base: base + self.sizes[i]].view(shape)


def _run_elementwise(ops, lookup, shapes, device, out_device, group=None, stats=None):
    """Executes the WSUM / SEQ_LERP / MEAN ops in one kernel launch (per rank).
    lookup(op, j) -> source tensor j of op; shapes[dst] -> torch.Size.  Returns {dst: fp32 tensor}."""
    import torch.distributed as dist

    lib = _lib.lib()
    trace = stats.get("trace") if stats is not None else None     # optional: host timestamps of the stages (seconds)
    import time as _time

    def mark(what):
        if trace is not None:
            trace.append((what, _time.perf_counter()))

    mark("enter")
    world = dist.get_world_size(group) if group is not None else 1
    rank = dist.get_rank(group) if group is not None else 0
    numel = {op.dst: int(torch.Size(shapes[op.dst]).numel()) for op in ops}
    layout = ShardLayout([numel[op.dst] for op in ops], world)
    out_off, shard_size = layout.offset, layout.shard_size
    mine = layout.mine(rank)

    # input arena for sources that are not already usable in place
    def in_place(t):
        return t.is_cuda and t.device == device and t.dtype == torch.float32 and t.is_contiguous()

    staged, in_total = [], 0
    for i in mine:
        for j in range(len(ops[i].srcs) + (1 if ops[i].central else 0)):
            t = lookup(ops[i], j)
            if tuple(t.shape) != tuple(shapes[ops[i].dst]):
                raise RuntimeError(f"{ops[i].dst}: source {j} has shape {tuple(t.shape)}, expected {tuple(shapes[ops[i].dst])}")
            if not in_place(t):
                staged.append((i, j, in_total, t))
                in_total += _round_up(t.numel())
    mark("scanned")
    arena_in = torch.empty(max(in_total, 1), dtype=torch.float32, device=device)
    arena_out = torch.empty(max(shard_size[rank], 1), dtype=torch.float32, device=device)
    staged_at = {(i, j): off for i, j, off, _ in staged}
    staged_by_op = {}
    for item in staged:
        staged_by_op.setdefault(item[0], []).append(item)

    def make_seg(i):
        op = ops[i]
        n_src = len(op.srcs) + (1 if op.central else 0)
        if n_src > _lib.MERGE_MAX_SRC:
            raise RuntimeError(f"{op.dst}: {n_src} sources exceed VLM_MERGE_MAX_SRC")
        seg = _lib.MergeSeg()
        seg.dst = arena_out.data_ptr() + out_off[i] * 4
        for j in range(n_src):
            if (i, j) in staged_at:
                seg.src[j] = arena_in.data_ptr() + staged_at[(i, j)] * 4
            else:
                t = lookup(op, j)
                keep.append(t)
                seg.src[j] = t.data_ptr()
        for j, c in enumerate(([0.0] if op.central else []) + list(op.coefs)):
            seg.coef[j] = c
        seg.n, seg.n_src, seg.mode = numel[op.dst], n_src, op.mode
        return seg

    keep = []
    cur = torch.cuda.current_stream(device)
    # Host checkpoints in, host tensors out: cut the targets into a few groups and overlap the H2D of group
    # g+1 with the kernel + D2H of group g (PCIe is full duplex; the kernel itself is ~0.2 ms).
    pipelined = world == 1 and out_device.type == "cpu" and in_total * 4 >= (128 << 20) and len(mine) >= 8
    ngroups = min(8, len(mine)) if pipelined else 1
    bounds = [len(mine) * g // ngroups for g in range(ngroups + 1)]
    h2d_stream = torch.cuda.Stream(device) if pipelined else cur
    d2h_stream = torch.cuda.Stream(device) if pipelined else cur
    mark("arenas")
    host = torch.empty(max(shard_size[rank], 1), dtype=torch.float32, pin_memory=True) if pipelined else None
    mark("pinned output")
    if pipelined:
        h2d_stream.wait_stream(cur)
        d2h_stream.wait_stream(cur)
    h2d = 0
    plans = []
    try:
        # 1. every group's host -> device copies go out first (asynchronous, one vlm_copy_batch per group, an event
        #    after each): the DMA engine starts at once and the segment tables below are built while it runs.
        #    (Measured on the B200 box, tools/pcie_probe.py + tools/merge_trace.py: 680 MB in + 340 MB out take 13.5 ms
        #    as two big copies running at once, 19.1 ms one after the other; this call takes 19.6 ms — 0.8 ms of host
        #    preparation, 15.6 ms until the last of the ~390 input copies has landed, 2 ms of tail.)
        ready = []
        for g in range(ngroups):
            idx = mine[bounds[g]: bounds[g + 1]]
            with torch.cuda.stream(h2d_stream):
                batch = []     # contiguous fp32 sources: one call for the whole group
                for i in idx:
                    for _, _, off, t in staged_by_op.get(i, ()):
                        src = t.detach()
                        h2d += src.numel() * 4 if not t.is_cuda else 0
                        if src.dtype == torch.float32 and src.is_contiguous():
                            keep.append(src)
                            batch.append((off * 4, src.data_ptr(), src.numel() * 4))
                            continue
                        src = src.reshape(-1)
                        if src.dtype != torch.float32:
                            src = src.float()
                        arena_in[off: off + src.numel()].copy_(src, non_blocking=True)
                if batch:
                    nb = len(batch)
                    offs = (ctypes.c_uint64 * nb)(*[b[0] for b in batch])
                    srcs = (ctypes.c_void_p * nb)(*[b[1] for b in batch])
                    sizes = (ctypes.c_uint64 * nb)(*[b[2] for b in batch])
                    _lib.check(lib.vlm_copy_batch(arena_in.data_ptr(), offs, srcs, sizes, nb, h2d_stream.cuda_stream))
                ev = torch.cuda.Event()
                ev.record(h2d_stream)
                ready.append(ev)
        mark("h2d enqueued")
        # 2. per group: segment table, kernel as soon as the group's inputs have landed, device -> host copy of its
        #    outputs on a third stream (PCIe is full duplex)
        for g in range(ngroups):
            idx = mine[bounds[g]: bounds[g + 1]]
            if not idx:
                continue
            segs = (_lib.MergeSeg * len(idx))(*[make_seg(i) for i in idx])
            plan = ctypes.c_void_p()
            _lib.check(lib.vlm_merge_plan_create(segs, len(idx), ctypes.byref(plan)))
            plans.append(plan)
            cur.wait_event(ready[g])
            _lib.check(lib.vlm_merge_plan_run(plan, cur.cuda_stream))
            if stats is not None:
                stats["merge_bytes"] = stats.get("merge_bytes", 0) + int(lib.vlm_merge_plan_bytes(plan))
            if pipelined:
                lo = out_off[idx[0]]
                hi = out_off[idx[-1]] + _round_up(numel[ops[idx[-1]].dst])
                d2h_stream.wait_stream(cur)
                with torch.cuda.stream(d2h_stream):
                    host[lo:hi].copy_(arena_out[lo:hi], non_blocking=True)
        mark("all enqueued")
    finally:
        cur.synchronize()
        mark("kernels done")
        if pipelined:
            h2d_stream.synchronize()
            d2h_stream.synchronize()
        for plan in plans:
            if plan:
                lib.vlm_merge_plan_destroy(plan)

    mark("copies done")
    # all-gather of the merged shards (the path's one exchange step)
    full = layout.gather(arena_out, rank, group)
    if pipelined:
        full = host
        if stats is not None:
            stats["d2h_bytes"] = stats.get("d2h_bytes", 0) + full.numel() * 4
            stats["pipelined_groups"] = ngroups
    elif out_device.type == "cpu":
        host = torch.empty(full.numel(), dtype=torch.float32, pin_memory=True)
        host.copy_(full, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
        full = host
        if stats is not None:
            stats["d2h_bytes"] = stats.get("d2h_bytes", 0) + full.numel() * 4
    if stats is not None:
        stats["h2d_bytes"] = stats.get("h2d_bytes", 0) + h2d
    out = {op.dst: layout.view(full, i, shapes[op.dst]) for i, op in enumerate(ops)}
    return out


def _assemble(state_dict, ops, computed):
    """Result dict in the reference's order: pass-through keys first, then the 13 targets per layer."""
    new = {k: v for k, v in state_dict.items() if is_passthrough_key(k)}
    for op in ops:
        new[op.dst] = state_dict[op.passthrough] if op.passthrough else computed[op.dst]
    return new


def _out_device(state_dict, ops, override=None, device=None):
    """Where the merged tensors go: where the inputs live (the reference's behaviour: CPU in, CPU out), unless the
    caller says otherwise.  Under a process group the gathered result is on every rank's GPU anyway; copying it to
    the host on EVERY rank is N device->host copies into the same host memory, so a launcher that only needs the
    host copy once passes out_device="cpu" on rank 0 and "cuda" elsewhere."""
    if override is not None:
        override = torch.device(override)
        return device if override.type == "cuda" else override
    for op in ops:
        for k in op.srcs:
            return state_dict[k].device
        if op.regmean:
            return state_dict[op.regmean[0][0]].device
    return torch.device("cpu")


def merge_weights(state_dict, config, device=None, num_layers=12, group=None, stats=None, out_device=None):
    """Interpolation merge.  config keys: merge_ratio, only_activate_used_experts,
    vlffn_start_layer_index, loss_names (src/vilt/config.py:141-149).
    out_device: None = where the inputs live; "cuda" = leave the merged tensors on the merge device; "cpu"."""
    device = _resolve_device(state_dict, device)
    ops = plan_merge_weights(state_dict.keys(), config, num_layers)
    todo = [op for op in ops if not op.passthrough]
    shapes = {op.dst: state_dict[op.srcs[0]].shape for op in todo}
    with torch.cuda.device(device):
        computed = _run_elementwise(todo, lambda op, j: state_dict[op.srcs[j]], shapes, device,
                                    _out_device(state_dict, todo, out_device, device), group, stats)
    return _assemble(state_dict, ops, computed)


def sum_task_vectors(state_dict, config, device=None, num_layers=12, group=None, stats=None, central_weight=None,
                     out_device=None):
    """Modality arithmetic with the reference's sequential semantics (SURVEY.md §8 a-7).  The centre is
    config['central_weight'] (a checkpoint path, as in the reference) unless a dict is passed.  Unlike the
    reference, the loaded centre is not mutated."""
    device = _resolve_device(state_dict, device)
    central = central_weight if central_weight is not None else _load(config["central_weight"])
    if "state_dict" in central:
        central = central["state_dict"]
    ops = plan_sum_task_vectors(state_dict.keys(), central.keys(), config, num_layers)
    todo = [op for op in ops if not op.passthrough]
    shapes = {op.dst: central[op.dst].shape for op in todo}

    def lookup(op, j):
        return central[op.dst] if j == 0 else state_dict[op.srcs[j - 1]]

    with torch.cuda.device(device):
        computed = _run_elementwise(todo, lookup, shapes, device, _out_device(state_dict, todo, out_device, device),
                                    group, stats)
    return _assemble(state_dict, ops, computed)


_SOLVE_STREAMS = {}   # device -> side streams of the concurrent RegMean path (libvlmerge keeps one solver context per stream)
_SUM_WORKSPACE = {}   # device -> flat fp64 workspace for the summed Grams, kept across calls (it only ever grows)


def _workspace(device, numel):
    ws = _SUM_WORKSPACE.get(device)
    if ws is None or ws.numel() < numel:
        _SUM_WORKSPACE[device] = None
        ws = _SUM_WORKSPACE[device] = torch.empty(int(numel), dtype=torch.float64, device=device)
    return ws


def _regmean_linears(lib, state_dict, grams, lin_ops, mine, cost, alpha, device, n_streams, results, stats=None):
    """The linear problems `mine` of regmean(): per problem vlm_gram_scale_accum per expert + vlm_regmean_rhs_diff per
    expert but the last (the difference form, see base_weight below), then vlm_spd_solve_right_async + vlm_widen_add, on n_streams CUDA streams (largest problem first, each to the least loaded stream;
    n_streams = 1: everything on the caller's stream, and `stats` receives the RHS / solve split from CUDA events).
    Every buffer is carved out BEFORE the streams fork — one fresh fp64 arena for the results (the returned tensors
    are views of it), one cached workspace for the summed Grams, operands staged on the caller's stream — so no
    allocation happens inside a side-stream context and a repeated call does the same work in the same time.
    One status read at the end.  A summed Gram that Cholesky rejects is solved again by pivoted LU
    (vlm_lu_solve_right), like the reference's torch.inverse (vilt_module.py:432,483); an exactly singular one
    raises LinAlgError as torch.inverse does."""
    import warnings

    cur = torch.cuda.current_stream(device)
    shapes = {idx: tuple(state_dict[lin_ops[idx].regmean[0][0]].shape) for idx in mine}
    acc_all = torch.empty(sum(o * i for o, i in shapes.values()), dtype=torch.float64, device=device)
    ws = _workspace(device, sum(i * i for _, i in shapes.values()))
    acc, summed = {}, {}
    a_off = s_off = 0
    for idx in mine:
        o, i = shapes[idx]
        acc[idx] = acc_all[a_off: a_off + o * i].view(o, i)
        summed[idx] = ws[s_off: s_off + i * i].view(i, i)
        a_off += o * i
        s_off += i * i
    # operands: used in place when resident (fp32 weights; fp32 or fp64 Grams), staged here otherwise
    staged = {}

    def operand(t, gram):
        key = (id(t), gram)
        if key not in staged:
            v = t.detach()
            if gram:
                if v.dtype not in (torch.float64, torch.float32):
                    v = v.double()
                v = v.to(device=device, non_blocking=True)
            else:
                v = v.to(device=device, dtype=torch.float32, non_blocking=True)
            staged[key] = v if v.stride(-1) == 1 and v.dim() == 2 else v.contiguous()
        return staged[key]

    for idx in mine:
        for wkey, gkey in lin_ops[idx].regmean:
            g = operand(grams[gkey], True)
            if tuple(g.shape) != (shapes[idx][1], shapes[idx][1]):
                raise RuntimeError(f"Gram {gkey} has shape {tuple(g.shape)}, expected {(shapes[idx][1],) * 2}")
            operand(state_dict[wkey], False)
    info = torch.zeros(len(lin_ops), 2, dtype=torch.int32, device=device)

    def base_weight(idx):
        """With M >= 2 experts: (sum_m W_m Ghat_m) S^-1 = W_base + (sum_{m != base} (W_m - W_base) Ghat_m) S^-1 with
        S = sum_m Ghat_m — one GEMM fewer than the formula as written (vilt_module.py:423-434), the same value in
        exact arithmetic.  The base is the last expert, when all weights share one pitch."""
        experts = lin_ops[idx].regmean
        if len(experts) < 2:
            return None
        ws = [operand(state_dict[wkey], False) for wkey, _ in experts]
        return ws[-1] if all(w.stride(0) == ws[-1].stride(0) for w in ws) else None

    def enqueue_rhs(idx, st):
        out_f, in_f = shapes[idx]
        base = base_weight(idx)
        experts = lin_ops[idx].regmean
        first = True
        for n, (wkey, gkey) in enumerate(experts):
            w, g = operand(state_dict[wkey], False), operand(grams[gkey], True)
            gdt = _lib.VLM_F64 if g.dtype == torch.float64 else _lib.VLM_F32
            _lib.check(lib.vlm_gram_scale_accum(g.data_ptr(), gdt, in_f, g.stride(0), alpha, summed[idx].data_ptr(),
                                                summed[idx].stride(0), int(n > 0), st))
            if base is None:
                _lib.check(lib.vlm_regmean_rhs(w.data_ptr(), out_f, in_f, w.stride(0), g.data_ptr(), gdt, g.stride(0),
                                               alpha, acc[idx].data_ptr(), acc[idx].stride(0), int(n > 0), st))
            elif n < len(experts) - 1:
                _lib.check(lib.vlm_regmean_rhs_diff(w.data_ptr(), base.data_ptr(), out_f, in_f, w.stride(0), g.data_ptr(),
                                                    gdt, g.stride(0), alpha, acc[idx].data_ptr(), acc[idx].stride(0),
                                                    int(not first), st))
                first = False

    def enqueue_finish(idx, st):
        """After the solve: add W_base back (see base_weight)."""
        base = base_weight(idx)
        if base is not None:
            out_f, in_f = shapes[idx]
            _lib.check(lib.vlm_widen_add(base.data_ptr(), out_f, in_f, base.stride(0), acc[idx].data_ptr(),
                                         acc[idx].stride(0), st))

    def enqueue_solve(idx, st):
        out_f, in_f = shapes[idx]
        _lib.check(lib.vlm_spd_solve_right_async(summed[idx].data_ptr(), in_f, summed[idx].stride(0), acc[idx].data_ptr(),
                                                 out_f, acc[idx].stride(0), info[idx].data_ptr(), st))
        enqueue_finish(idx, st)

    order = sorted(mine, key=lambda i: (-cost(lin_ops[i]), i))
    n_streams = max(1, min(int(n_streams), len(mine)))
    events = []
    if n_streams == 1:
        st = cur.cuda_stream
        for idx in order:
            if stats is not None:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ev[0].record(cur)
            enqueue_rhs(idx, st)
            if stats is not None:
                ev[1].record(cur)
            enqueue_solve(idx, st)
            if stats is not None:
                ev[2].record(cur)
                events.append(ev)
    else:
        pool = _SOLVE_STREAMS.setdefault(device, [])
        while len(pool) < n_streams:
            pool.append(torch.cuda.Stream(device))
        streams = pool[:n_streams]
        for st in streams:
            st.wait_stream(cur)
        load = [0] * n_streams
        for idx in order:
            k = min(range(n_streams), key=lambda j: (load[j], j))
            load[k] += cost(lin_ops[idx])
            enqueue_rhs(idx, streams[k].cuda_stream)
            enqueue_solve(idx, streams[k].cuda_stream)
        for st in streams:
            cur.wait_stream(st)
    status = info.cpu()                  # synchronises the caller's stream, hence all of the above
    if stats is not None:
        stats["solve_streams"] = n_streams
        if events:
            stats["rhs_seconds"] = stats.get("rhs_seconds", 0.0) + sum(e[0].elapsed_time(e[1]) for e in events) * 1e-3
            stats["solve_seconds"] = stats.get("solve_seconds", 0.0) + sum(e[1].elapsed_time(e[2]) for e in events) * 1e-3
    for idx in mine:
        potrf, potrs = int(status[idx, 0]), int(status[idx, 1])
        if potrf != 0:
            # Cholesky rejected the sum (not numerically positive definite): redo this problem with pivoted LU
            warnings.warn(f"{lin_ops[idx].dst}: summed Gram is not positive definite (leading minor {potrf}); "
                          "solving with pivoted LU like torch.inverse — calibrate with more rows than features or use "
                          "scaling_for_non_diag < 1", RuntimeWarning, stacklevel=3)
            enqueue_rhs(idx, cur.cuda_stream)
            out_f, in_f = shapes[idx]
            try:
                _lib.check(lib.vlm_lu_solve_right(summed[idx].data_ptr(), in_f, summed[idx].stride(0), acc[idx].data_ptr(),
                                                  out_f, acc[idx].stride(0), cur.cuda_stream))
            except _lib.VlmError as e:
                if e.code == _lib.ERR_NOT_SPD:  # the reference's torch.inverse raises on a singular sum too
                    raise torch.linalg.LinAlgError(f"{lin_ops[idx].dst}: {e}") from e
                raise
            enqueue_finish(idx, cur.cuda_stream)
            if stats is not None:
                stats["lu_fallbacks"] = stats.get("lu_fallbacks", 0) + 1
        elif potrs != 0:
            raise RuntimeError(f"{lin_ops[idx].dst}: cusolverDnDpotrs info {potrs}")
    for idx in mine:
        results[lin_ops[idx].dst] = acc[idx]


def _as_gram_dict(grams):
    """{name: Gram} of a dict or a GramCache (on its device).  Of a reduce-scattered cache every live name is listed,
    so that every rank plans the same problems, but only the Grams this rank owns hold sums and may be read."""
    if hasattr(grams, "state_dict") and hasattr(grams, "buffers"):  # a GramCache: stay on the device, fp32
        grams.finalize()
        return {n: grams.buffers[n] for n in grams.live_names()}
    return grams


def _regmean_cost(state_dict, op):
    o, i = state_dict[op.regmean[0][0]].shape
    return i * i * i // 3 + 2 * len(op.regmean) * o * i * i + 2 * o * i * i


def _regmean_sharding(state_dict, config, gram_names, world, num_layers):
    """regmean()'s plan and the cost-balanced ShardLayout of its linear problems over `world` ranks, plus the owner of
    every Gram a problem reads: (ops, lin_ops, layout, {gram name: rank})."""
    ops = plan_regmean(state_dict.keys(), gram_names, config, num_layers)
    lin_ops = [op for op in ops if not op.passthrough and op.regmean is not None]
    sizes = [int(state_dict[op.regmean[0][0]].numel()) for op in lin_ops]
    layout = ShardLayout(sizes, world, cost=lambda i: _regmean_cost(state_dict, lin_ops[i]), align=1)
    # plan_regmean gives every expert's linear its own Gram: each Gram has exactly one owner
    owners = {gram: layout.owner[idx] for idx, op in enumerate(lin_ops) for _, gram in op.regmean}
    return ops, lin_ops, layout, owners


def regmean_gram_owners(state_dict, config, gram_names, world, num_layers=12):
    """{Gram name: rank} — which rank's regmean(..., group=g) with a world of `world` ranks solves the one linear
    problem that reads each Gram (qkv <- attn.{m}, proj <- attn.{m}.proj, fc1 / fc2 <- mlp.{m}.fc1 / fc2).  Grams
    that no problem reads (the `v` / `l` Grams of the deep layers under a VQA config, for example) are not in the map.
    Pass every rank's agreed live names (GramCache.live_names() after calibration) and the arguments regmean() will
    get; GramCache.reduce_scatter(owners) then leaves each Gram's sum on its owner only."""
    return _regmean_sharding(state_dict, config, gram_names, int(world), num_layers)[3]


def regmean(state_dict, config, device=None, num_layers=12, group=None, stats=None, gram_matrices=None,
            solve_streams=8, out_device=None):
    """RegMean merge.  config keys: gram_matrices (path of the Gram file, as in the reference — or pass
    gram_matrices= a dict / GramCache), scaling_for_non_diag, vlffn_start_layer_index, loss_names.
    Linear weights come back fp64 like the reference's; biases / LayerNorms fp32.
    solve_streams: the independent per-linear problems (W*Ghat GEMMs + Cholesky solve) are spread over this many
    CUDA streams — one factorisation does not fill the GPU; 1 = strictly sequential (and the only mode in which
    `stats` receives the rhs / solve time split)."""
    import torch.distributed as dist

    device = _resolve_device(state_dict, device)
    lib = _lib.lib()
    if gram_matrices is None:
        gpath = config["gram_matrices"]
        # the packed fp32 container of gramfile.py, or the reference's own pickle of fp64 matrices
        gram_matrices = gramfile.load_packed(gpath, device) if gramfile.is_packed_file(gpath) else _load(gpath)
    alpha = float(config["scaling_for_non_diag"])
    if alpha == 1.0 and getattr(gram_matrices, "precision", None) in ("tf32", "tf32x3"):
        import warnings

        # measured on the B200 (DESIGN.md 4a): LayerNorm-fed linears come out 1e-2 off with single-pass TF32 Grams
        warnings.warn(f"regmean with scaling_for_non_diag = 1 on Grams cached with precision={gram_matrices.precision!r}: "
                      "the inverse of an unregularised Gram sum amplifies the tensor core's fp32 accumulation error; "
                      "calibrate with GramCache(precision='int8x4') (or 'fp64') for the reference's 1e-4",
                      RuntimeWarning, stacklevel=2)
    grams = _as_gram_dict(gram_matrices)
    world = dist.get_world_size(group) if group is not None else 1
    rank = dist.get_rank(group) if group is not None else 0
    ops, lin_ops, lin_layout, owners = _regmean_sharding(state_dict, config, grams.keys(), world, num_layers)
    scattered = getattr(gram_matrices, "owners", None)
    if scattered is not None and (scattered != owners or gram_matrices._rank != rank):
        raise ValueError("regmean: the GramCache was reduce_scatter()ed with a different owner map or rank than this "
                         f"call's (world {world}, rank {rank}, num_layers {num_layers}, this config): every rank holds only its own Gram "
                         "sums; scatter it with regmean_gram_owners() of the same arguments, or all_reduce() it")
    todo = [op for op in ops if not op.passthrough]
    mean_ops = [op for op in todo if op.regmean is None]
    out_device = _out_device(state_dict, todo, out_device, device)
    with torch.cuda.device(device):
        shapes = {op.dst: state_dict[op.srcs[0]].shape for op in mean_ops}
        computed = _run_elementwise(mean_ops, lambda op, j: state_dict[op.srcs[j]], shapes, device, out_device,
                                    group, stats)

        def cost(op):
            return _regmean_cost(state_dict, op)

        results = {}
        mine_lin = lin_layout.mine(rank)
        if mine_lin:
            _regmean_linears(lib, state_dict, grams, lin_ops, mine_lin, cost, alpha, device, solve_streams, results, stats)

        if world > 1:  # all-gather the solved weights: flat fp64, every rank knows every size
            local = torch.zeros(lin_layout.width, dtype=torch.float64, device=device)
            for idx in lin_layout.mine(rank):
                r = results[lin_ops[idx].dst]
                local[lin_layout.offset[idx]: lin_layout.offset[idx] + r.numel()].copy_(r.reshape(-1))
            gathered = lin_layout.gather(local, rank, group)
            for idx, op in enumerate(lin_ops):
                results[op.dst] = lin_layout.view(gathered, idx, state_dict[op.regmean[0][0]].shape)
        for op in lin_ops:
            computed[op.dst] = results[op.dst].to(out_device)
    return _assemble(state_dict, ops, computed)


class Merger:
    """Object form with the reference's calling convention: methods read self.hparams.config[...]
    (vilt_module.py:389,397,557,576,660...).  `ViLTransformerSS.merge_weights = Merger.merge_weights`
    style patching, or Merger(config).regmean(state_dict)."""

    def __init__(self, config, num_layers=12, device=None, group=None):
        """device=None: the device the state_dict lives on, else cuda:LOCAL_RANK under a launcher, else the current
        device (see _resolve_device)."""
        self.hparams = SimpleNamespace(config=config)
        self.num_layers, self.device, self.group = num_layers, device, group

    def merge_weights(self, state_dict):
        return merge_weights(state_dict, self.hparams.config, self.device, self.num_layers, self.group)

    def sum_task_vectors(self, state_dict):
        return sum_task_vectors(state_dict, self.hparams.config, self.device, self.num_layers, self.group)

    def regmean(self, state_dict):
        return regmean(state_dict, self.hparams.config, self.device, self.num_layers, self.group)

    def apply(self, state_dict):
        """The load-time dispatch of vilt_module.py:284-291."""
        cfg = self.hparams.config
        if cfg.get("merge_weights"):
            return self.merge_weights(state_dict)
        if cfg.get("sum_task_vectors"):
            return self.sum_task_vectors(state_dict)
        if cfg.get("regmean"):
            return self.regmean(state_dict)
        return state_dict


def independent(state_dict):
    """Merged tensors that come back on the CPU are views of ONE pinned host buffer (a single device->host copy):
    keeping any of them alive keeps the whole buffer, and torch.save of a subset serialises the shared storage.  This
    returns the same dict with every such view copied into its own ordinary tensor, like the reference's outputs."""
    seen = {}
    for v in state_dict.values():
        if torch.is_tensor(v) and v.device.type == "cpu":
            key = v.untyped_storage().data_ptr()
            seen[key] = seen.get(key, 0) + 1
    return {k: (v.clone() if torch.is_tensor(v) and v.device.type == "cpu" and
                (seen.get(v.untyped_storage().data_ptr(), 0) > 1 or v.is_pinned()) else v)
            for k, v in state_dict.items()}


__all__ = ["merge_weights", "sum_task_vectors", "regmean", "regmean_gram_owners", "Merger", "independent", "WSUM", "SEQ_LERP", "MEAN"]
