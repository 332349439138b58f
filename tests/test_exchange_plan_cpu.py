"""exchange_plan, the host side of GramCache.all_reduce() and reduce_scatter(), on CPU with the gloo backend (world 3):
buffer-set agreement, summed counters, owner-map checks, the packed layout and byte counts, and the collectives each
plan issues.  All cases run in one spawn; the tests check its results."""
import os
import socket
from collections import defaultdict

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from vl_merging_b200.gram import exchange_plan

WORLD = 3
COLLECTIVES = ("all_reduce", "all_gather_object", "all_gather", "broadcast", "reduce_scatter_tensor", "barrier")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _counting(fn):
    """Run fn() with every torch.distributed collective counted: (result or the exception raised, collective names)."""
    seen, orig = [], {n: getattr(dist, n) for n in COLLECTIVES}
    for n, f in orig.items():
        setattr(dist, n, lambda *a, _n=n, _f=f, **k: (seen.append(_n), _f(*a, **k))[1])
    try:
        try:
            out = fn()
        except ValueError as e:
            out = e
    finally:
        for n, f in orig.items():
            setattr(dist, n, f)
    return out, seen


def _summary(plan):
    return {k: getattr(plan, k) for k in ("names", "offsets", "sections", "width", "mine", "nbytes", "calls", "rows",
                                          "owners", "rank", "world")}


def _ragged(rank):
    """Rank r holds a (4 x 4, fired once, 3 rows), only<r> ((2 + r)^2, fired on rank r only) and never (fired nowhere)."""
    buffers = {"a": torch.ones(4, 4), f"only{rank}": torch.ones(2 + rank, 2 + rank), "never": torch.zeros(2, 2)}
    calls = defaultdict(int, {"a": 1, f"only{rank}": 1})
    rows = defaultdict(int, {"a": 3, f"only{rank}": 5 + rank})
    return buffers, calls, rows


def _job(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {}
    make32, make64 = (lambda d: torch.zeros(d, d)), (lambda d: torch.zeros(d, d, dtype=torch.float64))
    try:
        buffers, calls, rows = _ragged(rank)
        before = (dict(calls), dict(rows))
        plan, seen = _counting(lambda: exchange_plan(buffers, calls, rows, make=make32))
        res["ragged"] = _summary(plan)
        res["ragged_collectives"] = seen
        res["ragged_buffers"] = sorted(buffers)
        res["ragged_counters_kept"] = (dict(calls), dict(rows)) == before

        plan, seen = _counting(lambda: exchange_plan(buffers, calls, rows, symmetric=True))
        res["ragged_symmetric_nbytes"] = plan.nbytes

        plan, seen = _counting(lambda: exchange_plan({}, {}, {}))
        res["empty"], res["empty_collectives"] = _summary(plan), seen

        bufs = {} if rank == 0 else {"b": torch.ones(3, 3, dtype=torch.float64)}
        plan, _ = _counting(lambda: exchange_plan(bufs, {} if rank == 0 else {"b": 2}, {} if rank == 0 else {"b": 7},
                                                  make=make64))
        res["one_empty"], res["one_empty_buffers"] = _summary(plan), {n: g.dtype for n, g in bufs.items()}

        # reduce-scatter: live a (tri 10), b (3), c (6), e (15), z (1; owned by nobody)
        dims = {"a": 4, "b": 2, "c": 3, "e": 5, "z": 1}
        buffers = {n: torch.zeros(d, d) for n, d in dims.items()}
        calls, rows = {n: 1 for n in dims}, {n: 10 * (rank + 1) for n in dims}
        owners = {"e": 2, "c": 1, "b": 0, "a": 1}
        before = (dict(calls), dict(rows))
        plan, seen = _counting(lambda: exchange_plan(buffers, calls, rows, owners=owners))
        res["scatter"], res["scatter_collectives"] = _summary(plan), seen
        res["scatter_symmetric_nbytes"] = exchange_plan(buffers, calls, rows, owners=owners, symmetric=True).nbytes
        res["scatter_counters_kept"] = (dict(calls), dict(rows)) == before
        _, res["all_reduce_collectives"] = _counting(lambda: exchange_plan(buffers, calls, rows))

        bad = {"unknown_name": {**owners, "no.such.gram": 0},
               "rank_out_of_range": {**owners, "a": world},
               "negative_rank": {**owners, "a": -1},
               "not_an_int": {**owners, "a": 1.0},
               "differs_between_ranks": {**owners, "z": rank}}
        res["bad"] = {}
        for case, m in bad.items():
            out, seen = _counting(lambda: exchange_plan(buffers, calls, rows, owners=m))
            res["bad"][case] = (type(out).__name__, str(out), seen, (dict(calls), dict(rows)) == before)
        ret[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def results():
    ret = mp.Manager().dict()
    mp.spawn(_job, args=(WORLD, _free_port(), ret), nprocs=WORLD, join=True)
    return [ret[r] for r in range(WORLD)]


def test_all_reduce_plan_of_ragged_buffer_sets(results):
    for rank, r in enumerate(results):
        p = r["ragged"]
        # live names in agreed (sorted) order, back to back; `never` fired nowhere and does not travel
        assert p["names"] == p["mine"] == ["a", "only0", "only1", "only2"]
        assert p["offsets"] == [0, 10, 13, 19] and p["sections"] == [29] and p["width"] == 29
        assert p["nbytes"] == r["ragged_symmetric_nbytes"] == 29 * 4
        assert p["calls"] == {"a": 3, "never": 0, "only0": 1, "only1": 1, "only2": 1}
        assert p["rows"] == {"a": 9, "never": 0, "only0": 5, "only1": 6, "only2": 7}
        assert p["owners"] is None and (p["rank"], p["world"]) == (rank, WORLD)
        assert r["ragged_buffers"] == ["a", "never", "only0", "only1", "only2"]    # zero buffers for the missing names
        assert r["ragged_counters_kept"]


def test_all_reduce_plan_without_buffers(results):
    for r in results:
        p = r["empty"]
        assert p["names"] == p["mine"] == p["offsets"] == [] and p["sections"] == [0] and p["width"] == 0
        assert p["nbytes"] == 0 and p["calls"] == p["rows"] == {}
        assert r["empty_collectives"] == ["all_reduce"]          # the digest only: there are no counters to sum
        p = r["one_empty"]                                       # rank 0 holds nothing: it makes b with `make`
        assert p["names"] == ["b"] and p["nbytes"] == 6 * 8
        assert p["calls"] == {"b": 2 * (WORLD - 1)} and p["rows"] == {"b": 7 * (WORLD - 1)}
        assert r["one_empty_buffers"] == {"b": torch.float64}


def test_reduce_scatter_plan_layout_against_hand_computation(results):
    for rank, r in enumerate(results):
        p = r["scatter"]
        # stable sort by owner: b (owner 0), then a, c (owner 1, live order), then e (owner 2); z is not exchanged
        assert p["names"] == ["b", "a", "c", "e"]
        assert p["sections"] == [3, 10 + 6, 15] and p["width"] == 16
        assert p["offsets"] == [0, 16, 16 + 10, 32]
        assert p["mine"] == [["b"], ["a", "c"], ["e"]][rank]
        assert p["nbytes"] == WORLD * 16 * 4                    # NCCL: the whole padded [world x width] buffer
        assert r["scatter_symmetric_nbytes"] == [3, 16, 15][rank] * 4   # multimem: this rank's own triangles
        assert p["owners"] == {"e": 2, "c": 1, "b": 0, "a": 1}
        assert p["calls"] == {n: WORLD for n in "abcez"} and p["rows"] == {n: 60 for n in "abcez"}
        assert r["scatter_counters_kept"]


@pytest.mark.parametrize("case,message", [
    ("unknown_name", "owner map names 'no.such.gram', which is not a live Gram"),
    ("rank_out_of_range", f"owner {WORLD} of 'a' is not a rank of a {WORLD}-rank group"),
    ("negative_rank", f"owner -1 of 'a' is not a rank of a {WORLD}-rank group"),
    ("not_an_int", f"owner 1.0 of 'a' is not a rank of a {WORLD}-rank group"),
    ("differs_between_ranks", "the ranks passed different owner maps"),
])
def test_bad_owner_map_raises_on_every_rank_and_keeps_the_counters(results, case, message):
    for r in results:
        kind, text, seen, kept = r["bad"][case]
        assert kind == "ValueError" and message in text, text
        assert seen == ["all_reduce"] * 3                       # every rank issued the same collectives first
        assert kept


def test_collectives_per_plan(results):
    for r in results:
        assert r["all_reduce_collectives"] == ["all_reduce"] * 2     # buffer-set digest, counters
        assert r["scatter_collectives"] == ["all_reduce"] * 3        # buffer-set digest, counters, owner-map digest
        assert r["ragged_collectives"] == ["all_reduce", "all_gather_object", "all_reduce"]  # digests differ: the union
