"""GramCache.reduce_scatter() on real devices (NCCL, one process per GPU): every rank calibrates its own shard into pairs
of caches, all-reduces one of each pair and reduce-scatters the other by regmean_gram_owners, then compares the owned
Grams and the sharded regmean results.  Pairs: fp32 and int8x4 (fp64 Grams), plain (NCCL) and symmetric=True
(multimem).  2 ranks: one addition per element either way, so everything must match bit for bit; 4 ranks (where the
box has them): the reductions may add in a different order.  Also: a symmetric cache's all_reduce() that must refuse
leaves the cache as it was.  Skipped with fewer than 2 GPUs."""
import os
import socket
import tempfile
import warnings

import pytest
import torch

pytestmark = pytest.mark.gpu

LEGS = {"fp32": {}, "int8x4": {"precision": "int8x4"},
        "fp32_mc": {"symmetric": True}, "int8x4_mc": {"precision": "int8x4", "symmetric": True}}
CONFIG = dict(vlffn_start_layer_index=10, scaling_for_non_diag=1.0, loss_names={"irtr": 1.0, "vqa": 0, "nlvr2": 0})


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _raises(fn, exc):
    try:
        fn()
    except exc:
        return True
    return False


def _compare(whole, scat, sd, rank, world):
    """All-reduce `whole`, reduce-scatter `scat`, and report what the test asserts."""
    import torch.distributed as dist

    import vl_merging_b200 as vlm

    group = dist.group.WORLD
    owners = vlm.regmean_gram_owners(sd, CONFIG, scat.live_names(), world)
    whole.all_reduce()
    calls = dict(whole.calls)
    live = whole.live_names()
    res = {"bad_name": _raises(lambda: whole.reduce_scatter({**owners, "no.such.gram": 0}), ValueError),
           "bad_rank": _raises(lambda: whole.reduce_scatter({**owners, live[0]: world}), ValueError)}
    res["calls_kept"] = dict(whole.calls) == calls                       # a refused call changes no counter
    scat.reduce_scatter(owners)
    res["live_same"] = scat.live_names() == live and set(owners) == set(live)
    res["calls_same"] = dict(scat.calls) == calls
    res["owners_kept"] = scat.owners == owners
    mine = [n for n in live if owners[n] == rank]
    res["n_mine"] = len(mine)
    equal, sym, err = True, True, 0.0
    for n in mine:
        a, b = whole.gram(n), scat.gram(n)
        equal = equal and torch.equal(a, b)
        sym = sym and torch.equal(b, b.T)
        err = max(err, ((a.double() - b.double()).norm() / a.double().norm()).item())
    res.update(grams_equal=equal, sym=sym, gram_err=err)
    esz = whole.buffers[live[0]].element_size()
    section = [0] * world
    for n, r in owners.items():
        d = whole.buffers[n].shape[0]
        section[r] += d * (d + 1) // 2 * esz
    res["reduce_bytes"] = scat.last_reduce_bytes
    res["want_bytes"] = section[rank] if scat.symmetric else world * max(section)
    other = next(n for n in live if owners[n] != rank)
    with tempfile.TemporaryDirectory() as tmp:
        res["refuses"] = {
            "gram": _raises(lambda: scat.gram(other), RuntimeError),
            "state_dict": _raises(lambda: scat.state_dict(), RuntimeError),
            "save": _raises(lambda: scat.save(os.path.join(tmp, "g.pt")), RuntimeError),
            "save_packed": _raises(lambda: scat.save_packed(os.path.join(tmp, "g.vlmg")), RuntimeError),
            "all_reduce": _raises(lambda: scat.all_reduce(), RuntimeError),
            "accumulate": _raises(lambda: scat.accumulate(other, torch.ones(8, whole.buffers[other].shape[0],
                                                                            device=whole.device)), RuntimeError),
            "regmean_num_layers": _raises(lambda: vlm.regmean(sd, CONFIG, gram_matrices=scat, group=group,
                                                              num_layers=11), ValueError),
            "regmean_no_group": _raises(lambda: vlm.regmean(sd, CONFIG, gram_matrices=scat), ValueError),
        }
        res["wrote"] = os.listdir(tmp)
    for alpha in (1.0, 0.9):
        cfg = dict(CONFIG, scaling_for_non_diag=alpha)
        a = vlm.regmean(sd, cfg, gram_matrices=whole, group=group)
        b = vlm.regmean(sd, cfg, gram_matrices=scat, group=group)
        keys = [k for k in a if k.startswith("transformer.blocks.") and "gamma" not in k]
        res[f"regmean_equal_{alpha}"] = all(torch.equal(a[k], b[k]) for k in keys)
        res[f"regmean_err_{alpha}"] = max(((a[k].double() - b[k].double()).norm() /
                                           a[k].double().norm().clamp_min(1e-300)).item() for k in keys)
    scat.reset()
    res["reset"] = scat.owners is None and scat.gram(other).abs().max().item() == 0
    return res


def _outside_arena(model, rank):
    """A symmetric cache with a Gram outside its arena (a name register() did not know): all_reduce() must refuse on
    every rank before it sums a counter, and all_reduce(packed=False) must then give what a plain cache gives."""
    import vl_merging_b200 as vlm

    sym, plain = vlm.GramCache(symmetric=True), vlm.GramCache()
    for c in (sym, plain):
        c.register(model)
    gen = torch.Generator(device="cuda").manual_seed(90 + rank)
    for name in ("transformer.blocks.0.attn.v", "not.registered"):
        d = sym.buffers[name].shape[0] if name in sym.buffers else 64
        x = torch.randint(-4, 5, (37, d), generator=gen, device="cuda").float()   # exact Grams, in any summation order
        for c in (sym, plain):
            c.accumulate(name, x)

    def counts(c):
        return {n: v for n, v in c.calls.items() if v}, {n: v for n, v in c.rows.items() if v}

    before, refused = counts(sym), None
    try:
        sym.all_reduce()
    except RuntimeError as e:
        refused = str(e)
    res = {"refused": refused, "counters_kept": counts(sym) == before}
    sym.all_reduce(packed=False)
    plain.all_reduce()
    res["counters_equal"] = counts(sym) == counts(plain) and len(before[0]) == 2
    res["grams_equal"] = all(torch.equal(sym.gram(n), plain.gram(n)) for n in before[0])
    return res


def _worker(rank, world, port, ret):
    import torch.distributed as dist

    import vl_merging_b200 as vlm

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    warnings.simplefilter("ignore", RuntimeWarning)     # regmean at alpha = 1 on fp32 Grams warns
    try:
        cfg = vlm.vlmo_config("tiny")
        model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
        pairs = {}
        for leg, kw in LEGS.items():
            pairs[leg] = (vlm.GramCache(**kw), vlm.GramCache(**kw))
            for c in pairs[leg]:
                c.register(model)
        with torch.no_grad():    # this rank's shard: 4 x 197 image rows, 4 x 40 text rows per Gram
            model(vlm.synthetic_batch(4, cfg, seed=50 + rank, device="cuda"))
        sd = {k: v.detach() for k, v in model.state_dict().items()}
        out = {}
        for leg, (whole, scat) in pairs.items():
            try:
                out[leg] = _compare(whole, scat, sd, rank, world)
            except RuntimeError as e:
                if not (whole.symmetric and "multicast" in str(e)):
                    raise
                out[leg] = {"unsupported": str(e)}
        out["outside_arena"] = _outside_arena(model, rank)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module", params=[2, 4], ids=lambda w: f"{w}ranks")
def ranks(request):
    import torch.multiprocessing as mp

    world = request.param
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    return world, [ret[r] for r in range(world)]


def _check(ranks, leg):
    world, res = ranks
    if "unsupported" in res[0][leg]:
        pytest.skip(f"no multicast mapping on this system: {res[0][leg]['unsupported']}")
    fp64 = leg.startswith("int8x4")
    assert sum(r[leg]["n_mine"] for r in res) == 96
    for r in (r[leg] for r in res):
        assert r["bad_name"] and r["bad_rank"] and r["calls_kept"]
        assert r["live_same"] and r["calls_same"] and r["owners_kept"] and r["n_mine"] > 0
        assert r["sym"]
        if world == 2:
            assert r["grams_equal"], r["gram_err"]
        else:
            assert r["gram_err"] <= (1e-14 if fp64 else 1e-6)
        assert r["reduce_bytes"] == r["want_bytes"]
        assert all(r["refuses"].values()), r["refuses"]
        assert r["wrote"] == []
        assert r["reset"]
        if world == 2:
            assert r["regmean_equal_1.0"] and r["regmean_equal_0.9"], (r["regmean_err_1.0"], r["regmean_err_0.9"])
    if not leg.endswith("_mc"):
        assert len({r[leg]["reduce_bytes"] for r in res}) == 1      # one buffer of world x the largest section


@pytest.mark.parametrize("leg", ["fp32", "int8x4"])
def test_nccl_reduce_scatter_matches_all_reduce(ranks, leg):
    _check(ranks, leg)


@pytest.mark.parametrize("leg", ["fp32_mc", "int8x4_mc"])
def test_multimem_reduce_scatter_matches_all_reduce(ranks, leg):
    _check(ranks, leg)


def test_refused_symmetric_all_reduce_keeps_the_counters(ranks):
    _, res = ranks
    for r in (r["outside_arena"] for r in res):
        assert "outside the symmetric arena" in (r["refused"] or ""), r["refused"]
        assert r["counters_kept"]
        assert r["counters_equal"] and r["grams_equal"]
