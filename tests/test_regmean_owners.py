"""regmean_gram_owners: which rank's sharded regmean reads each Gram, the map GramCache.reduce_scatter() scatters by.
Pure host logic on the real VLMo-base and ViT-L (24-layer) shapes (meta tensors, no GPU)."""
import pytest
import torch

import vl_merging_b200 as vlm
from vl_merging_b200.merge import ShardLayout
from vl_merging_b200.plan import plan_regmean

MB = 1e6


def _geometry(size):
    cfg = vlm.vlmo_config(size)
    with torch.device("meta"):
        sd = vlm.VLMo(cfg).state_dict()
    return sd, cfg["num_layers"], cfg["vlffn_start_layer_index"]


@pytest.fixture(scope="module", params=["base", "large"])
def geometry(request):
    return (request.param,) + _geometry(request.param)


def _widths(sd, layers, mods=("v", "l"), deep_mods=None, start=None):
    """{Gram name: width} of the linears the calibration forward hooks (deep layers: deep_mods, if given)."""
    out = {}
    for i in range(layers):
        p = f"transformer.blocks.{i}."
        for m in (deep_mods if deep_mods is not None and i >= start else mods):
            for gram, weight in ((f"attn.{m}", f"attn.{m}.qkv.weight"), (f"attn.{m}.proj", f"attn.{m}.proj.weight"),
                                 (f"mlp.{m}.fc1", f"mlp.{m}.fc1.weight"), (f"mlp.{m}.fc2", f"mlp.{m}.fc2.weight")):
                out[p + gram] = sd[p + weight].shape[1]
    return out


def _config(start, task="irtr"):
    return dict(vlffn_start_layer_index=start, scaling_for_non_diag=1.0,
                loss_names={"irtr": int(task == "irtr"), "vqa": int(task == "vqa"), "nlvr2": 0})


def _parent_owners(sd, cfg, names, world, layers):
    """The assignment regmean() made before the owner map existed, restated: its linear problems, the same cost and
    the same cost-balanced ShardLayout, each problem's Grams on its rank."""
    ops = [op for op in plan_regmean(sd.keys(), names, cfg, layers) if not op.passthrough and op.regmean]

    def cost(op):
        o, i = sd[op.regmean[0][0]].shape
        return i * i * i // 3 + 2 * len(op.regmean) * o * i * i + 2 * o * i * i

    lay = ShardLayout([int(sd[op.regmean[0][0]].numel()) for op in ops], world, cost=lambda i: cost(ops[i]), align=1)
    pairs = [(g, lay.owner[idx]) for idx, op in enumerate(ops) for _, g in op.regmean]
    return pairs


@pytest.mark.parametrize("world", range(1, 9))
def test_every_read_gram_has_the_rank_regmean_assigns(geometry, world):
    _, sd, layers, start = geometry
    widths = _widths(sd, layers)
    cfg = _config(start)
    owners = vlm.regmean_gram_owners(sd, cfg, list(widths), world, num_layers=layers)
    pairs = _parent_owners(sd, cfg, list(widths), world, layers)
    assert len(pairs) == len({g for g, _ in pairs})                 # every Gram feeds exactly one problem
    assert owners == dict(pairs)
    assert set(owners) == set(widths)                               # irtr: every v / l Gram is read
    assert set(owners.values()) <= set(range(world))
    if world == 1:
        assert set(owners.values()) == {0}
    else:
        assert set(owners.values()) == set(range(world))            # every rank solves something


# (largest owner section, smallest) in MB of packed fp32 upper triangles
SECTIONS = {("base", 2): (269.1, 269.1), ("base", 4): (134.5, 134.5), ("base", 8): (80.2, 54.3),
            ("large", 2): (956.6, 956.6), ("large", 4): (478.3, 478.3), ("large", 8): (239.2, 239.2)}
TOTAL = {"base": 538.2, "large": 1913.3}


@pytest.mark.parametrize("world", [2, 4, 8])
def test_owner_sections(geometry, world):
    size, sd, layers, start = geometry
    widths = _widths(sd, layers)
    owners = vlm.regmean_gram_owners(sd, _config(start), list(widths), world, num_layers=layers)
    section = [0] * world
    for g, r in owners.items():
        section[r] += widths[g] * (widths[g] + 1) // 2 * 4
    assert round(sum(section) / MB, 1) == TOTAL[size]
    assert (round(max(section) / MB, 1), round(min(section) / MB, 1)) == SECTIONS[(size, world)]


def test_unread_grams_have_no_owner():
    sd, layers, start = _geometry("base")
    widths = _widths(sd, layers, deep_mods=("v", "l", "vl"), start=start)
    owners = vlm.regmean_gram_owners(sd, _config(start, "vqa"), list(widths), 4, num_layers=layers)
    deep_vl = {g for g in widths if int(g.split(".")[2]) >= start and (".vl" in g)}
    deep_v_l = {g for g in widths if int(g.split(".")[2]) >= start and ".vl" not in g}
    assert deep_vl and deep_v_l
    assert set(owners) == set(widths) - deep_v_l                    # the vqa plan reads only `vl` in the deep layers
    assert dict(_parent_owners(sd, _config(start, "vqa"), list(widths), 4, layers)) == owners


def test_owners_follow_num_layers_and_world():
    sd, layers, start = _geometry("base")
    names = list(_widths(sd, layers))
    a = vlm.regmean_gram_owners(sd, _config(start), names, 2, num_layers=layers)
    assert a != vlm.regmean_gram_owners(sd, _config(start), names, 4, num_layers=layers)
    assert a != vlm.regmean_gram_owners(sd, _config(start), names, 2, num_layers=layers - 1)
