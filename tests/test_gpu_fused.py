"""GPU: Gram caching on the fused vision-language route (type_id 2, SURVEY.md §8f rank 3).  The shallow `l` / `v`
experts are hooked on ROW SLICES h[:, :40] / h[:, 40:] of the joint sequence; GramCache reads them in place
through vlm_syrk_accum_strided (4-D tensor map) where the reference's reshape copies.  Checked against the
numpy oracle on the same activations and against golden vectors from the unmodified reference
(tests/golden/fused_tiny.npz); tolerances from BASELINE.json (Gram 1e-3, RegMean 1e-4 on identical Grams)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

import vl_merging_b200 as vlm

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
import oracle  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(HERE, "golden", "fused_tiny.npz")


def _rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _oracle_gram(x):
    store = oracle.new_gram_store()
    oracle.hook_gram_input(store, "g", x.detach().double().cpu().numpy())
    return store["g"]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("d", [768, 192, 200, 1024])
def test_row_slices_are_read_in_place(dtype, d):
    """Text slice [0, 40) and image slice [40, N) of a (B, N, D) activation, for 224- and 384-pixel images: vs the
    fp64 oracle on the slice, and vs the same kernel on a contiguous copy.  d = 200 has no whole 128-byte column
    groups (CUDA-core kernel, one launch per segment)."""
    torch.manual_seed(d)
    tol = 1e-3 if dtype == torch.float32 else 1e-5      # 16-bit products are exact: only the fp32 accumulation is left
    for b, n in ((6, 40 + 197), (4, 40 + 577)):
        h = torch.randn(b, n, d, device="cuda").to(dtype)
        for lo, hi in ((0, 40), (40, n), (3, 4), (3, 8)):       # (3, 8): 5-row segments, shorter than one K chunk
            x = h[:, lo:hi]
            assert not x.is_contiguous()
            cache = vlm.GramCache()
            before = vlm._lib.launch_count()
            cache.accumulate("s", x)
            cache.accumulate("s", x)
            launches = vlm._lib.launch_count() - before
            cache.accumulate("c", x.contiguous())
            cache.accumulate("c", x.contiguous())
            sd = cache.state_dict()
            want = 2 * _oracle_gram(x)
            assert _rel(sd["s"].numpy(), want) < tol, (b, n, lo, hi)
            assert _rel(sd["s"].numpy(), sd["c"].numpy()) < 2e-4
            if d != 200:
                assert launches == 2          # one launch per call: no copy kernel, no per-segment launches
            assert cache.rows["s"] == 2 * b * (hi - lo)


def test_deferred_row_slices_go_through_the_grouped_launch():
    torch.manual_seed(1)
    h = torch.randn(5, 237, 768, device="cuda")
    h2 = torch.randn(5, 237, 3072, device="cuda")
    cache = vlm.GramCache(defer_bytes=64 << 20)
    before = vlm._lib.launch_count()
    cache.accumulate("t", h[:, :40])
    cache.accumulate("i", h[:, 40:])
    cache.accumulate("whole", h)
    cache.accumulate("wide", h2[:, 40:])
    assert vlm._lib.launch_count() == before      # all pending
    cache.flush()
    assert vlm._lib.launch_count() == before + 1  # ONE grouped launch
    sd = cache.state_dict()
    for name, x in (("t", h[:, :40]), ("i", h[:, 40:]), ("whole", h), ("wide", h2[:, 40:])):
        assert _rel(sd[name].numpy(), _oracle_gram(x)) < 1e-3, name
    # at calibration size (64 x 617 tokens): each slice and a packed copy of it in one grouped launch, and the slice
    # through the immediate launch, against the packed copy's Gram
    big = torch.randn(64, 617, 768, device="cuda")
    for lo, hi in ((40, 617), (0, 40)):
        x = big[:, lo:hi]
        grouped, now = vlm.GramCache(defer_bytes=1 << 30), vlm.GramCache()
        grouped.accumulate("s", x)
        grouped.accumulate("c", x.contiguous())
        before = vlm._lib.launch_count()
        grouped.flush()
        assert vlm._lib.launch_count() == before + 1
        now.accumulate("s", x)
        packed = grouped.gram("c").double()
        for g in (grouped.gram("s"), now.gram("s")):
            assert ((g.double() - packed).norm() / packed.norm()).item() < 2e-4, (lo, hi)


def test_unaligned_or_odd_slices_fall_back_correctly():
    h = torch.randn(4, 50, 100, device="cuda")      # 400-byte rows: 16-byte aligned pitch, d not a whole group
    h3 = torch.randn(4, 50, 99, device="cuda")      # 396-byte rows: TMA cannot address -> CUDA-core kernel on a copy
    for t in (h, h3):
        x = t[:, 7:33]
        cache = vlm.GramCache()
        cache.accumulate("s", x)
        assert _rel(cache.state_dict()["s"].numpy(), _oracle_gram(x)) < 1e-3
    # broadcast batch dimension (stride 0): not a segment layout TMA can describe -> the generic copy path
    e = torch.randn(1, 40, 768, device="cuda").expand(4, 40, 768)
    cache = vlm.GramCache()
    cache.accumulate("e", e)
    assert _rel(cache.state_dict()["e"].numpy(), _oracle_gram(e)) < 1e-3
    # permuted (not a row slice): the generic copy path
    p = torch.randn(64, 8, 128, device="cuda").permute(1, 0, 2)
    cache = vlm.GramCache()
    cache.accumulate("p", p)
    assert _rel(cache.state_dict()["p"].numpy(), _oracle_gram(p)) < 1e-3


@pytest.fixture(scope="module")
def fused():
    z = np.load(GOLDEN)
    meta = json.loads(bytes(z["meta"]).decode())
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    cache = vlm.GramCache()
    cache.register(model, use_moe=True)
    with torch.no_grad():
        for bs, seed, pad in meta["calib_batches"]:
            ret = model.infer(vlm.synthetic_batch(bs, cfg, seed=seed, pad=pad, device="cuda"))
    cache.remove_hooks()
    return z, meta, cfg, model, cache, ret


def test_fused_route_grams_match_reference(fused):
    z, meta, cfg, model, cache, ret = fused
    assert np.abs(ret["cls_feats"].cpu().numpy() - z["calib/last_cls"]).max() < 1e-3
    grams = cache.state_dict()
    assert sorted(grams) == sorted(meta["gram_keys"])           # 88: v/l slices below layer 10, vl above
    for k in meta["gram_keys"]:
        g = grams[k].numpy()
        assert g.dtype == np.float64 and np.array_equal(g, g.T)
        fro, trace = z[f"gram/{k}/fro_trace"]
        assert np.linalg.norm(np.diag(g) - z[f"gram/{k}/diag"]) < 1e-3 * np.linalg.norm(z[f"gram/{k}/diag"]), k
        assert abs(np.linalg.norm(g) - fro) < 1e-3 * fro and abs(np.trace(g) - trace) < 1e-3 * trace, k
    for k in (f for f in z.files if f.startswith("gram_full/")):
        assert _rel(grams[k[len("gram_full/"):]].numpy(), z[k]) < 1e-3, k
    # rows seen: 7 samples x 40 text rows, x 197 image rows, x 237 joint rows
    assert cache.rows["transformer.blocks.0.attn.l"] == 7 * 40
    assert cache.rows["transformer.blocks.0.mlp.v.fc1"] == 7 * 197
    assert cache.rows["transformer.blocks.11.attn.vl"] == 7 * 237


@pytest.mark.parametrize("variant", ["vqa", "nlvr2"])
def test_regmean_of_fused_grams_matches_reference(fused, variant, tmp_path):
    z, meta, cfg, model, cache, _ = fused
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    mcfg = dict(vlffn_start_layer_index=cfg["vlffn_start_layer_index"], loss_names=meta["variants"][variant],
                scaling_for_non_diag=0.9)
    merged = vlm.regmean(sd, mcfg, gram_matrices=cache)
    pre = f"merged/{variant}/tensor/"
    for k in (f for f in z.files if f.startswith(pre)):
        got = merged[k[len(pre):]].cpu().numpy()[:8]
        tol = 5e-3 if k.endswith(".weight") and "norm" not in k else 1e-6   # linears consume OUR TF32 Grams
        assert _rel(got, z[k]) <= tol, (variant, k)
    # identical Grams on both sides (the reference-format fp64 file): RegMean itself to 1e-4
    cache.save(tmp_path / "g.pth")
    grams = {k: v.numpy() for k, v in torch.load(tmp_path / "g.pth", weights_only=False).items()}
    got = vlm.regmean({k: v.cpu() for k, v in sd.items()}, dict(mcfg, gram_matrices=str(tmp_path / "g.pth")))
    want = oracle.regmean({k: v.cpu().numpy() for k, v in sd.items()}, grams, mcfg)
    for k, w in want.items():
        if "transformer.blocks." in k and "gamma" not in k:
            assert _rel(got[k].numpy(), w) <= 1e-4, k
    ufo = vlm.VLMo(vlm.vlmo_config("tiny", use_moe=False)).eval().cuda()
    ufo.load_state_dict(merged, strict=False)
    bs, seed, pad = meta["eval_batch"]
    with torch.no_grad():
        out = ufo.infer(vlm.synthetic_batch(bs, cfg, seed=seed, pad=pad, device="cuda"))
    assert np.abs(out["cls_feats"].cpu().numpy() - z[f"merged/{variant}/cls"]).max() < 1e-3
