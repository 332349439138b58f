"""GPU: the packed Gram container end to end — pack / unpack / mirror kernels bit-exact against numpy, GramCache ->
packed file -> regmean identical to regmean on the live cache, and both conversions with the reference's
own Gram file (torch.save of fp64 matrices, src/cache_gram_matrices.py:349)."""
import os
import sys

import numpy as np
import pytest
import torch

import vl_merging_b200 as vlm
from vl_merging_b200 import _lib, gramfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gramfile import _write_by_hand  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype,code", [(torch.float32, 0), (torch.float64, 3)])
def test_batched_pack_unpack_bit_exact(dtype, code):
    """vlm_sym_pack_upper_batch / vlm_sym_unpack_batch / vlm_sym_mirror_batch: Grams of mixed widths in one launch each
    (the exchange buffer of GramCache.all_reduce, the packed Gram file, GramCache.finalize), fp32 and fp64, padded
    leading dimensions."""
    dims = [1, 31, 32, 33, 192, 768, 1000, 5, 256]
    torch.manual_seed(7)
    full = [torch.randn(d, d + (i % 3), dtype=dtype, device="cuda")[:, :d] for i, d in enumerate(dims)]
    upper = [torch.triu(a) + torch.tril(torch.full_like(a, float("nan")), -1) for a in full]
    upper = [torch.empty(d, d + (i % 3), dtype=dtype, device="cuda")[:, :d].copy_(u) for i, (d, u) in enumerate(zip(dims, upper))]
    sizes = [d * (d + 1) // 2 for d in dims]
    flat = torch.full((sum(sizes),), -7.0, dtype=dtype, device="cuda")
    lib, stream = _lib.lib(), torch.cuda.current_stream().cuda_stream
    items = _lib.sym_items(upper, flat)
    _lib.check(lib.vlm_sym_pack_upper_batch(items, len(dims), code, stream))
    got = flat.cpu().numpy()
    off = 0
    for a, d, sz in zip(full, dims, sizes):
        assert np.array_equal(got[off: off + sz], a.cpu().numpy()[np.triu_indices(d)]), d
        off += sz
    outs = [torch.full((d, d + 2), -1.0, dtype=dtype, device="cuda") for d in dims]
    _lib.check(lib.vlm_sym_unpack_batch(_lib.sym_items([o[:, :d] for o, d in zip(outs, dims)], flat), len(dims), code,
                                        stream))
    for a, o, d in zip(full, outs, dims):
        sym = (torch.triu(a) + torch.triu(a, 1).t()).cpu().numpy()
        assert np.array_equal(o.cpu().numpy()[:, :d], sym) and (o.cpu().numpy()[:, d:] == -1.0).all(), d
    assert lib.vlm_sym_pack_upper_batch(items, len(dims), 1, stream) == -1          # bf16 is not a Gram type
    # the mirror, in place: the NaNs below the diagonal become the transpose of the upper triangle; the upper triangle,
    # the diagonal and the padding columns stay as they are
    padded = [torch.randn(d, d + 1 + i % 3, dtype=dtype, device="cuda") for i, d in enumerate(dims)]
    for p, d in zip(padded, dims):
        p[:, :d] = torch.triu(p[:, :d]) + torch.tril(torch.full_like(p[:, :d], float("nan")), -1)
    before = [p.cpu().numpy() for p in padded]
    _lib.check(lib.vlm_sym_mirror_batch(_lib.sym_items([p[:, :d] for p, d in zip(padded, dims)]), len(dims), code, stream))
    for p, b, d in zip(padded, before, dims):
        got = p.cpu().numpy()
        assert np.array_equal(got[:, :d], np.triu(b[:, :d]) + np.triu(b[:, :d], 1).T), d
        assert np.array_equal(got[:, d:], b[:, d:]), d


def test_hand_written_file_loads(tmp_path):
    rng = np.random.default_rng(1)
    grams = {}
    for name, d in (("a", 5), ("b.fc2", 97), ("c", 256)):
        m = rng.standard_normal((d, d)).astype(np.float32)
        grams[name] = np.triu(m) + np.triu(m, 1).T
    _write_by_hand(tmp_path / "g", grams)
    got = gramfile.load_packed(tmp_path / "g")
    assert list(got) == list(grams)
    for k, g in grams.items():
        assert got[k].dtype == torch.float32 and got[k].is_cuda
        assert np.array_equal(got[k].cpu().numpy(), g)


@pytest.fixture(scope="module")
def calibrated():
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    cache = vlm.GramCache()
    cache.register(model, use_moe=True)
    with torch.no_grad():
        for seed in (1, 2):
            model(vlm.synthetic_batch(4, cfg, seed=seed, device="cuda"))
    cache.remove_hooks()
    return cfg, model, cache


def test_cache_to_packed_file_and_back(calibrated, tmp_path):
    cfg, model, cache = calibrated
    nbytes = cache.save_packed(tmp_path / "grams.vlmgram")
    assert nbytes == os.path.getsize(tmp_path / "grams.vlmgram")
    cache.save(tmp_path / "grams.pth")                                        # the reference's format
    assert nbytes < 0.26 * os.path.getsize(tmp_path / "grams.pth")
    entries, _ = gramfile.read_header(tmp_path / "grams.vlmgram")
    assert [e["name"] for e in entries] == cache.live_names()
    assert all(e["rows"] == cache.rows[e["name"]] and e["calls"] == 2 for e in entries)
    want = cache.state_dict()
    got32 = gramfile.load_packed(tmp_path / "grams.vlmgram")
    got64 = gramfile.load_packed(tmp_path / "grams.vlmgram", dtype=torch.float64)
    for k, w in want.items():
        assert torch.equal(got64[k].cpu(), w)                                 # fp32 values widened: exact
        assert torch.equal(got32[k].cpu().double(), w)


def test_regmean_reads_either_format(calibrated, tmp_path):
    cfg, model, cache = calibrated
    cache.save_packed(tmp_path / "g.vlmgram")
    cache.save(tmp_path / "g.pth")
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    mcfg = dict(vlffn_start_layer_index=10, loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0}, scaling_for_non_diag=0.9)
    live = vlm.regmean(sd, mcfg, gram_matrices=cache)
    packed = vlm.regmean(sd, dict(mcfg, gram_matrices=str(tmp_path / "g.vlmgram")))
    ref = vlm.regmean(sd, dict(mcfg, gram_matrices=str(tmp_path / "g.pth")))
    for k in live:
        assert torch.equal(live[k], packed[k]), k                             # same fp32 Grams: identical
        if live[k].dtype == torch.float64:
            assert (ref[k] - live[k]).norm() <= 1e-9 * live[k].norm(), k        # fp64 file: same values, fp64 RHS path
    assert sum(v.dtype == torch.float64 for v in live.values()) == 48


def test_conversion_to_and_from_the_reference_file(calibrated, tmp_path):
    cfg, model, cache = calibrated
    cache.save_packed(tmp_path / "g.vlmgram")
    gramfile.export_reference(tmp_path / "g.vlmgram", tmp_path / "exported.pth")
    exported = torch.load(tmp_path / "exported.pth", weights_only=False)       # what the reference's regmean reads
    want = cache.state_dict()
    assert list(exported) == list(want)
    for k, w in want.items():
        assert exported[k].dtype == torch.float64 and exported[k].device.type == "cpu"
        assert torch.equal(exported[k], w)
    gramfile.import_reference(tmp_path / "exported.pth", tmp_path / "again.vlmgram")
    again = gramfile.load_packed(tmp_path / "again.vlmgram", dtype=torch.float64)
    for k, w in want.items():
        assert torch.equal(again[k].cpu(), w)


def test_fp64_container_keeps_the_regmean_grade_grams_exactly(tmp_path):
    """A RegMean-grade cache (fp64 Gram buffers) writes the container in fp64 — half the reference file, every value
    kept — and regmean from that file equals regmean on the live cache; narrowing on load and the fp64 import of the
    reference's own file work too."""
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    cache = vlm.GramCache(precision="int8x4")
    cache.register(model, use_moe=True)
    with torch.no_grad():
        for seed in (5, 6, 7):
            model(vlm.synthetic_batch(8, cfg, seed=seed, device="cuda"))
    cache.remove_hooks()
    nbytes = cache.save_packed(tmp_path / "g64.vlmgram")
    cache.save(tmp_path / "g.pth")
    assert 0.49 < nbytes / os.path.getsize(tmp_path / "g.pth") < 0.52
    entries, _, fdtype = gramfile.read_header(tmp_path / "g64.vlmgram", with_dtype=True)
    assert fdtype == torch.float64 and [e["name"] for e in entries] == cache.live_names()
    want = cache.state_dict()
    got = gramfile.load_packed(tmp_path / "g64.vlmgram")
    got32 = gramfile.load_packed(tmp_path / "g64.vlmgram", dtype=torch.float32)
    for k, w in want.items():
        assert got[k].dtype == torch.float64 and torch.equal(got[k].cpu(), w)
        assert got32[k].dtype == torch.float32 and torch.equal(got32[k].cpu(), w.float())
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    mcfg = dict(vlffn_start_layer_index=10, loss_names={"irtr": 1, "vqa": 0, "nlvr2": 0}, scaling_for_non_diag=0.9)
    live = vlm.regmean(sd, mcfg, gram_matrices=cache)
    packed = vlm.regmean(sd, dict(mcfg, gram_matrices=str(tmp_path / "g64.vlmgram")))
    assert all(torch.equal(live[k], packed[k]) for k in live)
    gramfile.import_reference(tmp_path / "g.pth", tmp_path / "again64.vlmgram", dtype=torch.float64)
    again = gramfile.load_packed(tmp_path / "again64.vlmgram")
    assert all(torch.equal(again[k].cpu(), w) for k, w in want.items())
