"""vlm_sim_topk — the fused similarity + top-10 of the IRTR evaluation (objectives.py:684-710) — against torch on the
same features, and the recalls it yields against the oracle's, at odd sizes and at the COCO 5k x 25k size."""
import numpy as np
import pytest
import torch

import oracle
import vl_merging_b200 as vlm

pytestmark = pytest.mark.gpu


def _feats(m, n, d, dtype, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(m, d, device="cuda", generator=gen).to(dtype)
    b = torch.randn(n, d, device="cuda", generator=gen).to(dtype)
    return a, b


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("m,n,d", [(1, 1, 8), (7, 5, 64), (130, 300, 192), (128, 256, 768), (129, 257, 776), (300, 1000, 1024),
                                   (5000, 700, 768), (40, 9000, 768), (5000, 25000, 768)])
def test_sim_topk_matches_torch(m, n, d, dtype):
    a, b = _feats(m, n, d, dtype, seed=m * 31 + n)
    k = min(10, n)
    val, idx = vlm.sim_topk(a, b, k)
    scores = a.double() @ b.double().t()                  # exact products, fp64 sums: the ground truth
    want_val, want_idx = scores.topk(k, dim=1)
    assert val.shape == (m, k) and idx.shape == (m, k) and idx.dtype == torch.int64
    got_scores = torch.gather(scores, 1, idx)             # what the chosen columns really score
    # the kernel accumulates in fp32: it may swap two columns whose scores differ by rounding, nothing more
    assert torch.allclose(val.double(), got_scores, rtol=1e-5, atol=1e-4 * float(d) ** 0.5)
    assert torch.allclose(got_scores, want_val, rtol=1e-5, atol=2e-4 * float(d) ** 0.5)
    assert (idx == want_idx).float().mean() > 0.999
    assert bool((val[:, :-1] >= val[:, 1:]).all()) if k > 1 else True
    for r in range(min(m, 5)):                             # no column twice
        assert len(set(idx[r].tolist())) == k


def test_ties_prefer_the_lower_index():
    a = torch.ones(3, 64, device="cuda", dtype=torch.float16)
    b = torch.ones(600, 64, device="cuda", dtype=torch.float16)     # every score equal: 2+ column tiles, 1+ splits
    b[17] *= 2
    val, idx = vlm.sim_topk(a, b, 10)
    assert idx[0].tolist() == [17, 0, 1, 2, 3, 4, 5, 6, 7, 8]
    assert val[0].tolist() == [128.0] + [64.0] * 9


def test_fused_recalls_equal_oracle_at_coco_size():
    """5,000 images x 25,000 captions (5 per image): the six recalls of the fused path equal the oracle's
    (objectives.py:688-708 restated), which sorts the full fp32 score matrix."""
    gen = torch.Generator(device="cuda").manual_seed(11)
    n_img, per = 5000, 5
    base = torch.randn(n_img, 768, device="cuda", generator=gen)
    img = torch.nn.functional.normalize(base + 2.0 * torch.randn(n_img, 768, device="cuda", generator=gen), dim=-1).half()
    txt = torch.nn.functional.normalize(base.repeat_interleave(per, 0) +
                                        3.0 * torch.randn(n_img * per, 768, device="cuda", generator=gen), dim=-1).half()
    iids, tiids = np.arange(n_img), np.arange(n_img * per) // per
    recalls, (by_image, by_caption) = vlm.irtr_recall_fused(img, txt, iids, tiids)
    assert tuple(by_image.shape) == (5000, 10) and tuple(by_caption.shape) == (25000, 10)
    _, ref = oracle.irtr_recall(img.float().cpu().numpy(), txt.float().cpu().numpy(), iids, tiids)
    got = np.array([float(r) for r in recalls])
    assert 0.02 < got.min() and got.max() < 0.995
    assert np.allclose(got, np.array(ref, dtype=np.float64), atol=2.0 / n_img), (got, ref)
    # the unfused torch path (materialised scores + six topk calls) on the same features agrees as well
    _, plain = vlm.irtr_recall(img.float(), txt.float(), iids, tiids)
    assert np.allclose(got, np.array([float(r) for r in plain]), atol=2.0 / n_img)
    # fp32 features that fp16 holds exactly are narrowed back losslessly: same launches, same result
    again, _ = vlm.irtr_recall_fused(img.float(), txt.float(), iids, tiids)
    assert [float(r) for r in again] == [float(r) for r in recalls]
    with pytest.raises(RuntimeError):
        vlm.irtr_recall_fused(img.float()[:, :763], txt.float()[:, :763], iids, tiids)


def test_fp32_features_take_the_split_path_with_fp32_accuracy():
    """What infer_image_ft / infer_text_ft return (fp32: the normalisation promotes, even under autocast): three bf16
    planes per operand, six products, and the scores of the chosen columns match an fp64 recomputation to fp32
    accuracy — where a single bf16 pass would be off by 2^-9."""
    from vl_merging_b200.irtr import _split3

    gen = torch.Generator(device="cuda").manual_seed(5)
    a = torch.nn.functional.normalize(torch.randn(700, 768, device="cuda", generator=gen), dim=-1)
    b = torch.nn.functional.normalize(torch.randn(3000, 768, device="cuda", generator=gen), dim=-1)
    val, idx = vlm.sim_topk(_split3(a, True), _split3(b, False), 10)
    scores = a.double() @ b.double().t()
    want_val, want_idx = scores.topk(10, dim=1)
    assert (val.double() - torch.gather(scores, 1, idx)).abs().max() < 2e-6
    assert (torch.gather(scores, 1, idx) - want_val).abs().max() < 2e-6
    assert (idx == want_idx).float().mean() > 0.9995
    iids, tiids = np.arange(700), np.arange(3000) % 700
    recalls, _ = vlm.irtr_recall_fused(a, b, iids, tiids)
    _, ref = oracle.irtr_recall(a.cpu().numpy(), b.cpu().numpy(), iids, tiids)
    assert np.allclose([float(r) for r in recalls], np.array(ref, dtype=np.float64), atol=2.0 / 700)
