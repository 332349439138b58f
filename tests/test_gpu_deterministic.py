"""The deterministic Gram mode (vlm_set_deterministic, GramCache(deterministic=True)): every launch form still exact,
bit-identical from run to run, as accurate as the default mode, and bit-identical Gram files and RegMean results.

Exactness reuses the exactly summable inputs and the case lists of test_gpu_gram_kernels.py: in the deterministic mode
every kernel writes its partial tiles into workspace slots and one reduction launch adds them into G, so each launch
form is checked again, with its sentinels.  Determinism needs real-valued data (on exact data every order gives the same
bits): each form runs four times into fresh copies of the same G0, two of them while a matmul loop on another stream
competes for the SMs, so that the clusters start and finish in a different order.
"""
import contextlib

import pytest
import torch

import vl_merging_b200 as vlm
from sentinel_buffers import same_bits
from test_gpu_gram_kernels import (BF16, CODE, F16, F32, F64, SIMT, SINGLE, STRIDED, Member, Padded, Segmented,
                                   _single_id, exact_g0, exact_x, gram_twice, new_g, run_batch, split_exact_x,
                                   split_want, assert_exact_case, assert_upper_equal)
from vl_merging_b200 import _lib

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    return _lib.lib()


@contextlib.contextmanager
def deterministic(lib, on=True):
    prev = lib.vlm_get_deterministic()
    lib.vlm_set_deterministic(int(on))
    try:
        yield
    finally:
        lib.vlm_set_deterministic(prev)


# ---- 1. exactness survives ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", SINGLE, ids=_single_id)
def test_single_launch_is_exact(lib, case):
    dtype, rows, d, pitched = case
    e = {F32: 4, BF16: 2, F16: 2}[dtype]
    ldx, ldg, lead_x, lead_g = (d + 16 // e, d + 4, 16 // e, 4) if pitched else (d, d, 0, 0)
    x, x64, ex = exact_x(rows, d, dtype, seed=rows * 7 + d)
    xb = Padded(rows, d, ldx, dtype, fill=x, lead=lead_x)
    with deterministic(lib):
        gram_twice(lambda g: lib.vlm_syrk_accum(xb.ptr, CODE[dtype], rows, d, ldx, g.ptr, g.ld, None), x64, ex, d,
                   "det " + _single_id(case), ldg=ldg, g_lead=lead_g, seed=rows + d)
    assert xb.sentinels_intact()


@pytest.mark.parametrize("case", list(SIMT))
def test_cuda_core_fallback_is_exact(lib, case):
    dtype, rows, d, ldx, lead, ldg = SIMT[case]
    x, x64, ex = exact_x(rows, d, dtype, seed=rows + d)
    xb = Padded(rows, d, ldx, dtype, fill=x, lead=lead)
    with deterministic(lib):
        for fn in (lib.vlm_syrk_accum, lib.vlm_syrk_accum_simt):
            gram_twice(lambda g: fn(xb.ptr, CODE[dtype], rows, d, ldx, g.ptr, g.ld, None), x64, ex, d,
                       f"det {case} {fn.__name__}", ldg=ldg, seed=d)
    assert xb.sentinels_intact()


def test_cuda_core_many_row_slices_is_exact(lib):
    """More than one 2048-row slice (grid.z): several slots per tile."""
    rows, d = 9000, 200
    x, x64, ex = exact_x(rows, d, F32, seed=5)
    with deterministic(lib):
        gram_twice(lambda g: lib.vlm_syrk_accum_simt(x.data_ptr(), _lib.VLM_F32, rows, d, d, g.ptr, g.ld, None), x64, ex,
                   d, "det simt 9000 x 200", ldg=d + 1, seed=6)


@pytest.mark.parametrize("case", list(STRIDED))
def test_strided_segments_are_exact(lib, case):
    dtype, nseg, seg_rows, d, ldx, seg_stride, lead = STRIDED[case]
    rows = nseg * seg_rows
    x, x64, ex = exact_x(rows, d, dtype, seed=nseg * seg_rows + d)
    xs = Segmented(x, seg_rows, ldx, seg_stride, lead=lead)
    with deterministic(lib):
        gram_twice(lambda g: lib.vlm_syrk_accum_strided(xs.ptr, CODE[dtype], rows, d, ldx, seg_rows, seg_stride, g.ptr,
                                                        g.ld, None), x64, ex, d, "det " + case, ldg=d + 4, seed=nseg)
    assert xs.sentinels_intact()


def test_batch_text_tower_mix_is_exact(lib):
    shapes = [(2560, 768)] * 36 + [(2560, 3072)] * 12
    members = [Member(F32, r, d, seed=i) for i, (r, d) in enumerate(shapes)]
    with deterministic(lib):
        run_batch(lib, F32, members, list(range(len(members))), "det text tower")


def test_batch_small_is_exact(lib):
    shapes = [(256, 256), (300, 512), (33, 96), (4097, 32)]
    members = [Member(F32, r, d, seed=100 + i) for i, (r, d) in enumerate(shapes)]
    with deterministic(lib):
        run_batch(lib, F32, members, list(range(len(members))), "det small batch")


def test_batch_mixed_members_are_exact(lib):
    """Segmented members, individual fallbacks, rows = 0, and two members adding into the same G (their tiles share
    one reduction item)."""
    members = [
        Member(BF16, 64 * 40, 768, seed=1, seg=(40, 617 * 768)),
        Member(BF16, 16 * 577, 768, seed=2, lead=40 * 768, seg=(577, 617 * 768)),
        Member(BF16, 2560, 3072, seed=3),
        Member(BF16, 1000, 192, seed=4, lead=1),
        Member(BF16, 9 * 40, 256, seed=5, seg=(40, 40 * 256 + 4)),
        Member(BF16, 500, 96, seed=6),
        Member(BF16, 0, 64, seed=7),
        Member(BF16, 8193, 320, seed=8, ldx=328),
    ]
    members.append(Member(BF16, 65, 320, seed=9, exps=members[-1].e))
    with deterministic(lib):
        grams = run_batch(lib, BF16, members, [0, 1, 2, 3, 4, 5, 6, 7, 7], "det mixed batch")
    assert torch.equal(grams[6]["buf"].m, grams[6]["g0"].float())


@pytest.mark.parametrize("rows,d", [(36928, 768), (4097, 3072), (2049, 32)])
def test_split_gram_is_exact(lib, rows, d):
    x, hi, lo, e = split_exact_x(rows, d, seed=rows + d, density=min(1.0, 150 / rows))
    planes = torch.empty(2 * rows * d, dtype=F32, device="cuda")
    _lib.check(lib.vlm_tf32_split(x.data_ptr(), rows, d, d, 0, 0, planes.data_ptr(), None))
    g0 = exact_g0(d, e, seed=d, shift=12)
    want, abs_terms = split_want(hi, lo, g0)
    assert_exact_case(abs_terms, e, g0, want, shift=12)
    g = new_g(d, g0, ldg=d + 4, lead=4)
    with deterministic(lib):
        for _ in range(2):
            _lib.check(lib.vlm_syrk_accum(planes.data_ptr(), _lib.VLM_TF32X2, rows, d, d, g.ptr, g.ld, None))
    torch.cuda.synchronize()
    assert_upper_equal(g.m, want, f"det split r{rows} d{d}")
    assert g.sentinels_intact()


def _exact_f64_gram(lib, fn, rows, d, dtype, seg=None, what=""):
    """fp64 G (i8x4 or DMMA kernel) twice into an exact G0, sentinels around G and X."""
    x, x64, e = exact_x(rows, d, dtype, seed=rows + d)
    if seg is None:
        xb, ldx, seg_rows, seg_stride = Padded(rows, d, d, dtype, fill=x), d, 0, 0
    else:
        seg_rows, seg_stride = seg
        xb, ldx = Segmented(x, seg_rows, d, seg_stride), d
    g0 = exact_g0(d, e, seed=d)
    want = g0 + 2 * (x64.T @ x64)
    g = Padded(d, d, d + 2, F64, fill=g0, lead=2, sentinel=-777.25)
    scratch = torch.empty(max(1, lib.vlm_syrk_i8x4_scratch_bytes(rows, d)), dtype=torch.uint8, device="cuda")
    with deterministic(lib):
        for _ in range(2):
            if fn == "i8x4":
                _lib.check(lib.vlm_syrk_accum_i8x4(xb.ptr, CODE[dtype], rows, d, ldx, seg_rows, seg_stride,
                                                   scratch.data_ptr(), scratch.numel(), g.ptr, g.ld, None))
            else:
                _lib.check(lib.vlm_syrk_accum_f64(xb.ptr, CODE[dtype], rows, d, ldx, seg_rows, seg_stride, g.ptr, g.ld,
                                                  None))
    torch.cuda.synchronize()
    upper = torch.ones(d, d, dtype=torch.bool, device="cuda").triu()
    bad = (g.m != want) & upper
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} upper entries differ"
    assert g.sentinels_intact(), what
    assert xb.sentinels_intact(), what


@pytest.mark.parametrize("rows,d,dtype,seg", [(36928, 768, F32, None), (2560, 3072, F32, None), (300, 128, BF16, None),
                                              (64 * 577, 768, F16, (577, 617 * 768))],
                         ids=["phase-split-36928x768", "phases-chained-2560x3072", "small-bf16", "rowslice-f16"])
def test_int8x4_is_exact(lib, rows, d, dtype, seg):
    _exact_f64_gram(lib, "i8x4", rows, d, dtype, seg, f"det i8x4 {rows}x{d}")


@pytest.mark.parametrize("rows,d,dtype,seg", [(2560, 768, F32, None), (36928, 200, BF16, None),
                                              (64 * 40, 768, F32, (40, 617 * 768))],
                         ids=["2560x768", "unaligned-width", "rowslice"])
def test_fp64_is_exact(lib, rows, d, dtype, seg):
    _exact_f64_gram(lib, "f64", rows, d, dtype, seg, f"det f64 {rows}x{d}")


# ---- 2. determinism and accuracy on real-valued data ----------------------------------------------------------------

def _real(shape, dtype, seed, positive):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(*shape, generator=g, device="cuda")
    return (x.abs() if positive else x).to(dtype)


def _runs(call, g0, lib, n=4):
    """call(g) into fresh copies of g0, n times, runs 1 and 3 under a matmul loop on another stream; returns the Gs."""
    other = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device="cuda", dtype=torch.bfloat16)
    out = []
    for i in range(n):
        g = g0.clone()
        torch.cuda.synchronize()
        if i % 2:
            with torch.cuda.stream(other):
                for _ in range(30):
                    a = (a @ a).clamp_(-1, 1)
        with deterministic(lib):
            _lib.check(call(g))
        torch.cuda.synchronize()
        out.append(g)
    return out


def _rel_upper(g, ref):
    upper = torch.ones_like(ref, dtype=torch.bool).triu()
    return ((g.double() - ref)[upper].norm() / ref[upper].norm()).item()


TOL = {F32: 1e-3, BF16: 1e-4, F16: 1e-4}   # test_gpu_gram.py's bounds for the default mode
SHAPES = [(36928, 3072), (36928, 768), (2560, 768), (2560, 3072)]


@pytest.mark.parametrize("positive", [False, True], ids=["normal", "absnormal"])
@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("rows,d", SHAPES, ids=[f"{r}x{d}" for r, d in SHAPES])
def test_single_launch_is_deterministic(lib, rows, d, dtype, positive):
    x = _real((rows, d), dtype, seed=rows + d, positive=positive)
    g0 = _real((d, d), F32, seed=d, positive=False)
    gs = _runs(lambda g: lib.vlm_syrk_accum(x.data_ptr(), CODE[dtype], rows, d, d, g.data_ptr(), d, None), g0, lib)
    for i, g in enumerate(gs[1:], 1):
        assert same_bits(g, gs[0]), f"run {i} differs from run 0 in {int((g != gs[0]).sum())} entries"
    xd = x.double()
    assert _rel_upper(gs[0], g0.double() + xd.T @ xd) < TOL[dtype]


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
def test_row_slice_is_deterministic(lib, dtype):
    h = _real((64, 617, 768), dtype, seed=3, positive=True)
    x = h[:, 40:]
    g0 = torch.zeros(768, 768, device="cuda")
    gs = _runs(lambda g: lib.vlm_syrk_accum_strided(x.data_ptr(), CODE[dtype], 64 * 577, 768, 768, 577, 617 * 768,
                                                    g.data_ptr(), 768, None), g0, lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    xd = x.reshape(-1, 768).double()
    assert _rel_upper(gs[0], xd.T @ xd) < TOL[dtype]


def test_grouped_text_tower_is_deterministic(lib):
    shapes = [(2560, 768)] * 36 + [(2560, 3072)] * 12
    xs = [_real(s, F32, seed=i, positive=i % 2 == 1) for i, s in enumerate(shapes)]
    arena0 = torch.zeros(sum(d * d for _, d in shapes), device="cuda")

    def call(arena):
        probs = (_lib.SyrkProblem * len(shapes))()
        off = 0
        for q, x, (r, d) in zip(probs, xs, shapes):
            q.x, q.rows, q.ldx, q.d, q.g, q.ldg = x.data_ptr(), r, d, d, arena.data_ptr() + 4 * off, d
            off += d * d
        return lib.vlm_syrk_accum_batch(probs, len(shapes), _lib.VLM_F32, None)

    gs = _runs(call, arena0, lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    off = 0
    for i, (x, (_, d)) in enumerate(zip(xs, shapes)):
        if i % 11 == 0:
            xd = x.double()
            assert _rel_upper(gs[0][off:off + d * d].view(d, d), xd.T @ xd) < TOL[F32], i
        off += d * d


@pytest.mark.parametrize("rows,d", [(36928, 768), (2560, 3072)])
def test_int8x4_is_deterministic(lib, rows, d):
    x = _real((rows, d), F32, seed=rows, positive=True) * torch.linspace(0.02, 25.0, d, device="cuda")
    g0 = torch.zeros(d, d, dtype=F64, device="cuda")
    scratch = torch.empty(lib.vlm_syrk_i8x4_scratch_bytes(rows, d), dtype=torch.uint8, device="cuda")
    gs = _runs(lambda g: lib.vlm_syrk_accum_i8x4(x.data_ptr(), _lib.VLM_F32, rows, d, d, 0, 0, scratch.data_ptr(),
                                                 scratch.numel(), g.data_ptr(), d, None), g0, lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    xd = x.double()
    assert _rel_upper(gs[0], xd.T @ xd) < 1e-8


def test_fp64_is_deterministic(lib):
    rows, d = 2560, 768
    x = _real((rows, d), F32, seed=9, positive=False)
    g0 = torch.zeros(d, d, dtype=F64, device="cuda")
    gs = _runs(lambda g: lib.vlm_syrk_accum_f64(x.data_ptr(), _lib.VLM_F32, rows, d, d, 0, 0, g.data_ptr(), d, None),
               g0, lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    xd = x.double()
    assert _rel_upper(gs[0], xd.T @ xd) < 1e-13


def test_cuda_core_kernel_is_deterministic(lib):
    rows, d = 36928, 200
    x = _real((rows, d), F32, seed=10, positive=True)
    g0 = torch.zeros(d, d, device="cuda")
    gs = _runs(lambda g: lib.vlm_syrk_accum(x.data_ptr(), _lib.VLM_F32, rows, d, d, g.data_ptr(), d, None), g0, lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    xd = x.double()
    assert _rel_upper(gs[0], xd.T @ xd) < 1e-5


def test_split_is_deterministic(lib):
    rows, d = 36928, 768
    x = _real((rows, d), F32, seed=12, positive=True)
    planes = torch.empty(2 * rows * d, device="cuda")
    _lib.check(lib.vlm_tf32_split(x.data_ptr(), rows, d, d, 0, 0, planes.data_ptr(), None))
    g0 = torch.zeros(d, d, device="cuda")
    gs = _runs(lambda g: lib.vlm_syrk_accum(planes.data_ptr(), _lib.VLM_TF32X2, rows, d, d, g.data_ptr(), d, None), g0,
               lib)
    assert all(same_bits(g, gs[0]) for g in gs[1:])
    xd = x.double()
    assert _rel_upper(gs[0], xd.T @ xd) < 5e-5


# ---- 3. end to end: GramCache, Gram files, RegMean ------------------------------------------------------------------

@pytest.fixture(scope="module")
def recorded():
    """The tiny synthetic model, its state dict, and every hooked activation of three forwards, in hook order."""
    cfg = vlm.vlmo_config("tiny", num_layers=12)
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    acts, handles = [], []
    for name, mod in vlm.gram.select_hooked_modules(model, use_moe=True):
        handles.append(mod.register_forward_hook(
            lambda m, i, o, n=name: acts.append((n, (i[0] if isinstance(i, tuple) else i).detach().clone()))))
    with torch.no_grad():
        for seed in (3, 4, 5):      # 3 x 8 x 40 = 960 text rows: the summed text Grams are non-singular at alpha = 1
            model(vlm.synthetic_batch(8, cfg, seed=seed, device="cuda"))
    for h in handles:
        h.remove()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    return model, cfg, sd, acts


MCFG = dict(vlffn_start_layer_index=10, only_activate_used_experts=False, merge_ratio=0.5, sum_lambda=0.75,
            scaling_for_non_diag=1.0, loss_names={"irtr": 1.0, "vqa": 0, "nlvr2": 0})


def _replay(acts, **kw):
    cache = vlm.GramCache(deterministic=True, **kw)
    for name, x in acts:
        cache.accumulate(name, x)
    cache.flush()
    return cache


@pytest.mark.parametrize("defer", [0, 1 << 20], ids=["immediate", "deferred"])
@pytest.mark.parametrize("precision", ["tf32", "tf32x3", "fp64", "int8x4"])
def test_replayed_calibration_is_bit_identical(recorded, precision, defer, tmp_path):
    _, _, sd, acts = recorded
    a, b = _replay(acts, precision=precision, defer_bytes=defer), _replay(acts, precision=precision, defer_bytes=defer)
    assert a.deterministic and sorted(a.buffers) == sorted(b.buffers)
    for n in a.buffers:
        assert same_bits(a.buffers[n], b.buffers[n]), n
    files = []
    for c, tag in ((a, "a"), (b, "b")):      # same file names: torch.save's zip archive records its own name
        (tmp_path / tag).mkdir()
        c.save(tmp_path / tag / "grams.pt")
        c.save_packed(tmp_path / tag / "grams.vlmgram")
        files.append(((tmp_path / tag / "grams.pt").read_bytes(), (tmp_path / tag / "grams.vlmgram").read_bytes()))
    assert files[0][0] == files[1][0] and files[0][1] == files[1][1]
    ra, rb = vlm.regmean(sd, MCFG, gram_matrices=a), vlm.regmean(sd, MCFG, gram_matrices=b)
    assert sorted(ra) == sorted(rb)
    for k in ra:   # float tensors bit for bit; the integer buffers of the state dict (position indices) by value
        assert (same_bits(ra[k], rb[k]) if ra[k].is_floating_point() else torch.equal(ra[k], rb[k])), k


def test_side_stream_cache_is_bit_identical(recorded):
    _, _, _, acts = recorded
    a, b = _replay(acts, side_stream=True), _replay(acts, side_stream=True)
    torch.cuda.synchronize()
    for n in a.buffers:
        assert same_bits(a.buffers[n], b.buffers[n]), n


def test_cache_gram_matrices_forwards_the_option(recorded):
    model, cfg, _, _ = recorded
    batches = [vlm.synthetic_batch(4, cfg, seed=5, device="cuda", pad=True)]
    cache = vlm.cache_gram_matrices(model, batches, deterministic=True)
    assert cache.deterministic and len(cache.live_names()) > 0


# ---- 4. flag handling ------------------------------------------------------------------------------------------------

def test_flag_follows_torch_and_is_restored(lib):
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        assert vlm.GramCache().deterministic is True
        assert vlm.GramCache(deterministic=False).deterministic is False
    finally:
        torch.use_deterministic_algorithms(prev)
    assert vlm.GramCache().deterministic is prev
    x = torch.randn(300, 256, device="cuda")
    for before in (0, 1):
        lib.vlm_set_deterministic(before)
        try:
            for det in (False, True):
                cache = vlm.GramCache(deterministic=det, defer_bytes=1 << 20)
                cache.accumulate("g", x)
                assert lib.vlm_get_deterministic() == before
                cache.flush()
                assert lib.vlm_get_deterministic() == before
        finally:
            lib.vlm_set_deterministic(0)
