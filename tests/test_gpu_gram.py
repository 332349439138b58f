"""GPU parity of kernel (a) through GramCache (forward-hook API -> C ABI) against the oracle
(oracle.hook_gram_input: the reference's fp64 X^T X).  Tolerance from BASELINE.json: 1e-3 relative
Frobenius for fp32 activations (TF32 tensor cores, fp32 accumulate).  TMA rounds fp32 to TF32 on load, so the
error is unbiased rounding noise: <= 1e-3 on a handful of rows, ~3e-5 at calibration sizes (asserted below at
1e-4); bf16/f16 activations are exact on the tensor cores, what is left is the fp32 accumulation: 1e-4."""
import numpy as np
import pytest
import torch
import torch.nn as nn

import oracle
import vl_merging_b200 as vlm

pytestmark = pytest.mark.gpu
TOL = {torch.float32: 1e-3, torch.bfloat16: 1e-4, torch.float16: 1e-4}


def rel_fro(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _x(shape, dtype, seed, positive=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*shape, generator=g)
    if positive:
        x = x.abs() + 0.1  # post-GELU-like: non-zero mean
    return x.to(dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape,positive", [((4, 40, 768), False), ((3, 577, 768), True), ((2, 197, 3072), True),
                                            ((1, 1, 64), False), ((5, 7, 200), False), ((2, 33, 1000), True),
                                            ((1, 1000, 768), False), ((1, 1000, 768), True)])
def test_hook_matches_oracle(dtype, shape, positive):
    cache = vlm.GramCache()
    mod = nn.Identity()
    mod.module_name = "m"
    store = oracle.new_gram_store()
    for call in range(2):  # "+=" across calls
        x = _x(shape, dtype, seed=call, positive=positive)
        cache.hook_gram_input(mod, (x.cuda(),), None)      # tuple input, like nn.Module hooks deliver it
        oracle.hook_gram_input(store, "m", x.float().numpy())
    out = cache.state_dict()
    assert list(out.keys()) == ["m"]
    g = out["m"]
    assert g.dtype == torch.float64 and g.device.type == "cpu" and g.shape == (shape[-1], shape[-1])
    assert torch.equal(g, g.T)
    # up to a few thousand rows, the fp32 accumulation of exact 16-bit products stays 10x inside TOL
    assert rel_fro(g.numpy(), store["m"]) < (TOL[dtype] if dtype == torch.float32 else 1e-5)


def test_empty_ragged_and_unaligned_inputs():
    cache = vlm.GramCache()
    mod = nn.Identity()
    mod.module_name = "e"
    cache.hook_gram_input(mod, torch.zeros(0, 5, 128, device="cuda"), None)   # no rows: no-op
    assert cache.state_dict()["e"].abs().sum() == 0
    base = torch.randn(50, 264, device="cuda")
    views = [base[:, :256], base[:, 1:257], base[::2, 4:260]]   # padded pitch, misaligned start, strided rows
    store = oracle.new_gram_store()
    for i, v in enumerate(views):
        mod.module_name = f"v{i}"
        cache.hook_gram_input(mod, v, None)
        oracle.hook_gram_input(store, f"v{i}", v.cpu().numpy())
    out = cache.state_dict()
    for i in range(3):
        assert rel_fro(out[f"v{i}"].numpy(), store[f"v{i}"]) < 1e-3


def test_simt_and_tensor_core_paths_agree():
    x = _x((4, 577, 768), torch.float32, 3).cuda()
    a, b = vlm.GramCache(), vlm.GramCache(use_simt=True)
    a.accumulate("g", x)
    b.accumulate("g", x)
    ref = (x.double().reshape(-1, 768).T @ x.double().reshape(-1, 768)).cpu().numpy()
    assert rel_fro(b.state_dict()["g"].numpy(), ref) < 1e-5      # fp32 FMA kernel
    assert rel_fro(a.state_dict()["g"].numpy(), ref) < 1e-3      # TF32


@pytest.mark.parametrize("case", ["f32 start 4 bytes off", "f32 pitch d+1", "f32 d=200", "bf16 d=96"])
def test_syrk_accum_runs_the_cuda_core_kernel_outside_the_tensor_core_condition(case):
    """vlm_syrk_accum takes any alignment and width: an activation the CTA-pair kernel does not take runs, in one
    launch, on the CUDA-core kernel, bit for bit what vlm_syrk_accum_simt computes.  With at most 2048 rows that kernel
    has one row slice, so every output element is one atomic add onto zero: deterministic."""
    rows = 2000
    dtype, d, off, pitch = {"f32 start 4 bytes off": (torch.float32, 256, 1, 256),   # off, pitch in elements
                            "f32 pitch d+1": (torch.float32, 256, 0, 257),
                            "f32 d=200": (torch.float32, 200, 0, 200),
                            "bf16 d=96": (torch.bfloat16, 96, 0, 96)}[case]
    base = _x((rows * pitch + off,), torch.float32, 21).cuda().to(dtype)
    x = base[off:].view(rows, pitch)[:, :d]
    code = {torch.float32: vlm._lib.VLM_F32, torch.bfloat16: vlm._lib.VLM_BF16}[dtype]
    L = vlm._lib.lib()
    grams = []
    for fn in (L.vlm_syrk_accum, L.vlm_syrk_accum_simt):
        g = torch.zeros(d, d, device="cuda")
        before = vlm._lib.launch_count()
        rc = fn(x.data_ptr(), code, rows, d, pitch, g.data_ptr(), d, None)
        assert rc == 0, L.vlm_last_error()
        assert vlm._lib.launch_count() - before == 1
        grams.append(g)
    assert torch.equal(grams[0], grams[1])
    xd = x.double()
    assert rel_fro(grams[0].triu().cpu(), (xd.T @ xd).triu().cpu()) < 1e-5      # fp32 FMA


FULL_SIZE = [("tf32", torch.float32, 36928, 768), ("tf32", torch.float32, 36928, 3072), ("tf32", torch.bfloat16, 36928, 3072),
             ("tf32", torch.float16, 36928, 1024), ("tf32", torch.float32, 36928, 4096),
             ("tf32x3", torch.float32, 2560, 3072), ("tf32x3", torch.float32, 36928, 768), ("tf32x3", torch.float32, 36928, 3072),
             ("fp64", torch.float32, 2560, 768), ("fp64", torch.float32, 36928, 768), ("fp64", torch.float32, 36928, 3072),
             ("int8x4", torch.float32, 2560, 3072)]


@pytest.mark.parametrize("precision,dtype,rows,d", FULL_SIZE,
                         ids=[f"{p}-{str(t)[6:]}-{r}x{d}" for p, t, r, d in FULL_SIZE])
def test_full_size_properties(precision, dtype, rows, d):
    """BASELINE sizes (64 images x 577 tokens, 64 captions x 40 tokens) in the default mode and the RegMean-grade
    modes: fp64 torch Gram as checker + symmetry + trace identity."""
    x = (_x((rows, d), torch.float32, 11, positive=(d >= 3072)).cuda()).to(dtype)
    cache = vlm.GramCache(precision=precision)
    cache.accumulate("g", x.view(64, rows // 64, d))
    g = cache.gram("g")
    assert torch.equal(g, g.T)
    # tf32: 10x inside the BASELINE tolerance at calibration sizes, all dtypes
    row_tol, trace_tol = {"tf32": (1e-4, TOL[dtype]), "tf32x3": (5e-5, 5e-5), "fp64": (1e-13, 1e-13),
                          "int8x4": (1e-8, 1e-9)}[precision]
    xd = x.double()
    trace = (xd * xd).sum().item()
    assert abs(g.double().trace().item() - trace) / trace < trace_tol
    # 256 full rows of G in fp64 (the whole fp64 Gram of a 4096-wide activation would be 2 TFLOP)
    idx = torch.arange(0, d, max(1, d // 256), device="cuda")[:256]
    ref_rows = xd[:, idx].T @ xd
    err = (g.double()[idx] - ref_rows).norm() / ref_rows.norm()
    assert err.item() < row_tol


@pytest.mark.parametrize("dtype,d", [(torch.float32, 768), (torch.float32, 3072), (torch.float16, 3072), (torch.float32, 4096)])
def test_full_size_properties_int8x4(dtype, d):
    """The exact integer-tensor-core mode at BASELINE sizes: symmetry, the trace identity and 256 sampled rows against
    fp64 at 1e-8 (the RegMean-grade bar), and additivity over a split of the rows (each call picks its own column
    exponents, so the two results agree to the quantisation error, not bit for bit)."""
    rows = 36928
    x = (_x((rows, d), torch.float32, 12, positive=(d >= 3072)).cuda() * torch.linspace(0.02, 25.0, d, device="cuda")).to(dtype)
    cache = vlm.GramCache(precision="int8x4")
    cache.accumulate("g", x.view(64, 577, d))
    g = cache.gram("g")
    assert g.dtype == torch.float64 and torch.equal(g, g.T)
    xd = x.double()
    trace = (xd * xd).sum().item()
    assert abs(g.trace().item() - trace) / trace < 1e-9
    idx = torch.arange(0, d, max(1, d // 256), device="cuda")[:256]
    ref_rows = xd[:, idx].T @ xd
    assert ((g[idx] - ref_rows).norm() / ref_rows.norm()).item() < 1e-8
    halves = vlm.GramCache(precision="int8x4")
    halves.accumulate("g", x[: 32 * 577].view(32, 577, d))
    halves.accumulate("g", x[32 * 577:].view(32, 577, d))
    assert ((halves.gram("g") - g).norm() / g.norm()).item() < 1e-8


@pytest.mark.parametrize("precision", ["int8x4", "fp64", "tf32"])
def test_non_finite_activations_poison_their_row_and_column(precision):
    """An Inf or a NaN in an activation (fp16 overflow under autocast) makes row and column c of the reference's Gram
    non-finite (cache_gram_matrices.py:251-252).  Every mode must show it too — in particular the integer path, whose
    fixed-point digits could silently turn it into a finite number — and leave the other entries finite and right."""
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(8192, 256, device="cuda", generator=gen)
    x[17, 5] = float("inf")
    x[4000, 130] = float("nan")
    cache = vlm.GramCache(precision=precision)
    cache.accumulate("g", x)
    g = cache.gram("g").double()
    bad = torch.zeros(256, dtype=torch.bool, device="cuda")
    bad[[5, 130]] = True
    mask = bad[:, None] | bad[None, :]
    assert not torch.isfinite(g[mask]).any()
    assert torch.isfinite(g[~mask]).all()
    xd = x.double()
    ref = xd.T @ xd
    err = ((g[~mask] - ref[~mask]).norm() / ref[~mask].norm()).item()
    assert err < {"int8x4": 1e-8, "fp64": 1e-12, "tf32": 1e-3}[precision], err


def test_registration_and_reference_file_format(tmp_path):
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    cache = vlm.GramCache()
    names = cache.register(model, use_moe=True)
    assert len(names) == 116
    batch = vlm.synthetic_batch(2, cfg, seed=1, device="cuda")
    with torch.no_grad():
        model(batch)
    cache.remove_hooks()
    cache.save(tmp_path / "tmp.pth")
    loaded = torch.load(tmp_path / "tmp.pth", map_location="cpu", weights_only=False)
    assert len(loaded) == 96 and all(v.dtype == torch.float64 for v in loaded.values())
    assert loaded["transformer.blocks.0.attn.v"].shape == (192, 192)
    assert loaded["transformer.blocks.11.mlp.l.fc2"].shape == (768, 768)
    assert not any(".vl" in k for k in loaded)      # vl experts never run in IRTR calibration
    assert loaded["missing-key"] == 0.0             # still a defaultdict(float), like the reference's


def test_batched_launch_matches_individual_launches():
    """vlm_syrk_accum_batch through GramCache(defer_bytes=...): mixed shapes in one grid, incl. a column count that
    is not a whole number of 128-byte groups (issued individually) and two accumulations into the same Gram."""
    shapes = [(2560, 768), (2560, 3072), (40, 768), (333, 200), (1000, 1024), (2560, 768)]
    names = ["a", "b", "c", "odd", "e", "a"]
    xs = [_x(sh, torch.float32, 100 + i, positive=(i % 2 == 1)).cuda() for i, sh in enumerate(shapes)]
    now, later = vlm.GramCache(), vlm.GramCache(defer_bytes=64 << 20)
    for n, x in zip(names, xs):
        now.accumulate(n, x)
        later.accumulate(n, x)
    assert len(later._pending) == len(shapes)
    later.flush()
    assert not later._pending
    for n in set(names):
        a, b = now.gram(n).double(), later.gram(n).double()
        assert ((a - b).norm() / a.norm()).item() < 1e-6, n      # same arithmetic, different reduce-add order
    xd = torch.cat([xs[0], xs[5]]).double()
    ref = xd.T @ xd
    assert ((later.gram("a").double() - ref).norm() / ref.norm()).item() < 1e-3


def test_deferred_hooks_flush_after_each_forward():
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    a, b = vlm.GramCache(), vlm.GramCache(defer_bytes=1 << 40)   # defer everything
    a.register(model)
    b.register(model)
    with torch.no_grad():
        model(vlm.synthetic_batch(2, cfg, seed=3, device="cuda", pad=True))
    assert not b._pending                                      # flushed by the forward hook on the model
    ga, gb = a.state_dict(), b.state_dict()
    assert list(ga) == list(gb) and len(gb) == 96
    worst = max(((ga[k] - gb[k]).norm() / ga[k].norm()).item() for k in ga)
    assert worst < 1e-6, worst


def test_deferred_activation_modified_in_place_is_refused():
    """Deferral keeps a reference, not a copy: an in-place write before the flush would change the Gram silently.
    The version counter of the held tensor gives it away and flush() raises instead."""
    cache = vlm.GramCache(defer_bytes=1 << 30)
    x = torch.randn(4, 64, 128, device="cuda")
    cache.accumulate("a", x)
    cache.accumulate("b", torch.randn(256, 128, device="cuda"))
    x.mul_(2.0)                                   # e.g. an in-place residual / dropout after the hooked module
    with pytest.raises(RuntimeError, match="modified in place"):
        cache.flush()
    assert not cache._pending                     # nothing half-issued is left behind
    y = torch.randn(256, 128, device="cuda")
    cache.reset()
    cache.accumulate("a", y)                      # untouched activations still go through
    cache.flush()
    ref = y.double().T @ y.double()
    assert ((cache.gram("a").double() - ref).norm() / ref.norm()).item() < 1e-3


@pytest.mark.parametrize("precision", ["tf32x3", "fp64", "int8x4"])
def test_precision_modes_match_the_fp64_hook(precision):
    """The RegMean-grade Gram modes on the shapes of the hook path: 3-D inputs, a row slice of a (B, N, D) activation,
    bf16 inputs, an odd width (tf32x3: CUDA-core fallback; fp64: partial 128-column tiles, still on the cp.async path
    since 200 fp32 columns make 16-byte rows), immediate and grouped."""
    gen = torch.Generator(device="cuda").manual_seed(4)
    joint = torch.randn(6, 617, 256, device="cuda", generator=gen)
    joint64 = torch.randn(64, 617, 256, device="cuda", generator=gen) - 0.3     # big enough for the int8 path
    xs = {"plain": torch.randn(3, 577, 256, device="cuda", generator=gen), "slice": joint[:, 40:],
          "big": torch.randn(64, 577, 256, device="cuda", generator=gen) * torch.linspace(0.01, 30, 256, device="cuda"),
          "bigslice": joint64[:, 40:],
          "big_f16": (torch.randn(64, 577, 256, device="cuda", generator=gen) * torch.linspace(0.01, 30, 256, device="cuda")).half(),
          "bigslice_bf16": joint64.bfloat16()[:, 40:],         # int8x4 takes 16-bit activations too (widened exactly)
          "text": joint[:, :40], "bf16": torch.randn(1000, 128, device="cuda", generator=gen).bfloat16(),
          "odd": torch.randn(333, 200, device="cuda", generator=gen)}
    joint768 = torch.randn(4, 617, 768, device="cuda", generator=gen)
    xs.update({"d800": torch.rand(333, 800, device="cuda", generator=gen) + 0.25,    # a partial last 128-column block
               "tile": torch.randn(64, 128, device="cuda", generator=gen),
               "ragged": torch.randn(1000, 768, device="cuda", generator=gen),
               "slice768": joint768[:, 40:]})
    tol = {"fp64": 1e-13, "int8x4": 1e-7, "tf32x3": 5e-6}[precision]
    for defer in (0, 1 << 30):
        if precision != "tf32x3" and defer:
            continue
        cache = vlm.GramCache(precision=precision, defer_bytes=defer)
        for name, x in xs.items():
            cache.accumulate(name, x)
            cache.accumulate(name, x)
        cache.flush()
        for name, x in xs.items():
            x64 = x.double().reshape(-1, x.shape[-1])
            ref = 2 * (x64.T @ x64)
            g = cache.gram(name)
            assert g.dtype == (torch.float32 if precision == "tf32x3" else torch.float64)
            err = ((g.double() - ref).norm() / ref.norm()).item()
            if precision == "tf32x3" and name in ("bf16", "big", "bigslice", "big_f16", "bigslice_bf16"):
                tol_here = 5e-5      # what is left there is the tensor core's truncating fp32 accumulation (rows x 2^-25)
            elif precision == "tf32x3" and name in ("d800", "tile", "ragged", "slice768"):
                tol_here = 2e-6      # up to ~2300 rows the truncation stays this small
            else:
                tol_here = tol
            assert err < tol_here, (precision, defer, name, err)
            assert torch.equal(g, g.T)


@pytest.mark.parametrize("defer", [0, 1 << 40])
def test_side_stream_mode_matches_in_stream_launches(defer):
    """GramCache(side_stream=True): launches on a second stream, joined by flush() after every forward; the
    activations are freed by the forward long before the join, so this also exercises the keep-alive list."""
    cfg = vlm.vlmo_config("tiny")
    model = vlm.init_synthetic_(vlm.VLMo(cfg).eval(), seed=1).cuda()
    a, b = vlm.GramCache(), vlm.GramCache(defer_bytes=defer, side_stream=True)
    a.register(model)
    b.register(model)
    with torch.no_grad():
        for seed in (3, 4, 5):
            model(vlm.synthetic_batch(3, cfg, seed=seed, device="cuda", pad=True))
            model.infer(vlm.synthetic_batch(2, cfg, seed=seed + 10, device="cuda"))   # not model.__call__: no auto flush
            torch.empty(64 << 20, device="cuda").fill_(float("nan"))                   # churn the allocator
    assert not b._pending or defer
    ga, gb = a.state_dict(), b.state_dict()                     # state_dict() flushes and joins
    assert not b._side_keep and not b._pending
    assert list(ga) == list(gb)
    worst = max(((ga[k] - gb[k]).norm() / ga[k].norm()).item() for k in ga)
    assert worst < 1e-6, worst
    b.set_side_stream(False)
    assert b._side is None


def test_randomised_shape_sweep():
    """Seeded sweep over ragged shapes and dtypes: whole and partial 128-column blocks, row counts around the
    pipeline chunk (32 / 64 rows), widths that take the CTA-pair kernel (whole 128-byte groups) and widths that
    take the CUDA-core kernel, pitched inputs.  Checker: the reference hook's fp64 arithmetic in torch."""
    rng = np.random.default_rng(20261017)
    dtypes = [torch.float32, torch.bfloat16, torch.float16]
    for case in range(36):
        dtype = dtypes[case % 3]
        d = int(rng.choice([8, 32, 64, 96, 100, 128, 160, 200, 256, 264, 320, 512, 520, 768, 1000, 1024]))
        rows = int(rng.choice([1, 7, 31, 32, 33, 63, 64, 65, 127, 500, 1023, 4097, 9000]))
        pitch = d + int(rng.choice([0, 0, 8, 64]))
        base = _x((rows, pitch), torch.float32, 1000 + case, positive=bool(case % 2)).cuda().to(dtype)
        x = base[:, :d]
        cache = vlm.GramCache()
        cache.accumulate("g", x)
        cache.accumulate("g", x)
        xd = x.double()
        ref = 2 * (xd.T @ xd)
        got = cache.gram("g").double()
        err = ((got - ref).norm() / ref.norm()).item()
        assert torch.equal(got, got.T)
        assert err < TOL[dtype], (case, dtype, rows, d, pitch, err)
