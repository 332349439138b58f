"""The RegMean-grade kernels one by one, through the C ABI, against fp64 references.

RegMean inverts the summed Gram, so a small error in one tile of a Gram or of the right-hand side can decide whether
the merged weights stay within 1e-4 of the reference.  The end-to-end tests judge whole matrices by one relative
Frobenius norm, in which an error confined to a partial edge tile, a padded pitch or the diagonal of one tile
vanishes.  Here every entry is checked on its own:

* sentinels: every output (and every input) lives inside a larger allocation whose pad columns (ld > width), guard
  rows and lead-in elements are sentinels (sentinel_buffers.py): NaN around inputs, so that a stray read shows as a NaN
  in the result; a finite value, compared bit for bit, around outputs a kernel adds into, so that a stray write or a
  stray add shows.  Every address stays inside the allocation.
* element-wise bounds: a computed sum of n fp64 products, in any order, is within
  2 (n + 2) 2^-53 (|A| @ |B|)_ij of the exact one (the factor 2 also covers the fp64 reference itself).  A dropped,
  doubled or mis-scaled single term is an error of about (|A||B|)_ij / n, far above that.
* element-wise kernels (scale_G, widen-add) must be bit-exact: they do one rounded operation per step, the same ones
  torch does.
"""
import pytest
import torch

from sentinel_buffers import NAN, OUT_SENTINEL, Padded, Segmented
from vl_merging_b200 import _lib

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
F32, F64, BF16, F16 = torch.float32, torch.float64, torch.bfloat16, torch.float16
VLM_DTYPE = {F32: _lib.VLM_F32, BF16: _lib.VLM_BF16, F16: _lib.VLM_F16, F64: _lib.VLM_F64}
SHORT = {F32: "f32", F64: "f64", BF16: "bf16", F16: "f16"}


@pytest.fixture(scope="module")
def lib():
    return _lib.lib()


def _randn(*shape, seed, dtype=F64):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=F64).to(dtype).cuda()


def _sym(d, seed, dtype=F64):
    a = _randn(d, d, seed=seed)
    return (a + a.T + 4 * torch.eye(d, dtype=F64, device="cuda")).to(dtype)


def _check(rc):
    _lib.check(rc)
    torch.cuda.synchronize()


def _assert_within(got, ref, bound, mask=None, what=""):
    """|got - ref| <= bound entry by entry (NaN fails); mask: the entries that are checked."""
    ok = (got - ref).abs() <= bound
    if mask is not None:
        ok |= ~mask
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i, j = bad[0].tolist()
        ratio = ((got - ref).abs() / bound.clamp_min(1e-300))
        if mask is not None:
            ratio = ratio.masked_fill(~mask, 0)
        raise AssertionError(f"{what}: {bad.shape[0]} entries out of bound, first ({i}, {j}): got {got[i, j].item()!r}, "
                             f"ref {ref[i, j].item()!r}, bound {bound[i, j].item()!r}; worst |err|/bound "
                             f"{ratio.nan_to_num(float('inf')).max().item():.3g}")


def scaled_gram(g64, alpha):
    """scale_G of the reference: alpha * G off the diagonal, alpha * g + (1 - alpha) * g on it, each op rounded once."""
    out = g64 * alpha
    dg = torch.diagonal(g64)
    out.diagonal().copy_(dg * alpha + dg * (1.0 - alpha))
    return out


# ---- vlm_gram_scale_accum ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("alpha", [1.0, 0.9, 0.0, 0.37])
@pytest.mark.parametrize("d", [1, 7, 200, 768])
@pytest.mark.parametrize("gdt", [F32, F64], ids=SHORT.get)
def test_gram_scale_accum_is_bit_exact(lib, gdt, d, alpha, accumulate):
    g = Padded(d, d, d + 3, gdt, fill=_sym(d, seed=d, dtype=gdt))
    out0 = _randn(d, d, seed=d + 1)
    out = Padded(d, d, d + 5, F64, fill=out0, sentinel=OUT_SENTINEL)
    _check(lib.vlm_gram_scale_accum(g.ptr, VLM_DTYPE[gdt], d, g.ld, alpha, out.ptr, out.ld, accumulate, None))
    ref = scaled_gram(g.m.double(), alpha)
    if accumulate:
        ref = out0 + ref
    assert torch.equal(out.m, ref)
    assert out.sentinels_intact() and g.sentinels_intact()


# ---- vlm_widen_add -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rows,cols", [(1, 1), (7, 13), (200, 768), (1025, 3)])
def test_widen_add_is_bit_exact(lib, rows, cols):
    src = Padded(rows, cols, cols + 3, F32, fill=_randn(rows, cols, seed=rows, dtype=F32))
    dst0 = _randn(rows, cols, seed=cols)
    dst = Padded(rows, cols, cols + 1, F64, fill=dst0, sentinel=OUT_SENTINEL)
    _check(lib.vlm_widen_add(src.ptr, rows, cols, src.ld, dst.ptr, dst.ld, None))
    assert torch.equal(dst.m, dst0 + src.m.double())
    assert dst.sentinels_intact() and src.sentinels_intact()


# ---- vlm_regmean_rhs / vlm_regmean_rhs_diff ------------------------------------------------------------------------

def rhs_kernel_for(in_f, ldw, ldg, gdt, ldacc, ptrs):
    """The kernel regmean.cu selects (regmean_rhs_impl): the 128 x 128 cp.async pipeline needs in_f % 32 == 0, ldw % 4
    == 0, 16-byte G rows, an even ldacc and 16-byte aligned pointers; everything else takes the 64 x 64 kernel."""
    gelem = 8 if gdt == F64 else 4
    ok = in_f % 32 == 0 and ldw % 4 == 0 and ldg * gelem % 16 == 0 and ldacc % 2 == 0 and all(p % 16 == 0 for p in ptrs)
    return "pipelined" if ok else "fallback"


# id -> (out_f, in_f, G dtype, ldw, ldg, ldacc, acc lead-in, w_base lead-in): the lead-ins misalign by one element
RHS_CASES = {
    "pipelined-partialMN-nk5-f32": (200, 160, F32, 164, 168, 162, 0, 0),
    "pipelined-partialMN-nk5-f64": (200, 160, F64, 164, 162, 162, 0, 0),
    "pipelined-nk1-f32": (70, 32, F32, 36, 36, 34, 0, 0),
    "pipelined-nk2-f64": (130, 64, F64, 68, 66, 66, 0, 0),
    "pipelined-nk3-f32": (129, 96, F32, 96, 100, 98, 0, 0),
    "pipelined-real-768x3072-f32": (768, 3072, F32, 3076, 3076, 3074, 0, 0),
    "pipelined-real-2304x768-f64": (2304, 768, F64, 772, 770, 770, 0, 0),
    "fallback-width8-f64": (5, 8, F64, 9, 9, 9, 0, 0),
    "fallback-width100-f32": (130, 100, F32, 103, 101, 105, 0, 0),
    "fallback-width200-f64": (70, 200, F64, 203, 201, 201, 0, 0),
    "fallback-width200-f32": (200, 200, F32, 204, 204, 202, 0, 0),
    "fallback-ldw161-f32": (200, 160, F32, 161, 168, 162, 0, 0),
    "fallback-acc8Boff-f64": (200, 160, F64, 164, 162, 162, 1, 0),
    "fallback-wbase4Boff-f32": (200, 160, F32, 164, 168, 162, 0, 1),   # w aligned, w_base not: _diff only
}


@pytest.mark.parametrize("alpha", [1.0, 0.9])
@pytest.mark.parametrize("diff", [False, True], ids=["rhs", "rhs_diff"])
@pytest.mark.parametrize("case", list(RHS_CASES))
def test_regmean_rhs_matches_fp64_gemm(lib, case, diff, alpha):
    out_f, in_f, gdt, ldw, ldg, ldacc, acc_lead, wb_lead = RHS_CASES[case]
    if wb_lead and not diff:
        pytest.skip("w_base is only read by vlm_regmean_rhs_diff")
    seed = out_f * 7 + in_f
    w = Padded(out_f, in_f, ldw, F32, fill=_randn(out_f, in_f, seed=seed, dtype=F32))
    wb = Padded(out_f, in_f, ldw, F32, fill=w.m + 0.1 * _randn(out_f, in_f, seed=seed + 1, dtype=F32), lead=wb_lead)
    g = Padded(in_f, in_f, ldg, gdt, fill=_sym(in_f, seed=seed + 2, dtype=gdt))
    a = w.m.double() - wb.m.double() if diff else w.m.double()
    ghat = scaled_gram(g.m.double(), alpha)
    ref = a @ ghat
    absprod = a.abs() @ ghat.abs()
    acc0 = _randn(out_f, in_f, seed=seed + 3)
    for accumulate in (0, 1):
        # accumulate = 0 must not read acc: start from NaN there; accumulate = 1 adds onto a non-zero acc
        acc = Padded(out_f, in_f, ldacc, F64, fill=acc0 if accumulate else None, lead=acc_lead, sentinel=OUT_SENTINEL)
        if not accumulate:
            acc.m.fill_(NAN)
        ptrs = [w.ptr, g.ptr, acc.ptr] + ([wb.ptr] if diff else [])
        assert rhs_kernel_for(in_f, ldw, ldg, gdt, ldacc, ptrs) == case.split("-")[0]
        if diff:
            rc = lib.vlm_regmean_rhs_diff(w.ptr, wb.ptr, out_f, in_f, ldw, g.ptr, VLM_DTYPE[gdt], ldg, alpha, acc.ptr,
                                          acc.ld, accumulate, None)
        else:
            rc = lib.vlm_regmean_rhs(w.ptr, out_f, in_f, ldw, g.ptr, VLM_DTYPE[gdt], ldg, alpha, acc.ptr, acc.ld,
                                     accumulate, None)
        _check(rc)
        if accumulate:
            want, bound = acc0 + ref, 2 * (in_f + 2) * U * (absprod + acc0.abs())
        else:
            want, bound = ref, 2 * (in_f + 2) * U * absprod
        _assert_within(acc.m, want, bound, what=f"{case} accumulate={accumulate}")
        assert ((acc.m - want).norm() / want.norm()).item() < 1e-13   # and as a whole, in the norm regmean sees
        assert acc.sentinels_intact()
    assert w.sentinels_intact() and wb.sentinels_intact() and g.sentinels_intact()


# ---- vlm_spd_solve_right(_async) / vlm_lu_solve_right ---------------------------------------------------------------

def _spd(n, seed):
    """Q diag(lambda) Q^T with lambda in [1, 1e3], exactly symmetric."""
    q, _ = torch.linalg.qr(_randn(n, n, seed=seed))
    s = (q * torch.logspace(0, 3, n, dtype=F64, device="cuda")) @ q.T
    return (s + s.T) / 2


def _solve(lib, which, s_full, r_full):
    """X = R S^-1 through entry point `which` on pitched, sentinel-guarded copies; returns (rc, X, info words)."""
    in_f, out_f = s_full.shape[0], r_full.shape[0]
    s = Padded(in_f, in_f, in_f + 3, F64, fill=s_full)
    r = Padded(out_f, in_f, in_f + 5, F64, fill=r_full)
    info = torch.full((2,), -7, dtype=torch.int32, device="cuda")
    if which == "spd":
        rc = lib.vlm_spd_solve_right(s.ptr, in_f, s.ld, r.ptr, out_f, r.ld, None)
    elif which == "spd_async":
        rc = lib.vlm_spd_solve_right_async(s.ptr, in_f, s.ld, r.ptr, out_f, r.ld, info.data_ptr(), None)
    else:
        rc = lib.vlm_lu_solve_right(s.ptr, in_f, s.ld, r.ptr, out_f, r.ld, None)
    torch.cuda.synchronize()
    assert s.sentinels_intact() and r.sentinels_intact(), which
    return rc, r.m.clone(), info.tolist()


@pytest.mark.parametrize("out_f", [1, 13, 768])
@pytest.mark.parametrize("in_f", [8, 200, 768])
def test_solves_match_fp64_solve(lib, in_f, out_f):
    s_full = _spd(in_f, seed=in_f)
    r_full = _randn(out_f, in_f, seed=out_f)
    ref = torch.linalg.solve(s_full, r_full, left=False)
    for which in ("spd", "spd_async", "lu"):
        rc, x, info = _solve(lib, which, s_full, r_full)
        _lib.check(rc)
        if which == "spd_async":
            assert info == [0, 0]
        rel = ((x - ref).norm() / ref.norm()).item()
        resid = ((x @ s_full - r_full).norm() / (x.norm() * s_full.norm())).item()
        resid_r = ((x @ s_full - r_full).norm() / r_full.norm()).item()
        assert rel < 1e-11 and resid < 1e-13 and resid_r < 1e-10, (which, rel, resid, resid_r)


@pytest.mark.parametrize("in_f,k", [(8, 0), (200, 137), (768, 767)])
def test_solver_status_words(lib, in_f, k):
    """A negative pivot at k: potrf reports the leading minor k + 1; Cholesky fails, LU succeeds.  An exactly zero row
    and column make the matrix singular, which LU reports."""
    dg = torch.linspace(1, 10, in_f, dtype=F64, device="cuda")
    dg[k] = -1
    s_full = torch.diag(dg)
    r_full = _randn(13, in_f, seed=in_f)
    rc, _, info = _solve(lib, "spd_async", s_full, r_full)
    _lib.check(rc)
    assert info == [k + 1, 0]
    rc, _, _ = _solve(lib, "spd", s_full, r_full)
    assert rc == _lib.ERR_NOT_SPD
    rc, x, _ = _solve(lib, "lu", s_full, r_full)
    _lib.check(rc)
    ref = torch.linalg.solve(s_full, r_full, left=False)
    assert ((x - ref).norm() / ref.norm()).item() < 1e-14

    singular = _spd(in_f, seed=k)
    singular[k, :] = 0
    singular[:, k] = 0
    rc, _, _ = _solve(lib, "lu", singular, r_full)
    assert rc == _lib.ERR_NOT_SPD


# ---- vlm_syrk_accum_f64 --------------------------------------------------------------------------------------------

def f64_path_for(x_ptr, ldx, seg_stride, d, dtype):
    """The syrk_f64_kernel variant syrk_f64.cu selects: 16-byte cp.async chunks need x 16-byte aligned and ldx,
    seg_stride and d multiples of 16 bytes; otherwise every element is loaded on its own."""
    ev = 16 // torch.tensor([], dtype=dtype).element_size()
    return "vec" if x_ptr % 16 == 0 and ldx % ev == 0 and seg_stride % ev == 0 and d % ev == 0 else "scalar"


def _f64_gram_twice(lib, x_ptr, rows, d, ldx, seg_rows, seg_stride, dtype, x64, seed):
    """Two vlm_syrk_accum_f64 calls on the same X into a G that starts non-zero: upper triangle against
    G0 + 2 X^T X entry by entry, sentinels around G untouched."""
    g0 = _randn(d, d, seed=seed)
    g = Padded(d, d, d + 3, F64, fill=g0, sentinel=OUT_SENTINEL)
    for _ in range(2):
        _check(lib.vlm_syrk_accum_f64(x_ptr, VLM_DTYPE[dtype], rows, d, ldx, seg_rows, seg_stride, g.ptr, g.ld, None))
    # widened f32 / bf16 / f16 products are exact in fp64: only the 2 rows additions (and the one onto G0) round
    ref = g0 + 2 * (x64.T @ x64)
    bound = 2 * (2 * rows + 2) * U * (2 * (x64.abs().T @ x64.abs()) + g0.abs())
    upper = torch.ones(d, d, dtype=torch.bool, device="cuda").triu()
    _assert_within(g.m, ref, bound, mask=upper, what=f"syrk_f64 rows={rows} d={d}")
    assert g.sentinels_intact()   # below the diagonal is scratch by contract; outside the matrix is not


@pytest.mark.parametrize("rows", [1, 31, 32, 33, 257, 9000])
@pytest.mark.parametrize("d", [1, 100, 129, 200, 257])
@pytest.mark.parametrize("dtype", [F32, BF16, F16], ids=SHORT.get)
def test_syrk_f64_matches_fp64_gram(lib, dtype, d, rows):
    x = Padded(rows, d, d, dtype, fill=_randn(rows, d, seed=rows + d, dtype=dtype))   # NaN guard rows after X
    _f64_gram_twice(lib, x.ptr, rows, d, d, 0, 0, dtype, x.m.double(), seed=d)
    assert x.sentinels_intact()


# id -> (dtype, rows, d, ldx, lead-in elements): inputs that take the scalar-load kernel
F64_SCALAR_CASES = {
    "f32-start4Boff": (F32, 257, 128, 128, 1),
    "f32-ldx-d+1": (F32, 9000, 128, 129, 0),
    "bf16-d100": (BF16, 1000, 100, 100, 0),
    "f16-d200-ldx203": (F16, 577, 200, 203, 0),
}


@pytest.mark.parametrize("case", list(F64_SCALAR_CASES))
def test_syrk_f64_scalar_load_path(lib, case):
    dtype, rows, d, ldx, lead = F64_SCALAR_CASES[case]
    x = Padded(rows, d, ldx, dtype, fill=_randn(rows, d, seed=rows, dtype=dtype), lead=lead)
    assert f64_path_for(x.ptr, ldx, 0, d, dtype) == "scalar"
    _f64_gram_twice(lib, x.ptr, rows, d, ldx, 0, 0, dtype, x.m.double(), seed=rows)
    assert x.sentinels_intact()


# path -> (dtype, d, ldx, extra elements between segments): vec keeps every stride a multiple of 16 bytes; scalar is
# an f16 input whose seg_stride is odd
F64_SEG_LAYOUTS = {"vec": (F32, 128, 132, 8), "scalar": (F16, 96, 96, 3)}


@pytest.mark.parametrize("seg_rows,nseg", [(7, 50), (40, 30), (577, 16)])
@pytest.mark.parametrize("path", list(F64_SEG_LAYOUTS))
def test_syrk_f64_segmented_rows(lib, path, seg_rows, nseg):
    dtype, d, ldx, gap = F64_SEG_LAYOUTS[path]
    seg_stride = seg_rows * ldx + gap
    assert (seg_stride % 2 == 1) == (path == "scalar")
    rows = seg_rows * nseg
    x = Segmented(_randn(rows, d, seed=seg_rows, dtype=dtype), seg_rows, ldx, seg_stride)
    assert f64_path_for(x.ptr, ldx, seg_stride, d, dtype) == path
    _f64_gram_twice(lib, x.ptr, rows, d, ldx, seg_rows, seg_stride, dtype, x.rows.double(), seed=nseg)
    assert x.sentinels_intact()   # the input itself is untouched


# ---- vlm_syrk_accum_i8x4 -------------------------------------------------------------------------------------------

def _i8_input(rows, d, dtype, seed):
    """Random columns of scales e^-3 .. e^3, plus the columns where the pre-pass can go wrong: 0 all zero, 1 and 2 with
    a maximum of exactly 1.0 and 2^20 (2^15 for f16), 3 spanning 2^-20 .. 2^10, 4 f16 subnormals, 5 a maximum of
    2^-110, below the exponent clamp (zero in f16)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, d, generator=g, dtype=F64) * torch.exp(torch.rand(d, generator=g, dtype=F64) * 6 - 3)
    mid = rows // 2
    x[:, 0] = 0
    for c, top in ((1, 1.0), (2, 2.0 ** (15 if dtype == F16 else 20)), (5, 2.0 ** -110)):
        x[:, c] = (torch.rand(rows, generator=g, dtype=F64) * 2 - 1) * (0.75 * top)
        x[mid, c] = -top
    sign = torch.randint(0, 2, (rows,), generator=g).to(F64) * 2 - 1
    x[:, 3] = sign * 2.0 ** (torch.rand(rows, generator=g, dtype=F64) * 30 - 20)
    x[:, 4] = torch.randn(rows, generator=g, dtype=F64) * 2.0 ** -18
    return x.to(dtype).cuda()


def i8_bound(x64):
    """The error bound of one vlm_syrk_accum_i8x4 call, from the header's description of the kernel: column c is
    quantised with the step s_c = 2^(E_c - 26), E_c = the frexp exponent of its maximum clamped below at -100 (0 for
    a zero column); the three digit products with p + q >= 5 are dropped; the rest is fp64 additions."""
    rows = x64.shape[0]
    amax = x64.abs().amax(0)
    e = torch.where(amax > 0, torch.frexp(amax).exponent.clamp(min=-100), 0)
    s = torch.pow(2.0, (e - 26).to(F64))
    a = x64.abs()
    colsum = a.sum(0)
    return (s[None, :] / 2 * colsum[:, None] + s[:, None] / 2 * colsum[None, :]
            + rows * s[:, None] * s[None, :] * (0.25 + 2.0 ** 21) + 2 * rows * U * (a.T @ a))


def _i8_gram_twice(lib, x_ptr, rows, d, ldx, seg_rows, seg_stride, dtype, x64, seed):
    ldg = d + 2                                    # even: the epilogue's TMA needs 16-byte G rows
    g0 = _randn(d, d, seed=seed)
    g = Padded(d, d, ldg, F64, fill=g0, sentinel=OUT_SENTINEL)
    nbytes = lib.vlm_syrk_i8x4_scratch_bytes(rows, d)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        _check(lib.vlm_syrk_accum_i8x4(x_ptr, VLM_DTYPE[dtype], rows, d, ldx, seg_rows, seg_stride, scratch.data_ptr(),
                                       nbytes, g.ptr, g.ld, None))
    xtx = x64.T @ x64
    ref = g0 + 2 * xtx
    bound = 2 * i8_bound(x64) + 4 * U * (g0.abs() + 2 * (x64.abs().T @ x64.abs()))
    upper = torch.ones(d, d, dtype=torch.bool, device="cuda").triu()
    _assert_within(g.m, ref, bound, mask=upper, what=f"syrk_i8x4 rows={rows} d={d}")
    assert torch.equal(g.m[0], g0[0])   # column 0 is zero: all its digits are, so its Gram row gains exactly nothing
    assert g.sentinels_intact()


@pytest.mark.parametrize("rows", [1, 33, 4097, 20000])
@pytest.mark.parametrize("d", [128, 384, 640])
@pytest.mark.parametrize("dtype", [F32, F16, BF16], ids=SHORT.get)
def test_syrk_i8x4_within_its_error_bound(lib, dtype, d, rows):
    x = Padded(rows, d, d, dtype, fill=_i8_input(rows, d, dtype, seed=rows + d))
    _i8_gram_twice(lib, x.ptr, rows, d, d, 0, 0, dtype, x.m.double(), seed=d)
    assert x.sentinels_intact()


@pytest.mark.parametrize("dtype", [F32, BF16], ids=SHORT.get)
def test_syrk_i8x4_segmented_rows(lib, dtype):
    """The row slice h[:, 40:] of a (B, 617, d) activation: 577-row segments, read in place."""
    seg_rows, nseg, d = 577, 9, 384
    x = Segmented(_i8_input(seg_rows * nseg, d, dtype, seed=7), seg_rows, d, 617 * d, lead=40 * d)
    _i8_gram_twice(lib, x.ptr, seg_rows * nseg, d, d, seg_rows, 617 * d, dtype, x.rows.double(), seed=9)


# ---- the ids above name the kernels that actually run -----------------------------------------------------------

def test_selection_predicates_name_the_launched_kernels(lib):
    """rhs_kernel_for and f64_path_for mirror the library's selection; the profiler's kernel names confirm them."""
    from torch.profiler import ProfilerActivity, profile

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.key for e in prof.key_averages()]

    def rhs(ldw):
        w = Padded(64, 64, ldw, F32, fill=_randn(64, 64, seed=1, dtype=F32))
        g = Padded(64, 64, 64, F64, fill=_sym(64, seed=2))
        acc = Padded(64, 64, 64, F64)
        assert rhs_kernel_for(64, ldw, 64, F64, 64, [w.ptr, g.ptr, acc.ptr]) == ("pipelined" if ldw == 64 else "fallback")
        return kernels(lambda: _lib.check(lib.vlm_regmean_rhs(w.ptr, 64, 64, ldw, g.ptr, _lib.VLM_F64, 64, 0.9, acc.ptr,
                                                              64, 0, None)))

    names = rhs(64)
    assert any("regmean_rhs_pipelined_kernel" in n for n in names), names
    names = rhs(65)
    assert any("regmean_rhs_kernel" in n for n in names) and not any("pipelined" in n for n in names), names

    def syrk(ldx):
        x = Padded(64, 128, ldx, F32, fill=_randn(64, 128, seed=3, dtype=F32))
        g = Padded(128, 128, 128, F64, fill=torch.zeros(128, 128, dtype=F64, device="cuda"))
        assert f64_path_for(x.ptr, ldx, 0, 128, F32) == ("vec" if ldx == 128 else "scalar")
        return [n for n in kernels(lambda: _lib.check(lib.vlm_syrk_accum_f64(x.ptr, _lib.VLM_F32, 64, 128, ldx, 0, 0,
                                                                             g.ptr, 128, None)))
                if "syrk_f64_kernel" in n]

    for ldx, vec in ((128, True), (129, False)):
        names = syrk(ldx)
        # demangled "syrk_f64_kernel<float, true>" or mangled "...syrk_f64_kernelIfLb1EE..."
        assert len(names) == 1 and (("true>" in names[0] or "Lb1E" in names[0]) == vec), names
