"""The tensor-core Gram kernels (the CTA-pair kernel and its CUDA-core fallback) through the C ABI, bit for bit.

Every calibration Gram of the default precision comes from the CTA-pair kernel: fp32 activations rounded to TF32 by
TMA, bf16 / f16 ones as they are, fp32 accumulation in tensor memory, reduce-adds into an fp32 G.  With real-valued
data its error is a few 1e-4 of (|X|^T|X|)_ij, larger than the effect of one 32-row chunk dropped or doubled in one
piece of a stream-K schedule, of a reduce-add landing on the wrong slab, or of a truncating instead of a rounding
TMA conversion.  So these tests make the arithmetic exact and ask for equality:

* column c of X holds integers in [-7, 7] times 2^e_c: every value is exact in TF32, bf16 and f16 and every product
  is exact;
* entry (i, j) of the Gram is a sum of multiples of 2^(e_i + e_j).  While every partial sum stays below 2^21 of those
  units, fp32 holds it exactly in any order of addition, truncation included.  Each generator asserts that bound on
  |G0| + calls * (|X|^T|X|) and that every value lies on its grid, so that a later shape edit cannot make a case
  silently inexact.

Then every kernel and launch form must return exactly the fp64 G0 + 2 X^T X on the upper triangle (G starts from a
non-zero, integer-valued G0 and every call is made twice, so `+=` is checked too), and the finite sentinels around G
and the NaN sentinels around X must be intact (sentinel_buffers.py).  The ids name the kernel and the branch of the
work decomposition (build_pair_schedule in syrk_pair.cu) that runs.
"""
import pytest
import torch

from sentinel_buffers import OUT_SENTINEL, Padded, Segmented, same_bits
from vl_merging_b200 import _lib

pytestmark = pytest.mark.gpu

F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64
CODE = {F32: _lib.VLM_F32, BF16: _lib.VLM_BF16, F16: _lib.VLM_F16}
SHORT = {F32: "f32", BF16: "bf16", F16: "f16"}
ELEM = {F32: 4, BF16: 2, F16: 2}
LIMIT = 2 ** 21            # units of 2^(e_i + e_j) every partial sum stays below
B200_SMS = 148             # the schedule branches in the ids are those of a 148-SM B200 (74 CTA pairs)
SEG_CAP = 128              # chunks per accumulation (build_pair_schedule's seg_cap)
VLM_ERR_INVALID_ARG, VLM_ERR_ALIGNMENT, VLM_ERR_UNSUPPORTED = -1, -2, -3


@pytest.fixture(scope="module")
def lib():
    return _lib.lib()


def _check(rc):
    _lib.check(rc)
    torch.cuda.synchronize()


def chunk_rows(dtype):
    """Rows of X per pipeline stage (chunk_rows in syrk_pair.cu): 128 bytes of each column block."""
    return 128 // ELEM[dtype]


# ---- which kernel and which schedule branch runs ---------------------------------------------------------------------

def pair_supported(dtype, x_ptr, d, ldx, seg_stride, g_ptr, ldg):
    """syrk_pair_supported: the CTA-pair kernel takes whole 128-byte column groups, a 16-byte aligned X and G,
    16-byte row (and segment) pitches of X and ldg % 4 == 0; everything else runs on the CUDA-core kernel."""
    e = ELEM[dtype]
    return (d % (128 // e) == 0 and x_ptr % 16 == 0 and ldx * e % 16 == 0 and seg_stride * e % 16 == 0
            and g_ptr % 16 == 0 and ldg % 4 == 0)


def schedule_branch(kc, d, min_piece=0, nsm=B200_SMS):
    """The branches of build_pair_schedule for kc chunks and width d: T super-tiles over C = nsm / 2 clusters are
    dealt in whole rounds ("rounds"), or, when T < C, every tile is cut along K ("kcut"), or one or more rounds are
    followed by left-over tiles cut along K and interleaved into the last sweep ("round+leftover").  Left-over K pieces
    are at least 64 chunks long when kc >= 512 (or the grouped launch asks for it), else 8 ("min64" / "min8"); K
    ranges longer than seg_cap chunks are cut into segments that each end in a reduce-add ("segcap")."""
    c = nsm // 2
    nsb = (d + 255) // 256
    t = nsb * (nsb + 1) // 2
    rounds, rem = divmod(t, c)
    tags = ["rounds" if rem == 0 else "kcut" if rounds == 0 else "round+leftover"]
    if rem:
        tags.append(f"min{min_piece or (64 if kc >= 512 else 8)}")
    if kc > SEG_CAP:
        tags.append("segcap")
    return "-".join(tags)


def _nsm():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---- exact data -------------------------------------------------------------------------------------------------------

def col_exps(d, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi + 1, (d,), generator=g).to(F64).cuda()


EXPS = {F32: (-12, 12), BF16: (-12, 12), F16: (-14, 8)}   # f16: normal numbers only (subnormals: their own test)


def exact_x(rows, d, dtype, seed, exps=None):
    """X = V * 2^e, V integer in [-7, 7]: (x in dtype, the same values in fp64, e).  Asserts every value is exact in
    dtype."""
    e = col_exps(d, *EXPS[dtype], seed) if exps is None else exps
    gen = torch.Generator(device="cuda").manual_seed(seed)
    v = torch.randint(-7, 8, (rows, d), generator=gen, device="cuda", dtype=torch.int32).to(F64)
    x64 = v * torch.exp2(e)
    x = x64.to(dtype)
    assert torch.equal(x.double(), x64), "X is not exact in its element type"
    return x, x64, e


def exact_g0(d, e, seed, shift=0):
    """An integer-valued start G0: integers in [-64, 64] times 2^(e_i + e_j - shift)."""
    gen = torch.Generator(device="cuda").manual_seed(seed + 1_000_003)
    w = torch.randint(-64, 65, (d, d), generator=gen, device="cuda", dtype=torch.int32).to(F64)
    return w * torch.exp2(e[:, None] + e[None, :] - shift)


def assert_exact_case(abs_terms, e, g0, want, calls=2, shift=0):
    """The preconditions of an exact comparison: with unit_ij = 2^(e_i + e_j - shift), |G0| + calls * abs_terms (a
    bound on every partial sum, in any order) stays below 2^21 units, and G0 and the expected result lie on the grid."""
    unit = torch.exp2(e[:, None] + e[None, :] - shift)
    bound = (g0.abs() + calls * abs_terms) / unit
    assert bound.max().item() < LIMIT, f"case is not exact: partial sums reach {bound.max().item():.0f} units"
    for name, t in (("G0", g0), ("result", want)):
        q = t / unit
        assert torch.equal(q, q.round()), f"{name} is off its 2^(e_i+e_j) grid"


def assert_upper_equal(got, want, what):
    """got (fp32 G) equals want (fp64) exactly on the upper triangle."""
    d = want.shape[0]
    upper = torch.ones(d, d, dtype=torch.bool, device="cuda").triu()
    bad = (got.double() != want) & upper
    if bool(bad.any()):
        idx = bad.nonzero()
        i, j = idx[0].tolist()
        raise AssertionError(f"{what}: {idx.shape[0]} of {int(upper.sum())} upper entries differ; first ({i}, {j}): "
                             f"got {got[i, j].item()!r}, want {want[i, j].item()!r}; rows with a difference: "
                             f"{sorted(set(idx[:, 0].tolist()))[:8]}..., columns {sorted(set(idx[:, 1].tolist()))[:8]}...")


def new_g(d, g0, ldg=None, lead=0):
    return Padded(d, d, ldg or d, F32, fill=g0, lead=lead, sentinel=OUT_SENTINEL)


def gram_twice(call, x64, e, d, what, ldg=None, g_lead=0, seed=0):
    """call(g) twice into a G that starts at an exact G0; upper triangle == G0 + 2 X^T X, sentinels intact.  Returns
    the G buffer."""
    g0 = exact_g0(d, e, seed)
    want = g0 + 2 * (x64.T @ x64)
    assert_exact_case(x64.abs().T @ x64.abs(), e, g0, want)
    g = new_g(d, g0, ldg, g_lead)
    for _ in range(2):
        _check(call(g))
    assert_upper_equal(g.m, want, what)
    assert g.sentinels_intact(), f"{what}: a write or add outside G"
    return g


# ---- 1. single launch, vlm_syrk_accum ---------------------------------------------------------------------------------

# (dtype, rows, d, pitched): pitched = ldx > d, ldg = d + 4 and 16-byte lead-ins before X and G.  Widths with whole,
# partial (288 = 256 + 32, 416, 320 = 256 + 64) and nearly empty last super-tiles; rows around the chunk, the 128-chunk
# segment cap, and the calibration height 36928.
SINGLE = [
    (F32, 1, 32, False), (F32, 31, 96, True), (F32, 32, 160, False), (F32, 33, 288, True), (F32, 2560, 416, False),
    (F32, 4097, 768, True), (F32, 36928, 768, False), (F32, 2560, 1024, True), (F32, 36928, 3072, False),
    (F32, 4097, 3072, True), (F32, 2560, 4096, False), (F32, 33, 4096, True),
    (BF16, 1, 64, False), (BF16, 63, 192, True), (BF16, 64, 320, False), (BF16, 65, 768, True),
    (BF16, 2560, 3072, False), (BF16, 8193, 768, True), (BF16, 36928, 3072, True),
    (F16, 1, 64, True), (F16, 65, 192, False), (F16, 2560, 320, True), (F16, 8193, 3072, False),
    (F16, 36928, 768, False),
]


def _single_id(case):
    dtype, rows, d, pitched = case
    kc = -(-rows // chunk_rows(dtype))
    return f"pair-{SHORT[dtype]}-r{rows}-d{d}-{schedule_branch(kc, d)}-{'pitched' if pitched else 'dense'}"


def test_single_cases_reach_every_schedule_branch():
    tags = set()
    for c in SINGLE:
        dtype, rows, d, _ = c
        tags.update(schedule_branch(-(-rows // chunk_rows(dtype)), d).split("-"))
    assert {"kcut", "round+leftover", "min8", "min64", "segcap"} <= tags, tags


@pytest.mark.parametrize("case", SINGLE, ids=_single_id)
def test_single_launch_is_exact(lib, case):
    dtype, rows, d, pitched = case
    assert _nsm() == B200_SMS, "the ids name the schedule branches of a 148-SM B200"
    e = ELEM[dtype]
    ldx, ldg, lead_x, lead_g = (d + 16 // e, d + 4, 16 // e, 4) if pitched else (d, d, 0, 0)
    x, x64, ex = exact_x(rows, d, dtype, seed=rows * 7 + d)
    xb = Padded(rows, d, ldx, dtype, fill=x, lead=lead_x)
    g = gram_twice(lambda g: lib.vlm_syrk_accum(xb.ptr, CODE[dtype], rows, d, ldx, g.ptr, g.ld, None), x64, ex, d,
                   _single_id(case), ldg=ldg, g_lead=lead_g, seed=rows + d)
    assert pair_supported(dtype, xb.ptr, d, ldx, 0, g.ptr, g.ld)
    assert xb.sentinels_intact()


def test_f16_subnormal_columns_are_exact(lib):
    """f16 subnormals (|x| < 2^-14: exponents -24 .. -15 here, next to normal columns) on the kind::f16 tensor path:
    their products (down to 2^-48) are normal fp32 numbers, and the Gram must hold them exactly."""
    rows, d = 2560, 320
    ex = torch.cat([col_exps(d // 2, -24, -15, 5), col_exps(d - d // 2, -14, 4, 6)])
    x, x64, ex = exact_x(rows, d, F16, seed=11, exps=ex)
    assert bool((x.abs() < 2.0 ** -14).logical_and(x != 0).any())
    xb = Padded(rows, d, d, F16, fill=x)
    gram_twice(lambda g: lib.vlm_syrk_accum(xb.ptr, _lib.VLM_F16, rows, d, d, g.ptr, g.ld, None), x64, ex, d,
               "f16 subnormals", seed=3)


# ---- 2. the CUDA-core fallback -----------------------------------------------------------------------------------------

# id -> (dtype, rows, d, ldx, X lead-in elements, ldg)
SIMT = {
    "simt-f32-start4Boff": (F32, 2560, 128, 128, 1, 128),
    "simt-f32-ldx-odd": (F32, 577, 96, 97, 0, 96),
    "simt-f32-d200": (F32, 1000, 200, 200, 0, 200),
    "simt-bf16-d96": (BF16, 1000, 96, 96, 0, 96),
    "simt-f32-ldg-odd": (F32, 300, 256, 256, 0, 257),
}


@pytest.mark.parametrize("case", list(SIMT))
def test_cuda_core_fallback_is_exact(lib, case):
    dtype, rows, d, ldx, lead, ldg = SIMT[case]
    x, x64, ex = exact_x(rows, d, dtype, seed=rows + d)
    xb = Padded(rows, d, ldx, dtype, fill=x, lead=lead)
    results = []
    for fn in (lib.vlm_syrk_accum, lib.vlm_syrk_accum_simt):
        g = gram_twice(lambda g: fn(xb.ptr, CODE[dtype], rows, d, ldx, g.ptr, g.ld, None), x64, ex, d,
                       f"{case} {fn.__name__}", ldg=ldg, seed=d)
        assert not pair_supported(dtype, xb.ptr, d, ldx, 0, g.ptr, g.ld)
        results.append(g.m.triu())
    assert torch.equal(*results)
    assert xb.sentinels_intact()


# ---- 3. segmented rows, vlm_syrk_accum_strided ----------------------------------------------------------------------

# id -> (dtype, segments, rows per segment, d, ldx, seg_stride, lead-in elements); "pair4d" reads the segments
# through one 4-D tensor map, "perseg" (seg_stride * elem % 16 != 0) issues one vlm_syrk_accum per segment
STRIDED = {
    "pair4d-f32-text-40of617": (F32, 64, 40, 768, 768, 617 * 768, 0),
    "pair4d-f32-image-577of617": (F32, 64, 577, 768, 768, 617 * 768, 40 * 768),
    "pair4d-bf16-text-40of617": (BF16, 64, 40, 768, 768, 617 * 768, 0),
    "pair4d-bf16-image-577of617": (BF16, 64, 577, 768, 768, 617 * 768, 40 * 768),
    "pair4d-f32-5rows": (F32, 200, 5, 256, 260, 5 * 260 + 8, 0),
    "pair4d-bf16-5rows": (BF16, 150, 5, 192, 200, 5 * 200 + 16, 8),
    "pair4d-f32-wholechunks": (F32, 40, 64, 288, 288, 64 * 288 + 32, 0),
    "pair4d-bf16-wholechunks": (BF16, 30, 128, 192, 200, 128 * 200 + 16, 0),
    "perseg-f32-oddstride": (F32, 9, 40, 256, 256, 40 * 256 + 1, 0),
    "perseg-bf16-stride8B": (BF16, 9, 577, 384, 384, 577 * 384 + 4, 0),
}


@pytest.mark.parametrize("case", list(STRIDED))
def test_strided_segments_are_exact(lib, case):
    dtype, nseg, seg_rows, d, ldx, seg_stride, lead = STRIDED[case]
    rows = nseg * seg_rows
    x, x64, ex = exact_x(rows, d, dtype, seed=nseg * seg_rows + d)
    xs = Segmented(x, seg_rows, ldx, seg_stride, lead=lead)   # NaN in every gap between segments
    g = gram_twice(lambda g: lib.vlm_syrk_accum_strided(xs.ptr, CODE[dtype], rows, d, ldx, seg_rows, seg_stride,
                                                        g.ptr, g.ld, None), x64, ex, d, case, ldg=d + 4, seed=nseg)
    path = "pair4d" if pair_supported(dtype, xs.ptr, d, ldx, seg_stride, g.ptr, g.ld) else "perseg"
    assert path == case.split("-")[0]
    assert xs.sentinels_intact()


# ---- 4. grouped launch, vlm_syrk_accum_batch ------------------------------------------------------------------------

def batch_min_piece(problems, dtype, nsm=B200_SMS):
    """syrk_pair_batch_launch: K pieces of at least 64 chunks when the batch holds 8 such pieces per cluster."""
    bk = chunk_rows(dtype)
    work = sum((((d + 255) // 256) * ((d + 255) // 256 + 1) // 2) * (-(-rows // bk)) for rows, d in problems)
    return 64 if work >= 8 * 64 * (nsm // 2) else 0


class Member:
    """One problem of a grouped launch: X (plain or segmented, NaN-guarded) and the exact expected contribution."""

    def __init__(self, dtype, rows, d, seed, ldx=None, lead=0, seg=None, exps=None):
        self.rows, self.d = rows, d
        self.x, self.x64, self.e = exact_x(rows, d, dtype, seed=seed, exps=exps)
        self.ldx = ldx or d
        if seg is None:
            self.buf = Padded(rows, d, self.ldx, dtype, fill=self.x, lead=lead)
            self.seg_rows = self.seg_stride = 0
        else:
            self.seg_rows, self.seg_stride = seg
            self.buf = Segmented(self.x, self.seg_rows, self.ldx, self.seg_stride, lead=lead)


def run_batch(lib, dtype, members, targets, what):
    """members[i] adds into G targets[i] (an index: several members may share one G); every call twice."""
    grams = {}
    for t, m in zip(targets, members):
        if t not in grams:
            grams[t] = {"e": m.e, "d": m.d, "terms": 0, "abs": 0}
        grams[t]["terms"] = grams[t]["terms"] + m.x64.T @ m.x64
        grams[t]["abs"] = grams[t]["abs"] + m.x64.abs().T @ m.x64.abs()
    for t, gr in grams.items():
        gr["g0"] = exact_g0(gr["d"], gr["e"], seed=t)
        gr["want"] = gr["g0"] + 2 * gr["terms"]
        assert_exact_case(gr["abs"], gr["e"], gr["g0"], gr["want"])
        gr["buf"] = new_g(gr["d"], gr["g0"], ldg=gr["d"] + 4)
    probs = (_lib.SyrkProblem * len(members))()
    for q, t, m in zip(probs, targets, members):
        q.x, q.rows, q.ldx, q.d = m.buf.ptr, m.rows, m.ldx, m.d
        q.g, q.ldg = grams[t]["buf"].ptr, grams[t]["buf"].ld
        q.seg_rows, q.seg_stride = m.seg_rows, m.seg_stride
    for _ in range(2):
        _check(lib.vlm_syrk_accum_batch(probs, len(members), CODE[dtype], None))
    for t, gr in grams.items():
        assert_upper_equal(gr["buf"].m, gr["want"], f"{what}: G {t}")
        assert gr["buf"].sentinels_intact(), f"{what}: G {t}"
    for m in members:
        assert m.buf.sentinels_intact()
    return grams


def test_batch_text_tower_mix_is_exact(lib):
    """The text tower of one forward: 36 x [2560, 768] + 12 x [2560, 3072], the min_piece = 64 branch."""
    shapes = [(2560, 768)] * 36 + [(2560, 3072)] * 12
    assert batch_min_piece(shapes, F32) == 64
    members = [Member(F32, r, d, seed=i) for i, (r, d) in enumerate(shapes)]
    run_batch(lib, F32, members, list(range(len(members))), "text tower")


def test_batch_small_is_exact_and_matches_single_and_cuda_core_launches(lib):
    """A small batch (per-problem K pieces, the other branch): grouped, individual and CUDA-core Grams are all exact,
    hence bit-identical."""
    shapes = [(256, 256), (300, 512), (33, 96), (4097, 32)]
    assert batch_min_piece(shapes, F32) == 0
    members = [Member(F32, r, d, seed=100 + i) for i, (r, d) in enumerate(shapes)]
    grams = run_batch(lib, F32, members, list(range(len(members))), "small batch")
    for t, m in enumerate(members):
        for fn in (lib.vlm_syrk_accum, lib.vlm_syrk_accum_simt):
            g = new_g(m.d, grams[t]["g0"], ldg=m.d + 4)
            for _ in range(2):
                _check(fn(m.buf.ptr, _lib.VLM_F32, m.rows, m.d, m.ldx, g.ptr, g.ld, None))
            assert torch.equal(g.m.triu(), grams[t]["buf"].m.triu()), (t, fn.__name__)


def test_batch_mixed_members_are_exact(lib):
    """Segmented members, members that fall back to individual launches (misaligned start, odd segment stride, a
    width the pair kernel does not take), a rows = 0 member, two members adding into the same G, mixed widths."""
    members = [
        Member(BF16, 64 * 40, 768, seed=1, seg=(40, 617 * 768)),                       # text slice, 4-D map
        Member(BF16, 16 * 577, 768, seed=2, lead=40 * 768, seg=(577, 617 * 768)),       # image slice, 4-D map
        Member(BF16, 2560, 3072, seed=3),
        Member(BF16, 1000, 192, seed=4, lead=1),                                        # misaligned: CUDA cores
        Member(BF16, 9 * 40, 256, seed=5, seg=(40, 40 * 256 + 4)),                      # per-segment launches
        Member(BF16, 500, 96, seed=6),                                                  # d % 64 != 0: CUDA cores
        Member(BF16, 0, 64, seed=7),                                                    # nothing to add
        Member(BF16, 8193, 320, seed=8, ldx=328),
    ]
    members.append(Member(BF16, 65, 320, seed=9, exps=members[-1].e))                # same G as the one before
    targets = [0, 1, 2, 3, 4, 5, 6, 7, 7]
    grams = run_batch(lib, BF16, members, targets, "mixed batch")
    assert torch.equal(grams[6]["buf"].m, grams[6]["g0"].float())   # rows = 0: G untouched
    paths = [pair_supported(BF16, m.buf.ptr, m.d, m.ldx, m.seg_stride, grams[t]["buf"].ptr, grams[t]["buf"].ld)
             for t, m in zip(targets, members)]
    del paths[6]                                                                    # rows = 0: never launched
    assert paths == [True, True, True, False, False, False, True, True]


# ---- 5. TF32 rounding by TMA ----------------------------------------------------------------------------------------

def _bits(x):
    return x.view(torch.int32)


def rn_tf32(x):
    """Round fp32 to TF32, to nearest, ties to even (the sign-magnitude bit pattern rounds like the magnitude)."""
    b = _bits(x)
    return ((b + 0xFFF + ((b >> 13) & 1)) & ~0x1FFF).view(F32)


def rna_tf32(x):
    """cvt.rna.tf32.f32: round to nearest, ties away from zero."""
    return ((_bits(x) + 0x1000) & ~0x1FFF).view(F32)


def trunc_tf32(x):
    return (_bits(x) & ~0x1FFF).view(F32)


def f32_from_bits(b):
    """fp32 values from int64 bit patterns in [0, 2^32)."""
    return torch.where(b >= 1 << 31, b - (1 << 32), b).to(torch.int32).view(F32)


def full_mantissa_row(d, seed, lo=-20, hi=20):
    """One row of fp32 values with random 23-bit mantissas, signs and exponents in [lo, hi], no ties at the TF32
    rounding point."""
    g = torch.Generator().manual_seed(seed)
    mant = torch.randint(0, 1 << 23, (d,), generator=g, dtype=torch.int64)
    mant = torch.where((mant & 0x1FFF) == 0x1000, mant ^ 1, mant)
    exp = torch.randint(lo + 127, hi + 128, (d,), generator=g, dtype=torch.int64)
    sign = torch.randint(0, 2, (d,), generator=g, dtype=torch.int64)
    b = (sign << 31) | (exp << 23) | mant
    return f32_from_bits(b).reshape(1, d).cuda()


@pytest.mark.parametrize("d", [32, 288, 3072])
def test_tma_rounds_fp32_to_nearest_tf32(lib, d):
    """rows = 1: G = 2 outer(t) exactly (products of two TF32 values are exact in fp32), t = rn_tf32(x): pins the
    rounding conversion of the TFLOAT32 tensor map, which a truncating FLOAT32 map fails."""
    x = full_mantissa_row(d, seed=d)
    t = rn_tf32(x)
    assert bool((t != trunc_tf32(x)).any()) and torch.equal(t, rna_tf32(x))
    want = 2 * (t.double().T @ t.double())
    xb = Padded(1, d, d, F32, fill=x)
    g = new_g(d, torch.zeros(d, d, dtype=F64, device="cuda"))
    for _ in range(2):
        _check(lib.vlm_syrk_accum(xb.ptr, _lib.VLM_F32, 1, d, d, g.ptr, g.ld, None))
    assert_upper_equal(g.m, want, f"TF32 rounding d={d}")
    assert g.sentinels_intact() and xb.sentinels_intact()


def test_tma_tf32_tie_rule_is_recorded(lib, record_property, capsys):
    """Values exactly halfway between two TF32 numbers, with even and odd kept mantissas.  Column 0 is 1.0, so
    G[0, j] / 2 is the converted value of x_j.  The rule is reported, not asserted: each tie must only land on one of
    its two neighbours."""
    d = 64
    g = torch.Generator().manual_seed(9)
    mant = (torch.randint(0, 1 << 10, (d,), generator=g, dtype=torch.int64) << 13) | 0x1000
    exp = torch.randint(120, 135, (d,), generator=g, dtype=torch.int64)
    sign = torch.randint(0, 2, (d,), generator=g, dtype=torch.int64)
    b = (sign << 31) | (exp << 23) | mant
    b[0] = 0x3F800000
    x = f32_from_bits(b).reshape(1, d).cuda()
    xb = Padded(1, d, d, F32, fill=x)
    gb = new_g(d, torch.zeros(d, d, dtype=F64, device="cuda"))
    for _ in range(2):
        _check(lib.vlm_syrk_accum(xb.ptr, _lib.VLM_F32, 1, d, d, gb.ptr, gb.ld, None))
    conv = (gb.m[0:1, 1:] / 2)
    ties = x[:, 1:]
    even, away, down = rn_tf32(ties), rna_tf32(ties), trunc_tf32(ties)
    assert bool(((conv == away) | (conv == down)).all()), "a tie converted to neither neighbour"
    counts = {"ties": d - 1, "half-even": int((conv == even).sum()), "half-away": int((conv == away).sum()),
              "toward-zero": int((conv == down).sum())}
    record_property("tma_tf32_ties", counts)
    with capsys.disabled():
        print(f"\nTMA TFLOAT32 conversion of exact ties: {counts}")


# ---- 6. vlm_tf32_split ----------------------------------------------------------------------------------------------

def split_input(rows, d, seed):
    """fp32 values for the split: random mantissas, signs and exponents over most of the normal range (2^-100 ..
    2^127, so that lo = x - hi stays normal and nothing rounds past the largest float), one column of exact ties (even
    and odd kept mantissas) and one of exact ties of the low part."""
    g = torch.Generator().manual_seed(seed)
    mant = torch.randint(0, 1 << 23, (rows, d), generator=g, dtype=torch.int64)
    exp = torch.randint(27, 255, (rows, d), generator=g, dtype=torch.int64)
    sign = torch.randint(0, 2, (rows, d), generator=g, dtype=torch.int64)
    exp[:, :2] = exp[:, :2].clamp(max=253)
    mant[:, 0] = (mant[:, 0] & ~0x1FFF) | 0x1000                 # x itself halfway between two TF32 values
    mant[:, 1] = (mant[:, 1] & ~0x3) | 0x2                       # x - hi may be halfway between two TF32 values
    big = exp == 254
    mant = torch.where(big, mant & 0x7FE000, mant)               # the largest binade: nothing rounds up to infinity
    b = (sign << 31) | (exp << 23) | mant
    return f32_from_bits(b).cuda()


def split_planes_ref(x):
    hi = rna_tf32(x)
    return hi, rna_tf32(x - hi)


@pytest.mark.parametrize("layout", ["plain", "segmented"])
def test_tf32_split_matches_rna_emulation(lib, layout):
    rows, d = 1000, 96
    x = split_input(rows, d, seed=len(layout))
    if layout == "plain":
        xb = Padded(rows, d, d + 4, F32, fill=x, lead=4)
        seg_rows, seg_stride = 0, 0
    else:
        seg_rows, ldx = 40, d + 4
        seg_stride = seg_rows * ldx + 12
        xb = Segmented(x, seg_rows, ldx, seg_stride, lead=4)
    ldx = d + 4
    out = Padded(2 * rows, d, d, F32, sentinel=OUT_SENTINEL, guard=3)   # the two planes, then guard rows
    _check(lib.vlm_tf32_split(xb.ptr, rows, d, ldx, seg_rows, seg_stride, out.ptr, None))
    hi, lo = split_planes_ref(x)
    assert bool((_bits(x)[:, 0] & 0x1FFF == 0x1000).all()) and bool((lo != 0).any()) and bool((x < 0).any())
    assert same_bits(out.m[:rows], hi), "hi plane"
    assert same_bits(out.m[rows:], lo), "lo plane"
    assert out.sentinels_intact() and xb.sentinels_intact()


# ---- 7. split Gram, VLM_TF32X2 --------------------------------------------------------------------------------------

def split_exact_x(rows, d, seed, density):
    """Entries in {0, +-2^e_c, +-(1 + 2^-12) 2^e_c}: hi = +-2^e_c, lo = +-2^(e_c - 12).  Sparse enough that every
    column's squared sum stays far below 2^9, so that the Gram on the 2^(e_i + e_j - 12) grid stays below 2^21 units.
    Returns (x fp32, hi, lo in fp64, e)."""
    e = col_exps(d, -8, 8, seed)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.rand(rows, d, generator=gen, device="cuda", dtype=F64)
    sign = torch.where(torch.rand(rows, d, generator=gen, device="cuda", dtype=F64) < 0.5, -1.0, 1.0).to(F64)
    nz = u < density
    withlo = u < density / 2
    scale = torch.exp2(e)
    hi = torch.where(nz, sign, 0.0) * scale
    lo = torch.where(withlo, sign, 0.0) * scale * 2.0 ** -12
    x = (hi + lo).to(F32)
    assert torch.equal(x.double(), hi + lo)
    return x, hi, lo, e


def split_want(hi, lo, g0):
    terms = hi.T @ hi + hi.T @ lo + lo.T @ hi
    abs_terms = hi.abs().T @ hi.abs() + hi.abs().T @ lo.abs() + lo.abs().T @ hi.abs()
    return g0 + 2 * terms, abs_terms


def split_planes(lib, x, out_ptr):
    rows, d = x.shape
    _check(lib.vlm_tf32_split(x.data_ptr(), rows, d, d, 0, 0, out_ptr, None))


@pytest.mark.parametrize("rows,d", [(36928, 768), (4097, 3072), (2049, 32), (16, 96)])
def test_split_gram_is_exact(lib, rows, d):
    """G = G0 + 2 (hi'hi + hi'lo + lo'hi) exactly: both cross terms are there and lo'lo is not."""
    x, hi, lo, e = split_exact_x(rows, d, seed=rows + d, density=min(1.0, 150 / rows))
    assert bool((lo != 0).any())
    planes = torch.empty(2 * rows * d, dtype=F32, device="cuda")
    split_planes(lib, x, planes.data_ptr())
    assert torch.equal(planes[:rows * d].view(rows, d).double(), hi)
    assert torch.equal(planes[rows * d:].view(rows, d).double(), lo)
    g0 = exact_g0(d, e, seed=d, shift=12)
    want, abs_terms = split_want(hi, lo, g0)
    assert_exact_case(abs_terms, e, g0, want, shift=12)
    assert not torch.equal(want, g0 + 2 * (x.double().T @ x.double()))   # lo'lo matters on this data
    g = new_g(d, g0, ldg=d + 4, lead=4)
    for _ in range(2):
        _check(lib.vlm_syrk_accum(planes.data_ptr(), _lib.VLM_TF32X2, rows, d, d, g.ptr, g.ld, None))
    assert_upper_equal(g.m, want, f"split r{rows} d{d} {schedule_branch(-(-rows // 16), d)}")
    assert g.sentinels_intact()


def test_split_gram_grouped_is_exact(lib):
    """vlm_syrk_accum_batch with VLM_TF32X2: the planes of every problem back to back in one buffer."""
    shapes = [(2560, 768), (4097, 3072), (2049, 288), (2560, 768)]
    cases = [split_exact_x(r, d, seed=50 + i, density=min(1.0, 150 / r)) for i, (r, d) in enumerate(shapes)]
    planes = torch.empty(sum(2 * r * d for r, d in shapes), dtype=F32, device="cuda")
    probs = (_lib.SyrkProblem * len(shapes))()
    gs, wants = [], []
    off = 0
    for q, (r, d), (x, hi, lo, e) in zip(probs, shapes, cases):
        ptr = planes.data_ptr() + 4 * off
        split_planes(lib, x, ptr)
        off += 2 * r * d
        g0 = exact_g0(d, e, seed=r, shift=12)
        want, abs_terms = split_want(hi, lo, g0)
        assert_exact_case(abs_terms, e, g0, want, shift=12)
        g = new_g(d, g0, ldg=d + 4)
        q.x, q.rows, q.ldx, q.d, q.g, q.ldg, q.seg_rows, q.seg_stride = ptr, r, d, d, g.ptr, g.ld, 0, 0
        gs.append(g)
        wants.append(want)
    for _ in range(2):
        _check(lib.vlm_syrk_accum_batch(probs, len(shapes), _lib.VLM_TF32X2, None))
    for i, (g, want) in enumerate(zip(gs, wants)):
        assert_upper_equal(g.m, want, f"grouped split member {i}")
        assert g.sentinels_intact()


def test_split_gram_error_returns(lib):
    """The split planes exist only for the CTA-pair kernel: no silent CUDA-core fallback, G untouched."""
    rows = 64
    planes = torch.zeros(2 * rows * 64 + 4, dtype=F32, device="cuda")
    g0 = torch.ones(64, 64, dtype=F64, device="cuda")
    g = new_g(64, g0)
    p = planes.data_ptr()
    assert lib.vlm_syrk_accum(p, _lib.VLM_TF32X2, rows, 48, 48, g.ptr, g.ld, None) == VLM_ERR_UNSUPPORTED
    assert lib.vlm_syrk_accum(p + 4, _lib.VLM_TF32X2, rows, 64, 64, g.ptr, g.ld, None) == VLM_ERR_ALIGNMENT
    assert lib.vlm_syrk_accum_strided(p, _lib.VLM_TF32X2, rows, 64, 64, 32, 32 * 64, g.ptr, g.ld,
                                      None) == VLM_ERR_INVALID_ARG
    probs = (_lib.SyrkProblem * 1)()
    probs[0].x, probs[0].rows, probs[0].ldx, probs[0].d, probs[0].g, probs[0].ldg = p, rows, 48, 48, g.ptr, g.ld
    assert lib.vlm_syrk_accum_batch(probs, 1, _lib.VLM_TF32X2, None) == VLM_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(g.m, g0.float()) and g.sentinels_intact()


# ---- 8. the schedule cache -----------------------------------------------------------------------------------------

def test_schedule_cache_eviction_keeps_results_exact(lib):
    """1100 distinct chunk counts (more than twice the cache's 512 entries: two evictions, the second of which frees
    the schedules retired by the first) go through vlm_syrk_accum without a synchronisation in between, an i8x4 call
    (same cache) among them; then the first shape again, after its schedule was evicted."""
    d, n = 32, 1100
    x, x64, e = exact_x(32 * n, d, F32, seed=77)
    g0 = exact_g0(d, e, seed=1)
    chunk_grams = torch.einsum("kri,krj->kij", x64.view(n, 32, d), x64.view(n, 32, d))
    want = g0 + 2 * torch.cumsum(chunk_grams, 0)                  # k + 1 chunks: G0 + 2 X[:32(k+1)]^T X[:32(k+1)]
    assert_exact_case(x64.abs().T @ x64.abs(), e, g0, want[-1])
    g = g0.float().repeat(n + 1, 1, 1)
    xi, xi64, ei = exact_x(300, 128, F32, seed=78)
    gi0 = exact_g0(128, ei, seed=2)
    gi = Padded(128, 128, 130, F64, fill=gi0, sentinel=OUT_SENTINEL)
    scratch = torch.empty(lib.vlm_syrk_i8x4_scratch_bytes(300, 128), dtype=torch.uint8, device="cuda")
    for k in range(n):
        for _ in range(2):
            _lib.check(lib.vlm_syrk_accum(x.data_ptr(), _lib.VLM_F32, 32 * (k + 1), d, d, g[k].data_ptr(), d, None))
        if k == n // 2:
            for _ in range(2):
                _lib.check(lib.vlm_syrk_accum_i8x4(xi.data_ptr(), _lib.VLM_F32, 300, 128, 128, 0, 0, scratch.data_ptr(),
                                                   scratch.numel(), gi.ptr, gi.ld, None))
    for _ in range(2):
        _lib.check(lib.vlm_syrk_accum(x.data_ptr(), _lib.VLM_F32, 32, d, d, g[n].data_ptr(), d, None))
    torch.cuda.synchronize()
    upper = torch.ones(d, d, dtype=torch.bool, device="cuda").triu()
    bad = ((g[:n].double() != want) & upper).flatten(1).any(1)
    assert not bool(bad.any()), f"chunk counts with a wrong Gram: {(bad.nonzero()[:8, 0] + 1).tolist()}"
    assert_upper_equal(g[n], want[0], "first shape after eviction")
    wi = gi0 + 2 * (xi64.T @ xi64)
    assert not bool(((gi.m != wi) & torch.ones_like(wi, dtype=torch.bool).triu()).any()), "i8x4 Gram"
    assert gi.sentinels_intact()


# ---- 9. through GramCache ------------------------------------------------------------------------------------------

def _full_equal(got, want, what):
    bad = got.double() != want
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} entries differ, first {bad.nonzero()[0].tolist()}"


def test_gram_cache_default_precision_is_exact_end_to_end():
    """gram() of the default cache equals the full fp64 X^T X (the mirror included): plain 3-D input, row slices of a
    (B, 617, d) activation, a deferred group of mixed widths and dtypes, side-stream mode."""
    import vl_merging_b200 as vlm

    x3, x3_64, e3 = exact_x(4 * 617, 768, F32, seed=1)
    h, h64, eh = exact_x(8 * 617, 768, BF16, seed=2)
    h, h64 = h.view(8, 617, 768), h64.view(8, 617, 768)
    small = [exact_x(2560, 768, F32, seed=3), exact_x(2560, 3072, F32, seed=4), exact_x(40 * 16, 768, BF16, seed=5)]
    for kwargs in ({}, {"defer_bytes": 1 << 30}, {"side_stream": True}):
        cache = vlm.GramCache(**kwargs)
        for _ in range(2):
            cache.accumulate("plain3d", x3.view(4, 617, 768))
            cache.accumulate("text", h[:, :40])
            cache.accumulate("image", h[:, 40:])
            for i, (x, _, _) in enumerate(small):
                cache.accumulate(f"small{i}", x)
        t64, i64 = h64[:, :40].reshape(-1, 768), h64[:, 40:].reshape(-1, 768)
        inputs = {"plain3d": (x3_64, e3), "text": (t64, eh), "image": (i64, eh)}
        inputs.update({f"small{i}": (x64, e) for i, (_, x64, e) in enumerate(small)})
        for name, (x64, e) in inputs.items():
            want = 2 * (x64.T @ x64)
            g0 = torch.zeros_like(want)
            assert_exact_case(x64.abs().T @ x64.abs(), e, g0, want)
            _full_equal(cache.gram(name), want, f"GramCache({kwargs}) {name}")


@pytest.mark.parametrize("defer", [0, 1 << 30], ids=["immediate", "deferred"])
def test_gram_cache_tf32x3_is_exact_end_to_end(defer):
    """precision="tf32x3": split planes, then hi'hi + hi'lo + lo'hi; deferred, flush() packs the planes of the
    group back to back."""
    import vl_merging_b200 as vlm

    cache = vlm.GramCache(precision="tf32x3", defer_bytes=defer)
    shapes = {"a": (2560, 768), "b": (4097, 3072), "c": (1000, 768)}
    data = {n: split_exact_x(r, d, seed=r + d, density=min(1.0, 150 / r)) for n, (r, d) in shapes.items()}
    for _ in range(2):
        for n, (x, _, _, _) in data.items():
            cache.accumulate(n, x)
    for n, (x, hi, lo, e) in data.items():
        g0 = torch.zeros(x.shape[1], x.shape[1], dtype=F64, device="cuda")
        want, abs_terms = split_want(hi, lo, g0)
        assert_exact_case(abs_terms, e, g0, want, shift=12)
        _full_equal(cache.gram(n), want, f"tf32x3 {n}")


# ---- the ids above name the kernels that actually run --------------------------------------------------------------

def profiled_pair_launches():
    """For a dense (ldx = 128) and an odd-pitch (ldx = 129) fp32 X of width 128: {ldx: (pair_supported, names of the
    SYRK kernels torch.profiler saw vlm_syrk_accum launch)}."""
    from torch.profiler import ProfilerActivity, profile

    lib = _lib.lib()
    out = {}
    for ldx in (128, 129):
        x, _, _ = exact_x(64, 128, F32, seed=3)
        xb = Padded(64, 128, ldx, F32, fill=x)
        g = new_g(128, torch.zeros(128, 128, dtype=F64, device="cuda"))
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            _lib.check(lib.vlm_syrk_accum(xb.ptr, _lib.VLM_F32, 64, 128, ldx, g.ptr, g.ld, None))
            torch.cuda.synchronize()
        out[ldx] = (pair_supported(F32, xb.ptr, 128, ldx, 0, g.ptr, g.ld),
                    [e.key for e in prof.key_averages() if "syrk" in e.key])
    return out


def test_pair_predicate_names_the_launched_kernel():
    """pair_supported mirrors syrk_pair_supported; the profiler's kernel names confirm it.  The profile is taken in a
    child process: a torch.profiler session leaves CUPTI state behind in its process, after which a later session there
    (test_gpu_regmean_kernels.py's kernel-name check) can come back without any kernel records."""
    import json
    import os
    import subprocess
    import sys

    tests = os.path.dirname(os.path.abspath(__file__))
    code = (f"import json, sys; sys.path[:0] = {[os.path.dirname(tests), tests]!r}; "
            "import test_gpu_gram_kernels as t; print(json.dumps(t.profiled_pair_launches()))")
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    pair, names = got["128"]
    assert pair and any("syrk_2sm_kernel" in n for n in names) and not any("syrk_simt_kernel" in n for n in names), names
    pair, names = got["129"]
    assert not pair and any("syrk_simt_kernel" in n for n in names) and not any("syrk_2sm_kernel" in n for n in names), \
        names
