"""SYRK work decompositions (host logic of vlm_syrk_accum and vlm_syrk_accum_i8x4, no GPU): every (super-tile, chunk)
is covered exactly once, only upper-triangular tiles appear, makespans are near the ideal share."""
from collections import defaultdict

import pytest

import vl_merging_b200 as vlm

CASES = [(36928, 768, 4), (36928, 3072, 4), (2560, 768, 4), (2560, 3072, 2), (36928, 1024, 2), (36928, 4096, 4),
         (1, 8, 4), (64, 128, 4), (1000, 900, 4), (77, 200, 2), (5000, 129, 4)]


@pytest.mark.parametrize("rows,d,elem", [c for c in CASES if c[1] % (128 // c[2]) == 0])
def test_pair_schedule_covers_super_tiles_once(rows, d, elem):
    """CTA-pair kernel: every (super-tile, chunk) exactly once, b >= a, near-ideal makespan."""
    segs, off = vlm._lib.syrk_pair_schedule(rows, d, elem, 148)
    kc = (rows + 128 // elem - 1) // (128 // elem)
    nsb = (d + 255) // 256
    assert off[0] == 0 and off[-1] == len(segs) and 1 <= len(off) - 1 <= 74
    cover = defaultdict(list)
    costs = []
    for c in range(len(off) - 1):
        mine = segs[off[c]: off[c + 1]]
        costs.append(sum(k1 - k0 for _, _, k0, k1 in mine))
        for a, b, k0, k1 in mine:
            assert 0 <= a <= b < nsb and 0 <= k0 < k1 <= kc
            cover[(a, b)].append((k0, k1))
    assert set(cover) == {(a, b) for a in range(nsb) for b in range(a, nsb)}
    for ivs in cover.values():
        ivs.sort()
        assert ivs[0][0] == 0 and ivs[-1][1] == kc and all(x[1] == y[0] for x, y in zip(ivs, ivs[1:]))
    ideal = len(cover) * kc / 74
    assert max(costs) <= 1.25 * ideal + 16          # K-aligned tile ownership: makespan close to the ideal share
    assert max(k1 - k0 for _, _, k0, k1 in segs) <= 128   # accumulation cap (truncating fp32 accumulator)


def test_pair_schedule_is_k_aligned():
    """All clusters sweep K from the top of their tile together: in the first round every cluster's first
    segment starts at chunk 0, and whole tiles are owned by one cluster."""
    segs, off = vlm._lib.syrk_pair_schedule(36928, 3072, 4, 148)
    firsts = [segs[off[c]] for c in range(len(off) - 1)]
    assert all(f[2] == 0 for f in firsts)
    assert len({(f[0], f[1]) for f in firsts}) == len(firsts) == 74


@pytest.mark.parametrize("rows,d", [(36928, 768), (36928, 3072), (2560, 768), (2560, 3072), (36928, 1024), (36928, 4096),
                                    (100000, 256), (9216, 768), (64, 128), (200000, 768)])
def test_int8_schedule_runs_every_tile_once_per_phase(rows, d):
    """vlm_syrk_accum_i8x4: every (super-tile, phase) covers the K range exactly once; no segment is longer than the
    int32 accumulator is exact for (2^16 rows); phase 2 (128-row stages) is cut on multiples of 4 chunks; Grams with
    few tiles give every cluster ONE segment of one phase."""
    segs, off = vlm._lib.syrk_pair_schedule(rows, d, 1, 148)
    kc = (rows + 31) // 32
    nsb = (d + 255) // 256
    assert off[0] == 0 and off[-1] == len(segs) and 1 <= len(off) - 1 <= 74
    cover = defaultdict(list)
    for a, bp, k0, k1 in segs:
        b, ph = bp & 0xFFFF, bp >> 16
        assert 0 <= a <= b < nsb and ph in (0, 1, 2) and 0 <= k0 < k1 <= kc and k1 - k0 <= 2048
        cover[(a, b, ph)].append((k0, k1))
    assert set(cover) == {(a, b, ph) for a in range(nsb) for b in range(a, nsb) for ph in range(3)}
    for (a, b, ph), ivs in cover.items():
        ivs.sort()
        assert ivs[0][0] == 0 and ivs[-1][1] == kc and all(x[1] == y[0] for x, y in zip(ivs, ivs[1:]))
    ntile = nsb * (nsb + 1) // 2
    if 74 // ntile >= 3 and kc >= 64 and kc <= 2048:
        per_cluster = [segs[off[c]: off[c + 1]] for c in range(len(off) - 1)]
        if all(len(m) == 1 for m in per_cluster):                   # the phase-split form
            assert all(k0 % 4 == 0 for _, bp, k0, _ in segs if bp >> 16 == 2)
            assert len(per_cluster) <= 74 and len(per_cluster) >= 3 * ntile
    if (rows, d) in ((36928, 768), (2560, 768), (9216, 768)):
        assert all(off[c + 1] - off[c] == 1 for c in range(len(off) - 1))
