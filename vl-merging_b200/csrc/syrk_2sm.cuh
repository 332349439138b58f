// syrk_2sm.cuh — kernel (a), third generation: ONE tcgen05.mma.cta_group::2 instruction stream per CTA pair.
// Included by syrk_pair.cu (which owns the host side: tensor maps, schedules, launches) after its PTX wrappers.
//
// The pair kernel of syrk_pair.cu is paced by what an SM can take in per chunk (48 KB: its own A block, its own B
// block and the peer's multicast B block; 712 cycles against 548 cycles of tensor work, DESIGN.md 4a).  Here the
// two CTAs of a cluster execute one M = 256, N = 256 instruction together: CTA r holds row block 2a+r (its 128
// rows of A and of D) and column block 2b+r (its half of B); the tensor cores of the pair read the other half of
// B from the peer's shared memory.  32 KB per chunk per SM, no multicast, six 32 KB stages.
//
// Protocol (leader = cluster rank 0):
//   full[s]   lives in the LEADER.  Both CTAs' TMA loads (cp.async.bulk.tensor ... .cta_group::2) complete on it;
//             the leader's producer arms it with the bytes of both CTAs.  A peer load may complete before the
//             leader has armed the phase: the transaction count goes negative while the one pending arrival
//             keeps the phase open.
//   empty[s]  one per CTA, 1 arrival: the leader's tcgen05.commit.cta_group::2 multicast to both CTAs.
//   tfull[a]  one per CTA, 1 arrival: same multicast commit after the last MMA of a segment.
//   tempty[a] lives in the leader, 8 arrivals: one per epilogue warp of either CTA (the peer's arrive remotely).
// Only the leader's warp 1 issues MMAs.  Both CTAs walk the same segment list.
//
// SPLIT (fp32 only, "3xTF32"): X arrives as two planes {hi, lo} with hi = tf32(x), lo = tf32(x - hi)
// (vlm_tf32_split), described as a 4-D tensor {column in group, row, column group, plane}.  A chunk is 16 rows; one
// TMA box brings both planes of a block ([hi 8 KB][lo 8 KB]) and the issuer forms hi'hi + hi'lo + lo'hi: three MMAs
// per K step, 822 cycles of tensor work per 32 KB — the loop is tensor-bound.  What is dropped is lo'lo (2^-22
// relative) and the fp32 accumulation error of the tensor core, bounded as before by the segment length.
#pragma once

namespace vlm {
namespace {

constexpr int k2Stages = 6;
constexpr int k2StageBytes = 2 * kBlockBytes;  // [A][B]
constexpr int k2SmemBytes = k2Stages * k2StageBytes + 2 * kStagingBytes + 256 + 1024;

template <int ELEM_BYTES, bool SPLIT>
struct Geo2 {
  static constexpr int BK = SPLIT ? 16 : 128 / ELEM_BYTES;   // rows of X per stage
  static constexpr int GB = ELEM_BYTES;                      // column groups per 128-column block
  static constexpr int BOX_BYTES = BK * 128;                 // one column group of one plane (= LBO)
  static constexpr int PLANE_BYTES = GB * BOX_BYTES;         // one block of one plane: 16 KB, 8 KB when SPLIT
  static constexpr int UMMA_K = 32 / ELEM_BYTES;
  static constexpr int KSTEP_BYTES = UMMA_K * 128;
  static constexpr int NUM_K = BK / UMMA_K;                  // K steps per stage: 4, 2 when SPLIT
  static constexpr int LAYOUT_TYPE = ELEM_BYTES == 4 ? 1 : 2;
  static constexpr int SBO_BYTES = ELEM_BYTES == 4 ? 512 : 1024;
  static_assert(!SPLIT || ELEM_BYTES == 4, "the split mode is for fp32 activations");
  static_assert((SPLIT ? 2 : 1) * PLANE_BYTES == kBlockBytes, "block geometry");
};

__device__ __forceinline__ uint32_t mapa_rank(uint32_t cta_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// loads whose completion is counted on an mbarrier of EITHER CTA of the pair (shared::cluster address)
__device__ __forceinline__ void tma2_load_3d(const CUtensorMap* tm, uint32_t bar_cluster, void* smem_dst, int c0, int c1,
                                             int c2, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2),
      "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma2_load_4d(const CUtensorMap* tm, uint32_t bar_cluster, void* smem_dst, int c0, int c1,
                                             int c2, int c3, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tc2_commit_mcast(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)0x3)
               : "memory");
}
__device__ __forceinline__ void tmem2_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem2_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D fp32, A/B format fmt, both MN-major, M = 256 over the pair
__host__ __device__ constexpr uint32_t make_idesc2(int fmt, int n) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | (1u << 15) | (1u << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}
template <int FMT>
__device__ __forceinline__ void umma2(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                      uint32_t accumulate) {
  if constexpr (FMT == 2) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// BATCH = false: one problem, tensor maps in kernel parameters.  BATCH = true: the segments of several problems
// (e.g. all Grams of the text tower of one forward) share the grid; tensor maps live in global memory (`maps`:
// [2*pid] = X, [2*pid+1] = G), written by the host before the launch.  SPLIT: tm_x is the 4-D {hi, lo} map (see header); cps is ignored.
// DET (deterministic mode, syrk_det.cu): the G map (tm_g1, or every maps[2*pid+1]) describes the slot workspace, fp32
// {256 columns, slots * 256 rows}, and the segments are BatchSegs whose `slot` says where the partial goes.
template <int ELEM_BYTES, int FMT, bool BATCH, bool SPLIT, bool DET>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
syrk_2sm_kernel(const __grid_constant__ CUtensorMap tm_x1, const __grid_constant__ CUtensorMap tm_g1,
                const CUtensorMap* __restrict__ maps, const void* __restrict__ segs_raw,
                const int* __restrict__ seg_off, int d1, int cps1, int l2_hints) {
  using G = Geo2<ELEM_BYTES, SPLIT>;
  using Seg = typename std::conditional<BATCH || DET, BatchSeg, PairSeg>::type;
  const Seg* __restrict__ segs = static_cast<const Seg*>(segs_raw);
  auto map_x = [&](const Seg& sg) -> const CUtensorMap* {
    if constexpr (BATCH) return maps + 2 * sg.pid; else return &tm_x1;
  };
  auto map_g = [&](const Seg& sg) -> const CUtensorMap* {
    if constexpr (BATCH) return maps + 2 * sg.pid + 1; else return &tm_g1;
  };
  auto cols_of = [&](const Seg& sg) -> int {
    if constexpr (BATCH) return sg.d; else return d1;
  };
  auto cps_of = [&](const Seg& sg) -> int {
    if constexpr (SPLIT) return 0; else if constexpr (BATCH) return sg.cps; else return cps1;
  };
  constexpr int kRows = G::BK;
  constexpr int kBlk = kBlockBytes;
  constexpr int kNS = k2Stages;
  constexpr int kStageB = k2StageBytes;  // [A][B]
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* staging = smem + kNS * kStageB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + 2 * kStagingBytes);
  uint64_t* full = bars;                  // used in the leader only
  uint64_t* empty = bars + kNS;
  uint64_t* tfull = bars + 2 * kNS;
  uint64_t* tempty = bars + 2 * kNS + 2;  // used in the leader only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kNS + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int seg_begin = seg_off[cluster_id];
  const int seg_end = seg_off[cluster_id + 1];

  if (!BATCH && warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x1);
    tma_prefetch_desc(&tm_g1);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kNS; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem2_alloc(tmem_slot, kTmemCols);  // one warp of EACH CTA of the pair
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer (both CTAs): own A block + own half of B, completion counted in the leader =====
    int stage = 0;
    uint32_t phase = 0;
    int cur_pid = -1;
    const uint64_t pol_x = l2_policy(l2_hints & 3);
    const uint32_t full0 = mapa_rank(smem_u32(full), 0);
    for (int s = seg_begin; s < seg_end; ++s) {
      const Seg seg = segs[s];
      const CUtensorMap* tm_x = map_x(seg);
      if constexpr (BATCH) {
        if (seg.pid != cur_pid) {
          tensormap_acquire(tm_x);
          cur_pid = seg.pid;
        }
      }
      const bool diag = seg.sa == seg.sb;
      const int a_group = (2 * seg.sa + (int)rank) * G::GB;
      const int b_group = (2 * seg.sb + (int)rank) * G::GB;
      const uint32_t bytes_pair = (diag ? 2u : 4u) * kBlk;   // both CTAs: B (+ A) block each
      const int cps = cps_of(seg);
      int xseg = cps > 0 ? seg.k0 / cps : 0;
      int kin = seg.k0 - xseg * cps;
      for (int k = seg.k0; k < seg.k1; ++k) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (rank == 0) mbar_arrive_expect_tx(&full[stage], bytes_pair);
        uint8_t* sb = stage_base + stage * kStageB;
        const uint32_t bar = full0 + (uint32_t)stage * 8u;
        const int row = kin * kRows;
        if (SPLIT || cps > 0) {
          tma2_load_4d(tm_x, bar, sb + kBlk, 0, row, b_group, xseg, pol_x);
          if (!diag) tma2_load_4d(tm_x, bar, sb, 0, row, a_group, xseg, pol_x);
        } else {
          tma2_load_3d(tm_x, bar, sb + kBlk, 0, row, b_group, pol_x);
          if (!diag) tma2_load_3d(tm_x, bar, sb, 0, row, a_group, pol_x);
        }
        if (++kin == cps) {
          kin = 0;
          ++xseg;
        }
        if (++stage == kNS) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===== MMA issuer (leader only): the whole warp walks the loop, one elected lane issues =====
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t stage0 = smem_u32(stage_base);
    constexpr uint32_t kDescHi = (uint32_t)((G::SBO_BYTES >> 4) & 0x3FFF) | (1u << 14) | ((uint32_t)G::LAYOUT_TYPE << 29);
    constexpr uint32_t kDescLo = (uint32_t)((G::BOX_BYTES >> 4) & 0x3FFF) << 16;
    constexpr uint32_t idesc = make_idesc2(FMT, 256);
    for (int s = seg_begin; s < seg_end; ++s) {
      const Seg seg = segs[s];
      const int sa_t = __shfl_sync(0xffffffffu, seg.sa, 0), sb_t = __shfl_sync(0xffffffffu, seg.sb, 0);
      const int k0 = __shfl_sync(0xffffffffu, seg.k0, 0), k1 = __shfl_sync(0xffffffffu, seg.k1, 0);
      // diagonal super-tile: each CTA's A block IS its B block (one load); the pair forms all four blocks
      // and the peer's epilogue drops the one below the diagonal
      const uint32_t a_off = (sa_t == sb_t) ? kBlk : 0u;
      const uint32_t d_tmem = tmem_base + acc * kAccCols;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      for (int k = k0; k < k1; ++k) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t sb = stage0 + stage * kStageB;
        const uint32_t alo = (((sb + a_off) & 0x3FFFFu) >> 4) | kDescLo;
        const uint32_t blo = (((sb + kBlk) & 0x3FFFFu) >> 4) | kDescLo;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < G::NUM_K; ++kk) {
            const uint32_t st = kk * (G::KSTEP_BYTES >> 4);
            const uint64_t a_hi = ((uint64_t)kDescHi << 32) | (alo + st);
            const uint64_t b_hi = ((uint64_t)kDescHi << 32) | (blo + st);
            umma2<FMT>(d_tmem, a_hi, b_hi, idesc, (k > k0 || kk > 0) ? 1u : 0u);
            if constexpr (SPLIT) {
              const uint64_t a_lo = a_hi + (G::PLANE_BYTES >> 4);
              const uint64_t b_lo = b_hi + (G::PLANE_BYTES >> 4);
              umma2<FMT>(d_tmem, a_hi, b_lo, idesc, 1u);
              umma2<FMT>(d_tmem, a_lo, b_hi, idesc, 1u);
            }
          }
          tc2_commit_mcast(&empty[stage]);  // the slot is free in BOTH CTAs once these MMAs have read it
        }
        __syncwarp();
        if (++stage == kNS) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) tc2_commit_mcast(&tfull[acc]);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    // ===== epilogue (both CTAs): own 128 rows x 256 columns of the accumulator -> TMA reduce-add into G =====
    const int q = warp - 4;
    const int epi_tid = threadIdx.x - 128;
    const int row = q * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t slab_counter = 0;
    int cur_pid = -1;
    const uint64_t pol_g = l2_policy((l2_hints >> 2) & 3);
    const uint32_t tempty0 = mapa_rank(smem_u32(tempty), 0);
    for (int s = seg_begin; s < seg_end; ++s) {
      const Seg seg = segs[s];
      const CUtensorMap* tm_g = map_g(seg);
      const int d = cols_of(seg);
      if constexpr (BATCH) {
        if (epi_tid == 0 && seg.pid != cur_pid) {
          tensormap_acquire(tm_g);
          cur_pid = seg.pid;
        }
      }
      const bool diag = seg.sa == seg.sb;
      const int n_off = (diag && rank == 1) ? 1 : 0;   // peer on a diagonal tile: only block (2a+1, 2a+1)
      const int row0 = (2 * seg.sa + (int)rank) * 128;
      const int col0 = (2 * seg.sb + n_off) * 128;
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const int nslab = (row0 < d) ? min(4 * (2 - n_off), (d - col0 + 31) / 32) : 0;
      const bool last = (s == seg_end - 1);   // the stages are dead by now: one staging slot per slab
      for (int sl = 0; sl < nslab; ++sl) {
        uint8_t* buf = last ? stage_base + sl * kStagingBytes : staging + (slab_counter & 1) * kStagingBytes;
        if (!last) {
          if (epi_tid == 0) bulk_wait_group_read<1>();
          named_bar_sync(1, 128);
        }
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * kAccCols + n_off * 128 + sl * 32, v);
        tmem_ld_wait();
        const uint32_t rbase = smem_u32(buf) + row * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint32_t addr = rbase + ((uint32_t)(c ^ (row & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v[4 * c]), "r"(v[4 * c + 1]),
                       "r"(v[4 * c + 2]), "r"(v[4 * c + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (epi_tid == 0) {
          if constexpr (DET) {
            // this CTA's 128 rows of the slot: the segment that opens the slot stores, later segments of this
            // cluster on the same tile add.  Before adding, wait for COMPLETION (not just the source reads) of every
            // earlier bulk operation of this thread, the previous store / reduce-add into this slot among them: PTX
            // ISA, cp.async.bulk.wait_group — without .read, the wait lasts until the bulk async-groups are complete,
            // writes to their destinations included.  The adds into a slot are then in segment order.
            const int srow = (seg.slot >> 1) * 256 + (int)rank * 128, scol = n_off * 128 + sl * 32;
            if (seg.slot & 1) {
              if (sl == 0) bulk_wait_group<0>();
              tma_reduce_add_2d_hint(tm_g, buf, scol, srow, pol_g);
            } else {
              tma_store_2d_hint(tm_g, buf, scol, srow, pol_g);
            }
          } else {
            tma_reduce_add_2d_hint(tm_g, buf, col0 + sl * 32, row0, pol_g);
          }
          bulk_commit_group();
        }
        ++slab_counter;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty0 + (uint32_t)acc * 8u);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    // the staging memory must outlive the TMA engine's READS of it; the adds themselves complete before the grid does
    if (epi_tid == 0) bulk_wait_group_read<0>();
  }

  tc_fence_before();
  cluster_sync_all();  // the pair's MMAs read this CTA's shared memory and the peer arrives on the leader's barriers until here
  if (warp == 2) tmem2_dealloc(tmem_base, kTmemCols);
}

// fp32 -> {hi, lo} planes for the SPLIT kernel: hi = tf32(x) (round to nearest), lo = tf32(x - hi).
// x: rows x d with row pitch ldx, optionally segmented (seg_rows > 0: row r lives in segment r / seg_rows).
// out: [2][rows][d] contiguous.
__device__ __forceinline__ float to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__global__ void __launch_bounds__(256) tf32_split_kernel(const float* __restrict__ x, int64_t rows, int d, int64_t ldx,
                                                          int64_t seg_rows, int64_t seg_stride,
                                                          float* __restrict__ out) {
  const int d4 = d >> 2;
  const int64_t n4 = rows * d4;
  float4* hi = reinterpret_cast<float4*>(out);
  float4* lo = reinterpret_cast<float4*>(out + rows * (int64_t)d);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / d4;
    const int c = (int)(i - r * d4);
    const float* src = seg_rows > 0 ? x + (r / seg_rows) * seg_stride + (r % seg_rows) * ldx : x + r * ldx;
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + c);
    float4 h, l;
    h.x = to_tf32(v.x), h.y = to_tf32(v.y), h.z = to_tf32(v.z), h.w = to_tf32(v.w);
    l.x = to_tf32(v.x - h.x), l.y = to_tf32(v.y - h.y), l.z = to_tf32(v.z - h.z), l.w = to_tf32(v.w - h.w);
    hi[i] = h;
    lo[i] = l;
  }
}

}  // namespace
}  // namespace vlm
