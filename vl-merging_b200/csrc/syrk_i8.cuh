// syrk_i8.cuh — kernel (a), exact variant on the INTEGER tensor cores ("Ozaki" splitting), included by syrk_pair.cu.
//
// The RegMean-grade Gram needs ~1e-8 (DESIGN.md 4a: regmean amplifies Gram error a thousandfold on near-singular
// sums), which the fp32 accumulator of the floating-point tensor pipes cannot give at any segment length, and the
// fp64 DMMA path (syrk_f64.cu) gives at 30 TFLOP/s.  Integer MMAs accumulate EXACTLY:
//
//   x[r][c]  ~=  q[r][c] * 2^(E_c - 26),   q = rint(x * 2^(26 - E_c)),  |q| < 2^26,  2^E_c > max_r |x[r][c]|
//   q = D0 * 2^21 + D1 * 2^14 + D2 * 2^7 + D3,   balanced digits D_p in [-64, 64]   (four int8 planes)
//   G[i][j] = 2^(E_i + E_j - 52) * sum_{p,q} 2^(7 (6 - p - q)) * (D_p[:, i] . D_q[:, j])
//
// The dot products of digit planes are int8 x int8 -> int32 tensor-core products (tcgen05.mma kind::i8, exact: 2^12 per
// product); the thirteen pairs with p + q <= 4 are kept.  (Group 4 matters: its D_2 . D_2 term is a sum of SQUARES on
// the diagonal — with p + q <= 3 only, normally distributed activations came out 1.7e-7 off, on the B200 and in a numpy
// emulation alike.  What is dropped now is below 1e-9 of sqrt(G_ii G_jj).)  Pairs of one group s = p + q share a
// scale, so a segment accumulates one group per int32 TMEM accumulator, two groups at a time (below); its epilogue
// merges the two exactly (acc1 * 128 + acc0 < 2^39), scales by 2^(E_i + E_j - 10 - 7 s) and adds the doubles to the
// fp64 Gram with TMA reduce-adds (cp.reduce.async.bulk.tensor .add on an fp64 tensor map: the split-K reduction, the
// sum over groups and the `+=` across hook calls in one).  Quantisation error: 2^-27 of the column maximum per
// element, unbiased.
//
// Same CTA-pair structure as syrk_2sm_kernel (one tcgen05.mma.cta_group::2 stream, M = 256, N = 256; leader-owned
// full / tempty barriers; six 32 KB stages, MN-major SWIZZLE_128B planes).  Every MMA consumes one 4 KB plane of A
// and of B per CTA for 128 tensor cycles — 64 B/clk, the SM's ingest limit — unless loaded planes are reused, so a
// segment forms up to TWO groups at once, one per 256-column TMEM accumulator, in three phases per K range:
//   phase 0 (groups 4 and 3): a stage = 32 rows of all four planes ([A: 4 x 4 KB][B: 4 x 4 KB]), 7 MMAs per 32 KB;
//   phase 1 (groups 2 and 1): a stage = 32 rows of planes 0..2 ([A: 3 x 4 KB][B: 3 x 4 KB]), 5 MMAs per 24 KB;
//   phase 2 (group 0): a stage = 128 rows of plane 0 ([A: 16 KB][B: 16 KB]), 4 MMAs per 32 KB (ingest-bound, 1/13 of
//   the work);
// one TMA box per operand per stage (three tensor maps over the same planes).  The accumulators belong to the
// running segment, so its epilogue is not hidden; int32 holds 2^17 rows of a four-pair group, so segments are up to
// 65536 rows long and epilogues are rare.  Measured (ncu, 36928 x 3072): IMMA pipe 91.8 % of elapsed, 1.33 ms.
// History: one group per segment with 4 KB boxes: tensor pipe 43 %; per-element red.global.add.f64 epilogue (two per
// element per phase, ldexp): 1.51 ms — the SM retires ~0.8 atomics per clock, 22 us per phase and CTA.
#pragma once

namespace vlm {
namespace {

constexpr int kI8PlaneBytes = 32 * 128;   // 32 rows x 128 int8 columns
constexpr int kI8Planes = 4;
constexpr int kI8Phases = 3;              // {groups 4, 3}, {groups 2, 1}, {group 0}
constexpr int kI8SlabBytes = 16384;         // 128 rows x 16 fp64 columns: one TMA reduce-add box
constexpr int kI8SmemBytes = k2Stages * k2StageBytes + 2 * kI8SlabBytes + 1280 + 1024;   // stages, two slabs, barriers

struct I8Args {
  double* g;
  int64_t ldg;
  const int* exps;   // E_c per column
};

// D s32, A/B signed 8-bit, both MN-major, M = 256 over the pair
__host__ __device__ constexpr uint32_t make_idesc_i8(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(256 >> 4) << 24);
}
__device__ __forceinline__ void umma2_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// 2^e as a double, from its exponent bits (|e| < 1022: column exponents come from fp32 maxima); NaN for a poisoned
// column (exponent kI8Poison, minus whatever the caller subtracted from it)
__device__ __forceinline__ double i8_pow2(int e) {
  return e < -(1 << 19) ? __longlong_as_double(0x7ff8000000000000ll) : __hiloint2double((1023 + e) << 20, 0);
}

// segs: k in 32-row chunks, phase 0 (groups 4 and 3), 1 (groups 2 and 1) or 2 (group 0), width d; cps is always 0
// tm_g: G as a 2-D fp64 tensor, box 16 columns x 128 rows (the epilogue's TMA reduce-adds)
// DET (deterministic mode, syrk_det.cu): tm_g describes the slot workspace, fp64 {256 columns, slots * 256 rows}, and
// each segment's `slot` says where its partial goes (emit_slab).  The phases a cluster runs on one tile chain into one
// slot.
template <bool DET>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
syrk_i8x4_kernel(const __grid_constant__ CUtensorMap tm_p0, const __grid_constant__ CUtensorMap tm_p1,
                 const __grid_constant__ CUtensorMap tm_p2, const __grid_constant__ CUtensorMap tm_g,
                 const PairSeg* __restrict__ segs, const int* __restrict__ seg_off,
                 const __grid_constant__ I8Args args) {
  constexpr int kBlk = kBlockBytes;       // one operand of a stage
  constexpr int kNS = k2Stages;
  constexpr int kStageB = k2StageBytes;   // [A][B]
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* slab = smem + kNS * kStageB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(slab + 2 * kI8SlabBytes);
  uint64_t* full = bars;                  // used in the leader only
  uint64_t* empty = bars + kNS;
  uint64_t* tfull = bars + 2 * kNS;
  uint64_t* tempty = bars + 2 * kNS + 1;  // used in the leader only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kNS + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int seg_begin = seg_off[cluster_id];
  const int seg_end = seg_off[cluster_id + 1];

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_p0);
    tma_prefetch_desc(&tm_p1);
    tma_prefetch_desc(&tm_p2);
    tma_prefetch_desc(&tm_g);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kNS; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tfull, 1);
    mbar_init(tempty, 8);
    fence_barrier_init();
  }
  if (warp == 2) tmem2_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer (both CTAs): one box for its own A block, one for its own half of B =====
    int stage = 0;
    uint32_t phase = 0;
    const uint64_t pol_x = l2_evict_normal();
    const uint32_t full0 = mapa_rank(smem_u32(full), 0);
    for (int s = seg_begin; s < seg_end; ++s) {
      const PairSeg seg = segs[s];
      const int ph = seg.phase;
      const bool diag = seg.sa == seg.sb;
      const CUtensorMap* tm = ph == 0 ? &tm_p0 : ph == 1 ? &tm_p1 : &tm_p2;
      const int a_group = 2 * seg.sa + (int)rank;
      const int b_group = 2 * seg.sb + (int)rank;
      const uint32_t bytes_pair = (diag ? 2u : 4u) * (ph == 1 ? 3u * kI8PlaneBytes : (uint32_t)kBlk);
      for (int k = seg.k0; k < seg.k1; k += ph == 2 ? 4 : 1) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (rank == 0) mbar_arrive_expect_tx(&full[stage], bytes_pair);
        uint8_t* sb = stage_base + stage * kStageB;
        const uint32_t bar = full0 + (uint32_t)stage * 8u;
        tma2_load_4d(tm, bar, sb + kBlk, 0, k * 32, b_group, 0, pol_x);
        if (!diag) tma2_load_4d(tm, bar, sb, 0, k * 32, a_group, 0, pol_x);
        if (++stage == kNS) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===== MMA issuer (leader only) =====
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    const uint32_t stage0 = smem_u32(stage_base);
    // MN-major SWIZZLE_128B: 8-row atoms 1024 bytes apart (SBO); one 128-byte column group per CTA, LBO unused
    constexpr uint32_t kDescHi = (uint32_t)((1024 >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);
    constexpr uint32_t kDescLo = (uint32_t)((kI8PlaneBytes >> 4) & 0x3FFF) << 16;
    constexpr uint32_t idesc = make_idesc_i8(256);
    constexpr uint32_t kP = kI8PlaneBytes >> 4;     // 32 rows of one plane, in descriptor units
    for (int s = seg_begin; s < seg_end; ++s) {
      const PairSeg seg = segs[s];
      const int sa_t = __shfl_sync(0xffffffffu, seg.sa, 0), sb_t = __shfl_sync(0xffffffffu, seg.sb, 0);
      const int k0 = __shfl_sync(0xffffffffu, seg.k0, 0), k1 = __shfl_sync(0xffffffffu, seg.k1, 0);
      const int ph = __shfl_sync(0xffffffffu, seg.phase, 0);
      const uint32_t a_off = (sa_t == sb_t) ? kBlk : 0u;
      const uint32_t d_hi = tmem_base, d_lo = tmem_base + kAccCols;   // the higher / lower group of this phase
      mbar_wait(tempty, acc_phase ^ 1);
      tc_fence_after();
      for (int k = k0; k < k1; k += ph == 2 ? 4 : 1) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t sb = stage0 + stage * kStageB;
        const uint32_t alo = (((sb + a_off) & 0x3FFFFu) >> 4) | kDescLo;
        const uint32_t blo = (((sb + kBlk) & 0x3FFFFu) >> 4) | kDescLo;
        if (elect_one()) {
          auto mma = [&](uint32_t dst, uint32_t a_units, uint32_t b_units, uint32_t accumulate) {
            umma2_i8(dst, ((uint64_t)kDescHi << 32) | (alo + a_units), ((uint64_t)kDescHi << 32) | (blo + b_units), idesc,
                     accumulate);
          };
          const uint32_t first = (k == k0) ? 0u : 1u;
          if (ph == 0) {
            // planes p at p * 4 KB.  group 4: (1,3) (2,2) (3,1); group 3: (0,3) (1,2) (2,1) (3,0)
            mma(d_hi, 1 * kP, 3 * kP, first);
            mma(d_hi, 2 * kP, 2 * kP, 1u);
            mma(d_hi, 3 * kP, 1 * kP, 1u);
            mma(d_lo, 0 * kP, 3 * kP, first);
            mma(d_lo, 1 * kP, 2 * kP, 1u);
            mma(d_lo, 2 * kP, 1 * kP, 1u);
            mma(d_lo, 3 * kP, 0 * kP, 1u);
          } else if (ph == 1) {
            // planes 0..2.  group 2: (0,2) (1,1) (2,0); group 1: (0,1) (1,0)
            mma(d_hi, 0 * kP, 2 * kP, first);
            mma(d_hi, 1 * kP, 1 * kP, 1u);
            mma(d_hi, 2 * kP, 0 * kP, 1u);
            mma(d_lo, 0 * kP, 1 * kP, first);
            mma(d_lo, 1 * kP, 0 * kP, 1u);
          } else {
            // 128 rows of plane 0: up to four K steps of 32 rows, as many as still lie inside this segment's K range
            const int nks = min(4, k1 - k);
            for (int ks = 0; ks < nks; ++ks) mma(d_hi, ks * kP, ks * kP, ks == 0 ? first : 1u);
          }
          tc2_commit_mcast(&empty[stage]);
        }
        __syncwarp();
        if (++stage == kNS) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) tc2_commit_mcast(tfull);
      __syncwarp();
      acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    {
      // ===== epilogue (both CTAs): exact int32 sums of the phase's groups -> scaled fp64 -> TMA reduce-add into G =====
      // The two groups of a phase differ by 2^7 in scale: acc1 * 128 + acc0 is exact in 64-bit integers (< 2^39) and in
      // fp64, so a phase adds ONE double per element.  Scaling is by powers of two only (2^(E_row - 10 - 7 grp) and
      // 2^(E_col), built from their exponent bits).  Thread `row` writes 16 doubles of its accumulator row into a
      // 128-byte-swizzled slab; one cp.reduce.async.bulk.tensor (.add, fp64) per 128 x 16 slab carries it into G — the
      // per-element red.global.add.f64 of the first version ran at the SM's ~0.8 atomics per clock (22 us per phase).
      const int q = warp - 4;
      const int epi_tid = threadIdx.x - 128;
      const int row = q * 32 + lane;
      uint32_t acc_phase = 0;
      const uint32_t tempty0 = mapa_rank(smem_u32(tempty), 0);
      uint32_t slab_counter = 0;            // two slabs: the conversion of one overlaps the TMA engine's read of the other
      for (int s = seg_begin; s < seg_end; ++s) {
        const PairSeg seg = segs[s];
        const int ph = seg.phase, d = seg.d;
        const bool diag = seg.sa == seg.sb;
        const int n_off = (diag && rank == 1) ? 1 : 0;   // peer on a diagonal tile: only block (2a+1, 2a+1)
        const int row0 = (2 * seg.sa + (int)rank) * 128;
        const int col0 = (2 * seg.sb + n_off) * 128;
        const int grp = 4 - 2 * ph;                      // the group in accumulator 0 (the smaller scale of the phase)
        const bool two = ph != 2;
        mbar_wait(tfull, acc_phase);
        tc_fence_after();
        const double rscale = (row0 + row < d) ? i8_pow2(__ldg(args.exps + row0 + row) - 10 - 7 * grp) : 0.0;
        const int nslab = (row0 < d) ? min(8 * (2 - n_off), (d - col0 + 15) / 16) : 0;
        for (int sl = 0; sl < nslab; ++sl) {
          uint32_t v[16], w[16];
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + n_off * 128 + sl * 16;
          tmem_ld_32x32b_x16(taddr, v);
          if (two) tmem_ld_32x32b_x16(taddr + kAccCols, w);
          const int c0 = col0 + sl * 16;
          double val[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) val[j] = (c0 + j < d) ? i8_pow2(__ldg(args.exps + c0 + j)) * rscale : 0.0;
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const long long c = two ? (long long)(int)w[j] * 128 + (int)v[j] : (long long)(int)v[j];
            val[j] *= __ll2double_rn(c);
          }
          uint8_t* buf = slab + (slab_counter & 1) * kI8SlabBytes;
          if (epi_tid == 0) bulk_wait_group_read<1>();   // the slab issued two slabs ago has left shared memory
          named_bar_sync(1, 128);
          const uint32_t rbase = smem_u32(buf) + row * 128;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const uint32_t addr = rbase + ((uint32_t)(c ^ (row & 7)) << 4);
            asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(val[2 * c]), "d"(val[2 * c + 1]) : "memory");
          }
          fence_proxy_async_smem();
          named_bar_sync(1, 128);
          if (epi_tid == 0) emit_slab<DET, false>(&tm_g, buf, seg, c0, row0, sl == 0, 0);
          ++slab_counter;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty0);
        acc_phase ^= 1;
      }
      if (epi_tid == 0) bulk_wait_group_read<0>();
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem2_dealloc(tmem_base, kTmemCols);
}

// ---- pre-pass: column maxima -> exponents, then the four digit planes ---------------------------------------------
// X is fp32, or fp16 / bf16 (widened exactly: the reference calibrates under fp16 autocast, where the inputs of proj
// and fc2 are half precision)
template <typename T>
__device__ __forceinline__ const T* i8_row_ptr(const T* x, int64_t r, int64_t ldx, int64_t seg_rows, int64_t seg_stride) {
  return seg_rows > 0 ? x + (r / seg_rows) * seg_stride + (r % seg_rows) * ldx : x + r * ldx;
}
// columns 4 q .. 4 q + 3 of a row
__device__ __forceinline__ float4 i8_load4(const float* row, int q) { return __ldg(reinterpret_cast<const float4*>(row) + q); }
__device__ __forceinline__ float4 i8_load4(const __half* row, int q) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(row) + q);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 i8_load4(const __nv_bfloat16* row, int q) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(row) + q);
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}

// grid (d / 128, row slabs); thread t of 32 x 8: columns 4 (t & 31) .. +3 of the block, rows (t >> 5) + 8 i of the slab;
// four independent 16-byte loads in flight per thread (the pass is a pure HBM stream)
template <typename T>
__global__ void __launch_bounds__(256) i8_colmax_kernel(const T* __restrict__ x, int64_t rows, int d, int64_t ldx,
                                                        int64_t seg_rows, int64_t seg_stride, int64_t rows_per_slab,
                                                        unsigned* __restrict__ amax_bits) {
  const int cq = blockIdx.x * 32 + (threadIdx.x & 31);
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_slab, r1 = min(rows, r0 + rows_per_slab);
  // maxima of the BIT PATTERNS of |x| (non-negative floats order like their bit patterns; Inf and NaN order above
  // every finite value, where fmaxf would drop a NaN): a non-finite activation poisons its column (i8_exps_kernel)
  unsigned m0 = 0, m1 = 0, m2 = 0, m3 = 0;
  auto upd = [&](const float4& v) {
    m0 = max(m0, __float_as_uint(v.x) & 0x7fffffffu), m1 = max(m1, __float_as_uint(v.y) & 0x7fffffffu);
    m2 = max(m2, __float_as_uint(v.z) & 0x7fffffffu), m3 = max(m3, __float_as_uint(v.w) & 0x7fffffffu);
  };
  int64_t r = r0 + (threadIdx.x >> 5);
  for (; r + 24 < r1; r += 32) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      v[u] = i8_load4(i8_row_ptr(x, r + 8 * u, ldx, seg_rows, seg_stride), cq);
#pragma unroll
    for (int u = 0; u < 4; ++u) upd(v[u]);
  }
  for (; r < r1; r += 8) upd(i8_load4(i8_row_ptr(x, r, ldx, seg_rows, seg_stride), cq));
  // the block's 8 row groups are combined in shared memory first: one atomic per column per block (with one per
  // thread, ~1000 same-address atomics per column serialised in L2 and took longer than the pass over X)
  __shared__ uint4 red[8][32];
  red[threadIdx.x >> 5][threadIdx.x & 31] = make_uint4(m0, m1, m2, m3);
  __syncthreads();
  if (threadIdx.x < 128) {
    const unsigned* col = reinterpret_cast<const unsigned*>(&red[0][0]) + threadIdx.x;
    unsigned m = col[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = max(m, col[w * 128]);
    atomicMax(amax_bits + blockIdx.x * 128 + threadIdx.x, m);
  }
}

// E_c with 2^E_c > max |x[:, c]| (clamped below so that 2^(26 - E_c) is a finite float), and that scale as a float,
// written over the column maximum it was derived from.  A column holding an Inf or a NaN gets the exponent kI8Poison:
// its digits are zero and the epilogue turns its row and column of the Gram into NaN, as the reference's fp64 product
// would (cache_gram_matrices.py:251-252) — never a finite number.
constexpr int kI8Poison = -(1 << 20);
__global__ void i8_exps_kernel(unsigned* __restrict__ amax_bits_then_scales, int d, int* __restrict__ exps) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  const unsigned bits = amax_bits_then_scales[c];
  if (bits >= 0x7f800000u) {              // Inf or NaN somewhere in the column
    exps[c] = kI8Poison;
    amax_bits_then_scales[c] = 0;         // scale 0: the digits of the whole column are zero
    return;
  }
  const float m = __uint_as_float(bits);
  const int e = m > 0.f ? max(ilogbf(m) + 1, -100) : 0;
  exps[c] = e;
  amax_bits_then_scales[c] = (unsigned)(127 + 26 - e) << 23;   // the float 2^(26 - e)
}

// Four values of one row -> one char4 per digit plane.  t = rint(x * 2^(26 - E)), |t| <= 2^26; with the bias
// 64 (1 + 2^7 + 2^14) added, the plain base-128 digits of u are the balanced digits of t plus 64 (and u >> 21 is the
// top digit itself), so the four planes are bit fields of u: shifts, byte permutes and a per-byte "- 64".
__device__ __forceinline__ unsigned i8_pack_low_bytes(unsigned a0, unsigned a1, unsigned a2, unsigned a3) {
  return __byte_perm(__byte_perm(a0, a1, 0x0040), __byte_perm(a2, a3, 0x0040), 0x5410);
}
__device__ __forceinline__ unsigned i8_minus64_per_byte(unsigned w) {   // bytes in [0, 127] -> two's complement of (byte - 64)
  w = (w & 0x7f7f7f7fu) ^ 0x40404040u;
  return w | ((w & 0x40404040u) << 1);
}
__device__ __forceinline__ void i8_slice_store(const float4& v, const float4& sc, int8_t* __restrict__ dst, int64_t plane) {
  constexpr int kBias = 64 * (1 + 128 + 128 * 128);
  const unsigned u0 = (unsigned)(__float2int_rn(v.x * sc.x) + kBias), u1 = (unsigned)(__float2int_rn(v.y * sc.y) + kBias);
  const unsigned u2 = (unsigned)(__float2int_rn(v.z * sc.z) + kBias), u3 = (unsigned)(__float2int_rn(v.w * sc.w) + kBias);
  *reinterpret_cast<unsigned*>(dst + 3 * plane) = i8_minus64_per_byte(i8_pack_low_bytes(u0, u1, u2, u3));
  *reinterpret_cast<unsigned*>(dst + 2 * plane) = i8_minus64_per_byte(i8_pack_low_bytes(u0 >> 7, u1 >> 7, u2 >> 7, u3 >> 7));
  *reinterpret_cast<unsigned*>(dst + 1 * plane) = i8_minus64_per_byte(i8_pack_low_bytes(u0 >> 14, u1 >> 14, u2 >> 14, u3 >> 14));
  *reinterpret_cast<unsigned*>(dst) = i8_pack_low_bytes((unsigned)((int)u0 >> 21), (unsigned)((int)u1 >> 21),
                                                         (unsigned)((int)u2 >> 21), (unsigned)((int)u3 >> 21));
}
// block b: rows b, b + gridDim.x, ... (four rows per trip); thread t: column quads t, t + 256, ... of each row — no
// index division, 4 x 16 bytes in flight per thread
template <typename T>
__global__ void __launch_bounds__(256, 4) i8_slice_kernel(const T* __restrict__ x, int64_t rows, int d, int64_t ldx,
                                                       int64_t seg_rows, int64_t seg_stride,
                                                       const float* __restrict__ scales, int8_t* __restrict__ planes) {
  const int d4 = d >> 2;
  const int64_t plane = rows * (int64_t)d;
  const int64_t G = gridDim.x;
  for (int64_t r0 = blockIdx.x; r0 < rows; r0 += 4 * G) {
    const T* src[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) src[u] = i8_row_ptr(x, min(r0 + u * G, rows - 1), ldx, seg_rows, seg_stride);
    for (int cq = threadIdx.x; cq < d4; cq += 256) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = i8_load4(src[u], cq);
      const float4 e = __ldg(reinterpret_cast<const float4*>(scales) + cq);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (r0 + u * G < rows) i8_slice_store(v[u], e, planes + (r0 + u * G) * d + 4 * cq, plane);
    }
  }
}

}  // namespace
}  // namespace vlm
