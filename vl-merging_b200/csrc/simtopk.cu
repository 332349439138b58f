// simtopk.cu — SURVEY.md §8f rank 2: the retrieval step right after the merge, fused.
//
// compute_irtr_recall (src/vilt/modules/objectives.py:684-710) forms scores = img_cls_feats @ txt_cls_feats.t() —
// 5,000 x 25,000 for the COCO test split, 500 MB in fp32 — and then calls topk on it six times (k = 1, 5, 10 along
// both dimensions).  Only the ten best columns of every row are ever used.  This kernel computes the row-wise top-10
// of A * B^T straight from the tensor-core accumulators: the score matrix never exists.  The column-wise direction
// is the same kernel with the operands swapped (the GEMM is 0.19 TFLOP; recomputing it costs less than one pass over
// a materialised matrix).
//
//   A [m, d], B [n, d]: fp16 or bf16, row-major (K-major for the tensor core), what the towers produce under the
//   reference's autocast (:657,669).  Products are exact, accumulation fp32 in TMEM.
//   CTA (rb, sp): rows [128 rb, 128 rb + 128) of A against column tiles of 256 rows of B in split sp of `splits`
//   (so that 40 row blocks still fill 148 SMs); TMA (SWIZZLE_128B, K-major) -> 4 x 48 KB stages ->
//   tcgen05.mma.cta_group::1 kind::f16 M128 N256 K16 -> two 256-column TMEM accumulators; the epilogue thread of
//   row r reads its 256 scores (tcgen05.ld) while the next tile's MMAs run and keeps a sorted top-10 (value, column)
//   in registers: strict `>` against the current 10th, so of equal scores the lower column wins — the order of a
//   stable descending sort, which is what the oracle uses.
//   Output: [m][splits][10] values (descending; -inf padded) and int32 columns (-1 padded); the `splits` partial
//   lists of a row are merged by the caller (a stable sort of 10 * splits candidates).
#include <algorithm>

#include "common.cuh"
#include "umma.cuh"

namespace vlm {
namespace {

constexpr int kTop = 10;
constexpr int sTM = 128, sTN = 256, sTK = 64;      // tile: rows of A, rows of B, K elements (128 bytes of a 16-bit type)
constexpr int sStages = 4;
constexpr int sABytes = sTM * 128, sBBytes = sTN * 128;
constexpr int sStageBytes = sABytes + sBBytes;     // 48 KB
constexpr int sSmemBytes = sStages * sStageBytes + 256 + 1024;
constexpr int sThreads = 256;

// D fp32, A/B fmt (0 f16, 1 bf16), both K-major, M = 128
__host__ __device__ constexpr uint32_t make_idesc_kmajor(int fmt, int n) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

__global__ void __launch_bounds__(sThreads, 1)
sim_topk_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, int m, int n, int d,
                int fmt, int tiles_per_split, int splits, float* __restrict__ out_val, int* __restrict__ out_idx) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + sStages * sStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + sStages;
  uint64_t* tfull = bars + 2 * sStages;
  uint64_t* tempty = bars + 2 * sStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * sStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rb = blockIdx.x, sp = blockIdx.y;
  const int ntiles = (n + sTN - 1) / sTN;
  const int ct0 = sp * tiles_per_split, ct1 = min(ntiles, ct0 + tiles_per_split);
  const int nkb = (d + sTK - 1) / sTK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < sStages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 128);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    int stage = 0;
    uint32_t phase = 0;
    for (int ct = ct0; ct < ct1; ++ct)
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full[stage], sStageBytes);
        uint8_t* sb = smem + stage * sStageBytes;
        tma_load_2d(&tm_a, &full[stage], sb, kb * sTK, rb * sTM);
        tma_load_2d(&tm_b, &full[stage], sb + sABytes, kb * sTK, ct * sTN);
        if (++stage == sStages) {
          stage = 0;
          phase ^= 1;
        }
      }
  } else if (warp == 1) {
    // ===== MMA issuer: whole warp walks the loop, one elected lane issues =====
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    const uint32_t base = smem_u32(smem);
    // K-major SWIZZLE_128B: rows of 128 bytes, 8-row atoms 1024 bytes apart (SBO); LBO unused; one MMA = 32 bytes of K
    constexpr uint32_t kDescHi = (uint32_t)((1024 >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);
    constexpr uint32_t kDescLo = (uint32_t)((16 >> 4) & 0x3FFF) << 16;
    const uint32_t idesc = make_idesc_kmajor(fmt, sTN);
    for (int ct = ct0; ct < ct1; ++ct) {
      const uint32_t d_tmem = tmem_base + acc * sTN;
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t sa = base + stage * sStageBytes;
        const uint32_t alo = ((sa & 0x3FFFFu) >> 4) | kDescLo;
        const uint32_t blo = (((sa + sABytes) & 0x3FFFFu) >> 4) | kDescLo;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < sTK / 16; ++kk) {
            const uint64_t adesc = ((uint64_t)kDescHi << 32) | (alo + kk * (32 >> 4));
            const uint64_t bdesc = ((uint64_t)kDescHi << 32) | (blo + kk * (32 >> 4));
            umma<0>(d_tmem, adesc, bdesc, idesc, (kb > 0 || kk > 0) ? 1u : 0u);
          }
          tc_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == sStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) tc_commit(&tfull[acc]);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    // ===== epilogue: thread = one row of A; sorted top-10 over every column this CTA sees =====
    const int q = warp - 4;
    const int row = rb * sTM + q * 32 + lane;
    float val[kTop];
    int idx[kTop];
#pragma unroll
    for (int t = 0; t < kTop; ++t) {
      val[t] = -INFINITY;
      idx[t] = -1;
    }
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int ct = ct0; ct < ct1; ++ct) {
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const int col0 = ct * sTN;
#pragma unroll 1
      for (int c32 = 0; c32 < sTN / 32; ++c32) {
        if (col0 + c32 * 32 >= n) break;                 // uniform over the CTA
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * sTN + c32 * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float s = __uint_as_float(v[j]);
          const int col = col0 + c32 * 32 + j;
          if (col < n && s > val[kTop - 1]) {
            val[kTop - 1] = s;
            idx[kTop - 1] = col;
#pragma unroll
            for (int t = kTop - 1; t > 0; --t)
              if (val[t] > val[t - 1]) {
                const float fv = val[t];
                val[t] = val[t - 1];
                val[t - 1] = fv;
                const int iv = idx[t];
                idx[t] = idx[t - 1];
                idx[t - 1] = iv;
              }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (row < m) {
      float* ov = out_val + ((int64_t)row * splits + sp) * kTop;
      int* oi = out_idx + ((int64_t)row * splits + sp) * kTop;
#pragma unroll
      for (int t = 0; t < kTop; ++t) {
        ov[t] = val[t];
        oi[t] = idx[t];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

int encode_feat_map(const void* p, int dtype, int64_t rows, int d, int64_t ld, int box_rows, CUtensorMap* tm) {
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)sTK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(tm, dtype == VLM_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                      const_cast<void*>(p), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(features) failed: CUresult %d", (int)r);
  return 0;
}

}  // namespace
}  // namespace vlm

using namespace vlm;

extern "C" int vlm_sim_topk_splits(int64_t m, int64_t n) {
  int nsm = 0;
  if (device_sm_count(&nsm) != 0 || m <= 0 || n <= 0) return 1;
  const int64_t rbs = (m + sTM - 1) / sTM, ntiles = (n + sTN - 1) / sTN;
  int64_t splits = std::max<int64_t>(1, std::min<int64_t>(ntiles, (nsm + rbs - 1) / rbs));
  const int64_t tps = (ntiles + splits - 1) / splits;
  return (int)((ntiles + tps - 1) / tps);
}

extern "C" int vlm_sim_topk(const void* a, int64_t m, int64_t lda, const void* b, int64_t n, int64_t ldb, int d, int dtype,
                            float* out_val, int32_t* out_idx, int splits, void* stream) {
  VLM_REQUIRE(dtype == VLM_F16 || dtype == VLM_BF16, VLM_ERR_INVALID_ARG,
              "vlm_sim_topk: features must be VLM_F16 or VLM_BF16 (got %d)", dtype);
  VLM_REQUIRE(a && b && out_val && out_idx && m > 0 && n > 0 && d > 0 && lda >= d && ldb >= d, VLM_ERR_INVALID_ARG,
              "vlm_sim_topk: bad arguments");
  VLM_REQUIRE(m < ((int64_t)1 << 31) && n < ((int64_t)1 << 31), VLM_ERR_INVALID_ARG, "vlm_sim_topk: too many rows");
  VLM_REQUIRE((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0 && (lda % 8) == 0 &&
                  (ldb % 8) == 0,
              VLM_ERR_ALIGNMENT, "vlm_sim_topk: features must be 16-byte aligned with row pitches that are multiples of 8");
  if (int rc = require_sm100()) return rc;
  VLM_REQUIRE(splits == vlm_sim_topk_splits(m, n), VLM_ERR_INVALID_ARG,
              "vlm_sim_topk: splits must be vlm_sim_topk_splits(m, n) = %d (got %d)", vlm_sim_topk_splits(m, n), splits);
  CUtensorMap tm_a, tm_b;
  if (int rc = encode_feat_map(a, dtype, m, d, lda, sTM, &tm_a)) return rc;
  if (int rc = encode_feat_map(b, dtype, n, d, ldb, sTN, &tm_b)) return rc;
  const int ntiles = (int)((n + sTN - 1) / sTN);
  const int tps = (ntiles + splits - 1) / splits;
  VLM_CUDA(cudaFuncSetAttribute(sim_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sSmemBytes));
  dim3 grid((unsigned)((m + sTM - 1) / sTM), (unsigned)splits);
  sim_topk_kernel<<<grid, sThreads, sSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      tm_a, tm_b, (int)m, (int)n, d, dtype == VLM_BF16 ? 1 : 0, tps, splits, out_val, out_idx);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}
