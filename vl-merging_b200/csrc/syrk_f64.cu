// syrk_f64.cu — kernel (a), reference-precision variant: G += X^T X with fp64 products and fp64 accumulation on
// the fp64 tensor-core path (mma.sync m8n8k4 DMMA), G in fp64.
//
// Why it exists.  The reference hook casts the activation to fp64 before the product
// (src/cache_gram_matrices.py:251-252) and regmean inverts the summed Gram (src/vilt/modules/vilt_module.py:
// 432-434, :483-484).  The tcgen05 kernels accumulate in the tensor core's truncating fp32 accumulator: even with
// exact operands (bf16, or the 3xTF32 split) the Gram carries a ~2e-5 non-uniform shrink, and on inputs whose
// Gram has a small eigen-direction (LayerNorm outputs lie near an affine hyperplane: cond ~1e4-1e5) RegMean
// amplifies that to 1e-2 — measured on the B200, tests/test_gpu_regmean_chain.py.  No segment length fixes a
// truncating accumulator, so the RegMean-grade mode does what the reference does: fp64 throughout.
//
// Shape: 128 x 128 tiles of the block-upper triangle, 16 warps of 32 x 32 (4 x 4 m8n8k4 tiles each), K step 32 rows
// of X; the raw fp32 / bf16 / f16 rows of the two 128-column panels come in through a 3-stage cp.async pipeline and
// are widened when a fragment is read (X^T is A: A[m][k] = X[k][m], so both fragments read [k][column] and one
// pitch of 128 + 8 elements makes them bank-conflict free).  Rows are cut into `pieces` K ranges (grid.y) so that
// small Grams fill the GPU; every CTA adds its tile with red.global.add.f64 — the split-K reduction and the `+=`
// across hook calls in one mechanism, like the TMA reduce-add of the tcgen05 kernels.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "syrk.h"

namespace vlm {
namespace {

constexpr int FT = 128;       // tile edge
constexpr int FK = 32;        // rows of X per pipeline stage (two barriers per 32 rows cost 6 % at 16)
constexpr int FSTAGES = 3;
constexpr int FPITCH = FT + 8;

template <typename T>
struct F64Smem {
  T a[FSTAGES][FK][FPITCH];
  T b[FSTAGES][FK][FPITCH];
};

__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, bool valid) {
  const uint32_t d = smem_u32(smem_dst);
  const int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gmem_src), "r"(n) : "memory");
}
__device__ __forceinline__ void dmma_f64(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
__device__ __forceinline__ double widen(float v) { return (double)v; }
__device__ __forceinline__ double widen(__nv_bfloat16 v) { return (double)__bfloat162float(v); }
__device__ __forceinline__ double widen(__half v) { return (double)__half2float(v); }

// VEC: rows and columns allow 16-byte cp.async chunks (x 16-byte aligned, ldx / seg_stride / d multiples of 16 bytes)
// DET (deterministic mode, syrk_det.cu): g is the slot workspace; the CTA of tile blockIdx.x and K piece blockIdx.y
// stores its whole 128 x 128 tile into slot blockIdx.x * gridDim.y + blockIdx.y (ldg unused)
template <typename T, bool DET, bool VEC>
__global__ void __launch_bounds__(512, 1)
syrk_f64_kernel(const T* __restrict__ x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                double* __restrict__ g, int64_t ldg, int nb, int64_t rows_per_piece) {
  extern __shared__ __align__(16) uint8_t f64_smem_raw[];
  F64Smem<T>& sm = *reinterpret_cast<F64Smem<T>*>(f64_smem_raw);
  constexpr int EV = 16 / (int)sizeof(T);  // elements per 16-byte chunk
  // tile index -> (bi, bj), bj >= bi, row-major over the block-upper triangle
  int t = blockIdx.x, bi = 0;
  while (t >= nb - bi) {
    t -= nb - bi;
    ++bi;
  }
  const int bj = bi + t;
  const bool diag = bi == bj;
  const int a0 = bi * FT, b0 = bj * FT;
  const int64_t r_begin = (int64_t)blockIdx.y * rows_per_piece;
  const int64_t r_end = min(rows, r_begin + rows_per_piece);
  if (r_begin >= r_end) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = (warp >> 2) * 32, wn = (warp & 3) * 32;
  double c[4][4][2] = {};

  auto row_ptr = [&](int64_t r) -> const T* {
    return seg_rows > 0 ? x + (r / seg_rows) * seg_stride + (r % seg_rows) * ldx : x + r * ldx;
  };
  auto load_stage = [&](int slot, int64_t k0) {
    if constexpr (VEC) {
      constexpr int CPR = FT / EV;  // chunks per row of one panel
      for (int e = tid; e < (diag ? 1 : 2) * FK * CPR; e += 512) {
        const int panel = e / (FK * CPR), rem = e % (FK * CPR);
        const int kk = rem / CPR, ch = rem % CPR;
        const int col = (panel ? a0 : b0) + ch * EV;          // panel 0 = B columns (always), 1 = A columns
        const bool ok = (k0 + kk) < r_end && col < d;
        const T* src = ok ? row_ptr(k0 + kk) + col : x;
        cp_async16_zfill(panel ? &sm.a[slot][kk][ch * EV] : &sm.b[slot][kk][ch * EV], src, ok);
      }
    } else {
      for (int e = tid; e < (diag ? 1 : 2) * FK * FT; e += 512) {
        const int panel = e / (FK * FT), rem = e % (FK * FT);
        const int kk = rem / FT, cc = rem % FT;
        const int col = (panel ? a0 : b0) + cc;
        const bool ok = (k0 + kk) < r_end && col < d;
        const T v = ok ? row_ptr(k0 + kk)[col] : T(0.0f);
        if (panel) sm.a[slot][kk][cc] = v; else sm.b[slot][kk][cc] = v;
      }
    }
  };

  const int64_t nk = (r_end - r_begin + FK - 1) / FK;
  for (int s = 0; s < FSTAGES - 1; ++s) {
    if (s < nk) load_stage(s, r_begin + (int64_t)s * FK);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int64_t kt = 0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(FSTAGES - 2) : "memory");
    __syncthreads();
    if (kt + FSTAGES - 1 < nk) load_stage((int)((kt + FSTAGES - 1) % FSTAGES), r_begin + (kt + FSTAGES - 1) * FK);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int slot = (int)(kt % FSTAGES);
    const T(*pa)[FPITCH] = diag ? sm.b[slot] : sm.a[slot];
    const T(*pb)[FPITCH] = sm.b[slot];
#pragma unroll
    for (int ks = 0; ks < FK; ks += 4) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = widen(pa[ks + (lane & 3)][wm + i * 8 + (lane >> 2)]);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = widen(pb[ks + (lane & 3)][wn + j * 8 + (lane >> 2)]);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma_f64(c[i][j][0], c[i][j][1], a[i], b[j]);
    }
  }
  if constexpr (DET) {
    double* slot = g + ((size_t)blockIdx.x * gridDim.y + blockIdx.y) * FT * FT;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<double2*>(slot + (wm + i * 8 + (lane >> 2)) * FT + wn + j * 8 + (lane & 3) * 2) =
            make_double2(c[i][j][0], c[i][j][1]);
    return;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = a0 + wm + i * 8 + (lane >> 2);
      const int cc = b0 + wn + j * 8 + (lane & 3) * 2;
#pragma unroll
      for (int u = 0; u < 2; ++u)
        if (r < d && cc + u < d) atomicAdd(g + (int64_t)r * ldg + cc + u, c[i][j][u]);
    }
}

template <typename T>
int launch_f64(const T* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, double* g, int64_t ldg,
               cudaStream_t stream) {
  int nsm = 0;
  if (int rc = device_sm_count(&nsm)) return rc;
  const int nb = (d + FT - 1) / FT;
  const int64_t tiles = (int64_t)nb * (nb + 1) / 2;
  // K pieces.  CTAs take about the same time, so what matters is how full the LAST wave is: among the piece counts
  // that leave every CTA at least 8 K steps, take the one with the best wave efficiency tiles*p / (waves * SMs)
  // (ncu, 36928 x 768 with 609 CTAs = 4.1 waves: tensor pipe 82 % of active cycles but 70 % of elapsed).
  const int64_t p_max = std::max<int64_t>(1, std::min<int64_t>(rows / (8 * FK), 64));
  int64_t pieces = 1;
  double best = 0;
  for (int64_t p = 1; p <= p_max; ++p) {
    const int64_t ctas = tiles * p, waves = (ctas + nsm - 1) / nsm;
    const double eff = (double)ctas / (double)(waves * nsm);
    if (eff > best + 0.005) best = eff, pieces = p;
  }
  int64_t rpp = (rows + pieces - 1) / pieces;
  rpp = (rpp + FK - 1) / FK * FK;
  pieces = (rows + rpp - 1) / rpp;
  constexpr int ev = 16 / (int)sizeof(T);
  const bool vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && ldx % ev == 0 && seg_stride % ev == 0 && d % ev == 0;
  dim3 grid((unsigned)tiles, (unsigned)pieces);
  const int smem = (int)sizeof(F64Smem<T>);
  if (deterministic_mode()) {
    // tile t (row-major over the block-upper triangle, as the kernel numbers them): slots t * pieces .. + pieces
    std::vector<DetItem> items;
    for (int bi = 0, t = 0; bi < nb; ++bi)
      for (int bj = bi; bj < nb; ++bj, ++t)
        items.push_back({0, d, bi * FT, bj * FT, 0, (int)(t * pieces), (int)((t + 1) * pieces)});
    void* ws = nullptr;
    DetItem* d_items = nullptr;
    if (int rc = det_workspace((size_t)tiles * pieces * FT * FT * sizeof(double), &items, stream, &ws, &d_items)) return rc;
    auto kernel = vec ? syrk_f64_kernel<T, true, true> : syrk_f64_kernel<T, true, false>;
    VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<grid, 512, smem, stream>>>(x, rows, d, ldx, seg_rows, seg_stride, static_cast<double*>(ws), 0, nb, rpp);
    VLM_CUDA(cudaGetLastError());
    count_launch();
    if (int rc = det_reduce_launch(d_items, (int)items.size(), FT, true, ws, g, ldg, nullptr, stream)) return rc;
    VLM_CUDA(cudaFreeAsync(ws, stream));
    return 0;
  }
  if (vec) {
    auto kernel = syrk_f64_kernel<T, false, true>;
    VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<grid, 512, smem, stream>>>(x, rows, d, ldx, seg_rows, seg_stride, g, ldg, nb, rpp);
  } else {
    auto kernel = syrk_f64_kernel<T, false, false>;
    VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<grid, 512, smem, stream>>>(x, rows, d, ldx, seg_rows, seg_stride, g, ldg, nb, rpp);
  }
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace
}  // namespace vlm

using namespace vlm;

extern "C" int vlm_syrk_accum_f64(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                                  int64_t seg_stride, double* g, int64_t ldg, void* stream) {
  VLM_REQUIRE(dtype == VLM_F32 || dtype == VLM_BF16 || dtype == VLM_F16, VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_f64: dtype must be VLM_F32, VLM_BF16 or VLM_F16 (got %d)", dtype);
  VLM_REQUIRE(rows >= 0 && d > 0 && g != nullptr && ldg >= d, VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_f64: bad arguments (rows=%lld d=%d)", (long long)rows, d);
  VLM_REQUIRE(rows == 0 || (x != nullptr && ldx >= d), VLM_ERR_INVALID_ARG, "vlm_syrk_accum_f64: x is NULL or ldx < d");
  VLM_REQUIRE(seg_rows >= 0 && seg_stride >= 0 && (seg_rows == 0 || rows % seg_rows == 0), VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_f64: rows (%lld) must be a multiple of seg_rows (%lld)", (long long)rows,
              (long long)seg_rows);
  VLM_REQUIRE((reinterpret_cast<uintptr_t>(g) & 7) == 0, VLM_ERR_ALIGNMENT, "vlm_syrk_accum_f64: g must be 8-byte aligned");
  if (rows == 0) return 0;
  if (int rc = require_sm100()) return rc;
  if (seg_rows >= rows) seg_rows = 0;
  auto st = static_cast<cudaStream_t>(stream);
  if (dtype == VLM_F32) return launch_f64(static_cast<const float*>(x), rows, d, ldx, seg_rows, seg_stride, g, ldg, st);
  if (dtype == VLM_BF16)
    return launch_f64(static_cast<const __nv_bfloat16*>(x), rows, d, ldx, seg_rows, seg_stride, g, ldg, st);
  return launch_f64(static_cast<const __half*>(x), rows, d, ldx, seg_rows, seg_stride, g, ldg, st);
}
