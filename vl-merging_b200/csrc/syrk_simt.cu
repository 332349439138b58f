// syrk_simt.cu — CUDA-core Gram accumulation (device-side debug oracle / path for activations TMA
// cannot address).
// Same contract as the tensor-core kernel: G[r][c] += sum_k X[k][r]*X[k][c] for c >= r
// (src/cache_gram_matrices.py:246-254 of the reference computes the full fp64 matrix).
#include "common.cuh"
#include "syrk.h"

namespace vlm {

namespace {

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

constexpr int kTile = 64;   // output tile edge
constexpr int kKc = 16;     // rows per smem step
constexpr int kSplit = 2048;  // rows per grid.z slice

// grid: (nt, nt, ceil(rows / kSplit)); blocks with bx < by exit.  256 threads, 4x4 outputs each.
// DET (deterministic mode, syrk_det.cu): g is the slot workspace; the block of upper tile t (row-major over the
// upper triangle) and slice blockIdx.z stores its whole 64 x 64 tile into slot t * gridDim.z + blockIdx.z (ldg unused)
template <typename T, bool DET>
__global__ void __launch_bounds__(256)
syrk_simt_kernel(const T* __restrict__ x, int64_t rows, int d, int64_t ldx, float* __restrict__ g, int64_t ldg) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ float sa[kKc][kTile + 1];
  __shared__ float sb[kKc][kTile + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t r0 = (int64_t)blockIdx.z * kSplit;
  const int64_t r1 = min(rows, r0 + kSplit);
  float acc[4][4] = {};
  for (int64_t k0 = r0; k0 < r1; k0 += kKc) {
    for (int e = threadIdx.x; e < kKc * kTile; e += 256) {
      const int kk = e / kTile, c = e % kTile;
      const int64_t row = k0 + kk;
      const int ca = bi * kTile + c, cb = bj * kTile + c;
      sa[kk][c] = (row < r1 && ca < d) ? to_f32(x[row * ldx + ca]) : 0.f;
      sb[kk][c] = (row < r1 && cb < d) ? to_f32(x[row * ldx + cb]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kKc; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a[u] = sa[kk][ty * 4 + u];
        b[u] = sb[kk][tx * 4 + u];
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(a[u], b[v], acc[u][v]);
    }
    __syncthreads();
  }
  if constexpr (DET) {
    const int nt = gridDim.x, t = bi * nt - bi * (bi - 1) / 2 + (bj - bi);
    float* slot = g + ((size_t)t * gridDim.z + blockIdx.z) * kTile * kTile;
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<float4*>(slot + (ty * 4 + u) * kTile + tx * 4) =
          make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
    return;
  }
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int r = bi * kTile + ty * 4 + u, c = bj * kTile + tx * 4 + v;
      if (r < d && c < d && c >= r) atomicAdd(&g[(int64_t)r * ldg + c], acc[u][v]);
    }
}

template <bool DET>
void launch_simt(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg, dim3 grid,
                 cudaStream_t stream) {
  if (dtype == VLM_F32)
    syrk_simt_kernel<float, DET><<<grid, 256, 0, stream>>>(static_cast<const float*>(x), rows, d, ldx, g, ldg);
  else if (dtype == VLM_BF16)
    syrk_simt_kernel<__nv_bfloat16, DET>
        <<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), rows, d, ldx, g, ldg);
  else
    syrk_simt_kernel<__half, DET><<<grid, 256, 0, stream>>>(static_cast<const __half*>(x), rows, d, ldx, g, ldg);
}

}  // namespace

int syrk_simt_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                     cudaStream_t stream) {
  const int nt = (d + kTile - 1) / kTile;
  const int nz = (int)((rows + kSplit - 1) / kSplit);
  VLM_REQUIRE(nz <= 65535, VLM_ERR_INVALID_ARG, "vlm_syrk_accum_simt: rows too large");
  dim3 grid(nt, nt, nz);
  auto launch = [&](void* ws) -> int {
    if (ws)
      launch_simt<true>(x, dtype, rows, d, ldx, static_cast<float*>(ws), 0, grid, stream);
    else
      launch_simt<false>(x, dtype, rows, d, ldx, g, ldg, grid, stream);
    VLM_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  };
  if (!deterministic_mode()) return launch(nullptr);
  // upper tile t (row-major): slots t * nz .. + nz
  return det_grid_launch(d, kTile, nz, 2, false, g, ldg, stream, launch);
}

}  // namespace vlm
