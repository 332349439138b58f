// sympack.cu — the storage rule of every Gram, in three batched launches.
//
// A Gram is symmetric, and the SYRK kernels only ever form its upper triangle; the reference nevertheless
// writes the full matrix in fp64 (src/cache_gram_matrices.py:251,349: 2.15 GB for VLMo-base, 7.65 GB for ViT-L).
// Packed row-major upper triangle in fp32 — row r holds columns r..d-1 at offset r*d - r(r-1)/2 — is a quarter
// of that.  pack / unpack convert between a full Gram and that form (the on-disk container of gramfile.py and the
// exchange buffer of GramCache.all_reduce); mirror fills the lower triangle of a full Gram from its upper one, in
// place.  All three are HBM-bound copies; unpack and mirror go through 32x32 shared-memory tiles so that the mirrored
// half is written with coalesced rows too.
#include <vector>

#include "common.cuh"
#include "../../include/vlmerge.h"

namespace vlm {
namespace {

__device__ __forceinline__ int64_t packed_row_offset(int r, int d) {
  return (int64_t)r * d - ((int64_t)r * (r - 1)) / 2;
}

// All Grams of a cache in ONE launch (GramCache.all_reduce packs / unpacks 96 Grams, finalize mirrors them).  A block
// owns one 32-row BAND of one Gram and walks its tiles from the diagonal to the right edge with several independent
// loads in flight per thread: the first version (one 32 x 32 tile per block, 262 K blocks moving 8 KB each) ran at
// 1 TB/s — block turnover, not memory, was the limit.
struct SymItemDev {
  const void* full_c;   // pack: source; unpack: destination, mirror: read and written (cast away const)
  void* packed;
  int d;
  int first_band;       // index of this problem's first 32-row band in the flattened grid
  int64_t ld;
};

__device__ __forceinline__ SymItemDev locate_band(const SymItemDev* __restrict__ items, int n, int band, int* bi) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {            // the last item whose first_band <= band
    const int mid = (lo + hi + 1) >> 1;
    if (items[mid].first_band <= band) lo = mid; else hi = mid - 1;
  }
  const SymItemDev it = items[lo];
  *bi = band - it.first_band;
  return it;
}

// 8 warps x 4 rows; a row is one contiguous run on both sides; four 128-byte pieces in flight per warp
template <typename T>
__global__ void __launch_bounds__(256) sym_pack_batch_kernel(const SymItemDev* __restrict__ items, int n) {
  int bi;
  const SymItemDev it = locate_band(items, n, blockIdx.x, &bi);
  const T* __restrict__ g = static_cast<const T*>(it.full_c);
  T* __restrict__ packed = static_cast<T*>(it.packed);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int d = it.d;
  for (int rr = warp; rr < 32; rr += 8) {
    const int r = bi * 32 + rr;
    if (r >= d) break;
    const T* src = g + (int64_t)r * it.ld;
    T* dst = packed + packed_row_offset(r, d) - r;
    for (int c = r + lane; c < d; c += 128) {
      T v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (c + 32 * u < d) v[u] = src[c + 32 * u];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (c + 32 * u < d) dst[c + 32 * u] = v[u];
    }
  }
}

// the band's tiles two at a time: 8 independent loads per thread, then the rows of the tiles and, through shared memory,
// their mirror images
template <typename T>
__global__ void __launch_bounds__(256) sym_unpack_batch_kernel(const SymItemDev* __restrict__ items, int n) {
  int bi;
  const SymItemDev it = locate_band(items, n, blockIdx.x, &bi);
  const int d = it.d, nt = (d + 31) / 32;
  const T* __restrict__ packed = static_cast<const T*>(it.packed);
  T* __restrict__ out = static_cast<T*>(const_cast<void*>(it.full_c));
  __shared__ T tile[2][32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int bj0 = bi; bj0 < nt; bj0 += 2) {
    T v[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = bi * 32 + ty + 8 * k, c = (bj0 + u) * 32 + tx;
        v[u][k] = T(0);
        if (bj0 + u < nt && r < d && c < d)
          v[u][k] = (c >= r) ? packed[packed_row_offset(r, d) + (c - r)] : packed[packed_row_offset(c, d) + (r - c)];
      }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = bi * 32 + ty + 8 * k, c = (bj0 + u) * 32 + tx;
        if (bj0 + u < nt && r < d && c < d) out[(int64_t)r * it.ld + c] = v[u][k];
        tile[u][ty + 8 * k][tx] = v[u][k];
      }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (bj0 + u >= nt || bj0 + u == bi) continue;        // the diagonal tile was written whole above
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = (bj0 + u) * 32 + ty + 8 * k, c = bi * 32 + tx;    // mirrored position, below the diagonal
        if (r < d && c < d) out[(int64_t)r * it.ld + c] = tile[u][tx][ty + 8 * k];
      }
    }
    __syncthreads();
  }
}

// in place, the band's tiles two at a time through shared memory: the upper tiles are read and their transposes
// written below the diagonal (inside the diagonal tile only the elements below it)
template <typename T>
__global__ void __launch_bounds__(256) sym_mirror_batch_kernel(const SymItemDev* __restrict__ items, int n) {
  int bi;
  const SymItemDev it = locate_band(items, n, blockIdx.x, &bi);
  const int d = it.d, nt = (d + 31) / 32;
  T* g = static_cast<T*>(const_cast<void*>(it.full_c));
  __shared__ T tile[2][32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int bj0 = bi; bj0 < nt; bj0 += 2) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = bi * 32 + ty + 8 * k, c = (bj0 + u) * 32 + tx;
        tile[u][ty + 8 * k][tx] = (bj0 + u < nt && r < d && c < d) ? g[(int64_t)r * it.ld + c] : T(0);
      }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (bj0 + u >= nt) continue;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int rr = ty + 8 * k;
        const int r = (bj0 + u) * 32 + rr, c = bi * 32 + tx;      // mirrored position
        if (r < d && c < d && (bj0 + u != bi || tx < rr)) g[(int64_t)r * it.ld + c] = tile[u][tx][rr];
      }
    }
    __syncthreads();
  }
}

enum class SymOp { kPack, kUnpack, kMirror };

template <typename T>
void launch_sym(SymOp op, unsigned bands, const SymItemDev* items, int n, cudaStream_t s) {
  if (op == SymOp::kPack) sym_pack_batch_kernel<T><<<bands, 256, 0, s>>>(items, n);
  else if (op == SymOp::kUnpack) sym_unpack_batch_kernel<T><<<bands, 256, 0, s>>>(items, n);
  else sym_mirror_batch_kernel<T><<<bands, 256, 0, s>>>(items, n);
}

int sym_batch(const vlm_sym_item* items, int n, int dtype, SymOp op, cudaStream_t s, const char* who) {
  VLM_REQUIRE(items != nullptr && n >= 0, VLM_ERR_INVALID_ARG, "%s: bad arguments", who);
  VLM_REQUIRE(dtype == VLM_F32 || dtype == VLM_F64, VLM_ERR_INVALID_ARG, "%s: dtype must be VLM_F32 or VLM_F64 (got %d)", who, dtype);
  if (n == 0) return 0;
  std::vector<SymItemDev> host(n);
  int64_t bands = 0;
  for (int i = 0; i < n; ++i) {
    VLM_REQUIRE(items[i].full != nullptr && (items[i].packed != nullptr || op == SymOp::kMirror) && items[i].d > 0 &&
                    items[i].ld >= items[i].d,
                VLM_ERR_INVALID_ARG, "%s: bad item %d", who, i);
    VLM_REQUIRE(bands + (items[i].d + 31) / 32 < ((int64_t)1 << 31), VLM_ERR_INVALID_ARG, "%s: too many bands", who);
    host[i] = {items[i].full, items[i].packed, items[i].d, (int)bands, items[i].ld};
    bands += (items[i].d + 31) / 32;
  }
  SymItemDev* dev = nullptr;
  if (int rc = keep_async_pool()) return rc;
  VLM_CUDA(cudaMallocAsync(&dev, sizeof(SymItemDev) * n, s));
  VLM_CUDA(cudaMemcpyAsync(dev, host.data(), sizeof(SymItemDev) * n, cudaMemcpyHostToDevice, s));   // pageable: staged before return
  if (dtype == VLM_F32) launch_sym<float>(op, (unsigned)bands, dev, n, s);
  else launch_sym<double>(op, (unsigned)bands, dev, n, s);
  VLM_CUDA(cudaGetLastError());
  VLM_CUDA(cudaFreeAsync(dev, s));
  count_launch();
  return 0;
}

}  // namespace
}  // namespace vlm

using namespace vlm;

extern "C" int vlm_sym_pack_upper_batch(const vlm_sym_item* items, int n, int dtype, void* stream) {
  return sym_batch(items, n, dtype, SymOp::kPack, static_cast<cudaStream_t>(stream), "vlm_sym_pack_upper_batch");
}
extern "C" int vlm_sym_unpack_batch(const vlm_sym_item* items, int n, int dtype, void* stream) {
  return sym_batch(items, n, dtype, SymOp::kUnpack, static_cast<cudaStream_t>(stream), "vlm_sym_unpack_batch");
}
extern "C" int vlm_sym_mirror_batch(const vlm_sym_item* items, int n, int dtype, void* stream) {
  return sym_batch(items, n, dtype, SymOp::kMirror, static_cast<cudaStream_t>(stream), "vlm_sym_mirror_batch");
}
