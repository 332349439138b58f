// syrk_det.cu — the deterministic mode of the Gram launches (vlm_set_deterministic): the per-call slot workspace and
// the one reduction launch that adds each tile's slots into G in a fixed order.
//
// Every Gram kernel normally adds its partial tiles straight into G (TMA reduce-adds, atomicAdd), so the order of the
// additions is the order in which CTAs finish, and the fp32 / fp64 rounding of G varies from run to run.  In the
// deterministic mode each kernel writes a partial into a slot of its own instead (syrk_2sm.cuh, syrk_i8.cuh,
// syrk_f64.cu, syrk_simt.cu); the slots of a tile are numbered consecutively in schedule order, and the schedule is a
// pure function of (rows, d, dtype, SM count), so the sums below are the same bits in every run.
#include <algorithm>

#include "common.cuh"
#include "syrk.h"

namespace vlm {
namespace {

constexpr int kDetBand = 32;  // tile rows per CTA of the reduction

// grid (items, te / kDetBand), 256 threads; consecutive threads take consecutive columns (coalesced slot reads)
template <typename T>
__global__ void __launch_bounds__(256) syrk_det_reduce_kernel(const DetItem* __restrict__ items, const T* __restrict__ ws,
                                                              int te, T* g1, int64_t ldg1,
                                                              const DetGram* __restrict__ grams) {
  const DetItem it = items[blockIdx.x];
  T* g = grams ? static_cast<T*>(grams[it.pid].g) : g1;
  const int64_t ldg = grams ? grams[it.pid].ldg : ldg1;
  const size_t tile = (size_t)te * te;
  for (int e = threadIdx.x; e < kDetBand * te; e += blockDim.x) {
    const int lr = blockIdx.y * kDetBand + e / te, lc = e % te;
    const int r = it.row0 + lr, c = it.col0 + lc;
    if (r >= it.d || c >= it.d) continue;
    if (it.mode == 1 && lr >= 128 && lc < 128) continue;
    if (it.mode == 2 && c < r) continue;
    const T* p = ws + (size_t)it.slot_begin * tile + (size_t)lr * te + lc;
    T s = *p;
    for (int k = it.slot_begin + 1; k < it.slot_end; ++k) {
      p += tile;
      s += *p;
    }
    g[(int64_t)r * ldg + c] += s;
  }
}

}  // namespace

int det_workspace(size_t slot_bytes, const std::vector<DetItem>* items, cudaStream_t stream, void** ws,
                  DetItem** d_items) {
  if (int rc = keep_async_pool()) return rc;
  slot_bytes = (slot_bytes + 255) / 256 * 256;
  const size_t item_bytes = items ? items->size() * sizeof(DetItem) : 0;
  VLM_CUDA(cudaMallocAsync(ws, std::max<size_t>(1, slot_bytes + item_bytes), stream));
  if (items) {
    *d_items = reinterpret_cast<DetItem*>(static_cast<uint8_t*>(*ws) + slot_bytes);
    // pageable source: staged before the call returns; ordered on `stream` before the launches that read it
    VLM_CUDA(cudaMemcpyAsync(*d_items, items->data(), item_bytes, cudaMemcpyHostToDevice, stream));
  }
  return 0;
}

int det_reduce_launch(const DetItem* d_items, int nitems, int te, bool f64, const void* ws, void* g1, int64_t ldg1,
                      const DetGram* grams, cudaStream_t stream) {
  if (nitems == 0) return 0;
  const dim3 grid((unsigned)nitems, (unsigned)(te / kDetBand));
  if (f64)
    syrk_det_reduce_kernel<double><<<grid, 256, 0, stream>>>(d_items, static_cast<const double*>(ws), te,
                                                              static_cast<double*>(g1), ldg1, grams);
  else
    syrk_det_reduce_kernel<float><<<grid, 256, 0, stream>>>(d_items, static_cast<const float*>(ws), te,
                                                             static_cast<float*>(g1), ldg1, grams);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace vlm
