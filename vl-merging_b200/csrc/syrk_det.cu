// syrk_det.cu — the deterministic mode of the Gram launches (vlm_set_deterministic): the per-call slot workspace and
// the one reduction launch that adds each tile's slots into G in a fixed order.
//
// Every Gram kernel normally adds its partial tiles straight into G (TMA reduce-adds, atomicAdd), so the order of the
// additions is the order in which CTAs finish, and the fp32 / fp64 rounding of G varies from run to run.  In the
// deterministic mode each kernel writes a partial into a slot of its own instead (syrk_2sm.cuh, syrk_i8.cuh,
// syrk_f64.cu, syrk_simt.cu); the slots of a tile are numbered consecutively in schedule order, and the schedule is a
// pure function of (rows, d, dtype, SM count), so the sums below are the same bits in every run.
//
// det_launch is the one launch sequence of the mode, for every Gram kernel: workspace, the kernel's launch, reduction,
// and the workspace freed again whatever fails on the way.  The CTA-pair kernels describe their slots to TMA (the slot
// map stands in for their G map); the fp64 and CUDA-core kernels, whose grids are regular tile grids, go through
// det_grid_launch.
#include <algorithm>
#include <vector>

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

namespace {
int det_reduce_launch(const DetReduce& red, int te, bool f64, const void* ws, cudaStream_t stream) {
  if (red.nitems == 0) return 0;
  const dim3 grid((unsigned)red.nitems, (unsigned)(te / kDetBand));
  if (f64)
    syrk_det_reduce_kernel<double><<<grid, 256, 0, stream>>>(red.d_items, static_cast<const double*>(ws), te,
                                                              static_cast<double*>(red.g), red.ldg, red.grams);
  else
    syrk_det_reduce_kernel<float><<<grid, 256, 0, stream>>>(red.d_items, static_cast<const float*>(ws), te,
                                                             static_cast<float*>(red.g), red.ldg, red.grams);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}
}  // namespace

int det_launch(int nslots, int te, bool f64, const std::vector<DetItem>* items, DetReduce red, CUtensorMap* slot_map,
               cudaStream_t stream, const std::function<int(void*)>& launch) {
  if (int rc = keep_async_pool()) return rc;
  const size_t slot_bytes = ((size_t)nslots * te * te * (f64 ? 8 : 4) + 255) / 256 * 256;
  const size_t item_bytes = items ? items->size() * sizeof(DetItem) : 0;
  void* ws = nullptr;
  VLM_CUDA(cudaMallocAsync(&ws, std::max<size_t>(1, slot_bytes + item_bytes), stream));
  auto run = [&]() -> int {
    if (items) {
      red.d_items = reinterpret_cast<const DetItem*>(static_cast<uint8_t*>(ws) + slot_bytes);
      red.nitems = (int)items->size();
      // pageable source: staged before the call returns; ordered on `stream` before the launches that read it
      VLM_CUDA(cudaMemcpyAsync(const_cast<DetItem*>(red.d_items), items->data(), item_bytes, cudaMemcpyHostToDevice,
                               stream));
    }
    if (slot_map) {
      if (int rc = encode_matrix_map(slot_map, f64, ws, (int64_t)nslots * te, te, te)) return rc;
    }
    if (int rc = launch(ws)) return rc;
    return det_reduce_launch(red, te, f64, ws, stream);
  };
  if (int rc = run()) {
    cudaFreeAsync(ws, stream);  // the error that stopped the sequence is the one reported
    return rc;
  }
  VLM_CUDA(cudaFreeAsync(ws, stream));
  return 0;
}

int det_grid_launch(int d, int te, int pieces, int mode, bool f64, void* g, int64_t ldg, cudaStream_t stream,
                    const std::function<int(void*)>& launch) {
  const int nb = (d + te - 1) / te;
  std::vector<DetItem> items;
  for (int bi = 0, t = 0; bi < nb; ++bi)
    for (int bj = bi; bj < nb; ++bj, ++t)
      items.push_back({0, d, bi * te, bj * te, mode, t * pieces, (t + 1) * pieces, 0});
  return det_launch((int)items.size() * pieces, te, f64, &items, {nullptr, 0, g, ldg, nullptr}, nullptr, stream,
                    launch);
}

}  // namespace vlm
