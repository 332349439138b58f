// symreduce.cu — the data-parallel exchange step of Gram caching as ONE kernel over NVSwitch multicast memory.
//
// GramCache.all_reduce() sums the per-rank Gram arenas (the reference has no such step: every DDP rank overwrites the
// same file, src/cache_gram_matrices.py:349).  Its default form is pack -> NCCL all-reduce -> unpack: three passes over
// a staging buffer.  When the arena lives in symmetric memory with a multicast mapping (torch symmetric memory:
// cuMulticast objects behind it), the same result needs no staging at all:
//
//   * the 32-row bands of every live Gram (from the diagonal to the right edge) are dealt to the ranks (band bi of
//     Gram i: rank (i + bi) mod world);
//   * the owner of a band reads it with multimem.ld_reduce.add — ONE load returns the sum over all ranks' arenas, formed
//     inside the switch (SASS: LDGMC.ADD) — and writes it back with multimem.st, which the switch broadcasts into every
//     rank's arena; the lower triangles are then mirrored locally (vlm_sym_mirror_batch, one launch).
//
// pack + reduce-scatter + all-gather + unpack in one launch; every element of the upper triangles crosses NVLink once
// in each direction, and every rank ends up with bit-identical Grams (one owner computes each value).  The launch must be bracketed by cross-rank barriers (GramCache does that with the
// symmetric-memory handle's barrier): all ranks' SYRK launches before, nobody reads a Gram until all stores landed.
//
// vlm_sym_reduce_multimem is the reduce-scatter form (GramCache.reduce_scatter): every Gram has one owner rank, which
// reads it the same way and keeps the sum in its own arena only (plain stores, no broadcast).
#include <vector>

#include "common.cuh"
#include "../../include/vlmerge.h"

namespace vlm {
namespace {

struct SpanDev {
  uint64_t offset_bytes;   // of the Gram inside the arena
  int d;
  int first_band;          // index of this Gram's first 32-row band in the flattened grid
  int64_t ld;
};

__device__ __forceinline__ float4 mc_ld_reduce(const float* p) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void mc_st(float* p, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
__device__ __forceinline__ double mc_ld_reduce(const double* p) {
  double v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void mc_st(double* p, double v) {
  asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

__device__ __forceinline__ SpanDev locate_band(const SpanDev* __restrict__ spans, int n, int band, int* item, int* bi) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {            // the last span whose first_band <= band
    const int mid = (lo + hi + 1) >> 1;
    if (spans[mid].first_band <= band) lo = mid; else hi = mid - 1;
  }
  *item = lo;
  *bi = band - spans[lo].first_band;
  return spans[lo];
}

// Band (item, bi) — rows 32 bi .. 32 bi + 31 of Gram `item`, from the diagonal tile to the right edge — belongs to rank
// (item + bi) % world; the other ranks' blocks exit at once.  A warp owns four rows of the band and walks each from
// column 32 bi to d in fully contiguous pieces: 32 lanes x 16 bytes per multimem instruction, four instructions in
// flight (multimem.ld_reduce x 4, then multimem.st x 4).  The sums go back into every rank's arena through the
// switch; the lower triangles are mirrored locally afterwards (vlm_sym_mirror_batch), so every element of the
// upper triangles crosses NVLink once in each direction.  (A first version dealt 32 x 32 tiles to the ranks: 128-byte
// runs, 1.9 ms for the 538 MB of VLMo-base at N = 2.)
//
// kLocal (vlm_sym_reduce_multimem, the reduce-scatter form): the caller passes only the spans it owns, so every band is
// its own; the sums go to local_base + offset with plain stores instead of the multimem.st broadcast.
template <typename T, typename V, int VE, bool kLocal>   // V: the access type (float4 / double), VE elements each
__global__ void __launch_bounds__(256) sym_allreduce_mc_kernel(uint8_t* __restrict__ mc_base, const SpanDev* __restrict__ spans,
                                                                int n, int rank, int world, uint8_t* __restrict__ local_base) {
  int item, bi;
  const SpanDev sp = locate_band(spans, n, blockIdx.x, &item, &bi);
  if (!kLocal && (item + bi) % world != rank) return;
  const int d = sp.d;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T* g = reinterpret_cast<T*>(mc_base + sp.offset_bytes);
  T* out = kLocal ? reinterpret_cast<T*>(local_base + sp.offset_bytes) : g;
  constexpr int kStep = 32 * VE;            // elements per warp instruction
  for (int rr = warp; rr < 32; rr += 8) {
    const int r = bi * 32 + rr;
    if (r >= d) break;
    T* row = g + (int64_t)r * sp.ld;
    T* out_row = out + (int64_t)r * sp.ld;
    for (int c = bi * 32 + lane * VE; c < d; c += 4 * kStep) {
      V s[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (c + u * kStep < d) s[u] = mc_ld_reduce(row + c + u * kStep);   // d % VE == 0 (host): a vector is in or out
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (c + u * kStep >= d) continue;
        if (kLocal)
          *reinterpret_cast<V*>(out_row + c + u * kStep) = s[u];
        else
          mc_st(row + c + u * kStep, s[u]);
      }
    }
  }
}

int upload_spans(const vlm_sym_span* spans, int n, int dtype, const char* who, cudaStream_t s, SpanDev** dev, int64_t* bands) {
  std::vector<SpanDev> host(n);
  *bands = 0;
  for (int i = 0; i < n; ++i) {
    VLM_REQUIRE(spans[i].d > 0 && spans[i].ld >= spans[i].d, VLM_ERR_INVALID_ARG, "%s: bad span %d", who, i);
    // multimem accesses are 16 bytes wide in fp32 (8 in fp64) and must be naturally aligned
    VLM_REQUIRE(spans[i].offset_bytes % 16 == 0 && (dtype == VLM_F64 || (spans[i].d % 4 == 0 && spans[i].ld % 4 == 0)),
                VLM_ERR_ALIGNMENT, "%s: span %d needs a 16-byte aligned offset and, in fp32, d and ld multiples of 4", who, i);
    const int64_t nt = (spans[i].d + 31) / 32;
    VLM_REQUIRE(*bands + nt < ((int64_t)1 << 31), VLM_ERR_INVALID_ARG, "%s: too many bands", who);
    host[i] = {spans[i].offset_bytes, spans[i].d, (int)*bands, spans[i].ld};
    *bands += nt;
  }
  if (int rc = keep_async_pool()) return rc;
  VLM_CUDA(cudaMallocAsync(dev, sizeof(SpanDev) * n, s));
  VLM_CUDA(cudaMemcpyAsync(*dev, host.data(), sizeof(SpanDev) * n, cudaMemcpyHostToDevice, s));   // pageable: staged before return
  return 0;
}

}  // namespace
}  // namespace vlm

using namespace vlm;

// Both entry points: argument checks, span upload, one launch.  kLocal: see sym_allreduce_mc_kernel.
template <bool kLocal>
static int launch_mc(const char* who, void* multicast_base, void* local_base, const vlm_sym_span* spans, int n, int dtype,
                     int rank, int world, void* stream) {
  VLM_REQUIRE(dtype == VLM_F32 || dtype == VLM_F64, VLM_ERR_INVALID_ARG, "%s: dtype must be VLM_F32 or VLM_F64 (got %d)",
              who, dtype);
  if (n == 0) return 0;
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SpanDev* dev = nullptr;
  int64_t bands = 0;
  if (int rc = upload_spans(spans, n, dtype, who, s, &dev, &bands)) return rc;
  uint8_t* mc = static_cast<uint8_t*>(multicast_base);
  uint8_t* local = static_cast<uint8_t*>(local_base);
  if (dtype == VLM_F32)
    sym_allreduce_mc_kernel<float, float4, 4, kLocal><<<(unsigned)bands, 256, 0, s>>>(mc, dev, n, rank, world, local);
  else
    sym_allreduce_mc_kernel<double, double, 1, kLocal><<<(unsigned)bands, 256, 0, s>>>(mc, dev, n, rank, world, local);
  VLM_CUDA(cudaGetLastError());
  VLM_CUDA(cudaFreeAsync(dev, s));
  count_launch();
  return 0;
}

extern "C" int vlm_sym_allreduce_multimem(void* multicast_base, const vlm_sym_span* spans, int n, int dtype, int rank,
                                          int world, void* stream) {
  VLM_REQUIRE(multicast_base != nullptr && spans != nullptr && n >= 0 && world >= 1 && rank >= 0 && rank < world,
              VLM_ERR_INVALID_ARG, "vlm_sym_allreduce_multimem: bad arguments");
  return launch_mc<false>("vlm_sym_allreduce_multimem", multicast_base, nullptr, spans, n, dtype, rank, world, stream);
}

extern "C" int vlm_sym_reduce_multimem(void* multicast_base, void* local_base, const vlm_sym_span* spans, int n, int dtype,
                                       void* stream) {
  VLM_REQUIRE(multicast_base != nullptr && local_base != nullptr && spans != nullptr && n >= 0, VLM_ERR_INVALID_ARG,
              "vlm_sym_reduce_multimem: bad arguments");
  // the plain stores are as wide as the multimem loads: the local arena needs the same alignment as the multicast one
  VLM_REQUIRE(reinterpret_cast<uintptr_t>(local_base) % 16 == 0, VLM_ERR_ALIGNMENT,
              "vlm_sym_reduce_multimem: local_base must be 16-byte aligned");
  return launch_mc<true>("vlm_sym_reduce_multimem", multicast_base, local_base, spans, n, dtype, 0, 1, stream);
}
