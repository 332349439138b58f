// syrk_pair.cu — host side of kernel (a), the CTA-pair SYRK (device code: syrk_2sm.cuh): tensor maps, the
// K-aligned work decomposition, schedule cache, single and batched launches, and the fp32 -> {hi, lo} split.
//
// Work unit = a 256 x 256 SUPER-TILE (a, b), b >= a, of the block-upper triangle of G, computed by a cluster of two
// CTAs with ONE tcgen05.mma.cta_group::2 instruction stream (M = 256 over the pair): CTA r holds row block 2a+r
// (its 128 rows of A and of the accumulator) and column block 2b+r (its half of B).  X is described to TMA as a 3-D
// tensor {column in group, row, column group} (strides: element, row pitch, 128 B), so ONE cp.async.bulk.tensor box
// {128 B, BK rows, groups per block} fetches a whole 128-column block in exactly the [group][row][128 B] order of
// the canonical MN-major UMMA layout: 2 TMA instructions and 32 KB per CTA per stage.  Widths that are not whole
// 128-byte column groups, and operands TMA cannot address, run on the CUDA-core kernel instead (syrk_simt.cu; the
// condition is syrk_pair_supported).  History (DESIGN.md 4a): a single-CTA kernel (removed), then CTA pairs with two
// cta_group::1 streams and TMA multicast (48 KB taken in per SM per stage: ingest-bound at 84 % tensor pipe), then
// this one (93 %).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <map>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "syrk.h"
#include "umma.cuh"

namespace vlm {

namespace {

constexpr int kStagingBytes = 16384;
constexpr int kThreads = 256;
constexpr int kTmemCols = 512;
constexpr int kAccCols = 256;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// L2 eviction policies (createpolicy): the activation X is a stream that is only re-read within a short window
// (by the other clusters sweeping the same rows), the Gram tiles are re-read and re-written by every K segment's
// reduce-add for the whole launch.
__device__ __forceinline__ uint64_t l2_policy(int kind) {  // 0 evict_normal, 1 evict_first, 2 evict_last
  uint64_t p;
  if (kind == 1)
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2)
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_reduce_add_2d_hint(const CUtensorMap* tm, const void* smem_src, int c0, int c1,
                                                       uint64_t pol) {
  asm volatile(
      "cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
      ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(pol)
      : "memory");
}

__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* tm, const void* smem_src, int c0, int c1,
                                                  uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(pol)
               : "memory");
}

// One unit of work of a cluster in a BATCHED launch (several independent Gram problems in one grid): as PairSeg,
// plus which problem it belongs to (index into the tensor-map array) and that problem's column count.
// cps = chunks per row segment of a segmented activation (0: contiguous rows, 3-D tensor map).
// slot (deterministic mode only, where single launches use this layout too): workspace slot << 1 | 1 if an earlier
// segment of the same cluster already wrote that slot (det_slots).
struct BatchSeg {
  int32_t sa, sb, k0, k1, pid, d, cps, slot;
};
__device__ __forceinline__ void tensormap_acquire(const CUtensorMap* tm) {
  asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

}  // namespace
}  // namespace vlm

#include "syrk_2sm.cuh"
#include "syrk_i8.cuh"

namespace vlm {
namespace {
// d_segs: PairSegs, or in the deterministic mode BatchSegs with workspace slots, plus the reduction's tile list
struct DeviceSchedule2 {
  int nclusters = 0;
  void* d_segs = nullptr;
  int* d_off = nullptr;
  DetItem* d_items = nullptr;
  int nitems = 0, nslots = 0;
};
std::mutex g_mu2;
// (device, chunks, d, chunk rows or -8 for int8, SMs, deterministic)
typedef std::tuple<int, int64_t, int, int, int, bool> ScheduleKey;
std::map<ScheduleKey, DeviceSchedule2> g_sched2;
// schedules evicted from the cache: freed at the NEXT eviction, after a device synchronisation, never while a
// launch that was handed their pointers may still be pending (the lock is held from lookup to launch)
std::vector<DeviceSchedule2> g_retired2;

// Deterministic mode: gives every (problem, super-tile, cluster) a workspace slot of its own.  The slots of one tile
// are numbered consecutively in schedule order (cluster by cluster, each cluster's segments in order), which is the
// order the reduction adds them in.  Sets seg.slot = slot << 1 | (1 when an earlier segment of the same cluster opened
// the slot: that one stores, the later ones add); returns the number of slots and one DetItem per tile.  same_g (grouped
// launches): problem p adds into the G of problem same_g[p] <= p, so that problems sharing a G share its tiles' items.
int det_slots(std::vector<BatchSeg>* segs, const std::vector<int>& off, std::vector<DetItem>* items,
              const std::vector<int>* same_g = nullptr) {
  std::map<std::tuple<int, int, int>, int> tile_of;  // (G, super row, super column) -> index into items
  std::vector<std::vector<int>> opened;              // per tile: its temporary slot ids, in schedule order
  std::vector<int> temp(segs->size());
  int ntemp = 0;
  items->clear();
  for (size_t c = 0; c + 1 < off.size(); ++c) {
    std::map<int, int> mine;  // tile -> temporary slot id of this cluster
    for (int s = off[c]; s < off[c + 1]; ++s) {
      BatchSeg& q = (*segs)[s];
      const int sb = q.sb & 0xFFFF;  // (the int8 schedule keeps the phase in the bits above)
      const int gp = same_g ? (*same_g)[q.pid] : q.pid;
      auto t = tile_of.emplace(std::make_tuple(gp, q.sa, sb), (int)items->size());
      if (t.second) {
        items->push_back({gp, q.d, q.sa * 256, sb * 256, q.sa == sb ? 1 : 0, 0, 0, 0});
        opened.emplace_back();
      }
      const int tile = t.first->second;
      auto m = mine.find(tile);
      if (m == mine.end()) {
        mine.emplace(tile, ntemp);
        opened[tile].push_back(ntemp);
        temp[s] = ntemp++;
        q.slot = 0;
      } else {
        temp[s] = m->second;
        q.slot = 1;
      }
    }
  }
  std::vector<int> final_id(ntemp);
  int next = 0;
  for (size_t t = 0; t < items->size(); ++t) {
    (*items)[t].slot_begin = next;
    for (int id : opened[t]) final_id[id] = next++;
    (*items)[t].slot_end = next;
  }
  for (size_t s = 0; s < segs->size(); ++s) (*segs)[s].slot |= final_id[temp[s]] << 1;
  return next;
}

// The device copy of the schedule `build` makes for `key`, built and uploaded on first use.  Call with g_mu2 held
// until the launch that reads it is enqueued.  Deterministic keys: as BatchSegs of one problem of width d (cps chunks
// per row segment) with their workspace slots.
template <typename Build>
int cached_schedule(const ScheduleKey& key, Build build, cudaStream_t stream, const DeviceSchedule2** out, int d = 0,
                    int cps = 0) {
  auto it = g_sched2.find(key);
  if (it == g_sched2.end()) {
    if (g_sched2.size() >= 512) {  // ragged workloads (a new row count every call): start over, do not grow forever
      VLM_CUDA(cudaDeviceSynchronize());  // launches that read the schedules retired LAST time have finished
      for (auto& ds : g_retired2) {
        cudaFree(ds.d_segs);
        cudaFree(ds.d_off);
        cudaFree(ds.d_items);
      }
      g_retired2.clear();
      for (auto& kv : g_sched2) g_retired2.push_back(kv.second);
      g_sched2.clear();
    }
    std::vector<PairSeg> segs;
    std::vector<int> off;
    build(&segs, &off);
    DeviceSchedule2 ds;
    ds.nclusters = (int)off.size() - 1;
    const void* seg_src = segs.data();
    size_t seg_bytes = segs.size() * sizeof(PairSeg);
    std::vector<BatchSeg> bsegs;
    std::vector<DetItem> items;
    if (std::get<5>(key)) {
      for (const PairSeg& s : segs) bsegs.push_back({s.sa, s.sb, s.k0, s.k1, 0, d, cps, 0});
      ds.nslots = det_slots(&bsegs, off, &items);
      ds.nitems = (int)items.size();
      seg_src = bsegs.data();
      seg_bytes = bsegs.size() * sizeof(BatchSeg);
      VLM_CUDA(cudaMalloc(&ds.d_items, std::max<size_t>(1, items.size()) * sizeof(DetItem)));
      VLM_CUDA(cudaMemcpyAsync(ds.d_items, items.data(), items.size() * sizeof(DetItem), cudaMemcpyHostToDevice, stream));
    }
    VLM_CUDA(cudaMalloc(&ds.d_segs, std::max<size_t>(1, seg_bytes)));
    VLM_CUDA(cudaMalloc(&ds.d_off, off.size() * sizeof(int)));
    VLM_CUDA(cudaMemcpyAsync(ds.d_segs, seg_src, seg_bytes, cudaMemcpyHostToDevice, stream));
    VLM_CUDA(cudaMemcpyAsync(ds.d_off, off.data(), off.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    VLM_CUDA(cudaStreamSynchronize(stream));
    it = g_sched2.emplace(key, ds).first;
  }
  *out = &it->second;
  return 0;
}

// The slot workspace of the deterministic mode as a 2-D TMA tensor {256 columns, slots * 256 rows}, with the box and
// swizzle of the G map it stands in for (fp32: 32 x 128, fp64: 16 x 128)
int encode_slot_map(EncodeTiledFn encode, void* ws, int nslots, bool f64, CUtensorMap* tm) {
  const int elem = f64 ? 8 : 4;
  cuuint64_t gdim[2] = {256, (cuuint64_t)nslots * 256};
  cuuint64_t gstr[1] = {(cuuint64_t)256 * elem};
  cuuint32_t box[2] = {(cuuint32_t)(128 / elem), 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(tm, f64 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ws, gdim, gstr, box,
                      estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(slot workspace) failed: CUresult %d", (int)r);
  return 0;
}

inline int elem_bytes(int dtype) { return (dtype == VLM_F32 || dtype == VLM_TF32X2) ? 4 : 2; }
// rows of X per pipeline stage = schedule chunk
inline int chunk_rows(int dtype) { return dtype == VLM_TF32X2 ? 16 : 128 / elem_bytes(dtype); }

// X as a 3-D tensor {column in group, row, column group} (strides: row pitch, 128 bytes); G as a 2-D fp32 tensor.
// seg_rows > 0: 4-D, {column in group, row in segment, column group, segment}.
// VLM_TF32X2: 4-D, {column in group, row, column group, plane}, planes rows * ldx elements apart, and one box
// fetches both planes of a 128-column block for 16 rows.
int encode_maps(EncodeTiledFn encode, const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                int64_t seg_stride, float* g, int64_t ldg, CUtensorMap* tm_x, CUtensorMap* tm_g) {
  const int elem = elem_bytes(dtype);
  const int bk = chunk_rows(dtype), gc = 128 / elem;
  {
    // fp32 activations are described to TMA as TFLOAT32: the copy engine then ROUNDS each value to TF32 on its
    // way into shared memory.  With the plain FLOAT32 element type the tensor core truncates the low 13
    // mantissa bits of both operands instead, a systematic -6.8e-4 relative bias on every Gram (measured on the
    // B200, 36928 x 3072: rel. Frobenius error 7.6e-4 truncated vs 2.5e-5 rounded, same speed).
    // (The planes of VLM_TF32X2 hold TF32 values already: the conversion is then the identity.)
    const CUtensorMapDataType dt = elem == 4             ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32
                                   : dtype == VLM_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                       : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const bool split = dtype == VLM_TF32X2;
    const bool segmented = !split && seg_rows > 0;
    const int rank = (split || segmented) ? 4 : 3;
    cuuint64_t gdim[4] = {(cuuint64_t)gc, (cuuint64_t)(segmented ? seg_rows : rows), (cuuint64_t)(d / gc),
                          (cuuint64_t)(split ? 2 : segmented ? rows / seg_rows : 1)};
    cuuint64_t gstr[3] = {(cuuint64_t)ldx * elem, 128, (cuuint64_t)(split ? rows * ldx : seg_stride) * elem};
    cuuint32_t box[4] = {(cuuint32_t)gc, (cuuint32_t)bk, (cuuint32_t)elem /* groups per 128-column block */,
                         (cuuint32_t)(split ? 2 : 1)};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUtensorMapSwizzle swz = elem == 4 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
    CUresult r = encode(tm_x, dt, rank, const_cast<void*>(x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(X, %d-D) failed: CUresult %d", rank, (int)r);
  }
  {
    cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)d};
    cuuint64_t gstr[1] = {(cuuint64_t)ldg * 4};
    cuuint32_t box[2] = {32, 128};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(tm_g, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, g, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(G) failed: CUresult %d", (int)r);
  }
  return 0;
}

// device scratch for batched launches: a small ring per (device, stream); reuse is ordered by the stream itself
struct Scratch {
  void* ptr[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t cap[4] = {0, 0, 0, 0};
  int next = 0;
};
std::map<std::pair<int, cudaStream_t>, Scratch> g_scratch;

// bits 0-1: policy of the X loads, bits 2-3: policy of the G reduce-adds (0 normal, 1 evict_first, 2 evict_last)
int l2_hints() {
  static const int v = [] {
    const char* e = getenv("VLM_SYRK_L2_HINTS");
    return e ? atoi(e) : (2 << 2);
  }();
  return v;
}

typedef void (*PairKernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap*, const void*, const int*, int, int,
                           int);
template <bool BATCH, bool DET>
PairKernel pick_kernel(int dtype) {
  if (dtype == VLM_TF32X2) return syrk_2sm_kernel<4, 2, BATCH, true, DET>;
  if (dtype == VLM_F32) return syrk_2sm_kernel<4, 2, BATCH, false, DET>;
  if (dtype == VLM_BF16) return syrk_2sm_kernel<2, 1, BATCH, false, DET>;
  return syrk_2sm_kernel<2, 0, BATCH, false, DET>;
}

}  // namespace

// Work decomposition for the CTA-pair kernel: K-ALIGNED tile ownership.
//
// Every cluster sweeps the rows of X from the top for "its" super-tile, so at any moment all clusters read
// the same thin band of rows: X streams from HBM once, every re-read (each column block is used by ~nsb
// tiles) hits L2, and no row panel has to fit in L2.  T super-tiles over C clusters:
//   * T >= C: floor(T/C) rounds of whole tiles (cluster c owns tiles c, c+C, ...), then the T mod C
//     left-over tiles are cut along K into C equal shares (stream-K) so that nobody idles;
//   * T <  C: every tile is cut along K into m = floor(C/T) equal pieces with the SAME boundaries for all
//     tiles (clusters on different tiles then stay aligned in K); T*m clusters are used.
// With at least one round, a cluster's left-over pieces are merged into its last sweep next to the own-tile
// segment covering the same rows (see below), so they too read the band of X that is in L2.  The reduce-adds
// into G carry an L2 evict_last policy: each tile is re-read and re-written by every K segment while ~45 MB of X
// stream through L2 in between (ncu, 36928 x 3072 fp32: DRAM read+write 636 MB without either, 526 MB with both).
// A K range longer than seg_cap chunks is processed as consecutive segments of at most seg_cap chunks:
// each ends with its own reduce-add into G (hidden behind the next segment's mainloop by the double-
// buffered TMEM accumulator), which bounds the tensor core's truncating fp32 accumulation.
// Measured against the alternatives on the B200 (36928 x 3072 fp32): panel-major stream-K with chunk-granular
// shares 672 TFLOP/s (many short segments whose 128 KB epilogues cannot hide), this schedule 753-758; an L2
// look-ahead prefetch (cp.async.bulk.prefetch.tensor) cost 8 %, half-height stages x 8 cost 14 %.  (Numbers of the
// multicast pair kernel of round 1; the cta_group::2 kernel keeps the schedule unchanged.)
void build_pair_schedule(int64_t kc, int d, int nclusters_max, std::vector<PairSeg>* segs, std::vector<int>* off,
                         int64_t seg_cap_arg, int64_t min_piece_arg) {
  // chunks per accumulation: 4096 fp32 rows / 8192 16-bit rows.  Measured on the B200 with all-positive
  // activations 36928 x 3072: cap 128 / 256 / 512 / none -> rel. error 7.6e-4 / 7.8e-4 / 8.2e-4 / 1.0e-3 (fp32),
  // 2.2e-5 / 5.0e-5 / 8.8e-5 (bf16), at 742 / 753 / 766 / 779 TFLOP/s.
  int64_t seg_cap = seg_cap_arg > 0 ? seg_cap_arg : 128;
  if (const char* e = getenv("VLM_SYRK_SEG_CHUNKS")) seg_cap = std::max(1, atoi(e));
  const int nsb = (d + 255) / 256;
  struct T {
    int a, b;
  };
  std::vector<T> tiles;
  for (int a = 0; a < nsb; ++a)
    for (int b = a; b < nsb; ++b) tiles.push_back({a, b});
  const int64_t ntile = (int64_t)tiles.size();
  const int64_t min_chunks = 8;  // do not cut a K range below this: every piece pays a 128 KB epilogue per CTA
  const int C = nclusters_max;
  std::vector<std::vector<PairSeg>> per;
  auto emit = [&](int c, const T& t, int64_t k0, int64_t k1) {
    if (k1 <= k0) return;
    const int64_t pieces = (k1 - k0 + seg_cap - 1) / seg_cap;
    for (int64_t i = 0; i < pieces; ++i) {
      const int64_t a = k0 + (k1 - k0) * i / pieces, b = k0 + (k1 - k0) * (i + 1) / pieces;
      per[c].push_back({t.a, t.b, (int)a, (int)b});
    }
  };
  per.resize(C);
  const int64_t rounds = ntile / C;  // whole tiles per cluster, all clusters sweeping K from 0 together
  for (int64_t r = 0; r < rounds; ++r)
    for (int c = 0; c < C; ++c) emit(c, tiles[r * C + c], 0, kc);
  // The R = T mod C left-over tiles (all T tiles when T < C) are cut along K into P equal pieces with the
  // same boundaries for every tile; the (piece, tile) items are dealt round-robin in piece-major order,
  // so concurrently processed items belong to the same one or two pieces (K-aligned).  P minimises the
  // makespan ceil(R*P/C)/P among piece lengths between min_chunks.. and seg_cap chunks.
  const int64_t rem = ntile - rounds * C;
  if (rem > 0) {
    const int64_t p_lo = std::max<int64_t>(1, (kc + seg_cap - 1) / seg_cap);
    // shortest K piece: 64 chunks for long sweeps, min_chunks for short ones when the problem runs alone (it has to
    // fill the GPU by itself); a grouped launch with plenty of other work asks for 64 throughout (min_piece_arg), so
    // that a 2560-row Gram is not cut into 8-chunk pieces whose 128 KB epilogues take longer than their mainloops
    const int64_t min_piece = min_piece_arg > 0 ? min_piece_arg : (kc >= 8 * 64 ? 64 : min_chunks);
    const int64_t p_hi = std::max<int64_t>(p_lo, kc / min_piece);
    int64_t best_p = p_lo;
    double best = 1e30;
    for (int64_t p = p_lo; p <= p_hi; ++p) {
      const double makespan = (double)((rem * p + C - 1) / C) / (double)p;
      if (makespan < best - 1e-9) best = makespan, best_p = p;
    }
    // With at least one round of whole tiles, a left-over piece is not appended after the sweep (by then its rows
    // have long left L2: X is streamed once per round) but INTERLEAVED into the cluster's last sweep, right after
    // the own-tile segment that covers the same rows — every cluster keeps reading the one band of X that is in L2.
    std::vector<std::vector<PairSeg>> sweep;
    static const bool interleave_on = [] {
      const char* e = getenv("VLM_SYRK_INTERLEAVE");
      return e ? atoi(e) != 0 : true;
    }();
    const bool interleave = interleave_on && rounds > 0;
    if (interleave) {
      sweep.resize(C);
      for (int c = 0; c < C; ++c) {
        const size_t n_last = (size_t)((kc + seg_cap - 1) / seg_cap);  // segments of the last whole tile
        sweep[c].assign(per[c].end() - n_last, per[c].end());
        per[c].resize(per[c].size() - n_last);
      }
    }
    int64_t q = 0;
    for (int64_t p = 0; p < best_p; ++p)
      for (int64_t t = 0; t < rem; ++t, ++q)
        emit((int)(q % C), tiles[rounds * C + t], kc * p / best_p, kc * (p + 1) / best_p);
    if (interleave) {
      for (int c = 0; c < C; ++c) {
        // per[c] = earlier rounds + this cluster's left-over pieces (ascending k0); merge them into the sweep
        const size_t n_before = (size_t)(rounds - 1) * (size_t)((kc + seg_cap - 1) / seg_cap);
        std::vector<PairSeg> pieces(per[c].begin() + n_before, per[c].end());
        per[c].resize(n_before);
        size_t i = 0;
        for (const PairSeg& own : sweep[c]) {
          per[c].push_back(own);
          while (i < pieces.size() && pieces[i].k0 < own.k1) per[c].push_back(pieces[i++]);
        }
        while (i < pieces.size()) per[c].push_back(pieces[i++]);
      }
    }
  }
  while (!per.empty() && per.back().empty()) per.pop_back();  // clusters without work are not launched
  segs->clear();
  off->assign(1, 0);
  for (auto& v : per) {
    segs->insert(segs->end(), v.begin(), v.end());
    off->push_back((int)segs->size());
  }
}

// Host view for the CPU tests: segments as {super_row, super_col, k0, k1} per cluster.
void build_syrk_pair_schedule_host(int64_t kc, int d, int nsm, std::vector<int32_t>* flat, std::vector<int>* off) {
  std::vector<PairSeg> segs;
  build_pair_schedule(kc, d, nsm / 2, &segs, off);
  flat->clear();
  for (const PairSeg& s : segs) {
    flat->push_back(s.sa);
    flat->push_back(s.sb);
    flat->push_back(s.k0);
    flat->push_back(s.k1);
  }
}

// Host view of the int8 schedule (kc in 32-row chunks): {super_row, super_col | phase << 16, k0, k1} per cluster.
static void build_i8_schedule(int64_t kc, int d, int C, std::vector<PairSeg>* segs, std::vector<int>* off);
void build_syrk_i8_schedule_host(int64_t kc, int d, int nsm, std::vector<int32_t>* flat, std::vector<int>* off) {
  std::vector<PairSeg> segs;
  build_i8_schedule(kc, d, nsm / 2, &segs, off);
  flat->clear();
  for (const PairSeg& s : segs) {
    flat->push_back(s.sa);
    flat->push_back(s.sb);
    flat->push_back(s.k0);
    flat->push_back(s.k1);
  }
}

bool syrk_pair_supported(int dtype, const void* x, int d, int64_t ldx, int64_t seg_stride, const float* g, int64_t ldg) {
  const int elem = elem_bytes(dtype);
  return d % (128 / elem) == 0 &&  // whole 128-byte column groups (the 3-D tensor map needs them)
         (reinterpret_cast<uintptr_t>(x) & 15) == 0 && ((ldx * elem) & 15) == 0 && ((seg_stride * elem) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(g) & 15) == 0 && (ldg & 3) == 0;
}

// chunks per row segment (0 = contiguous) and in total
static inline void seg_chunks(int64_t rows, int64_t seg_rows, int bk, int64_t* cps, int64_t* kc) {
  if (seg_rows > 0) {
    *cps = (seg_rows + bk - 1) / bk;
    *kc = (rows / seg_rows) * *cps;
  } else {
    *cps = 0;
    *kc = (rows + bk - 1) / bk;
  }
}

int syrk_pair_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                    float* g, int64_t ldg, cudaStream_t stream) {
  const int bk = chunk_rows(dtype);
  VLM_REQUIRE(rows < (int64_t)1 << 31, VLM_ERR_INVALID_ARG, "vlm_syrk_accum: rows too large");
  if (seg_rows >= rows || dtype == VLM_TF32X2) seg_rows = 0;  // one segment: plain rows
  int dev = 0, nsm = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  if (int rc = device_sm_count(&nsm)) return rc;
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  int64_t cps, kc;
  seg_chunks(rows, seg_rows, bk, &cps, &kc);
  VLM_REQUIRE(kc < (int64_t)1 << 30, VLM_ERR_INVALID_ARG, "vlm_syrk_accum: too many row chunks");
  CUtensorMap tm_x, tm_g;
  if (int rc = encode_maps(encode, x, dtype, rows, d, ldx, seg_rows, seg_stride, g, ldg, &tm_x, &tm_g)) return rc;
  const int smem = k2SmemBytes;
  const bool det = deterministic_mode();
  PairKernel kernel = det ? pick_kernel<false, true>(dtype) : pick_kernel<false, false>(dtype);

  // lookup and launch under one lock: an eviction by another host thread cannot free a schedule between the two
  std::lock_guard<std::mutex> lk(g_mu2);
  const DeviceSchedule2* sched = nullptr;
  if (int rc = cached_schedule(std::make_tuple(dev, kc, d, bk, nsm, det),
                               [&](std::vector<PairSeg>* segs, std::vector<int>* off) {
                                 build_pair_schedule(kc, d, nsm / 2, segs, off);
                               },
                               stream, &sched, d, (int)cps))
    return rc;
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  void* ws = nullptr;
  if (det) {
    if (int rc = det_workspace((size_t)sched->nslots * 256 * 256 * 4, nullptr, stream, &ws, nullptr)) return rc;
    if (int rc = encode_slot_map(encode, ws, sched->nslots, false, &tm_g)) {
      cudaFreeAsync(ws, stream);
      return rc;
    }
  }
  kernel<<<2 * sched->nclusters, kThreads, smem, stream>>>(tm_x, tm_g, nullptr, sched->d_segs, sched->d_off, d, (int)cps,
                                                           l2_hints());
  VLM_CUDA(cudaGetLastError());
  count_launch();
  if (det) {
    if (int rc = det_reduce_launch(sched->d_items, sched->nitems, 256, false, ws, g, ldg, nullptr, stream)) return rc;
    VLM_CUDA(cudaFreeAsync(ws, stream));
  }
  return 0;
}

int tf32_split_launch(const float* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, float* out,
                      cudaStream_t stream) {
  int nsm = 0;
  if (int rc = device_sm_count(&nsm)) return rc;
  if (seg_rows >= rows) seg_rows = 0;
  const int64_t n4 = rows * (d / 4);
  const int64_t blocks = std::min<int64_t>((n4 + 255) / 256, (int64_t)nsm * 8);
  tf32_split_kernel<<<(unsigned)std::max<int64_t>(1, blocks), 256, 0, stream>>>(x, rows, d, ldx, seg_rows, seg_stride, out);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// Exact Gram on the integer tensor cores (syrk_i8.cuh).  scratch: [4 planes: 4 * rows * d bytes][exps: d ints]
// [column maxima: d uints], 16-byte aligned.
size_t syrk_i8x4_scratch_bytes(int64_t rows, int d) { return (size_t)4 * rows * d + (size_t)8 * d + 64; }

// The int8 schedule: every (tile, K range) of the floating-point schedule runs once per phase.  When there are fewer
// (tile, phase) pairs than clusters (768-wide Grams: 6 tiles), the clusters of a tile are divided among its phases
// instead — each cluster then runs ONE segment of ONE phase and pays one pipeline fill and one exposed epilogue, not
// three (ncu, 36928 x 768: IMMA pipe 64 % of elapsed with three; A/B on the B200, profiles/r02_syrk_i8x4_cases.log:
// 2560 x 768 0.063 -> 0.043 ms, 9216 x 768 0.086 -> 0.069, 36928 x 768 0.209 -> 0.196).  Phase weights = tensor time per 32 rows in units
// of one MMA (phase 2 is ingest-bound: a little over one).
static void build_i8_schedule(int64_t kc, int d, int C, std::vector<PairSeg>* segs, std::vector<int>* off) {
  const int nsb = (d + 255) / 256;
  const int T = nsb * (nsb + 1) / 2;
  segs->clear();
  off->assign(1, 0);
  const int m = (int)std::min<int64_t>(C / T, kc / 6);    // clusters per tile; no K piece much below 8 chunks (measured: 2560 x 768 is fastest with all 12)
  if (m >= 3 && kc >= 64) {
    const double w[3] = {7.0, 5.0, 1.15};
    const double fixed = 200.0;              // pipeline fill + exposed epilogue of one segment, in 32-row MMA units
    int best[3] = {0, 0, 0};
    double best_t = 1e30;
    for (int n0 = 1; n0 <= m - 2; ++n0)
      for (int n1 = 1; n0 + n1 <= m - 1; ++n1) {
        const int n2 = m - n0 - n1;
        const double t = std::max(w[0] / n0, std::max(w[1] / n1, w[2] / n2));
        if (t < best_t - 1e-12) best_t = t, best[0] = n0, best[1] = n1, best[2] = n2;
      }
    const double t_split = best_t * (double)kc + fixed;
    const double t_all = (w[0] + w[1] + w[2]) / m * (double)kc + 3 * fixed;
    if (t_split < t_all) {
      for (int a = 0; a < nsb; ++a)
        for (int b = a; b < nsb; ++b)
          for (int ph = 0; ph < kI8Phases; ++ph)
            for (int i = 0; i < best[ph]; ++i) {
              // phase 2 consumes 128-row stages: cut its K range on multiples of 4 chunks
              const int64_t g = ph == 2 ? 4 : 1, units = (kc + g - 1) / g;
              const int64_t k0 = std::min(kc, units * i / best[ph] * g), k1 = std::min(kc, units * (i + 1) / best[ph] * g);
              if (k1 > k0) {
                // int32 accumulation is exact for 2^17 rows; 2048 chunks = 65536 rows per segment
                for (int64_t k = k0; k < k1; k += 2048)
                  segs->push_back({a, b | (ph << 16), (int)k, (int)std::min(k1, k + 2048)});
                off->push_back((int)segs->size());
              }
            }
      return;
    }
  }
  std::vector<PairSeg> base;
  std::vector<int> boff;
  // int32 accumulation of a four-pair group is exact for 2^17 rows (|digit| <= 64); 2048 chunks = 65536 rows per
  // segment keeps the (exposed) epilogues rare
  build_pair_schedule(kc, d, C, &base, &boff, 2048);
  for (size_t c = 0; c + 1 < boff.size(); ++c) {
    for (int i = boff[c]; i < boff[c + 1]; ++i)
      for (int ph = 0; ph < kI8Phases; ++ph) segs->push_back({base[i].sa, base[i].sb | (ph << 16), base[i].k0, base[i].k1});
    off->push_back((int)segs->size());
  }
}

template <typename T>
static int i8_prepass(const T* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, unsigned* amax,
                      int* exps, int8_t* planes, int nsm, cudaStream_t stream) {
  // column maxima -> exponents (+ the float scales, written over the maxima) -> digit planes
  VLM_CUDA(cudaMemsetAsync(amax, 0, sizeof(unsigned) * d, stream));
  const int64_t slabs = std::max<int64_t>(1, std::min<int64_t>((rows + 255) / 256, (int64_t)nsm * 16 / std::max(1, d / 128)));
  const int64_t rps = (rows + slabs - 1) / slabs;
  i8_colmax_kernel<T><<<dim3((unsigned)(d / 128), (unsigned)((rows + rps - 1) / rps)), 256, 0, stream>>>(
      x, rows, d, ldx, seg_rows, seg_stride, rps, amax);
  i8_exps_kernel<<<(d + 255) / 256, 256, 0, stream>>>(amax, d, exps);
  i8_slice_kernel<T><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(rows, (int64_t)nsm * 4)), 256, 0, stream>>>(
      x, rows, d, ldx, seg_rows, seg_stride, reinterpret_cast<const float*>(amax), planes);
  VLM_CUDA(cudaGetLastError());
  count_launch(3);
  return 0;
}

int syrk_i8x4_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                     void* scratch, double* g, int64_t ldg, cudaStream_t stream) {
  int dev = 0, nsm = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  if (int rc = device_sm_count(&nsm)) return rc;
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  if (seg_rows >= rows) seg_rows = 0;
  int8_t* planes = static_cast<int8_t*>(scratch);
  int* exps = reinterpret_cast<int*>(planes + (((size_t)4 * rows * d + 15) & ~(size_t)15));
  unsigned* amax = reinterpret_cast<unsigned*>(exps + d);
  int rc;
  if (dtype == VLM_F32)
    rc = i8_prepass(static_cast<const float*>(x), rows, d, ldx, seg_rows, seg_stride, amax, exps, planes, nsm, stream);
  else if (dtype == VLM_F16)
    rc = i8_prepass(static_cast<const __half*>(x), rows, d, ldx, seg_rows, seg_stride, amax, exps, planes, nsm, stream);
  else
    rc = i8_prepass(static_cast<const __nv_bfloat16*>(x), rows, d, ldx, seg_rows, seg_stride, amax, exps, planes, nsm, stream);
  if (rc) return rc;

  // three views of the planes: 32 rows of all four (groups 4, 3), 32 rows of planes 0..2 (groups 2, 1), 128 rows of
  // plane 0 (group 0)
  CUtensorMap tm_p[3];
  for (int ph = 0; ph < 3; ++ph) {
    const cuuint32_t np = ph == 0 ? 4 : ph == 1 ? 3 : 1;
    cuuint64_t gdim[4] = {128, (cuuint64_t)rows, (cuuint64_t)(d / 128), np};
    cuuint64_t gstr[3] = {(cuuint64_t)d, 128, (cuuint64_t)rows * d};
    cuuint32_t box[4] = {128, (cuuint32_t)(ph == 2 ? 128 : 32), 1, np};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = encode(&tm_p[ph], CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, planes, gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(int8 planes) failed: CUresult %d", (int)r);
  }
  // G as a 2-D fp64 tensor for the epilogue's TMA reduce-adds: box = 16 columns (128 bytes) x 128 rows
  CUtensorMap tm_g;
  {
    cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)d};
    cuuint64_t gstr[1] = {(cuuint64_t)ldg * 8};
    cuuint32_t box[2] = {16, 128};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&tm_g, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, g, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(G fp64) failed: CUresult %d", (int)r);
  }
  const int64_t kc = (rows + 31) / 32;
  VLM_REQUIRE(kc < (int64_t)1 << 30, VLM_ERR_INVALID_ARG, "vlm_syrk_accum_i8x4: too many row chunks");
  const bool det = deterministic_mode();
  std::lock_guard<std::mutex> lk(g_mu2);
  const DeviceSchedule2* sched = nullptr;
  if (int rc = cached_schedule(std::make_tuple(dev, kc, d, -8, nsm, det),  // chunk rows -8: the int8 schedule
                               [&](std::vector<PairSeg>* segs, std::vector<int>* off) {
                                 build_i8_schedule(kc, d, nsm / 2, segs, off);
                               },
                               stream, &sched, d))
    return rc;
  const int smem = kI8SmemBytes;
  auto kernel = det ? syrk_i8x4_kernel<true> : syrk_i8x4_kernel<false>;
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  void* ws = nullptr;
  if (det) {
    if (int rc = det_workspace((size_t)sched->nslots * 256 * 256 * 8, nullptr, stream, &ws, nullptr)) return rc;
    if (int rc = encode_slot_map(encode, ws, sched->nslots, true, &tm_g)) {
      cudaFreeAsync(ws, stream);
      return rc;
    }
  }
  I8Args args{g, ldg, exps};
  kernel<<<2 * sched->nclusters, kThreads, smem, stream>>>(tm_p[0], tm_p[1], tm_p[2], tm_g, sched->d_segs, sched->d_off, d,
                                                           args);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  if (det) {
    if (int rc = det_reduce_launch(sched->d_items, sched->nitems, 256, true, ws, g, ldg, nullptr, stream)) return rc;
    VLM_CUDA(cudaFreeAsync(ws, stream));
  }
  return 0;
}

int syrk_pair_batch_launch(const vlm_syrk_problem* probs, int n, int dtype, cudaStream_t stream) {
  const int bk = chunk_rows(dtype);
  int dev = 0, nsm = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  if (int rc = device_sm_count(&nsm)) return rc;
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  const int C = nsm / 2;
  std::vector<CUtensorMap> maps(2 * (size_t)n);
  std::vector<std::vector<BatchSeg>> per(C);
  std::vector<int64_t> load(C, 0);
  // per-shape schedule (segments, per-cluster offsets, shares sorted heaviest first): a batch usually repeats a
  // handful of shapes (36 x [2560, 768] + 12 x [2560, 3072] for the text tower), so it is built once per shape
  struct ShapeSched {
    std::vector<PairSeg> segs;
    std::vector<int> off;
    std::vector<std::pair<int64_t, int>> shares;
  };
  std::map<std::pair<int64_t, int>, ShapeSched> by_shape;
  // total work of the batch in (tile, chunk) units: with at least ~8 pieces of 64 chunks per cluster there is no need
  // to cut short K ranges finely (ncu of the text group, 36 x [2560, 768] + 12 x [2560, 3072]: tensor pipe 72 % of
  // elapsed with 8-chunk pieces — 2,640 segments whose epilogues outlast their mainloops)
  int64_t batch_work = 0;
  for (int p = 0; p < n; ++p) {
    const int64_t nsb = (probs[p].d + 255) / 256;
    batch_work += nsb * (nsb + 1) / 2 * ((probs[p].rows + bk - 1) / bk);
  }
  const int64_t min_piece = batch_work >= (int64_t)8 * 64 * C ? 64 : 0;
  for (int p = 0; p < n; ++p) {
    const vlm_syrk_problem& q = probs[p];
    VLM_REQUIRE(q.rows < (int64_t)1 << 31, VLM_ERR_INVALID_ARG, "vlm_syrk_accum: rows too large");
    const int64_t seg_rows = (dtype != VLM_TF32X2 && q.seg_rows > 0 && q.seg_rows < q.rows) ? q.seg_rows : 0;
    if (int rc = encode_maps(encode, q.x, dtype, q.rows, q.d, q.ldx, seg_rows, q.seg_stride, q.g, q.ldg, &maps[2 * p],
                             &maps[2 * p + 1]))
      return rc;
    int64_t cps, kc;
    seg_chunks(q.rows, seg_rows, bk, &cps, &kc);
    auto found = by_shape.find({kc, q.d});
    if (found == by_shape.end()) {
      ShapeSched ss;
      build_pair_schedule(kc, q.d, C, &ss.segs, &ss.off, 0, min_piece);
      for (int c = 0; c + 1 < (int)ss.off.size(); ++c) {
        int64_t cost = 0;
        for (int s = ss.off[c]; s < ss.off[c + 1]; ++s) cost += ss.segs[s].k1 - ss.segs[s].k0;
        ss.shares.push_back({cost, c});
      }
      std::sort(ss.shares.begin(), ss.shares.end(),
                [](auto& a, auto& b) { return a.first > b.first || (a.first == b.first && a.second < b.second); });
      found = by_shape.emplace(std::make_pair(kc, q.d), std::move(ss)).first;
    }
    const std::vector<PairSeg>& segs = found->second.segs;
    const std::vector<int>& off = found->second.off;
    const std::vector<std::pair<int64_t, int>>& shares = found->second.shares;
    // this problem's per-cluster shares go to the least loaded clusters, heaviest share first
    std::vector<int> order(C);
    for (int c = 0; c < C; ++c) order[c] = c;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return load[a] < load[b]; });
    for (size_t i = 0; i < shares.size(); ++i) {
      const int dst = order[i % C], c = shares[i].second;
      for (int s = off[c]; s < off[c + 1]; ++s)
        per[dst].push_back({segs[s].sa, segs[s].sb, segs[s].k0, segs[s].k1, p, q.d, (int)cps, 0});
      load[dst] += shares[i].first;
    }
  }
  int ncl = C;
  while (ncl > 0 && per[ncl - 1].empty()) --ncl;  // (clusters are filled least-loaded first, so gaps are rare)
  std::vector<BatchSeg> flat;
  std::vector<int> foff(1, 0);
  for (int c = 0; c < ncl; ++c) {
    flat.insert(flat.end(), per[c].begin(), per[c].end());
    foff.push_back((int)flat.size());
  }
  if (flat.empty()) return 0;
  // deterministic mode: every problem's G map is replaced by the map of the one slot workspace, and the reduction's
  // tile list and the problems' G pointers follow the segments in the table
  const bool det = deterministic_mode();
  std::vector<DetItem> items;
  std::vector<DetGram> grams;
  void* ws = nullptr;
  if (det) {
    std::vector<int> same_g(n);
    for (int p = 0; p < n; ++p) {
      same_g[p] = p;
      for (int q = 0; q < p; ++q)
        if (probs[q].g == probs[p].g && probs[q].ldg == probs[p].ldg) {
          same_g[p] = q;
          break;
        }
      grams.push_back({probs[p].g, probs[p].ldg});
    }
    const int nslots = det_slots(&flat, foff, &items, &same_g);
    if (int rc = det_workspace((size_t)nslots * 256 * 256 * 4, nullptr, stream, &ws, nullptr)) return rc;
    CUtensorMap tm_ws;
    if (int rc = encode_slot_map(encode, ws, nslots, false, &tm_ws)) {
      cudaFreeAsync(ws, stream);
      return rc;
    }
    for (int p = 0; p < n; ++p) maps[2 * p + 1] = tm_ws;
  }
  const size_t maps_bytes = maps.size() * sizeof(CUtensorMap);
  const size_t off_bytes = ((foff.size() * sizeof(int)) + 127) / 128 * 128;
  const size_t seg_bytes = flat.size() * sizeof(BatchSeg);
  const size_t item_bytes = items.size() * sizeof(DetItem), gram_bytes = grams.size() * sizeof(DetGram);
  const size_t total = maps_bytes + off_bytes + seg_bytes + item_bytes + gram_bytes;
  std::vector<uint8_t> host(total);
  memcpy(host.data(), maps.data(), maps_bytes);
  memcpy(host.data() + maps_bytes, foff.data(), foff.size() * sizeof(int));
  memcpy(host.data() + maps_bytes + off_bytes, flat.data(), seg_bytes);
  if (det) {
    memcpy(host.data() + maps_bytes + off_bytes + seg_bytes, items.data(), item_bytes);
    memcpy(host.data() + maps_bytes + off_bytes + seg_bytes + item_bytes, grams.data(), gram_bytes);
  }
  uint8_t* dptr = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_mu2);
    Scratch& sc = g_scratch[{dev, stream}];
    const int i = sc.next;
    sc.next = (sc.next + 1) % 4;
    if (sc.cap[i] < total) {
      if (sc.ptr[i]) VLM_CUDA(cudaFree(sc.ptr[i]));  // synchronises: nothing in flight can still read it
      sc.cap[i] = std::max<size_t>(total * 2, 1 << 18);
      VLM_CUDA(cudaMalloc(&sc.ptr[i], sc.cap[i]));
    }
    dptr = static_cast<uint8_t*>(sc.ptr[i]);
  }
  // pageable source: staged before the call returns; ordered on `stream` before the kernel below
  VLM_CUDA(cudaMemcpyAsync(dptr, host.data(), total, cudaMemcpyHostToDevice, stream));
  const int smem = k2SmemBytes;
  PairKernel kernel = det ? pick_kernel<true, true>(dtype) : pick_kernel<true, false>(dtype);
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  kernel<<<2 * ncl, kThreads, smem, stream>>>(maps[0], maps[1], reinterpret_cast<const CUtensorMap*>(dptr),
                                              dptr + maps_bytes + off_bytes,
                                              reinterpret_cast<const int*>(dptr + maps_bytes), 0, 0, l2_hints());
  VLM_CUDA(cudaGetLastError());
  count_launch();
  if (det) {
    const uint8_t* d_items = dptr + maps_bytes + off_bytes + seg_bytes;
    if (int rc = det_reduce_launch(reinterpret_cast<const DetItem*>(d_items), (int)items.size(), 256, false, ws, nullptr,
                                   0, reinterpret_cast<const DetGram*>(d_items + item_bytes), stream))
      return rc;
    VLM_CUDA(cudaFreeAsync(ws, stream));
  }
  return 0;
}

}  // namespace vlm
