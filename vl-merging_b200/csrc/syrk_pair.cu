// syrk_pair.cu — host side of kernel (a), the CTA-pair SYRK (device code: syrk_2sm.cuh, syrk_i8.cuh): tensor maps,
// the K-aligned work decomposition, the one plan builder and segment record of every CTA-pair launch, the plan cache,
// single, grouped and int8x4 launches, and the fp32 -> {hi, lo} split.
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
#include <cstring>
#include <utility>
#include <map>
#include <mutex>
#include <tuple>
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
// L2 eviction policies (createpolicy): the activation X is a stream that is only re-read within a short window (by
// the other clusters sweeping the same rows); the floating-point kernel's Gram tiles are re-read and re-written by
// every K segment's reduce-add for the whole launch (evict_last; see build_pair_schedule).
__device__ __forceinline__ uint64_t l2_evict_normal() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// One unit of work of a CLUSTER, the one record of every CTA-pair kernel (syrk_2sm_kernel, syrk_i8x4_kernel):
// super-tile (sa, sb) in 256-column units, row chunks [k0, k1) of problem pid (index into a grouped launch's tensor
// maps, else 0) of width d with cps chunks per row segment (0: contiguous rows, 3-D tensor map); phase: the int8
// kernel's phase (else 0); slot (deterministic mode only): workspace slot << 1 | 1 if an earlier segment of the same
// cluster already wrote that slot (det_slots).
struct PairSeg {
  int32_t sa, sb, k0, k1, pid, d, cps, phase, slot;
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

inline int elem_bytes(int dtype) { return (dtype == VLM_F32 || dtype == VLM_TF32X2) ? 4 : 2; }
// rows of X per pipeline stage = schedule chunk
inline int chunk_rows(int dtype) { return dtype == VLM_TF32X2 ? 16 : 128 / elem_bytes(dtype); }

// X as a 3-D tensor {column in group, row, column group} (strides: row pitch, 128 bytes).
// seg_rows > 0: 4-D, {column in group, row in segment, column group, segment}.
// VLM_TF32X2: 4-D, {column in group, row, column group, plane}, planes rows * ldx elements apart, and one box
// fetches both planes of a 128-column block for 16 rows.
int encode_x_map(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                 CUtensorMap* tm_x) {
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  const int elem = elem_bytes(dtype);
  const int bk = chunk_rows(dtype), gc = 128 / elem;
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
  return 0;
}

// device scratch for batched launches: a small ring per (device, stream); reuse is ordered by the stream itself
struct Scratch {
  void* ptr[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t cap[4] = {0, 0, 0, 0};
  int next = 0;
};
std::map<std::pair<int, cudaStream_t>, Scratch> g_scratch;

typedef void (*PairKernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap*, const PairSeg*, const int*);
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
// seg_cap_arg: chunks per accumulation (0: 128); min_piece_arg: shortest K piece a left-over tile is cut into (0: 64
// chunks for long sweeps, 8 for short ones).  Every segment carries width d; pid, cps, phase and slot are left 0.
static void build_pair_schedule(int64_t kc, int d, int nclusters_max, std::vector<PairSeg>* segs, std::vector<int>* off,
                                int64_t seg_cap_arg = 0, int64_t min_piece_arg = 0) {
  // chunks per accumulation: 4096 fp32 rows / 8192 16-bit rows.  Measured on the B200 with all-positive
  // activations 36928 x 3072: cap 128 / 256 / 512 / none -> rel. error 7.6e-4 / 7.8e-4 / 8.2e-4 / 1.0e-3 (fp32),
  // 2.2e-5 / 5.0e-5 / 8.8e-5 (bf16), at 742 / 753 / 766 / 779 TFLOP/s.
  const int64_t seg_cap = seg_cap_arg > 0 ? seg_cap_arg : 128;
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
      per[c].push_back({t.a, t.b, (int)a, (int)b, 0, d});
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
    const bool interleave = rounds > 0;
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
                  segs->push_back({a, b, (int)k, (int)std::min(k1, k + 2048), 0, d, 0, ph});
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
      for (int ph = 0; ph < kI8Phases; ++ph) {
        segs->push_back(base[i]);
        segs->back().phase = ph;
      }
    off->push_back((int)segs->size());
  }
}

// ---- the plan of a CTA-pair launch ---------------------------------------------------------------------------------

namespace {

// One Gram of a CTA-pair launch: kc row chunks of width d, cps chunks per row segment (0: contiguous rows); same_g:
// the first Gram of the launch that adds into the same G (its own index if none), whose reduction tiles it shares
struct PlanGram {
  int64_t kc;
  int d, cps, same_g;
};
// The work of one launch: segments cluster by cluster (cluster c runs segs[off[c] .. off[c + 1])), and in the
// deterministic mode the reduction's tiles and the number of workspace slots
struct PairPlan {
  std::vector<PairSeg> segs;
  std::vector<int> off;
  std::vector<DetItem> items;
  int nslots = 0;
};
enum class PlanKind { kSingle, kInt8, kGrouped };

// Deterministic mode: gives every (G, super-tile, cluster) a workspace slot of its own.  The slots of one tile are
// numbered consecutively in schedule order (cluster by cluster, each cluster's segments in order), which is the order
// the reduction adds them in.  Sets seg.slot = slot << 1 | (1 when an earlier segment of the same cluster opened the
// slot: that one stores, the later ones add; the int8 phases of a tile chain so); fills plan->items with one DetItem
// per tile and returns the number of slots.
int det_slots(PairPlan* plan, const std::vector<PlanGram>& grams) {
  std::vector<PairSeg>& segs = plan->segs;
  std::map<std::tuple<int, int, int>, int> tile_of;  // (G, super row, super column) -> index into items
  std::vector<std::vector<int>> opened;              // per tile: its temporary slot ids, in schedule order
  std::vector<int> temp(segs.size());
  int ntemp = 0;
  plan->items.clear();
  for (size_t c = 0; c + 1 < plan->off.size(); ++c) {
    std::map<int, int> mine;  // tile -> temporary slot id of this cluster
    for (int s = plan->off[c]; s < plan->off[c + 1]; ++s) {
      PairSeg& q = segs[s];
      const int gp = grams[q.pid].same_g;
      auto t = tile_of.emplace(std::make_tuple(gp, q.sa, q.sb), (int)plan->items.size());
      if (t.second) {
        plan->items.push_back({gp, q.d, q.sa * 256, q.sb * 256, q.sa == q.sb ? 1 : 0, 0, 0, 0});
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
  for (size_t t = 0; t < plan->items.size(); ++t) {
    plan->items[t].slot_begin = next;
    for (int id : opened[t]) final_id[id] = next++;
    plan->items[t].slot_end = next;
  }
  for (size_t s = 0; s < segs.size(); ++s) segs[s].slot |= final_id[temp[s]] << 1;
  return next;
}

// The one plan builder of the CTA-pair launches, over C clusters.  kSingle / kInt8: the schedule of the one Gram
// (build_pair_schedule / build_i8_schedule).  kGrouped: every Gram is scheduled as if it ran alone (once per shape;
// min_piece: see build_pair_schedule), and its per-cluster shares go to the least loaded clusters, heaviest share
// first.  det: the workspace slots and reduction tiles as well (det_slots).
PairPlan build_plan(PlanKind kind, const std::vector<PlanGram>& grams, int C, bool det, int64_t min_piece = 0) {
  PairPlan plan;
  if (kind != PlanKind::kGrouped) {
    const PlanGram& q = grams[0];
    if (kind == PlanKind::kInt8)
      build_i8_schedule(q.kc, q.d, C, &plan.segs, &plan.off);
    else
      build_pair_schedule(q.kc, q.d, C, &plan.segs, &plan.off);
    for (PairSeg& s : plan.segs) s.cps = q.cps;
  } else {
    std::vector<std::vector<PairSeg>> per(C);
    std::vector<int64_t> load(C, 0);
    // per-shape schedule (segments, per-cluster offsets, shares sorted heaviest first): a batch usually repeats a
    // handful of shapes (36 x [2560, 768] + 12 x [2560, 3072] for the text tower), so it is built once per shape
    struct ShapeSched {
      std::vector<PairSeg> segs;
      std::vector<int> off;
      std::vector<std::pair<int64_t, int>> shares;
    };
    std::map<std::pair<int64_t, int>, ShapeSched> by_shape;
    for (int p = 0; p < (int)grams.size(); ++p) {
      const PlanGram& q = grams[p];
      auto found = by_shape.find({q.kc, q.d});
      if (found == by_shape.end()) {
        ShapeSched ss;
        build_pair_schedule(q.kc, q.d, C, &ss.segs, &ss.off, 0, min_piece);
        for (int c = 0; c + 1 < (int)ss.off.size(); ++c) {
          int64_t cost = 0;
          for (int s = ss.off[c]; s < ss.off[c + 1]; ++s) cost += ss.segs[s].k1 - ss.segs[s].k0;
          ss.shares.push_back({cost, c});
        }
        std::sort(ss.shares.begin(), ss.shares.end(),
                  [](auto& a, auto& b) { return a.first > b.first || (a.first == b.first && a.second < b.second); });
        found = by_shape.emplace(std::make_pair(q.kc, q.d), std::move(ss)).first;
      }
      const ShapeSched& ss = found->second;
      // this Gram's per-cluster shares go to the least loaded clusters, heaviest share first
      std::vector<int> order(C);
      for (int c = 0; c < C; ++c) order[c] = c;
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return load[a] < load[b]; });
      for (size_t i = 0; i < ss.shares.size(); ++i) {
        const int dst = order[i % C], c = ss.shares[i].second;
        for (int s = ss.off[c]; s < ss.off[c + 1]; ++s) {
          per[dst].push_back(ss.segs[s]);
          per[dst].back().pid = p;
          per[dst].back().cps = q.cps;
        }
        load[dst] += ss.shares[i].first;
      }
    }
    int ncl = C;
    while (ncl > 0 && per[ncl - 1].empty()) --ncl;  // (clusters are filled least-loaded first, so gaps are rare)
    plan.off.assign(1, 0);
    for (int c = 0; c < ncl; ++c) {
      plan.segs.insert(plan.segs.end(), per[c].begin(), per[c].end());
      plan.off.push_back((int)plan.segs.size());
    }
  }
  if (det) plan.nslots = det_slots(&plan, grams);
  return plan;
}

// The device copy of a single launch's plan
struct DevicePlan {
  int nclusters = 0;
  PairSeg* d_segs = nullptr;
  int* d_off = nullptr;
  DetItem* d_items = nullptr;
  int nitems = 0, nslots = 0;
};
std::mutex g_mu2;
// (device, chunks, d, chunk rows or -8 for int8, SMs, deterministic, chunks per row segment)
typedef std::tuple<int, int64_t, int, int, int, bool, int> PlanKey;
std::map<PlanKey, DevicePlan> g_plans;
// plans evicted from the cache: freed at the NEXT eviction, after a device synchronisation, never while a launch that
// was handed their pointers may still be pending (the lock is held from lookup to launch)
std::vector<DevicePlan> g_retired;

// The plan of a single launch of q on the current device, built and uploaded on first use.  chunk_rows: rows of X per
// chunk, or -8 for the int8 schedule.  Call with g_mu2 held until the launch that reads it is enqueued.
int cached_plan(int chunk_rows, const PlanGram& q, bool det, cudaStream_t stream, const DevicePlan** out) {
  int dev = 0, nsm = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  if (int rc = device_sm_count(&nsm)) return rc;
  const PlanKey key(dev, q.kc, q.d, chunk_rows, nsm, det, q.cps);
  auto it = g_plans.find(key);
  if (it == g_plans.end()) {
    if (g_plans.size() >= 512) {  // ragged workloads (a new row count every call): start over, do not grow forever
      VLM_CUDA(cudaDeviceSynchronize());  // launches that read the plans retired LAST time have finished
      for (auto& dp : g_retired) {
        cudaFree(dp.d_segs);
        cudaFree(dp.d_off);
        cudaFree(dp.d_items);
      }
      g_retired.clear();
      for (auto& kv : g_plans) g_retired.push_back(kv.second);
      g_plans.clear();
    }
    const PairPlan plan = build_plan(chunk_rows < 0 ? PlanKind::kInt8 : PlanKind::kSingle, {q}, nsm / 2, det);
    DevicePlan dp;
    dp.nclusters = (int)plan.off.size() - 1;
    dp.nitems = (int)plan.items.size();
    dp.nslots = plan.nslots;
    const size_t seg_bytes = plan.segs.size() * sizeof(PairSeg), item_bytes = plan.items.size() * sizeof(DetItem);
    if (det) {
      VLM_CUDA(cudaMalloc(&dp.d_items, std::max<size_t>(1, item_bytes)));
      VLM_CUDA(cudaMemcpyAsync(dp.d_items, plan.items.data(), item_bytes, cudaMemcpyHostToDevice, stream));
    }
    VLM_CUDA(cudaMalloc(&dp.d_segs, std::max<size_t>(1, seg_bytes)));
    VLM_CUDA(cudaMalloc(&dp.d_off, plan.off.size() * sizeof(int)));
    VLM_CUDA(cudaMemcpyAsync(dp.d_segs, plan.segs.data(), seg_bytes, cudaMemcpyHostToDevice, stream));
    VLM_CUDA(cudaMemcpyAsync(dp.d_off, plan.off.data(), plan.off.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    VLM_CUDA(cudaStreamSynchronize(stream));
    it = g_plans.emplace(key, dp).first;
  }
  *out = &it->second;
  return 0;
}

}  // namespace

void syrk_schedule_host(int64_t kc, int d, int nsm, bool int8, std::vector<int32_t>* flat, std::vector<int>* off) {
  const PairPlan plan = build_plan(int8 ? PlanKind::kInt8 : PlanKind::kSingle, {{kc, d, 0, 0}}, nsm / 2, false);
  flat->clear();
  for (const PairSeg& s : plan.segs) flat->insert(flat->end(), {s.sa, s.sb | s.phase << 16, s.k0, s.k1});
  *off = plan.off;
}

int encode_matrix_map(CUtensorMap* tm, bool f64, void* ptr, int64_t rows, int64_t cols, int64_t pitch) {
  EncodeTiledFn encode = nullptr;
  if (int rc = tensor_map_encoder(&encode)) return rc;
  const int elem = f64 ? 8 : 4;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)pitch * elem};
  cuuint32_t box[2] = {(cuuint32_t)(128 / elem), 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(tm, f64 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ptr, gdim, gstr, box,
                      estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VLM_REQUIRE(r == CUDA_SUCCESS, VLM_ERR_DRIVER, "cuTensorMapEncodeTiled(%s matrix, %lld x %lld) failed: CUresult %d",
              f64 ? "fp64" : "fp32", (long long)rows, (long long)cols, (int)r);
  return 0;
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
  int64_t cps, kc;
  seg_chunks(rows, seg_rows, bk, &cps, &kc);
  VLM_REQUIRE(kc < (int64_t)1 << 30, VLM_ERR_INVALID_ARG, "vlm_syrk_accum: too many row chunks");
  CUtensorMap tm_x, tm_g;
  if (int rc = encode_x_map(x, dtype, rows, d, ldx, seg_rows, seg_stride, &tm_x)) return rc;
  if (int rc = encode_matrix_map(&tm_g, false, g, d, d, ldg)) return rc;
  const bool det = deterministic_mode();
  PairKernel kernel = det ? pick_kernel<false, true>(dtype) : pick_kernel<false, false>(dtype);
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k2SmemBytes));

  // lookup and launch under one lock: an eviction by another host thread cannot free a plan between the two
  std::lock_guard<std::mutex> lk(g_mu2);
  const DevicePlan* plan = nullptr;
  if (int rc = cached_plan(bk, {kc, d, (int)cps, 0}, det, stream, &plan)) return rc;
  auto launch = [&](void*) -> int {
    kernel<<<2 * plan->nclusters, kThreads, k2SmemBytes, stream>>>(tm_x, tm_g, nullptr, plan->d_segs, plan->d_off);
    VLM_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  };
  if (!det) return launch(nullptr);
  return det_launch(plan->nslots, 256, false, nullptr, {plan->d_items, plan->nitems, g, ldg, nullptr}, &tm_g, stream,
                    launch);
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
  int nsm = 0;
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
  if (int rc = encode_matrix_map(&tm_g, true, g, d, d, ldg)) return rc;
  const int64_t kc = (rows + 31) / 32;
  VLM_REQUIRE(kc < (int64_t)1 << 30, VLM_ERR_INVALID_ARG, "vlm_syrk_accum_i8x4: too many row chunks");
  const bool det = deterministic_mode();
  auto kernel = det ? syrk_i8x4_kernel<true> : syrk_i8x4_kernel<false>;
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kI8SmemBytes));
  std::lock_guard<std::mutex> lk(g_mu2);
  const DevicePlan* plan = nullptr;
  if (int rc = cached_plan(-8, {kc, d, 0, 0}, det, stream, &plan)) return rc;  // chunk rows -8: the int8 schedule
  const I8Args args{g, ldg, exps};
  auto launch = [&](void*) -> int {
    kernel<<<2 * plan->nclusters, kThreads, kI8SmemBytes, stream>>>(tm_p[0], tm_p[1], tm_p[2], tm_g, plan->d_segs,
                                                                     plan->d_off, args);
    VLM_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  };
  if (!det) return launch(nullptr);
  return det_launch(plan->nslots, 256, true, nullptr, {plan->d_items, plan->nitems, g, ldg, nullptr}, &tm_g, stream,
                    launch);
}

int syrk_pair_batch_launch(const vlm_syrk_problem* probs, int n, int dtype, cudaStream_t stream) {
  const int bk = chunk_rows(dtype);
  int dev = 0, nsm = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  if (int rc = device_sm_count(&nsm)) return rc;
  const int C = nsm / 2;
  const bool det = deterministic_mode();
  std::vector<CUtensorMap> maps(2 * (size_t)n);
  std::vector<PlanGram> grams(n);
  // total work of the batch in (tile, chunk) units: with at least ~8 pieces of 64 chunks per cluster there is no need
  // to cut short K ranges finely (ncu of the text group, 36 x [2560, 768] + 12 x [2560, 3072]: tensor pipe 72 % of
  // elapsed with 8-chunk pieces — 2,640 segments whose epilogues outlast their mainloops)
  int64_t batch_work = 0;
  for (int p = 0; p < n; ++p) {
    const vlm_syrk_problem& q = probs[p];
    VLM_REQUIRE(q.rows < (int64_t)1 << 31, VLM_ERR_INVALID_ARG, "vlm_syrk_accum: rows too large");
    if (int rc = encode_x_map(q.x, dtype, q.rows, q.d, q.ldx, q.seg_rows, q.seg_stride, &maps[2 * p])) return rc;
    if (int rc = encode_matrix_map(&maps[2 * p + 1], false, q.g, q.d, q.d, q.ldg)) return rc;
    int64_t cps, kc;
    seg_chunks(q.rows, q.seg_rows, bk, &cps, &kc);
    grams[p] = {kc, q.d, (int)cps, p};
    for (int o = 0; det && o < p; ++o)
      if (probs[o].g == q.g && probs[o].ldg == q.ldg) {
        grams[p].same_g = o;
        break;
      }
    const int64_t nsb = (q.d + 255) / 256;
    batch_work += nsb * (nsb + 1) / 2 * ((q.rows + bk - 1) / bk);
  }
  const PairPlan plan = build_plan(PlanKind::kGrouped, grams, C, det, batch_work >= (int64_t)8 * 64 * C ? 64 : 0);
  if (plan.segs.empty()) return 0;
  // deterministic mode: the reduction reads its tiles and the problems' G pointers from the table as well
  std::vector<DetGram> targets;
  for (int p = 0; det && p < n; ++p) targets.push_back({probs[p].g, probs[p].ldg});
  const size_t maps_bytes = maps.size() * sizeof(CUtensorMap);
  const size_t off_bytes = ((plan.off.size() * sizeof(int)) + 127) / 128 * 128;
  const size_t seg_bytes = ((plan.segs.size() * sizeof(PairSeg)) + 127) / 128 * 128;
  const size_t item_bytes = plan.items.size() * sizeof(DetItem), target_bytes = targets.size() * sizeof(DetGram);
  const size_t total = maps_bytes + off_bytes + seg_bytes + item_bytes + target_bytes;
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
  PairKernel kernel = det ? pick_kernel<true, true>(dtype) : pick_kernel<true, false>(dtype);
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k2SmemBytes));
  CUtensorMap tm_ws;
  auto launch = [&](void*) -> int {
    // deterministic mode: every problem's G map is replaced by the map of the one slot workspace
    for (int p = 0; det && p < n; ++p) maps[2 * p + 1] = tm_ws;
    std::vector<uint8_t> host(total);
    memcpy(host.data(), maps.data(), maps_bytes);
    memcpy(host.data() + maps_bytes, plan.off.data(), plan.off.size() * sizeof(int));
    memcpy(host.data() + maps_bytes + off_bytes, plan.segs.data(), plan.segs.size() * sizeof(PairSeg));
    if (det) {
      memcpy(host.data() + maps_bytes + off_bytes + seg_bytes, plan.items.data(), item_bytes);
      memcpy(host.data() + maps_bytes + off_bytes + seg_bytes + item_bytes, targets.data(), target_bytes);
    }
    // pageable source: staged before the call returns; ordered on `stream` before the kernel below
    VLM_CUDA(cudaMemcpyAsync(dptr, host.data(), total, cudaMemcpyHostToDevice, stream));
    kernel<<<(unsigned)(2 * (plan.off.size() - 1)), kThreads, k2SmemBytes, stream>>>(
        maps[0], maps[1], reinterpret_cast<const CUtensorMap*>(dptr),
        reinterpret_cast<const PairSeg*>(dptr + maps_bytes + off_bytes),
        reinterpret_cast<const int*>(dptr + maps_bytes));
    VLM_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  };
  if (!det) return launch(nullptr);
  const uint8_t* d_items = dptr + maps_bytes + off_bytes + seg_bytes;
  return det_launch(plan.nslots, 256, false, nullptr,
                    {reinterpret_cast<const DetItem*>(d_items), (int)plan.items.size(), nullptr, 0,
                     reinterpret_cast<const DetGram*>(d_items + item_bytes)},
                    &tm_ws, stream, launch);
}

}  // namespace vlm
