// api.cu — C-ABI entry points declared in include/vlmerge.h (argument validation, error state) for
// the Gram path; merge.cu and regmean.cu define their own entry points.
#include <cstdarg>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "syrk.h"

namespace vlm {

std::atomic<uint64_t> g_launches{0};

std::string& last_error_ref() {
  static thread_local std::string msg;
  return msg;
}

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error_ref() = buf;
  return code;
}

namespace {
std::mutex g_dev_mu;
int g_sm_count[64] = {};
int g_cc_major[64] = {};
}  // namespace

int device_sm_count(int* out) {
  int dev = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  VLM_REQUIRE(dev >= 0 && dev < 64, VLM_ERR_UNSUPPORTED, "device index %d out of range", dev);
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (g_sm_count[dev] == 0) {
    VLM_CUDA(cudaDeviceGetAttribute(&g_sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
    VLM_CUDA(cudaDeviceGetAttribute(&g_cc_major[dev], cudaDevAttrComputeCapabilityMajor, dev));
  }
  *out = g_sm_count[dev];
  return 0;
}

int tensor_map_encoder(EncodeTiledFn* out) {
  // the driver's entry point, the same for every thread: a race between two first lookups stores it twice
  static std::atomic<EncodeTiledFn> encode{nullptr};
  if (!encode.load(std::memory_order_acquire)) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    VLM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    VLM_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, VLM_ERR_DRIVER,
                "cuTensorMapEncodeTiled not available from the driver");
    encode.store(reinterpret_cast<EncodeTiledFn>(fn), std::memory_order_release);
  }
  *out = encode.load(std::memory_order_acquire);
  return 0;
}

// The small descriptor tables of the batched launches come from cudaMallocAsync.  With its default release threshold
// (0) the pool hands its memory back to the driver at every synchronisation and the next call pays a real allocation
// (~0.3 ms, measured around the pack / unpack launches of GramCache.all_reduce): keep the pool's memory instead.
int keep_async_pool() {
  static bool done[64] = {};
  int dev = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (dev >= 0 && dev < 64 && !done[dev]) {
    cudaMemPool_t pool;
    VLM_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t threshold = UINT64_MAX;
    VLM_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
    done[dev] = true;
  }
  return 0;
}

int require_sm100() {
  int nsm = 0, dev = 0;
  if (int rc = device_sm_count(&nsm)) return rc;
  VLM_CUDA(cudaGetDevice(&dev));
  VLM_REQUIRE(g_cc_major[dev] == 10, VLM_ERR_UNSUPPORTED,
              "libvlmerge is built for sm_100a only (device compute capability major = %d)", g_cc_major[dev]);
  return 0;
}

namespace {
int check_syrk_args(const char* who, const void* x, int dtype, int64_t rows, int d, int64_t ldx, const float* g,
                    int64_t ldg) {
  VLM_REQUIRE(dtype == VLM_F32 || dtype == VLM_BF16 || dtype == VLM_F16 || dtype == VLM_TF32X2, VLM_ERR_INVALID_ARG,
              "%s: dtype must be VLM_F32, VLM_BF16, VLM_F16 or VLM_TF32X2 (got %d)", who, dtype);
  VLM_REQUIRE(rows >= 0 && d > 0, VLM_ERR_INVALID_ARG, "%s: rows=%lld d=%d", who, (long long)rows, d);
  VLM_REQUIRE(g != nullptr && ldg >= d, VLM_ERR_INVALID_ARG, "%s: g is NULL or ldg < d", who);
  VLM_REQUIRE(rows == 0 || (x != nullptr && ldx >= d), VLM_ERR_INVALID_ARG, "%s: x is NULL or ldx < d", who);
  return 0;
}
}  // namespace

}  // namespace vlm

using namespace vlm;

namespace vlm {
namespace {
thread_local bool t_deterministic = false;
}  // namespace
bool deterministic_mode() { return t_deterministic; }
}  // namespace vlm

extern "C" int vlm_version(void) { return VLM_ABI_VERSION; }
extern "C" const char* vlm_last_error(void) { return last_error_ref().c_str(); }
extern "C" uint64_t vlm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" int vlm_set_deterministic(int on) {
  t_deterministic = on != 0;
  return 0;
}
extern "C" int vlm_get_deterministic(void) { return t_deterministic ? 1 : 0; }

namespace {
int check_segments(const char* who, int64_t rows, int64_t seg_rows, int64_t seg_stride) {
  VLM_REQUIRE(seg_rows > 0 && rows % seg_rows == 0, VLM_ERR_INVALID_ARG,
              "%s: rows (%lld) must be a multiple of seg_rows (%lld)", who, (long long)rows, (long long)seg_rows);
  VLM_REQUIRE(seg_stride >= 0, VLM_ERR_INVALID_ARG, "%s: seg_stride < 0", who);
  return 0;
}

// The fp32-accumulating Gram entry points, and how a Gram of theirs runs
enum class Entry { kAccum, kStrided, kBatch };
enum class GramPath { kNone, kPair, kPerSegment, kSimt };

// The one router of vlm_syrk_accum, _strided and _batch.  Validates every problem, normalises its row segments
// (afterwards seg_rows > 0 only for two or more segments, never for VLM_TF32X2) and picks its path: the CTA-pair
// kernel, one launch per segment where that kernel cannot read the segments in one launch, or the CUDA-core kernel.
// Only then does anything run.  vlm_syrk_accum_strided asks for its segments, which must divide the rows; a vlm_syrk_problem
// with seg_rows outside (0, rows), or of VLM_TF32X2 planes, is one run of rows.  kBatch: the Grams for the CTA-pair
// kernel share one grouped launch.
int syrk_route(Entry entry, const vlm_syrk_problem* probs, int n, int dtype, cudaStream_t stream) {
  static const char* const kWho[] = {"vlm_syrk_accum", "vlm_syrk_accum_strided", "vlm_syrk_accum_batch"};
  const char* who = kWho[(int)entry];
  std::vector<vlm_syrk_problem> qs(probs, probs + n);
  std::vector<GramPath> paths(n, GramPath::kNone);
  bool any = false;
  for (int p = 0; p < n; ++p) {
    vlm_syrk_problem& q = qs[p];
    if (int rc = check_syrk_args(who, q.x, dtype, q.rows, q.d, q.ldx, q.g, q.ldg)) return rc;
    if (q.rows == 0) continue;
    const bool strided = entry == Entry::kStrided;
    bool segmented = q.seg_rows > 0 && q.seg_rows < q.rows && (strided || dtype != VLM_TF32X2);
    if (strided || segmented) {
      if (int rc = check_segments(who, q.rows, q.seg_rows, q.seg_stride)) return rc;
    }
    VLM_REQUIRE(!segmented || dtype != VLM_TF32X2, VLM_ERR_INVALID_ARG,
                "%s: VLM_TF32X2 planes are packed by vlm_tf32_split, they have no row segments", who);
    if (!segmented) q.seg_rows = q.seg_stride = 0;
    const bool pair = syrk_pair_supported(dtype, q.x, q.d, q.ldx, q.seg_stride, q.g, q.ldg);
    if (dtype == VLM_TF32X2) {  // the planes exist only for the CTA-pair kernel
      VLM_REQUIRE(pair || entry != Entry::kBatch, VLM_ERR_UNSUPPORTED,
                  "%s: VLM_TF32X2 needs d %% 32 == 0 and 16-byte aligned planes", who);
      VLM_REQUIRE(q.d % 32 == 0, VLM_ERR_UNSUPPORTED,
                  "%s: VLM_TF32X2 needs d %% 32 == 0 (got %d); use vlm_syrk_accum_simt on the fp32 activation", who,
                  q.d);
      VLM_REQUIRE(pair, VLM_ERR_ALIGNMENT,
                  "%s: VLM_TF32X2 planes and g must be 16-byte aligned with ldx and ldg multiples of 4", who);
    }
    paths[p] = pair ? GramPath::kPair : segmented ? GramPath::kPerSegment : GramPath::kSimt;
    any = true;
  }
  if (!any) return 0;
  if (int rc = require_sm100()) return rc;
  std::vector<vlm_syrk_problem> grouped;
  for (int p = 0; p < n; ++p) {
    const vlm_syrk_problem& q = qs[p];
    int rc = 0;
    if (paths[p] == GramPath::kPair && entry == Entry::kBatch) {
      grouped.push_back(q);
    } else if (paths[p] == GramPath::kPair) {
      rc = syrk_pair_launch(q.x, dtype, q.rows, q.d, q.ldx, q.seg_rows, q.seg_stride, q.g, q.ldg, stream);
    } else if (paths[p] == GramPath::kSimt) {
      rc = syrk_simt_launch(q.x, dtype, q.rows, q.d, q.ldx, q.g, q.ldg, stream);
    } else if (paths[p] == GramPath::kPerSegment) {
      // row segments the CTA-pair kernel cannot read in one launch: each segment is a Gram of its own
      const int elem = dtype == VLM_F32 ? 4 : 2;
      for (int64_t s = 0; s < q.rows / q.seg_rows && rc == 0; ++s) {
        const char* xs = static_cast<const char*>(q.x) + (size_t)s * q.seg_stride * elem;
        rc = syrk_pair_supported(dtype, xs, q.d, q.ldx, 0, q.g, q.ldg)
                 ? syrk_pair_launch(xs, dtype, q.seg_rows, q.d, q.ldx, 0, 0, q.g, q.ldg, stream)
                 : syrk_simt_launch(xs, dtype, q.seg_rows, q.d, q.ldx, q.g, q.ldg, stream);
      }
    }
    if (rc) return rc;
  }
  if (grouped.empty()) return 0;
  return syrk_pair_batch_launch(grouped.data(), (int)grouped.size(), dtype, stream);
}
}  // namespace

extern "C" int vlm_syrk_accum(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                              void* stream) {
  const vlm_syrk_problem q{x, rows, ldx, g, ldg, d, 0, 0, 0};
  return syrk_route(Entry::kAccum, &q, 1, dtype, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_syrk_accum_strided(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                                      int64_t seg_stride, float* g, int64_t ldg, void* stream) {
  const vlm_syrk_problem q{x, rows, ldx, g, ldg, d, 0, seg_rows, seg_stride};
  return syrk_route(Entry::kStrided, &q, 1, dtype, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_syrk_accum_batch(const vlm_syrk_problem* probs, int n, int dtype, void* stream) {
  VLM_REQUIRE(n >= 0 && (probs != nullptr || n == 0), VLM_ERR_INVALID_ARG, "vlm_syrk_accum_batch: bad arguments");
  return syrk_route(Entry::kBatch, probs, n, dtype, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_syrk_accum_simt(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                                   void* stream) {
  if (int rc = check_syrk_args("vlm_syrk_accum_simt", x, dtype, rows, d, ldx, g, ldg)) return rc;
  if (rows == 0) return 0;
  return syrk_simt_launch(x, dtype, rows, d, ldx, g, ldg, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_tf32_split(const float* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                              float* out, void* stream) {
  VLM_REQUIRE(rows >= 0 && d > 0 && d % 4 == 0 && out != nullptr && (rows == 0 || (x != nullptr && ldx >= d)),
              VLM_ERR_INVALID_ARG, "vlm_tf32_split: bad arguments (rows=%lld d=%d)", (long long)rows, d);
  VLM_REQUIRE(seg_rows >= 0 && seg_stride >= 0 && (seg_rows == 0 || rows % seg_rows == 0), VLM_ERR_INVALID_ARG,
              "vlm_tf32_split: rows (%lld) must be a multiple of seg_rows (%lld)", (long long)rows, (long long)seg_rows);
  VLM_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx & 3) == 0 && (seg_stride & 3) == 0 &&
                  (reinterpret_cast<uintptr_t>(out) & 15) == 0,
              VLM_ERR_ALIGNMENT, "vlm_tf32_split: x / out must be 16-byte aligned, ldx and seg_stride multiples of 4");
  if (rows == 0) return 0;
  if (int rc = require_sm100()) return rc;
  return tf32_split_launch(x, rows, d, ldx, seg_rows, seg_stride, out, static_cast<cudaStream_t>(stream));
}

extern "C" uint64_t vlm_syrk_i8x4_scratch_bytes(int64_t rows, int d) {
  return (rows > 0 && d > 0) ? (uint64_t)syrk_i8x4_scratch_bytes(rows, d) : 0;
}

extern "C" int vlm_syrk_accum_i8x4(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                                   int64_t seg_stride, void* scratch, uint64_t scratch_bytes, double* g, int64_t ldg,
                                   void* stream) {
  VLM_REQUIRE(dtype == VLM_F32 || dtype == VLM_F16 || dtype == VLM_BF16, VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_i8x4: dtype must be VLM_F32, VLM_F16 or VLM_BF16 (got %d)", dtype);
  VLM_REQUIRE(rows >= 0 && d > 0 && g != nullptr && ldg >= d && (rows == 0 || (x != nullptr && ldx >= d)),
              VLM_ERR_INVALID_ARG, "vlm_syrk_accum_i8x4: bad arguments (rows=%lld d=%d)", (long long)rows, d);
  VLM_REQUIRE(d % 128 == 0, VLM_ERR_UNSUPPORTED,
              "vlm_syrk_accum_i8x4: d must be a multiple of 128 (got %d); use vlm_syrk_accum_f64", d);
  VLM_REQUIRE(seg_rows >= 0 && seg_stride >= 0 && (seg_rows == 0 || rows % seg_rows == 0), VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_i8x4: rows (%lld) must be a multiple of seg_rows (%lld)", (long long)rows, (long long)seg_rows);
  VLM_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx & 3) == 0 && (seg_stride & 3) == 0 &&
                  (reinterpret_cast<uintptr_t>(scratch) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 &&
                  (ldg & 1) == 0,
              VLM_ERR_ALIGNMENT,
              "vlm_syrk_accum_i8x4: x / scratch / g must be 16-byte aligned, ldx and seg_stride multiples of 4, ldg even");
  VLM_REQUIRE(rows < ((int64_t)1 << 31), VLM_ERR_INVALID_ARG, "vlm_syrk_accum_i8x4: rows too large");
  if (rows == 0) return 0;
  VLM_REQUIRE(scratch != nullptr && scratch_bytes >= syrk_i8x4_scratch_bytes(rows, d), VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_i8x4: scratch too small (%llu bytes, need %llu)", (unsigned long long)scratch_bytes,
              (unsigned long long)syrk_i8x4_scratch_bytes(rows, d));
  if (int rc = require_sm100()) return rc;
  return syrk_i8x4_launch(x, dtype, rows, d, ldx, seg_rows, seg_stride, scratch, g, ldg, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_syrk_pair_schedule_host(int64_t rows, int d, int elem_bytes, int nsm, int32_t* segs_out, int cap,
                                           int32_t* off_out, int off_cap, int* ncluster_out) {
  VLM_REQUIRE(rows > 0 && d > 0 && (elem_bytes == 1 || elem_bytes == 2 || elem_bytes == 4) && nsm > 1 && ncluster_out,
              VLM_ERR_INVALID_ARG, "vlm_syrk_pair_schedule_host: bad arguments");
  const int bk = elem_bytes == 1 ? 32 : 128 / elem_bytes;  // int8: the 32-row chunks of the int8 schedule
  std::vector<int32_t> flat;
  std::vector<int> off;
  syrk_schedule_host((rows + bk - 1) / bk, d, nsm, elem_bytes == 1, &flat, &off);
  *ncluster_out = (int)off.size() - 1;
  VLM_REQUIRE((int)flat.size() <= 4 * cap && (int)off.size() <= off_cap, VLM_ERR_INVALID_ARG,
              "vlm_syrk_pair_schedule_host: output capacity too small (%d segments)", (int)flat.size() / 4);
  for (size_t i = 0; i < flat.size(); ++i) segs_out[i] = flat[i];
  for (size_t i = 0; i < off.size(); ++i) off_out[i] = off[i];
  return (int)flat.size() / 4;
}
