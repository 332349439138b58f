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
  static EncodeTiledFn encode = nullptr;
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    VLM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    VLM_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, VLM_ERR_DRIVER,
                "cuTensorMapEncodeTiled not available from the driver");
    encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *out = encode;
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

extern "C" int vlm_syrk_accum(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                              void* stream) {
  if (int rc = check_syrk_args("vlm_syrk_accum", x, dtype, rows, d, ldx, g, ldg)) return rc;
  if (rows == 0) return 0;
  if (int rc = require_sm100()) return rc;
  const bool pair = syrk_pair_supported(dtype, x, d, ldx, 0, g, ldg);
  if (dtype == VLM_TF32X2) {  // the planes exist only for the CTA-pair kernel
    VLM_REQUIRE(d % 32 == 0, VLM_ERR_UNSUPPORTED,
                "vlm_syrk_accum: VLM_TF32X2 needs d %% 32 == 0 (got %d); use vlm_syrk_accum_simt on the fp32 activation", d);
    VLM_REQUIRE(pair, VLM_ERR_ALIGNMENT,
                "vlm_syrk_accum: VLM_TF32X2 planes and g must be 16-byte aligned with ldx and ldg multiples of 4");
  }
  if (pair) return syrk_pair_launch(x, dtype, rows, d, ldx, 0, 0, g, ldg, static_cast<cudaStream_t>(stream));
  return syrk_simt_launch(x, dtype, rows, d, ldx, g, ldg, static_cast<cudaStream_t>(stream));
}

namespace {
int check_segments(const char* who, int dtype, int64_t rows, int64_t seg_rows, int64_t seg_stride) {
  VLM_REQUIRE(seg_rows > 0 && rows % seg_rows == 0, VLM_ERR_INVALID_ARG,
              "%s: rows (%lld) must be a multiple of seg_rows (%lld)", who, (long long)rows, (long long)seg_rows);
  VLM_REQUIRE(seg_stride >= 0, VLM_ERR_INVALID_ARG, "%s: seg_stride < 0", who);
  (void)dtype;
  return 0;
}
}  // namespace

extern "C" int vlm_syrk_accum_strided(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                                      int64_t seg_stride, float* g, int64_t ldg, void* stream) {
  if (int rc = check_syrk_args("vlm_syrk_accum_strided", x, dtype, rows, d, ldx, g, ldg)) return rc;
  if (rows == 0) return 0;
  if (int rc = check_segments("vlm_syrk_accum_strided", dtype, rows, seg_rows, seg_stride)) return rc;
  if (seg_rows == rows) return vlm_syrk_accum(x, dtype, rows, d, ldx, g, ldg, stream);
  VLM_REQUIRE(dtype != VLM_TF32X2, VLM_ERR_INVALID_ARG,
              "vlm_syrk_accum_strided: VLM_TF32X2 planes are packed by vlm_tf32_split, they have no row segments");
  if (int rc = require_sm100()) return rc;
  if (syrk_pair_supported(dtype, x, d, ldx, seg_stride, g, ldg))
    return syrk_pair_launch(x, dtype, rows, d, ldx, seg_rows, seg_stride, g, ldg, static_cast<cudaStream_t>(stream));
  // row segments the CTA-pair kernel cannot read in one launch: one vlm_syrk_accum per segment
  const int elem = dtype == VLM_F32 ? 4 : 2;
  for (int64_t s = 0; s < rows / seg_rows; ++s) {
    const char* xs = static_cast<const char*>(x) + (size_t)s * seg_stride * elem;
    if (int rc = vlm_syrk_accum(xs, dtype, seg_rows, d, ldx, g, ldg, stream)) return rc;
  }
  return 0;
}

extern "C" int vlm_syrk_accum_batch(const vlm_syrk_problem* probs, int n, int dtype, void* stream) {
  VLM_REQUIRE(n >= 0 && (probs != nullptr || n == 0), VLM_ERR_INVALID_ARG, "vlm_syrk_accum_batch: bad arguments");
  if (n == 0) return 0;
  if (int rc = require_sm100()) return rc;
  std::vector<vlm_syrk_problem> grouped;
  for (int p = 0; p < n; ++p) {
    const vlm_syrk_problem& q = probs[p];
    if (int rc = check_syrk_args("vlm_syrk_accum_batch", q.x, dtype, q.rows, q.d, q.ldx, q.g, q.ldg)) return rc;
    if (q.rows == 0) continue;
    const bool segmented = dtype != VLM_TF32X2 && q.seg_rows > 0 && q.seg_rows < q.rows;
    const bool pair = syrk_pair_supported(dtype, q.x, q.d, q.ldx, segmented ? q.seg_stride : 0, q.g, q.ldg);
    VLM_REQUIRE(dtype != VLM_TF32X2 || pair, VLM_ERR_UNSUPPORTED,
                "vlm_syrk_accum_batch: VLM_TF32X2 needs d %% 32 == 0 and 16-byte aligned planes");
    if (segmented) {
      if (int rc = check_segments("vlm_syrk_accum_batch", dtype, q.rows, q.seg_rows, q.seg_stride)) return rc;
    }
    if (pair) {
      grouped.push_back(q);
    } else if (segmented) {
      if (int rc = vlm_syrk_accum_strided(q.x, dtype, q.rows, q.d, q.ldx, q.seg_rows, q.seg_stride, q.g, q.ldg, stream))
        return rc;
    } else if (int rc = vlm_syrk_accum(q.x, dtype, q.rows, q.d, q.ldx, q.g, q.ldg, stream)) {
      return rc;
    }
  }
  if (grouped.empty()) return 0;
  return syrk_pair_batch_launch(grouped.data(), (int)grouped.size(), dtype, static_cast<cudaStream_t>(stream));
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
  const int bk = 128 / elem_bytes;
  std::vector<int32_t> flat;
  std::vector<int> off;
  if (elem_bytes == 1)
    build_syrk_i8_schedule_host((rows + 31) / 32, d, nsm, &flat, &off);
  else
    build_syrk_pair_schedule_host((rows + bk - 1) / bk, d, nsm, &flat, &off);
  *ncluster_out = (int)off.size() - 1;
  VLM_REQUIRE((int)flat.size() <= 4 * cap && (int)off.size() <= off_cap, VLM_ERR_INVALID_ARG,
              "vlm_syrk_pair_schedule_host: output capacity too small (%d segments)", (int)flat.size() / 4);
  for (size_t i = 0; i < flat.size(); ++i) segs_out[i] = flat[i];
  for (size_t i = 0; i < off.size(); ++i) off_out[i] = off[i];
  return (int)flat.size() / 4;
}
