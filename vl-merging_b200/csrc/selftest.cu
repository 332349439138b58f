// selftest.cu — native smoke/benchmark of libvlmerge on a B200, independent of Python.
//   build/selftest [quick|full]
// For every kernel it checks the result against a host fp64 computation (or the SIMT kernel for
// the large SYRK shapes) and prints one line per case: rel. Frobenius error, time, TFLOP/s or GB/s.
// Exit code = number of failed cases.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <functional>
#include <utility>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <vector>

#include "../../include/vlmerge.h"

#define CK(x)                                                                             \
  do {                                                                                    \
    cudaError_t e_ = (x);                                                                 \
    if (e_ != cudaSuccess) {                                                              \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__);     \
      exit(99);                                                                           \
    }                                                                                     \
  } while (0)
#define VK(x)                                                              \
  do {                                                                     \
    int r_ = (x);                                                          \
    if (r_ != 0) {                                                         \
      printf("vlm error %d: %s (%s:%d)\n", r_, vlm_last_error(), __FILE__, __LINE__); \
      exit(98);                                                            \
    }                                                                      \
  } while (0)

static uint64_t g_rng = 0x9E3779B97F4A7C15ull;
static inline float frand() {  // uniform (-1, 1)
  g_rng = g_rng * 6364136223846793005ull + 1442695040888963407ull;
  return (float)((g_rng >> 40) & 0xFFFFFF) / 8388608.0f - 1.0f;
}

static int g_fail = 0;

// the lower triangle of one d x d Gram (pitch ld) from its upper one
static void mirror(void* g, int d, int64_t ld, int dtype) {
  const vlm_sym_item it = {g, nullptr, d, 0, ld};
  VK(vlm_sym_mirror_batch(&it, 1, dtype, nullptr));
}

struct Timer {
  cudaEvent_t a, b;
  Timer() {
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
  }
  void start() { CK(cudaEventRecord(a)); }
  float stop() {
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms;
    CK(cudaEventElapsedTime(&ms, a, b));
    return ms;
  }
};

// ---- SYRK ----------------------------------------------------------------------------------
template <typename T>
static void fill_x(std::vector<T>& h, int mode);
template <>
void fill_x<float>(std::vector<float>& h, int mode) {
  for (auto& v : h) {
    float f = frand();
    v = mode == 1 ? fabsf(f) + 0.25f : f;
  }
}
template <>
void fill_x<__nv_bfloat16>(std::vector<__nv_bfloat16>& h, int mode) {
  for (auto& v : h) {
    float f = frand();
    v = __float2bfloat16(mode == 1 ? fabsf(f) + 0.25f : f);
  }
}
template <>
void fill_x<__half>(std::vector<__half>& h, int mode) {
  for (auto& v : h) {
    float f = frand();
    v = __float2half(mode == 1 ? fabsf(f) + 0.25f : f);
  }
}
static inline double to_d(float v) { return v; }
static inline double to_d(__nv_bfloat16 v) { return __bfloat162float(v); }
static inline double to_d(__half v) { return __half2float(v); }

// compares the upper triangle of two d x d matrices; returns rel. Frobenius error
static double upper_rel_err(const std::vector<float>& a, const std::vector<double>& ref, int d, double* max_abs,
                            int* wr, int* wc) {
  double num = 0, den = 0;
  *max_abs = 0;
  *wr = *wc = -1;
  for (int r = 0; r < d; ++r)
    for (int c = r; c < d; ++c) {
      const double x = a[(size_t)r * d + c], y = ref[(size_t)r * d + c];
      const double e = x - y;
      num += e * e;
      den += y * y;
      if (fabs(e) > *max_abs) {
        *max_abs = fabs(e);
        *wr = r;
        *wc = c;
      }
    }
  return sqrt(num / (den > 0 ? den : 1));
}

template <typename T>
static void syrk_case(const char* name, int dtype, int64_t rows, int d, int mode, bool host_ref, int iters,
                      double tol) {
  const int64_t ldx = d;
  std::vector<T> hx((size_t)rows * d);
  fill_x<T>(hx, mode);
  T* dx;
  float *g_tc, *g_ref;
  CK(cudaMalloc(&dx, hx.size() * sizeof(T)));
  CK(cudaMalloc(&g_tc, (size_t)d * d * 4));
  CK(cudaMalloc(&g_ref, (size_t)d * d * 4));
  CK(cudaMemcpy(dx, hx.data(), hx.size() * sizeof(T), cudaMemcpyHostToDevice));
  CK(cudaMemset(g_tc, 0, (size_t)d * d * 4));
  CK(cudaMemset(g_ref, 0, (size_t)d * d * 4));

  std::vector<double> ref((size_t)d * d, 0.0);
  std::vector<int> sample_rows;  // host fp64 reference restricted to these rows when !host_ref
  if (host_ref) {
    for (int64_t k = 0; k < rows; ++k) {
      const T* xr = &hx[(size_t)k * d];
      for (int r = 0; r < d; ++r) {
        const double a = to_d(xr[r]);
        double* o = &ref[(size_t)r * d];
        for (int c = r; c < d; ++c) o[c] += a * to_d(xr[c]);
      }
    }
  } else {
    // exact fp64 rows on the host (12 rows spread over the row blocks) ...
    for (int t = 0; t < 12; ++t) sample_rows.push_back((int)(((int64_t)t * 2654435761ll + 17) % d));
    for (int r : sample_rows) {
      double* o = &ref[(size_t)r * d];
      for (int c = 0; c < d; ++c) o[c] = 0;
      for (int64_t k = 0; k < rows; ++k) {
        const T* xr = &hx[(size_t)k * d];
        const double a = to_d(xr[r]);
        for (int c = r; c < d; ++c) o[c] += a * to_d(xr[c]);
      }
    }
    // ... and the CUDA-core kernel over the whole matrix (fp32 accumulation: looser check)
    VK(vlm_syrk_accum_simt(dx, dtype, rows, d, ldx, g_ref, d, nullptr));
    CK(cudaDeviceSynchronize());
  }

  // two accumulating calls: checks "+=" across calls as well (reference doubled)
  VK(vlm_syrk_accum(dx, dtype, rows, d, ldx, g_tc, d, nullptr));
  VK(vlm_syrk_accum(dx, dtype, rows, d, ldx, g_tc, d, nullptr));
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("SYRK %-28s KERNEL FAILED: %s\n", name, cudaGetErrorString(e));
    exit(97);
  }
  std::vector<float> out((size_t)d * d);
  CK(cudaMemcpy(out.data(), g_tc, out.size() * 4, cudaMemcpyDeviceToHost));
  for (auto& v : ref) v *= 2.0;
  double max_abs = 0;
  int wr = -1, wc = -1;
  double err;
  double simt_err = 0;
  if (host_ref) {
    err = upper_rel_err(out, ref, d, &max_abs, &wr, &wc);
  } else {
    double num = 0, den = 0;
    for (int r : sample_rows)
      for (int c = r; c < d; ++c) {
        const double e = out[(size_t)r * d + c] - ref[(size_t)r * d + c];
        num += e * e;
        den += ref[(size_t)r * d + c] * ref[(size_t)r * d + c];
        if (fabs(e) > max_abs) max_abs = fabs(e), wr = r, wc = c;
      }
    err = sqrt(num / den);
    std::vector<float> simt((size_t)d * d);
    CK(cudaMemcpy(simt.data(), g_ref, simt.size() * 4, cudaMemcpyDeviceToHost));
    num = den = 0;
    for (int r = 0; r < d; ++r)
      for (int c = r; c < d; ++c) {
        const double y = 2.0 * simt[(size_t)r * d + c];
        const double e = out[(size_t)r * d + c] - y;
        num += e * e;
        den += y * y;
      }
    simt_err = sqrt(num / den);
    if (simt_err > 3e-3) err = simt_err;  // whole-matrix sanity: a misplaced tile shows up here
  }

  // finalize: mirror check
  mirror(g_tc, d, d, VLM_F32);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out.data(), g_tc, out.size() * 4, cudaMemcpyDeviceToHost));
  size_t asym = 0;
  for (int r = 0; r < d; ++r)
    for (int c = 0; c < r; ++c) asym += out[(size_t)r * d + c] != out[(size_t)c * d + r];

  float ms = 0;
  if (iters > 0) {
    Timer t;
    for (int i = 0; i < 3; ++i) VK(vlm_syrk_accum(dx, dtype, rows, d, ldx, g_tc, d, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum(dx, dtype, rows, d, ldx, g_tc, d, nullptr));
    ms = t.stop() / iters;
  }
  const double flops = (double)rows * d * (d + 1.0);  // symmetric count
  const bool ok = err <= tol && asym == 0 && std::isfinite(err);
  printf("SYRK %-28s rows=%-6lld d=%-5d relF=%.3e vs_simt=%.1e maxabs=%.3e@(%d,%d) asym=%zu  %.3f ms  %.1f TFLOP/s(sym)  %s\n",
         name, (long long)rows, d, err, simt_err, max_abs, wr, wc, asym, ms, ms > 0 ? flops / ms * 1e-9 : 0.0,
         ok ? "OK" : "FAIL");
  if (!ok) {
    ++g_fail;
    // a few samples to help diagnose layout mistakes
    for (int r = 0; r < 2; ++r)
      for (int c : {r, r + 1, 31, 32, 127, 128, 255, 256}) {
        if (c < d && c >= r) printf("   G[%d][%d] got %.6g want %.6g\n", r, c, out[(size_t)r * d + c], ref[(size_t)r * d + c]);
      }
  }
  CK(cudaFree(dx));
  CK(cudaFree(g_tc));
  CK(cudaFree(g_ref));
}



// Split-precision Gram (vlm_tf32_split + VLM_TF32X2): host fp64 Gram of the whole matrix (host_ref) or of 12
// sample rows; optionally a row-segmented source (nseg > 1: rows = nseg * seg_rows out of n_tok-row items).
static void syrk_split_case(const char* name, int nseg, int n_tok, int off, int seg_rows, int d, int mode, bool host_ref,
                            int iters, double tol) {
  std::vector<float> hx((size_t)nseg * n_tok * d);
  fill_x<float>(hx, mode);
  const int64_t rows = (int64_t)nseg * seg_rows;
  float *dx, *planes, *g;
  CK(cudaMalloc(&dx, hx.size() * 4));
  CK(cudaMalloc(&planes, (size_t)2 * rows * d * 4));
  CK(cudaMalloc(&g, (size_t)d * d * 4));
  CK(cudaMemcpy(dx, hx.data(), hx.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(g, 0, (size_t)d * d * 4));
  const float* slice = dx + (size_t)off * d;
  auto xrow = [&](int64_t k) { return &hx[(((size_t)(k / seg_rows)) * n_tok + off + (k % seg_rows)) * d]; };
  std::vector<int> rs;
  if (host_ref) for (int r = 0; r < d; ++r) rs.push_back(r);
  else for (int t = 0; t < 12; ++t) rs.push_back((int)(((int64_t)t * 2654435761ll + 17) % d));
  std::vector<double> ref((size_t)d * d, 0.0);
  for (int r : rs) {
    double* o = &ref[(size_t)r * d];
    for (int c = 0; c < d; ++c) o[c] = 0;
    for (int64_t k = 0; k < rows; ++k) {
      const float* xr = xrow(k);
      const double a = xr[r];
      for (int c = r; c < d; ++c) o[c] += a * (double)xr[c];
    }
  }
  VK(vlm_tf32_split(slice, rows, d, d, nseg > 1 ? seg_rows : 0, (int64_t)n_tok * d, planes, nullptr));
  VK(vlm_syrk_accum(planes, VLM_TF32X2, rows, d, d, g, d, nullptr));
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("SPLIT %-27s KERNEL FAILED: %s\n", name, cudaGetErrorString(e));
    exit(97);
  }
  std::vector<float> out((size_t)d * d);
  CK(cudaMemcpy(out.data(), g, out.size() * 4, cudaMemcpyDeviceToHost));
  double num = 0, den = 0, max_abs = 0;
  for (int r : rs)
    for (int c = r; c < d; ++c) {
      const double df = out[(size_t)r * d + c] - ref[(size_t)r * d + c];
      num += df * df;
      den += ref[(size_t)r * d + c] * ref[(size_t)r * d + c];
      if (fabs(df) > max_abs) max_abs = fabs(df);
    }
  const double err = sqrt(num / den);
  float ms_split = 0, ms_syrk = 0;
  if (iters > 0) {
    Timer t;
    for (int i = 0; i < 2; ++i) VK(vlm_syrk_accum(planes, VLM_TF32X2, rows, d, d, g, d, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum(planes, VLM_TF32X2, rows, d, d, g, d, nullptr));
    ms_syrk = t.stop() / iters;
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_tf32_split(slice, rows, d, d, nseg > 1 ? seg_rows : 0, (int64_t)n_tok * d, planes, nullptr));
    ms_split = t.stop() / iters;
  }
  const double flops = (double)rows * d * (d + 1.0);
  const bool ok = err <= tol && std::isfinite(err);
  printf("SPLIT %-27s rows=%-6lld d=%-5d relF=%.3e maxabs=%.3e  split %.3f ms + syrk %.3f ms  %.1f TFLOP/s(sym, 1x count)  %s\n",
         name, (long long)rows, d, err, max_abs, ms_split, ms_syrk, ms_syrk > 0 ? flops / (ms_syrk + ms_split) * 1e-9 : 0.0,
         ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  CK(cudaFree(dx));
  CK(cudaFree(planes));
  CK(cudaFree(g));
}


// Reference-precision Gram (vlm_syrk_accum_f64): host fp64 Gram of the whole matrix (host_ref) or of 12 sample rows;
// optionally a row-segmented source.  Two accumulating calls (checks "+=" and the split-K reduction), then the mirror.
template <typename T>
static void syrk_f64_case(const char* name, int dtype, int nseg, int n_tok, int off, int seg_rows, int d, int mode,
                          bool host_ref, int iters, double tol) {
  std::vector<T> hx((size_t)nseg * n_tok * d);
  fill_x<T>(hx, mode);
  const int64_t rows = (int64_t)nseg * seg_rows;
  T* dx;
  double* g;
  CK(cudaMalloc(&dx, hx.size() * sizeof(T)));
  CK(cudaMalloc(&g, (size_t)d * d * 8));
  CK(cudaMemcpy(dx, hx.data(), hx.size() * sizeof(T), cudaMemcpyHostToDevice));
  CK(cudaMemset(g, 0, (size_t)d * d * 8));
  const T* slice = dx + (size_t)off * d;
  auto xrow = [&](int64_t k) { return &hx[(((size_t)(k / seg_rows)) * n_tok + off + (k % seg_rows)) * d]; };
  std::vector<int> rs;
  if (host_ref) for (int r = 0; r < d; ++r) rs.push_back(r);
  else for (int t = 0; t < 12; ++t) rs.push_back((int)(((int64_t)t * 2654435761ll + 17) % d));
  std::vector<double> ref((size_t)d * d, 0.0);
  for (int r : rs) {
    double* o = &ref[(size_t)r * d];
    for (int c = 0; c < d; ++c) o[c] = 0;
    for (int64_t k = 0; k < rows; ++k) {
      const T* xr = xrow(k);
      const double a = to_d(xr[r]);
      for (int c = r; c < d; ++c) o[c] += a * to_d(xr[c]);
    }
  }
  const int64_t sr = nseg > 1 ? seg_rows : 0;
  VK(vlm_syrk_accum_f64(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, g, d, nullptr));
  VK(vlm_syrk_accum_f64(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, g, d, nullptr));
  mirror(g, d, d, VLM_F64);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("F64   %-27s KERNEL FAILED: %s\n", name, cudaGetErrorString(e));
    exit(97);
  }
  std::vector<double> out((size_t)d * d);
  CK(cudaMemcpy(out.data(), g, out.size() * 8, cudaMemcpyDeviceToHost));
  double num = 0, den = 0;
  size_t asym = 0;
  for (int r : rs)
    for (int c = r; c < d; ++c) {
      const double want = 2.0 * ref[(size_t)r * d + c];
      const double df = out[(size_t)r * d + c] - want;
      num += df * df;
      den += want * want;
      asym += out[(size_t)c * d + r] != out[(size_t)r * d + c];
    }
  const double err = sqrt(num / den);
  float ms = 0;
  if (iters > 0) {
    Timer t;
    VK(vlm_syrk_accum_f64(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, g, d, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum_f64(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, g, d, nullptr));
    ms = t.stop() / iters;
  }
  const double flops = (double)rows * d * (d + 1.0);
  const bool ok = err <= tol && asym == 0 && std::isfinite(err);
  printf("F64   %-27s rows=%-6lld d=%-5d relF=%.3e asym=%zu  %.3f ms  %.2f TFLOP/s(sym)  %s\n", name, (long long)rows, d, err,
         asym, ms, ms > 0 ? flops / ms * 1e-9 : 0.0, ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  CK(cudaFree(dx));
  CK(cudaFree(g));
}


// Exact Gram on the integer tensor cores (vlm_syrk_accum_i8x4): host fp64 Gram of the whole matrix (host_ref) or of 12 sample rows;
// optionally a row-segmented source.  Two accumulating calls (checks "+=" and the split-K reduction), then the mirror.
template <typename T>
static void syrk_i8_case(const char* name, int dtype, int nseg, int n_tok, int off, int seg_rows, int d, int mode,
                          bool host_ref, int iters, double tol) {
  std::vector<T> hx((size_t)nseg * n_tok * d);
  fill_x<T>(hx, mode);
  const int64_t rows = (int64_t)nseg * seg_rows;
  T* dx;
  double* g;
  CK(cudaMalloc(&dx, hx.size() * sizeof(T)));
  CK(cudaMalloc(&g, (size_t)d * d * 8));
  void* scratch;
  const uint64_t sbytes = vlm_syrk_i8x4_scratch_bytes(rows, d);
  CK(cudaMalloc(&scratch, sbytes));
  CK(cudaMemcpy(dx, hx.data(), hx.size() * sizeof(T), cudaMemcpyHostToDevice));
  CK(cudaMemset(g, 0, (size_t)d * d * 8));
  const T* slice = dx + (size_t)off * d;
  auto xrow = [&](int64_t k) { return &hx[(((size_t)(k / seg_rows)) * n_tok + off + (k % seg_rows)) * d]; };
  std::vector<int> rs;
  if (host_ref) for (int r = 0; r < d; ++r) rs.push_back(r);
  else for (int t = 0; t < 12; ++t) rs.push_back((int)(((int64_t)t * 2654435761ll + 17) % d));
  std::vector<double> ref((size_t)d * d, 0.0);
  for (int r : rs) {
    double* o = &ref[(size_t)r * d];
    for (int c = 0; c < d; ++c) o[c] = 0;
    for (int64_t k = 0; k < rows; ++k) {
      const T* xr = xrow(k);
      const double a = to_d(xr[r]);
      for (int c = r; c < d; ++c) o[c] += a * to_d(xr[c]);
    }
  }
  const int64_t sr = nseg > 1 ? seg_rows : 0;
  VK(vlm_syrk_accum_i8x4(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, scratch, sbytes, g, d, nullptr));
  VK(vlm_syrk_accum_i8x4(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, scratch, sbytes, g, d, nullptr));
  mirror(g, d, d, VLM_F64);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("I8X4  %-27s KERNEL FAILED: %s\n", name, cudaGetErrorString(e));
    exit(97);
  }
  std::vector<double> out((size_t)d * d);
  CK(cudaMemcpy(out.data(), g, out.size() * 8, cudaMemcpyDeviceToHost));
  double num = 0, den = 0;
  size_t asym = 0;
  for (int r : rs)
    for (int c = r; c < d; ++c) {
      const double want = 2.0 * ref[(size_t)r * d + c];
      const double df = out[(size_t)r * d + c] - want;
      num += df * df;
      den += want * want;
      asym += out[(size_t)c * d + r] != out[(size_t)r * d + c];
    }
  const double err = sqrt(num / den);
  float ms = 0;
  if (iters > 0) {
    Timer t;
    VK(vlm_syrk_accum_i8x4(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, scratch, sbytes, g, d, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum_i8x4(slice, dtype, rows, d, d, sr, (int64_t)n_tok * d, scratch, sbytes, g, d, nullptr));
    ms = t.stop() / iters;
  }
  const double flops = (double)rows * d * (d + 1.0);
  const bool ok = err <= tol && asym == 0 && std::isfinite(err);
  printf("I8X4  %-27s rows=%-6lld d=%-5d relF=%.3e asym=%zu  %.3f ms  %.2f TFLOP/s(sym)  %s\n", name, (long long)rows, d, err,
         asym, ms, ms > 0 ? flops / ms * 1e-9 : 0.0, ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  CK(cudaFree(dx));
  CK(cudaFree(g));
  CK(cudaFree(scratch));
}



// Grouped launch of n1 problems (rows1 x d1) + n2 problems (rows2 x d2), all fp32, distinct activations and Grams:
// correctness of every Gram against the single-launch kernel, and the rate of the group (what GramCache's deferred
// flush issues: e.g. 9 x [36928, 768] for a slice of the image tower, 36 x [2560, 768] + 12 x [2560, 3072] for the text tower).
static void syrk_batch_case(int n1, int64_t rows1, int d1, int n2, int64_t rows2, int d2, int iters) {
  const int n = n1 + n2;
  std::vector<vlm_syrk_problem> pr(n);
  std::vector<float*> xs(n), gs(n), refs(n);
  double flops = 0;
  for (int p = 0; p < n; ++p) {
    const int64_t rows = p < n1 ? rows1 : rows2;
    const int d = p < n1 ? d1 : d2;
    std::vector<float> hx((size_t)rows * d);
    fill_x<float>(hx, p & 1);
    CK(cudaMalloc(&xs[p], hx.size() * 4));
    CK(cudaMemcpy(xs[p], hx.data(), hx.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMalloc(&gs[p], (size_t)d * d * 4));
    CK(cudaMalloc(&refs[p], (size_t)d * d * 4));
    CK(cudaMemset(gs[p], 0, (size_t)d * d * 4));
    CK(cudaMemset(refs[p], 0, (size_t)d * d * 4));
    pr[p] = vlm_syrk_problem{xs[p], rows, d, gs[p], d, d, 0, 0, 0};
    flops += (double)rows * d * (d + 1.0);
    VK(vlm_syrk_accum(xs[p], VLM_F32, rows, d, d, refs[p], d, nullptr));
  }
  VK(vlm_syrk_accum_batch(pr.data(), n, VLM_F32, nullptr));
  CK(cudaDeviceSynchronize());
  double worst = 0;
  for (int p = 0; p < n; ++p) {
    const int d = p < n1 ? d1 : d2;
    std::vector<float> a((size_t)d * d), b((size_t)d * d);
    CK(cudaMemcpy(a.data(), gs[p], a.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b.data(), refs[p], b.size() * 4, cudaMemcpyDeviceToHost));
    double num = 0, den = 0;
    for (int r = 0; r < d; ++r)
      for (int c = r; c < d; ++c) {
        const double e = (double)a[(size_t)r * d + c] - b[(size_t)r * d + c];
        num += e * e;
        den += (double)b[(size_t)r * d + c] * b[(size_t)r * d + c];
      }
    worst = std::max(worst, sqrt(num / den));
  }
  float ms = 0;
  if (iters > 0) {
    Timer t;
    for (int i = 0; i < 2; ++i) VK(vlm_syrk_accum_batch(pr.data(), n, VLM_F32, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum_batch(pr.data(), n, VLM_F32, nullptr));
    ms = t.stop() / iters;
  }
  const bool ok = worst < 5e-5;   // same kernel, same operands: only segment boundaries and the order of the reduce-adds differ
  printf("BATCH %d x [%lld, %d] + %d x [%lld, %d]  vs single launches relF=%.2e  %.3f ms  %.1f TFLOP/s(sym)  %s\n", n1,
         (long long)rows1, d1, n2, (long long)rows2, d2, worst, ms, ms > 0 ? flops / ms * 1e-9 : 0.0, ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  for (int p = 0; p < n; ++p) {
    CK(cudaFree(xs[p]));
    CK(cudaFree(gs[p]));
    CK(cudaFree(refs[p]));
  }
}


// Fused similarity + top-10 (vlm_sim_topk) against a host computation: m x n scores of fp16 features, ten best
// columns per row (ties: lower column first).
static void simtopk_case(int m, int n, int d, int iters) {
  std::vector<__half> ha((size_t)m * d), hb((size_t)n * d);
  for (auto& v : ha) v = __float2half(frand());
  for (auto& v : hb) v = __float2half(frand());
  __half *da, *db;
  CK(cudaMalloc(&da, ha.size() * 2));
  CK(cudaMalloc(&db, hb.size() * 2));
  CK(cudaMemcpy(da, ha.data(), ha.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(db, hb.data(), hb.size() * 2, cudaMemcpyHostToDevice));
  const int splits = vlm_sim_topk_splits(m, n);
  float* dv;
  int* di;
  CK(cudaMalloc(&dv, (size_t)m * splits * 10 * 4));
  CK(cudaMalloc(&di, (size_t)m * splits * 10 * 4));
  VK(vlm_sim_topk(da, m, d, db, n, d, d, VLM_F16, dv, di, splits, nullptr));
  CK(cudaDeviceSynchronize());
  std::vector<float> hv((size_t)m * splits * 10);
  std::vector<int> hi((size_t)m * splits * 10);
  CK(cudaMemcpy(hv.data(), dv, hv.size() * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hi.data(), di, hi.size() * 4, cudaMemcpyDeviceToHost));
  int bad = 0;
  const int rows_checked = std::min(m, 64);
  std::vector<double> sc(n);
  for (int r = 0; r < rows_checked; ++r) {
    const int row = (int)(((int64_t)r * 2654435761ll) % m);
    for (int c = 0; c < n; ++c) {
      double acc = 0;
      for (int k = 0; k < d; ++k) acc += (double)__half2float(ha[(size_t)row * d + k]) * __half2float(hb[(size_t)c * d + k]);
      sc[c] = acc;
    }
    // merge the split lists of this row, then compare with the host's top-k by SCORE (fp32 accumulation may swap near-ties)
    std::vector<std::pair<float, int>> got;
    for (int t = 0; t < splits * 10; ++t)
      if (hi[((size_t)row * splits) * 10 + t] >= 0) got.push_back({hv[((size_t)row * splits) * 10 + t], hi[((size_t)row * splits) * 10 + t]});
    std::stable_sort(got.begin(), got.end(), [](auto& a, auto& b) { return a.first > b.first; });
    std::vector<double> want(sc);
    std::sort(want.begin(), want.end(), std::greater<double>());
    const int k = std::min(10, n);
    if ((int)got.size() < k) {
      ++bad;
      continue;
    }
    for (int t = 0; t < k; ++t) {
      const int c = got[t].second;
      if (c < 0 || c >= n || fabs(sc[c] - want[t]) > 1e-3 * sqrt((double)d) || fabs(got[t].first - sc[c]) > 1e-3 * sqrt((double)d)) ++bad;
    }
  }
  float ms = 0;
  if (iters > 0) {
    Timer t;
    VK(vlm_sim_topk(da, m, d, db, n, d, d, VLM_F16, dv, di, splits, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_sim_topk(da, m, d, db, n, d, d, VLM_F16, dv, di, splits, nullptr));
    ms = t.stop() / iters;
  }
  printf("SIMTOPK m=%-6d n=%-6d d=%-5d splits=%d mismatches=%d  %.3f ms  %.1f TFLOP/s  %s\n", m, n, d, splits, bad, ms,
         ms > 0 ? 2.0 * m * n * d / ms * 1e-9 : 0.0, bad == 0 ? "OK" : "FAIL");
  if (bad) ++g_fail;
  CK(cudaFree(da));
  CK(cudaFree(db));
  CK(cudaFree(dv));
  CK(cudaFree(di));
}

// Row-sliced activation: the view h[:, off:off+seg_rows] of an (nseg, n_tok, d) tensor, read in place
// (vlm_syrk_accum_strided, and the same problem through vlm_syrk_accum_batch) against a host fp64 Gram of the
// slice (host_ref) or the contiguous kernel on a packed copy of the slice.
template <typename T>
static void syrk_strided_case(const char* name, int dtype, int nseg, int n_tok, int off, int seg_rows, int d,
                              bool host_ref, int iters, double tol) {
  std::vector<T> hx((size_t)nseg * n_tok * d);
  fill_x<T>(hx, 0);
  const int64_t rows = (int64_t)nseg * seg_rows;
  std::vector<T> packed((size_t)rows * d);
  for (int s = 0; s < nseg; ++s)
    memcpy(&packed[(size_t)s * seg_rows * d], &hx[((size_t)s * n_tok + off) * d], (size_t)seg_rows * d * sizeof(T));
  T *dx, *dp;
  float *g1, *g2, *g3;
  CK(cudaMalloc(&dx, hx.size() * sizeof(T)));
  CK(cudaMalloc(&dp, packed.size() * sizeof(T)));
  CK(cudaMemcpy(dx, hx.data(), hx.size() * sizeof(T), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dp, packed.data(), packed.size() * sizeof(T), cudaMemcpyHostToDevice));
  for (float** g : {&g1, &g2, &g3}) {
    CK(cudaMalloc(g, (size_t)d * d * 4));
    CK(cudaMemset(*g, 0, (size_t)d * d * 4));
  }
  const T* slice = dx + (size_t)off * d;
  VK(vlm_syrk_accum_strided(slice, dtype, rows, d, d, seg_rows, (int64_t)n_tok * d, g1, d, nullptr));
  vlm_syrk_problem pr[2];
  memset(pr, 0, sizeof(pr));
  pr[0].x = slice, pr[0].rows = rows, pr[0].ldx = d, pr[0].g = g2, pr[0].ldg = d, pr[0].d = d;
  pr[0].seg_rows = seg_rows, pr[0].seg_stride = (int64_t)n_tok * d;
  pr[1].x = dp, pr[1].rows = rows, pr[1].ldx = d, pr[1].g = g3, pr[1].ldg = d, pr[1].d = d;  // contiguous twin
  VK(vlm_syrk_accum_batch(pr, 2, dtype, nullptr));
  CK(cudaDeviceSynchronize());
  std::vector<float> o1((size_t)d * d), o2((size_t)d * d), o3((size_t)d * d);
  CK(cudaMemcpy(o1.data(), g1, o1.size() * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(o2.data(), g2, o2.size() * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(o3.data(), g3, o3.size() * 4, cudaMemcpyDeviceToHost));
  std::vector<double> ref((size_t)d * d, 0.0);
  if (host_ref) {
    for (int64_t k = 0; k < rows; ++k) {
      const T* xr = &packed[(size_t)k * d];
      for (int r = 0; r < d; ++r) {
        const double a = to_d(xr[r]);
        double* o = &ref[(size_t)r * d];
        for (int c = r; c < d; ++c) o[c] += a * to_d(xr[c]);
      }
    }
  } else {
    for (size_t i = 0; i < ref.size(); ++i) ref[i] = o3[i];  // contiguous kernel on the packed copy
  }
  double ma = 0;
  int wr = -1, wc = -1;
  const double e1 = upper_rel_err(o1, ref, d, &ma, &wr, &wc);
  const double e2 = upper_rel_err(o2, ref, d, &ma, &wr, &wc);
  float ms = 0, ms_packed = 0;
  if (iters > 0) {
    Timer t;
    for (int i = 0; i < 3; ++i)
      VK(vlm_syrk_accum_strided(slice, dtype, rows, d, d, seg_rows, (int64_t)n_tok * d, g1, d, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i)
      VK(vlm_syrk_accum_strided(slice, dtype, rows, d, d, seg_rows, (int64_t)n_tok * d, g1, d, nullptr));
    ms = t.stop() / iters;
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_syrk_accum(dp, dtype, rows, d, d, g3, d, nullptr));
    ms_packed = t.stop() / iters;
  }
  const bool ok = e1 <= tol && e2 <= tol && std::isfinite(e1) && std::isfinite(e2);
  printf("SYRK-STRIDED %-24s segs=%d x %d rows (of %d) d=%-5d relF=%.3e batch=%.3e  %.3f ms (packed copy: %.3f ms)  %s\n",
         name, nseg, seg_rows, n_tok, d, e1, e2, ms, ms_packed, ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  CK(cudaFree(dx));
  CK(cudaFree(dp));
  CK(cudaFree(g1));
  CK(cudaFree(g2));
  CK(cudaFree(g3));
}

// ---- symmetric storage (sympack.cu): pack, unpack and mirror of one Gram with a padded pitch ------------------
// `g` and `out` start as copies of one random matrix; pack g, unpack into out, mirror g: both must then hold the
// symmetric matrix of g's upper triangle, with the padding columns untouched.
template <typename T>
static void pack_case(int d, int pad) {
  const int dtype = sizeof(T) == 4 ? VLM_F32 : VLM_F64;
  const int64_t ld = d + pad;
  std::vector<T> h((size_t)d * ld);
  for (auto& v : h) v = frand();
  T *g, *packed, *out;
  const size_t np = (size_t)d * (d + 1) / 2;
  CK(cudaMalloc(&g, h.size() * sizeof(T)));
  CK(cudaMalloc(&packed, np * sizeof(T)));
  CK(cudaMalloc(&out, h.size() * sizeof(T)));
  CK(cudaMemcpy(g, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(out, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  vlm_sym_item it = {g, packed, d, 0, ld};
  VK(vlm_sym_pack_upper_batch(&it, 1, dtype, nullptr));
  it.full = out;
  VK(vlm_sym_unpack_batch(&it, 1, dtype, nullptr));
  mirror(g, d, ld, dtype);
  CK(cudaDeviceSynchronize());
  std::vector<T> hp(np), hu(h.size()), hm(h.size());
  CK(cudaMemcpy(hp.data(), packed, np * sizeof(T), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hu.data(), out, hu.size() * sizeof(T), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hm.data(), g, hm.size() * sizeof(T), cudaMemcpyDeviceToHost));
  size_t bad = 0, k = 0;
  for (int r = 0; r < d; ++r)
    for (int c = r; c < d; ++c, ++k) bad += hp[k] != h[(size_t)r * ld + c];
  for (int r = 0; r < d; ++r)
    for (int c = 0; c < ld; ++c) {
      const T want = c < r ? h[(size_t)c * ld + r] : h[(size_t)r * ld + c];
      bad += hu[(size_t)r * ld + c] != want;
      bad += hm[(size_t)r * ld + c] != want;
    }
  printf("PACK %s d=%-5d ld=%-5lld mismatches=%zu  %s\n", dtype == VLM_F32 ? "f32" : "f64", d, (long long)ld, bad,
         bad == 0 ? "OK" : "FAIL");
  if (bad) ++g_fail;
  CK(cudaFree(g));
  CK(cudaFree(packed));
  CK(cudaFree(out));
}

// ---- merge ---------------------------------------------------------------------------------
static void merge_case(const char* name, int mode, int n_src, size_t n, size_t misalign, int iters) {
  std::vector<std::vector<float>> hs(n_src, std::vector<float>(n));
  for (auto& v : hs)
    for (auto& x : v) x = frand();
  float coef[4] = {0.5f, 0.5f, 1.0f / 3, 0.25f};
  if (mode == VLM_MERGE_SEQ_LERP) coef[1] = coef[2] = coef[3] = 0.75f;
  std::vector<float*> ds(n_src);
  for (int m = 0; m < n_src; ++m) {
    CK(cudaMalloc(&ds[m], (n + 8) * 4));
    CK(cudaMemcpy(ds[m] + misalign, hs[m].data(), n * 4, cudaMemcpyHostToDevice));
  }
  float* dd;
  CK(cudaMalloc(&dd, (n + 8) * 4));
  vlm_merge_seg seg;
  memset(&seg, 0, sizeof(seg));
  seg.dst = dd + misalign;
  for (int m = 0; m < n_src; ++m) {
    seg.src[m] = ds[m] + misalign;
    seg.coef[m] = coef[m];
  }
  seg.n = n;
  seg.n_src = n_src;
  seg.mode = mode;
  // split into several segments to exercise the chunk table
  std::vector<vlm_merge_seg> segs;
  size_t off = 0;
  const size_t parts[4] = {n / 2, n / 4, n > 777 ? (size_t)777 : (size_t)0, 0};
  for (int p = 0; p < 4; ++p) {
    size_t len = p == 3 ? n - off : (parts[p] / 4) * 4;
    if (len == 0) continue;
    vlm_merge_seg s2 = seg;
    s2.dst = seg.dst + off;
    for (int m = 0; m < n_src; ++m) s2.src[m] = seg.src[m] + off;
    s2.n = len;
    segs.push_back(s2);
    off += len;
  }
  vlm_merge_plan* plan;
  VK(vlm_merge_plan_create(segs.data(), (int)segs.size(), &plan));
  VK(vlm_merge_plan_run(plan, nullptr));
  CK(cudaDeviceSynchronize());
  std::vector<float> out(n);
  CK(cudaMemcpy(out.data(), dd + misalign, n * 4, cudaMemcpyDeviceToHost));
  size_t bad = 0;
  for (size_t i = 0; i < n; ++i) {
    volatile float acc;
    if (mode == VLM_MERGE_WSUM) {
      acc = coef[0] * hs[0][i];
      for (int m = 1; m < n_src; ++m) {
        volatile float p = coef[m] * hs[m][i];
        acc = acc + p;
      }
    } else if (mode == VLM_MERGE_SEQ_LERP) {
      acc = hs[0][i];
      for (int m = 1; m < n_src; ++m) {
        volatile float dlt = hs[m][i] - acc;
        volatile float p = coef[m] * dlt;
        acc = acc + p;
      }
    } else {
      acc = hs[0][i];
      for (int m = 1; m < n_src; ++m) acc = acc + hs[m][i];
      acc = acc / (float)n_src;
    }
    bad += memcmp((const void*)&acc, &out[i], 4) != 0;
  }
  float ms = 0;
  if (iters > 0) {
    Timer t;
    for (int i = 0; i < 3; ++i) VK(vlm_merge_plan_run(plan, nullptr));
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_merge_plan_run(plan, nullptr));
    ms = t.stop() / iters;
  }
  const double gb = (double)vlm_merge_plan_bytes(plan) * 1e-9;
  printf("MERGE %-24s n=%-10zu src=%d misalign=%zu mismatches=%zu  %.3f ms  %.0f GB/s  %s\n", name, n, n_src,
         misalign, bad, ms, ms > 0 ? gb / (ms * 1e-3) : 0.0, bad == 0 ? "OK" : "FAIL");
  if (bad) ++g_fail;
  VK(vlm_merge_plan_destroy(plan));
  for (auto p : ds) CK(cudaFree(p));
  CK(cudaFree(dd));
}

// ---- regmean -------------------------------------------------------------------------------
static void regmean_case(int out_f, int in_f, double alpha) {
  // G = Y^T Y + I (SPD), W random
  const int rows = in_f + 64;
  std::vector<double> y((size_t)rows * in_f), G((size_t)in_f * in_f, 0.0);
  for (auto& v : y) v = frand();
  for (int k = 0; k < rows; ++k)
    for (int r = 0; r < in_f; ++r)
      for (int c = 0; c < in_f; ++c) G[(size_t)r * in_f + c] += y[(size_t)k * in_f + r] * y[(size_t)k * in_f + c];
  std::vector<float> W((size_t)out_f * in_f);
  for (auto& v : W) v = frand();
  std::vector<double> Gh(G);
  for (int r = 0; r < in_f; ++r)
    for (int c = 0; c < in_f; ++c)
      Gh[(size_t)r * in_f + c] =
          r == c ? alpha * G[(size_t)r * in_f + c] + (1 - alpha) * G[(size_t)r * in_f + c] : alpha * G[(size_t)r * in_f + c];
  std::vector<double> R((size_t)out_f * in_f, 0.0);
  for (int o = 0; o < out_f; ++o)
    for (int k = 0; k < in_f; ++k) {
      const double w = W[(size_t)o * in_f + k];
      for (int c = 0; c < in_f; ++c) R[(size_t)o * in_f + c] += w * Gh[(size_t)k * in_f + c];
    }
  double *dG, *dS, *dR;
  float* dW;
  CK(cudaMalloc(&dG, G.size() * 8));
  CK(cudaMalloc(&dS, G.size() * 8));
  CK(cudaMalloc(&dR, R.size() * 8));
  CK(cudaMalloc(&dW, W.size() * 4));
  CK(cudaMemcpy(dG, G.data(), G.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dW, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
  VK(vlm_gram_scale_accum(dG, VLM_F64, in_f, in_f, alpha, dS, in_f, 0, nullptr));
  VK(vlm_regmean_rhs(dW, out_f, in_f, in_f, dG, VLM_F64, in_f, alpha, dR, in_f, 0, nullptr));
  CK(cudaDeviceSynchronize());
  std::vector<double> gotR(R.size()), gotS(G.size());
  CK(cudaMemcpy(gotR.data(), dR, R.size() * 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(gotS.data(), dS, G.size() * 8, cudaMemcpyDeviceToHost));
  double num = 0, den = 0, sbad = 0;
  for (size_t i = 0; i < R.size(); ++i) {
    num += (gotR[i] - R[i]) * (gotR[i] - R[i]);
    den += R[i] * R[i];
  }
  for (size_t i = 0; i < G.size(); ++i) sbad += gotS[i] != Gh[i];
  const double rhs_err = sqrt(num / den);
  // solve: X = R * S^-1  =>  X * S == R
  VK(vlm_spd_solve_right(dS, in_f, in_f, dR, out_f, in_f, nullptr));
  std::vector<double> X(R.size());
  CK(cudaMemcpy(X.data(), dR, R.size() * 8, cudaMemcpyDeviceToHost));
  num = 0;
  for (int o = 0; o < out_f; ++o)
    for (int c = 0; c < in_f; ++c) {
      double acc = 0;
      for (int k = 0; k < in_f; ++k) acc += X[(size_t)o * in_f + k] * Gh[(size_t)k * in_f + c];
      const double e = acc - R[(size_t)o * in_f + c];
      num += e * e;
    }
  const double solve_err = sqrt(num / den);
  // difference form: (W - W2) * Ghat through vlm_regmean_rhs_diff, then + W2 through vlm_widen_add
  std::vector<float> W2(W.size());
  for (auto& v : W2) v = frand();
  float* dW2;
  CK(cudaMalloc(&dW2, W2.size() * 4));
  CK(cudaMemcpy(dW2, W2.data(), W2.size() * 4, cudaMemcpyHostToDevice));
  VK(vlm_regmean_rhs_diff(dW, dW2, out_f, in_f, in_f, dG, VLM_F64, in_f, alpha, dR, in_f, 0, nullptr));
  VK(vlm_widen_add(dW2, out_f, in_f, in_f, dR, in_f, nullptr));
  CK(cudaMemcpy(X.data(), dR, R.size() * 8, cudaMemcpyDeviceToHost));
  double dnum = 0, dden = 0;
  for (int o = 0; o < out_f; ++o)
    for (int c = 0; c < in_f; ++c) {
      double acc = W2[(size_t)o * in_f + c];
      for (int k = 0; k < in_f; ++k)
        acc += ((double)W[(size_t)o * in_f + k] - (double)W2[(size_t)o * in_f + k]) * Gh[(size_t)k * in_f + c];
      const double e = X[(size_t)o * in_f + c] - acc;
      dnum += e * e;
      dden += acc * acc;
    }
  const double diff_err = sqrt(dnum / dden);
  CK(cudaFree(dW2));
  const bool ok = rhs_err < 1e-13 && sbad == 0 && solve_err < 1e-10 && diff_err < 1e-13;
  printf("REGMEAN out=%d in=%d alpha=%.2f rhs_relF=%.2e scaleG_mismatch=%.0f solve_residual=%.2e diff_form_relF=%.2e  %s\n",
         out_f, in_f, alpha, rhs_err, sbad, solve_err, diff_err, ok ? "OK" : "FAIL");
  if (!ok) ++g_fail;
  CK(cudaFree(dG));
  CK(cudaFree(dS));
  CK(cudaFree(dR));
  CK(cudaFree(dW));
}

int main(int argc, char** argv) {
  const bool full = argc > 1 && !strcmp(argv[1], "full");
  if (argc >= 2 && !strcmp(argv[1], "overhead")) {  // host cost of one vlm_syrk_accum call (tiny problem, async)
    float *dx, *dg;
    CK(cudaMalloc(&dx, 64 * 128 * 4));
    CK(cudaMalloc(&dg, 128 * 128 * 4));
    CK(cudaMemset(dx, 0, 64 * 128 * 4));
    CK(cudaMemset(dg, 0, 128 * 128 * 4));
    for (int i = 0; i < 10; ++i) VK(vlm_syrk_accum(dx, VLM_F32, 64, 128, 128, dg, 128, nullptr));
    CK(cudaDeviceSynchronize());
    const int n = 2000;
    timespec t0, t1, t2;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int i = 0; i < n; ++i) VK(vlm_syrk_accum(dx, VLM_F32, 64, 128, 128, dg, 128, nullptr));
    clock_gettime(CLOCK_MONOTONIC, &t1);
    CK(cudaDeviceSynchronize());
    clock_gettime(CLOCK_MONOTONIC, &t2);
    auto us = [](timespec a, timespec b) { return (b.tv_sec - a.tv_sec) * 1e6 + (b.tv_nsec - a.tv_nsec) * 1e-3; };
    printf("OVERHEAD vlm_syrk_accum: %.2f us/call to enqueue (host), %.2f us/call until drained (GPU-bound)\n",
           us(t0, t1) / n, us(t0, t2) / n);
    return 0;
  }
  if (argc >= 2 && !strcmp(argv[1], "merge")) {  // only the VLMo-base sized merges (for ncu captures)
    merge_case("wsum2 85M (base ufo)", VLM_MERGE_WSUM, 2, 85045248, 0, 5);
    merge_case("seqlerp3 85M", VLM_MERGE_SEQ_LERP, 3, 85045248, 0, 5);
    return g_fail;
  }
  if (argc >= 5 && !strcmp(argv[1], "rhs")) {  // selftest rhs <out_f> <in_f> <iters>: kernel (c) timing, fp32 Gram in
    const int out_f = atoi(argv[2]), in_f = atoi(argv[3]), iters = atoi(argv[4]);
    std::vector<float> W((size_t)out_f * in_f), Gm((size_t)in_f * in_f);
    for (auto& v : W) v = frand();
    for (auto& v : Gm) v = frand();
    float *dW, *dG;
    double* dR;
    CK(cudaMalloc(&dW, W.size() * 4));
    CK(cudaMalloc(&dG, Gm.size() * 4));
    CK(cudaMalloc(&dR, W.size() * 8));
    CK(cudaMemcpy(dW, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dG, Gm.data(), Gm.size() * 4, cudaMemcpyHostToDevice));
    for (int i = 0; i < 2; ++i) VK(vlm_regmean_rhs(dW, out_f, in_f, in_f, dG, VLM_F32, in_f, 0.9, dR, in_f, 0, nullptr));
    Timer t;
    t.start();
    for (int i = 0; i < iters; ++i) VK(vlm_regmean_rhs(dW, out_f, in_f, in_f, dG, VLM_F32, in_f, 0.9, dR, in_f, i > 0, nullptr));
    const float ms = t.stop() / iters;
    // spot check one row against the host
    std::vector<double> got(in_f);
    VK(vlm_regmean_rhs(dW, out_f, in_f, in_f, dG, VLM_F32, in_f, 0.9, dR, in_f, 0, nullptr));
    CK(cudaMemcpy(got.data(), dR + (size_t)(out_f - 1) * in_f, in_f * 8, cudaMemcpyDeviceToHost));
    double num = 0, den = 0;
    for (int c = 0; c < in_f; ++c) {
      double acc = 0;
      for (int k = 0; k < in_f; ++k) {
        const double g = Gm[(size_t)k * in_f + c];
        acc += (double)W[(size_t)(out_f - 1) * in_f + k] * (k == c ? 0.9 * g + (1 - 0.9) * g : 0.9 * g);
      }
      num += (acc - got[c]) * (acc - got[c]);
      den += acc * acc;
    }
    printf("RHS out=%d in=%d  %.3f ms  %.2f TFLOP/s fp64  row_relerr=%.2e\n", out_f, in_f, ms,
           2.0 * out_f * in_f * (double)in_f / ms * 1e-9, sqrt(num / den));
    return 0;
  }
  if (argc >= 6 && !strcmp(argv[1], "case")) {  // selftest case <f32|bf16|f16> <rows> <d> <iters> [positive]
    const int64_t rows = atoll(argv[3]);
    const int d = atoi(argv[4]), iters = atoi(argv[5]), mode = argc > 6 ? atoi(argv[6]) : 0;
    if (!strcmp(argv[2], "f32")) syrk_case<float>("case f32", VLM_F32, rows, d, mode, false, iters, 2e-3);
    else if (!strcmp(argv[2], "bf16")) syrk_case<__nv_bfloat16>("case bf16", VLM_BF16, rows, d, mode, false, iters, 1e-4);
    else syrk_case<__half>("case f16", VLM_F16, rows, d, mode, false, iters, 1e-4);
    return g_fail;
  }
  if (argc >= 6 && !strcmp(argv[1], "simtopk")) {  // selftest simtopk <m> <n> <d> <iters>
    simtopk_case(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]));
    return g_fail;
  }
  if (argc >= 9 && !strcmp(argv[1], "batch")) {  // selftest batch <n1> <rows1> <d1> <n2> <rows2> <d2> <iters>
    syrk_batch_case(atoi(argv[2]), atoll(argv[3]), atoi(argv[4]), atoi(argv[5]), atoll(argv[6]), atoi(argv[7]), atoi(argv[8]));
    return g_fail;
  }
  if (argc >= 5 && !strcmp(argv[1], "i8x4")) {  // selftest i8x4 <rows> <d> <iters> [positive] [f32|f16|bf16]
    const int rows = atoi(argv[2]), d = atoi(argv[3]), iters = atoi(argv[4]), mode = argc > 5 ? atoi(argv[5]) : 0;
    const char* dt = argc > 6 ? argv[6] : "f32";
    if (!strcmp(dt, "f16")) syrk_i8_case<__half>("case f16", VLM_F16, 1, rows, 0, rows, d, mode, false, iters, 1e-7);
    else if (!strcmp(dt, "bf16")) syrk_i8_case<__nv_bfloat16>("case bf16", VLM_BF16, 1, rows, 0, rows, d, mode, false, iters, 1e-7);
    else syrk_i8_case<float>("case f32", VLM_F32, 1, rows, 0, rows, d, mode, false, iters, 1e-7);
    return g_fail;
  }
  if (argc >= 6 && !strcmp(argv[1], "f64")) {  // selftest f64 <f32|bf16> <rows> <d> <iters> [positive]
    const int rows = atoi(argv[3]), d = atoi(argv[4]), iters = atoi(argv[5]), mode = argc > 6 ? atoi(argv[6]) : 0;
    if (!strcmp(argv[2], "f32")) syrk_f64_case<float>("case f32", VLM_F32, 1, rows, 0, rows, d, mode, false, iters, 1e-13);
    else syrk_f64_case<__nv_bfloat16>("case bf16", VLM_BF16, 1, rows, 0, rows, d, mode, false, iters, 1e-13);
    return g_fail;
  }
  if (argc >= 5 && !strcmp(argv[1], "split")) {  // selftest split <rows> <d> <iters> [positive]
    syrk_split_case("case tf32x3", 1, atoi(argv[2]), 0, atoi(argv[2]), atoi(argv[3]), argc > 5 ? atoi(argv[5]) : 0, false,
                    atoi(argv[4]), 5e-5);
    return g_fail;
  }
  if (argc >= 2 && !strcmp(argv[1], "pack")) {  // pack / unpack / mirror kernels only (for compute-sanitizer)
    for (int d : {1, 31, 33, 192, 768, 1000}) {
      pack_case<float>(d, d % 2 ? 3 : 0);
      pack_case<double>(d, d % 2 ? 3 : 0);
    }
    return g_fail;
  }
  if (argc >= 9 && !strcmp(argv[1], "strided")) {  // selftest strided <f32|bf16> <nseg> <n_tok> <off> <seg_rows> <d> <iters>
    const int nseg = atoi(argv[3]), n_tok = atoi(argv[4]), off = atoi(argv[5]), seg_rows = atoi(argv[6]);
    const int d = atoi(argv[7]), iters = atoi(argv[8]);
    if (!strcmp(argv[2], "f32"))
      syrk_strided_case<float>("strided f32", VLM_F32, nseg, n_tok, off, seg_rows, d, false, iters, 2e-4);
    else
      syrk_strided_case<__nv_bfloat16>("strided bf16", VLM_BF16, nseg, n_tok, off, seg_rows, d, false, iters, 2e-4);
    return g_fail;
  }
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("device: %s, %d SMs, cc %d.%d, vlm abi %d\n", prop.name, prop.multiProcessorCount, prop.major, prop.minor,
         vlm_version());

  // merge first: simplest kernel
  merge_case("wsum2", VLM_MERGE_WSUM, 2, 1 << 20, 0, 0);
  merge_case("wsum3", VLM_MERGE_WSUM, 3, (1 << 20) + 3, 0, 0);
  merge_case("seqlerp3", VLM_MERGE_SEQ_LERP, 3, (1 << 18) + 1, 0, 0);
  merge_case("seqlerp4", VLM_MERGE_SEQ_LERP, 4, (1 << 18), 0, 0);
  merge_case("mean2", VLM_MERGE_MEAN, 2, 4099, 0, 0);
  merge_case("mean3-misaligned", VLM_MERGE_MEAN, 3, 70001, 1, 0);
  merge_case("wsum2-misaligned", VLM_MERGE_WSUM, 2, 70001, 3, 0);

  for (int d : {1, 33, 768}) {
    pack_case<float>(d, d % 2 ? 3 : 0);
    pack_case<double>(d, d % 2 ? 3 : 0);
  }

  regmean_case(96, 128, 1.0);
  regmean_case(200, 192, 0.9);
  regmean_case(70, 100, 0.9);     // the 64 x 64 kernel (in_f not a multiple of 32)

  // SYRK: small shapes against a host fp64 Gram
  syrk_case<float>("f32 1 tile", VLM_F32, 64, 128, 0, true, 0, 2e-3);
  syrk_case<float>("f32 wide tile", VLM_F32, 200, 256, 0, true, 0, 2e-3);
  syrk_case<float>("f32 d=768 ragged rows", VLM_F32, 1000, 768, 0, true, 0, 2e-3);
  syrk_case<float>("f32 d=200 CUDA-core route", VLM_F32, 333, 200, 1, true, 0, 2e-3);
  syrk_case<float>("f32 d=900 CUDA-core route", VLM_F32, 130, 900, 0, true, 0, 2e-3);
  syrk_case<__nv_bfloat16>("bf16 d=768", VLM_BF16, 1000, 768, 0, true, 0, 1e-5);
  syrk_case<__half>("f16 d=768 positive", VLM_F16, 1000, 768, 1, true, 0, 1e-5);
  syrk_case<__nv_bfloat16>("bf16 d=200 CUDA-core route", VLM_BF16, 77, 200, 1, true, 0, 1e-5);
  syrk_case<float>("f32 d=768 positive", VLM_F32, 2560, 768, 1, true, 0, 2e-3);

  // reference precision (fp64 DMMA)
  syrk_f64_case<float>("f32 1 tile", VLM_F32, 1, 64, 0, 64, 128, 0, true, 0, 1e-13);
  syrk_f64_case<float>("f32 d=768 ragged rows", VLM_F32, 1, 1000, 0, 1000, 768, 0, true, 0, 1e-13);
  syrk_f64_case<float>("f32 d=203 odd (scalar path)", VLM_F32, 1, 333, 0, 333, 203, 1, true, 0, 1e-13);
  syrk_f64_case<__nv_bfloat16>("bf16 d=200 ragged", VLM_BF16, 1, 77, 0, 77, 200, 1, true, 0, 1e-13);
  syrk_f64_case<__half>("f16 d=768", VLM_F16, 1, 1000, 0, 1000, 768, 0, true, 0, 1e-13);
  syrk_f64_case<float>("f32 image slice", VLM_F32, 4, 617, 40, 577, 768, 0, true, 0, 1e-13);
  syrk_f64_case<float>("f32 text d=768", VLM_F32, 1, 2560, 0, 2560, 768, 0, false, 20, 1e-13);
  syrk_f64_case<float>("f32 image d=768", VLM_F32, 1, 36928, 0, 36928, 768, 0, false, 10, 1e-13);
  syrk_f64_case<float>("f32 image d=3072", VLM_F32, 1, 36928, 0, 36928, 3072, 1, false, 3, 1e-13);

  // exact Gram on the integer tensor cores
  syrk_i8_case<float>("i8x4 1 tile", VLM_F32, 1, 64, 0, 64, 128, 0, true, 0, 1e-7);
  syrk_i8_case<float>("i8x4 d=768 ragged rows", VLM_F32, 1, 1000, 0, 1000, 768, 0, true, 0, 1e-7);
  syrk_i8_case<float>("i8x4 d=384 positive", VLM_F32, 1, 333, 0, 333, 384, 1, true, 0, 1e-7);
  syrk_i8_case<float>("i8x4 image slice", VLM_F32, 4, 617, 40, 577, 768, 0, true, 0, 1e-7);
  syrk_i8_case<__half>("i8x4 f16 d=768", VLM_F16, 1, 1000, 0, 1000, 768, 0, true, 0, 1e-7);
  syrk_i8_case<__nv_bfloat16>("i8x4 bf16 slice d=256", VLM_BF16, 3, 100, 20, 64, 256, 1, true, 0, 1e-7);
  syrk_i8_case<float>("i8x4 text d=3072", VLM_F32, 1, 2560, 0, 2560, 3072, 1, false, 10, 1e-7);
  syrk_i8_case<float>("i8x4 image d=768", VLM_F32, 1, 36928, 0, 36928, 768, 0, false, 10, 1e-7);
  syrk_i8_case<float>("i8x4 image d=3072", VLM_F32, 1, 36928, 0, 36928, 3072, 1, false, 5, 1e-7);

  // split precision (3xTF32)
  syrk_split_case("tf32x3 1 tile", 1, 64, 0, 64, 128, 0, true, 0, 2e-6);
  syrk_split_case("tf32x3 d=768 ragged rows", 1, 1000, 0, 1000, 768, 0, true, 0, 2e-6);
  syrk_split_case("tf32x3 d=800 positive", 1, 333, 0, 333, 800, 1, true, 0, 2e-6);
  syrk_split_case("tf32x3 image slice", 4, 617, 40, 577, 768, 0, true, 0, 2e-6);
  syrk_split_case("tf32x3 text d=3072", 1, 2560, 0, 2560, 3072, 1, false, 20, 5e-5);
  syrk_split_case("tf32x3 image d=768", 1, 36928, 0, 36928, 768, 0, false, 20, 5e-5);
  syrk_split_case("tf32x3 image d=3072", 1, 36928, 0, 36928, 3072, 1, false, 10, 5e-5);

  // row-sliced activations of the fused vision-language route: text rows [0, 40), image rows [40, 617)
  syrk_strided_case<float>("f32 text slice", VLM_F32, 8, 617, 0, 40, 768, true, 0, 2e-3);
  syrk_strided_case<float>("f32 image slice", VLM_F32, 4, 617, 40, 577, 768, true, 0, 2e-3);
  syrk_strided_case<__nv_bfloat16>("bf16 image slice", VLM_BF16, 4, 617, 40, 577, 768, true, 0, 1e-5);
  syrk_strided_case<float>("f32 d=200 CUDA-core route", VLM_F32, 3, 50, 7, 33, 200, true, 0, 2e-3);
  syrk_strided_case<float>("f32 image slice x64", VLM_F32, 64, 617, 40, 577, 768, false, 20, 2e-4);
  syrk_strided_case<float>("f32 text slice x64", VLM_F32, 64, 617, 0, 40, 768, false, 20, 2e-4);

  // retrieval step: fused similarity + top-10
  simtopk_case(130, 300, 192, 0);
  simtopk_case(5000, 25000, 768, 5);

  // grouped launches: a small mixed group for correctness
  syrk_batch_case(3, 1000, 768, 2, 333, 256, 0);

  // hot shapes: SIMT kernel as the reference, timed
  syrk_case<float>("f32 text d=768", VLM_F32, 2560, 768, 0, false, 20, 2e-3);
  syrk_case<float>("f32 text d=3072", VLM_F32, 2560, 3072, 1, false, 20, 2e-3);
  syrk_case<float>("f32 image d=768", VLM_F32, 36928, 768, 0, false, 20, 2e-3);
  syrk_case<float>("f32 image d=3072", VLM_F32, 36928, 3072, 1, false, 10, 2e-3);
  syrk_case<__nv_bfloat16>("bf16 image d=768", VLM_BF16, 36928, 768, 0, false, 20, 1e-4);
  syrk_case<__nv_bfloat16>("bf16 image d=3072", VLM_BF16, 36928, 3072, 1, false, 10, 1e-4);
  if (full) {
    syrk_case<float>("f32 image d=1024", VLM_F32, 36928, 1024, 0, false, 20, 2e-3);
    syrk_case<float>("f32 image d=4096", VLM_F32, 36928, 4096, 1, false, 10, 2e-3);
    syrk_case<__half>("f16 image d=4096", VLM_F16, 36928, 4096, 1, false, 10, 1e-4);
  }

  // merge bandwidth at the VLMo-base size: 2 sources x 85 M elements -> 1.02 GB moved
  merge_case("wsum2 85M (base ufo)", VLM_MERGE_WSUM, 2, 85045248, 0, 20);
  merge_case("seqlerp3 85M", VLM_MERGE_SEQ_LERP, 3, 85045248, 0, 20);

  printf("launches=%llu failed=%d\n", (unsigned long long)vlm_launch_count(), g_fail);
  return g_fail;
}
