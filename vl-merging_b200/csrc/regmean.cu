// regmean.cu — kernel (c): the RegMean right-hand side  acc (+)= W * Ghat  and the summed, scaled
// Gram, both fp64 like the reference (src/vilt/modules/vilt_module.py:388-392 scale_G, :423-424 and
// :474-475 `summed_gram += G; later_weight += W.double() @ G`), plus the SPD solve that replaces
// `matmul(later_weight, torch.inverse(summed_gram))` (:432-434, :483-484) through cuSOLVER.
//
// The GEMM runs on the fp64 tensor-core path (mma.sync m8n8k4 DMMA): RegMean multiplies by the
// inverse of an ill-conditioned Gram sum afterwards, so the right-hand side keeps the reference's
// precision instead of a split-TF32 approximation.  scale_G is fused into the operand load:
// Ghat[k][n] = alpha*G[k][n] off the diagonal and alpha*g + (1-alpha)*g on it (the reference's own
// rounding), so the scaled Gram is never materialised.
#include <dlfcn.h>

#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

namespace vlm {
namespace {

__device__ __forceinline__ double scaled_g(double g, bool on_diag, double alpha, double one_minus_alpha) {
  const double a = __dmul_rn(alpha, g);
  return on_diag ? __dadd_rn(a, __dmul_rn(one_minus_alpha, g)) : a;
}

template <typename GT>
__global__ void __launch_bounds__(256)
gram_scale_accum_kernel(const GT* __restrict__ g, int d, int64_t ldg, double alpha, double oma,
                        double* __restrict__ out, int64_t ldo, int accumulate) {
  const int64_t n = (int64_t)d * d;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / d), c = (int)(e % d);
    const double v = scaled_g((double)g[(int64_t)r * ldg + c], r == c, alpha, oma);
    double* o = out + (int64_t)r * ldo + c;
    *o = accumulate ? __dadd_rn(*o, v) : v;
  }
}

// acc[M x N] (+)= W[M x K] * Ghat[K x N], K == N == in_f.  Block tile 64x64, K step 16, 4 warps
// (2x2), each warp 32x32 = 4x4 m8n8k4 tiles.
constexpr int BM = 64, BN = 64, BKK = 16;

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

template <typename GT>
__global__ void __launch_bounds__(128)
regmean_rhs_kernel(const float* __restrict__ w, const float* __restrict__ w_sub, int M, int K, int64_t ldw,
                   const GT* __restrict__ g, int64_t ldg, double alpha, double oma, double* __restrict__ acc,
                   int64_t ldacc, int accumulate) {
  __shared__ double sa[2][BM][BKK + 1];  // W tile, widened
  __shared__ double sb[2][BKK][BN + 1];  // Ghat tile
  // blockIdx.x walks the rows of W (fast), blockIdx.y the columns of G: blocks that run together share one
  // 16 x 64 column strip of G per K step, so G (up to 67 MB fp32 for in_f = 4096) streams from HBM once
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int N = K;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
  double c[4][4][2] = {};

  auto load_tiles = [&](int buf, int k0) {
    for (int e = threadIdx.x; e < BM * BKK; e += 128) {
      const int r = e / BKK, kk = e % BKK;
      const int gm = m0 + r, gk = k0 + kk;
      double v = 0.0;
      if (gm < M && gk < K) {
        v = (double)w[(int64_t)gm * ldw + gk];
        if (w_sub) v -= (double)w_sub[(int64_t)gm * ldw + gk];    // exact: both widen exactly, the difference rounds once
      }
      sa[buf][r][kk] = v;
    }
    for (int e = threadIdx.x; e < BKK * BN; e += 128) {
      const int kk = e / BN, cc = e % BN;
      const int gk = k0 + kk, gn = n0 + cc;
      sb[buf][kk][cc] =
          (gk < K && gn < N) ? scaled_g((double)g[(int64_t)gk * ldg + gn], gk == gn, alpha, oma) : 0.0;
    }
  };

  const int nk = (K + BKK - 1) / BKK;
  load_tiles(0, 0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < nk) load_tiles(buf ^ 1, (kt + 1) * BKK);
#pragma unroll
    for (int ks = 0; ks < BKK; ks += 4) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sa[buf][wm + i * 8 + (lane >> 2)][ks + (lane & 3)];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = sb[buf][ks + (lane & 3)][wn + j * 8 + (lane >> 2)];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma(c[i][j][0], c[i][j][1], a[i], b[j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = m0 + wm + i * 8 + (lane >> 2);
      const int cc = n0 + wn + j * 8 + (lane & 3) * 2;
#pragma unroll
      for (int u = 0; u < 2; ++u)
        if (r < M && cc + u < N) {
          double* o = acc + (int64_t)r * ldacc + cc + u;
          *o = accumulate ? __dadd_rn(*o, c[i][j][u]) : c[i][j][u];
        }
    }
}

// Pipelined variant for the real layer shapes (K a multiple of 32, 16-byte aligned rows): 128x128 block tile,
// 16 warps of 32x32, raw fp32 / fp64 tiles brought in by a 3-stage cp.async pipeline; widening to fp64 and
// scale_G happen when a fragment is read from shared memory, so no converted copy is ever stored.
constexpr int TM = 128, TN = 128, TK = 32, TSTAGES = 3;
constexpr int W_PITCH = TK + 4;  // floats: fragment reads hit 32 distinct banks

template <typename GT, bool SUB>
struct RhsSmem {
  static constexpr int G_PITCH = TN + (sizeof(GT) == 4 ? 8 : 4);  // conflict-free k-major fragment reads
  float w[TSTAGES][TM][W_PITCH];
  GT g[TSTAGES][TK][G_PITCH];
  float w_sub[SUB ? TSTAGES : 1][SUB ? TM : 1][SUB ? W_PITCH : 4];   // SUB: the tile of the subtracted weight
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
  const uint32_t d = smem_u32(smem_dst);
  const int n = valid ? 16 : 0;  // src-size 0: zero-fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gmem_src), "r"(n) : "memory");
}

// SUB: the left operand is W - W_sub (same pitch), formed in fp64 when a fragment is read.
template <typename GT, bool SUB>
__global__ void __launch_bounds__(512, 1)
regmean_rhs_pipelined_kernel(const float* __restrict__ w, const float* __restrict__ w_sub, int M, int K, int64_t ldw,
                             const GT* __restrict__ g, int64_t ldg, double alpha, double oma, double* __restrict__ acc,
                             int64_t ldacc, int accumulate) {
  extern __shared__ __align__(16) uint8_t rhs_smem_raw[];
  RhsSmem<GT, SUB>& sm = *reinterpret_cast<RhsSmem<GT, SUB>*>(rhs_smem_raw);
  constexpr int GV = 16 / sizeof(GT);  // G elements per 16-byte chunk
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;  // x walks W rows: co-running blocks share G strips
  const int N = K;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = (warp >> 2) * 32, wn = (warp & 3) * 32;
  double c[4][4][2] = {};

  auto load_stage = [&](int slot, int kt) {
    const int k0 = kt * TK;
    for (int e = tid; e < TM * (TK / 4); e += 512) {  // W tile: 128 rows x 32 floats = 1024 16-byte chunks
      const int r = e / (TK / 4), ch = e % (TK / 4);
      const bool ok = (m0 + r) < M && k0 < K;
      cp_async16(&sm.w[slot][r][ch * 4], w + (int64_t)(ok ? m0 + r : 0) * ldw + (ok ? k0 : 0) + ch * 4, ok);
      if constexpr (SUB)
        cp_async16(&sm.w_sub[slot][r][ch * 4], w_sub + (int64_t)(ok ? m0 + r : 0) * ldw + (ok ? k0 : 0) + ch * 4, ok);
    }
    constexpr int chunks_per_row = TN / GV;
    for (int e = tid; e < TK * chunks_per_row; e += 512) {  // G tile: 32 rows x 128 columns
      const int kk = e / chunks_per_row, ch = e % chunks_per_row;
      const bool ok = k0 < K && (n0 + ch * GV) < N;
      cp_async16(&sm.g[slot][kk][ch * GV], g + (int64_t)(ok ? k0 + kk : 0) * ldg + (ok ? n0 + ch * GV : 0), ok);
    }
  };

  const int nk = K / TK;
  for (int s = 0; s < TSTAGES - 1; ++s) {
    if (s < nk) load_stage(s, s);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int kt = 0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(TSTAGES - 2) : "memory");
    __syncthreads();
    if (kt + TSTAGES - 1 < nk) load_stage((kt + TSTAGES - 1) % TSTAGES, kt + TSTAGES - 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int slot = kt % TSTAGES;
#pragma unroll
    for (int ks = 0; ks < TK; ks += 4) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a[i] = (double)sm.w[slot][wm + i * 8 + (lane >> 2)][ks + (lane & 3)];
        if constexpr (SUB) a[i] -= (double)sm.w_sub[slot][wm + i * 8 + (lane >> 2)][ks + (lane & 3)];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int kk = ks + (lane & 3), nn = wn + j * 8 + (lane >> 2);
        b[j] = scaled_g((double)sm.g[slot][kk][nn], kt * TK + kk == n0 + nn, alpha, oma);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma(c[i][j][0], c[i][j][1], a[i], b[j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = m0 + wm + i * 8 + (lane >> 2);
      const int cc = n0 + wn + j * 8 + (lane & 3) * 2;
      if (r < M && cc < N) {  // N is even here, so the pair is either fully inside or fully outside
        double2* o = reinterpret_cast<double2*>(acc + (int64_t)r * ldacc + cc);
        double2 v = make_double2(c[i][j][0], c[i][j][1]);
        if (accumulate) {
          const double2 old = *o;
          v.x = __dadd_rn(old.x, v.x);
          v.y = __dadd_rn(old.y, v.y);
        }
        *o = v;
      }
    }
}

// ---- cuSOLVER through dlopen (off the hot path; keeps libvlmerge loadable without it) ----------
typedef void* cusolverDnHandle_t;
typedef int cusolverStatus_t;
struct Cusolver {
  void* lib = nullptr;
  cusolverStatus_t (*create)(cusolverDnHandle_t*) = nullptr;
  cusolverStatus_t (*set_stream)(cusolverDnHandle_t, cudaStream_t) = nullptr;
  cusolverStatus_t (*potrf_bufsize)(cusolverDnHandle_t, int, int, double*, int, int*) = nullptr;
  cusolverStatus_t (*potrf)(cusolverDnHandle_t, int, int, double*, int, double*, int, int*) = nullptr;
  cusolverStatus_t (*potrs)(cusolverDnHandle_t, int, int, int, const double*, int, double*, int, int*) = nullptr;
  cusolverStatus_t (*getrf_bufsize)(cusolverDnHandle_t, int, int, double*, int, int*) = nullptr;
  cusolverStatus_t (*getrf)(cusolverDnHandle_t, int, int, double*, int, double*, int*, int*) = nullptr;
  cusolverStatus_t (*getrs)(cusolverDnHandle_t, int, int, int, const double*, int, const int*, double*, int, int*) = nullptr;
};
Cusolver g_cs;
std::mutex g_cs_mu;

int load_cusolver() {
  if (g_cs.lib) return 0;
  const char* names[] = {"libcusolver.so.11", "libcusolver.so", "/usr/local/cuda/lib64/libcusolver.so.11",
                         "libcusolver.so.12"};
  for (const char* n : names) {
    g_cs.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_cs.lib) break;
  }
  VLM_REQUIRE(g_cs.lib != nullptr, VLM_ERR_DRIVER, "cannot dlopen libcusolver: %s", dlerror());
#define VLM_SYM(field, name)                                              \
  g_cs.field = reinterpret_cast<decltype(g_cs.field)>(dlsym(g_cs.lib, name)); \
  VLM_REQUIRE(g_cs.field != nullptr, VLM_ERR_DRIVER, "libcusolver lacks %s", name)
  VLM_SYM(create, "cusolverDnCreate");
  VLM_SYM(set_stream, "cusolverDnSetStream");
  VLM_SYM(potrf_bufsize, "cusolverDnDpotrf_bufferSize");
  VLM_SYM(potrf, "cusolverDnDpotrf");
  VLM_SYM(potrs, "cusolverDnDpotrs");
  VLM_SYM(getrf_bufsize, "cusolverDnDgetrf_bufferSize");
  VLM_SYM(getrf, "cusolverDnDgetrf");
  VLM_SYM(getrs, "cusolverDnDgetrs");
#undef VLM_SYM
  return 0;
}

}  // namespace
}  // namespace vlm

using namespace vlm;

extern "C" int vlm_gram_scale_accum(const void* g, int g_dtype, int d, int64_t ldg, double alpha, double* out,
                                    int64_t ldo, int accumulate, void* stream) {
  VLM_REQUIRE(g && out && d > 0 && ldg >= d && ldo >= d, VLM_ERR_INVALID_ARG, "vlm_gram_scale_accum: bad arguments");
  VLM_REQUIRE(g_dtype == VLM_F64 || g_dtype == VLM_F32, VLM_ERR_INVALID_ARG,
              "vlm_gram_scale_accum: g_dtype must be VLM_F64 or VLM_F32");
  const int64_t n = (int64_t)d * d;
  int nsm = 0;
  if (int rc = device_sm_count(&nsm)) return rc;
  const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)nsm * 8);
  auto s = static_cast<cudaStream_t>(stream);
  if (g_dtype == VLM_F64)
    gram_scale_accum_kernel<double>
        <<<grid, 256, 0, s>>>(static_cast<const double*>(g), d, ldg, alpha, 1.0 - alpha, out, ldo, accumulate);
  else
    gram_scale_accum_kernel<float>
        <<<grid, 256, 0, s>>>(static_cast<const float*>(g), d, ldg, alpha, 1.0 - alpha, out, ldo, accumulate);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

namespace vlm {
namespace {
template <typename GT, bool SUB>
int launch_rhs_pipelined(const float* w, const float* w_sub, int out_f, int in_f, int64_t ldw, const void* g, int64_t ldg,
                         double alpha, double* acc, int64_t ldacc, int accumulate, cudaStream_t s) {
  dim3 grid((out_f + TM - 1) / TM, (in_f + TN - 1) / TN);
  auto kernel = regmean_rhs_pipelined_kernel<GT, SUB>;
  VLM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RhsSmem<GT, SUB>)));
  kernel<<<grid, 512, sizeof(RhsSmem<GT, SUB>), s>>>(w, w_sub, out_f, in_f, ldw, static_cast<const GT*>(g), ldg, alpha,
                                                     1.0 - alpha, acc, ldacc, accumulate);
  return 0;
}

int regmean_rhs_impl(const char* who, const float* w, const float* w_sub, int out_f, int in_f, int64_t ldw, const void* g,
                     int g_dtype, int64_t ldg, double alpha, double* acc, int64_t ldacc, int accumulate, void* stream) {
  VLM_REQUIRE(w && g && acc && out_f > 0 && in_f > 0 && ldw >= in_f && ldg >= in_f && ldacc >= in_f,
              VLM_ERR_INVALID_ARG, "%s: bad arguments", who);
  VLM_REQUIRE(g_dtype == VLM_F64 || g_dtype == VLM_F32, VLM_ERR_INVALID_ARG, "%s: g_dtype must be VLM_F64 or VLM_F32", who);
  auto s = static_cast<cudaStream_t>(stream);
  const int gelem = g_dtype == VLM_F64 ? 8 : 4;
  const bool pipelined = in_f % TK == 0 && (ldw % 4) == 0 && ((ldg * gelem) % 16) == 0 && (ldacc % 2) == 0 &&
                         (reinterpret_cast<uintptr_t>(w) % 16) == 0 && (reinterpret_cast<uintptr_t>(w_sub) % 16) == 0 &&
                         (reinterpret_cast<uintptr_t>(g) % 16) == 0 && (reinterpret_cast<uintptr_t>(acc) % 16) == 0;
  if (pipelined) {
    int rc;
    if (g_dtype == VLM_F64)
      rc = w_sub ? launch_rhs_pipelined<double, true>(w, w_sub, out_f, in_f, ldw, g, ldg, alpha, acc, ldacc, accumulate, s)
                 : launch_rhs_pipelined<double, false>(w, w_sub, out_f, in_f, ldw, g, ldg, alpha, acc, ldacc, accumulate, s);
    else
      rc = w_sub ? launch_rhs_pipelined<float, true>(w, w_sub, out_f, in_f, ldw, g, ldg, alpha, acc, ldacc, accumulate, s)
                 : launch_rhs_pipelined<float, false>(w, w_sub, out_f, in_f, ldw, g, ldg, alpha, acc, ldacc, accumulate, s);
    if (rc) return rc;
    VLM_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  dim3 grid((out_f + BM - 1) / BM, (in_f + BN - 1) / BN);
  if (g_dtype == VLM_F64)
    regmean_rhs_kernel<double><<<grid, 128, 0, s>>>(w, w_sub, out_f, in_f, ldw, static_cast<const double*>(g), ldg, alpha,
                                                    1.0 - alpha, acc, ldacc, accumulate);
  else
    regmean_rhs_kernel<float><<<grid, 128, 0, s>>>(w, w_sub, out_f, in_f, ldw, static_cast<const float*>(g), ldg, alpha,
                                                   1.0 - alpha, acc, ldacc, accumulate);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

__global__ void __launch_bounds__(256) widen_add_kernel(const float* __restrict__ src, int rows, int cols, int64_t lds,
                                                        double* __restrict__ dst, int64_t ldd) {
  const int64_t n = (int64_t)rows * cols;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / cols, c = e - r * cols;
    dst[r * ldd + c] = __dadd_rn(dst[r * ldd + c], (double)src[r * lds + c]);
  }
}

// potrf's status word can miss a pivot that is not positive: a 768 x 768 diagonal matrix whose last entry is -1
// factors with status 0 and a NaN at the end of the diagonal (B200, cuSOLVER of CUDA 12.8).  Every diagonal entry of
// a Cholesky factor is finite and positive, so the factor itself says whether potrf succeeded: if the status is 0
// and an entry is not, report the first such pivot (1-based, as potrf does).  One block, stream-ordered.
__global__ void __launch_bounds__(256) potrf_status_kernel(const double* __restrict__ l, int n, int64_t ld,
                                                           int* __restrict__ info) {
  __shared__ int first;
  if (threadIdx.x == 0) first = n;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = l[(int64_t)i * ld + i];
    if (!(v > 0.0 && isfinite(v))) atomicMin(&first, i);
  }
  __syncthreads();
  if (threadIdx.x == 0 && *info == 0 && first < n) *info = first + 1;
}
}  // namespace
}  // namespace vlm

extern "C" int vlm_regmean_rhs(const float* w, int out_f, int in_f, int64_t ldw, const void* g, int g_dtype,
                               int64_t ldg, double alpha, double* acc, int64_t ldacc, int accumulate, void* stream) {
  return regmean_rhs_impl("vlm_regmean_rhs", w, nullptr, out_f, in_f, ldw, g, g_dtype, ldg, alpha, acc, ldacc, accumulate,
                          stream);
}

extern "C" int vlm_regmean_rhs_diff(const float* w, const float* w_base, int out_f, int in_f, int64_t ldw, const void* g,
                                    int g_dtype, int64_t ldg, double alpha, double* acc, int64_t ldacc, int accumulate,
                                    void* stream) {
  VLM_REQUIRE(w_base != nullptr, VLM_ERR_INVALID_ARG, "vlm_regmean_rhs_diff: w_base is NULL");
  return regmean_rhs_impl("vlm_regmean_rhs_diff", w, w_base, out_f, in_f, ldw, g, g_dtype, ldg, alpha, acc, ldacc,
                          accumulate, stream);
}

extern "C" int vlm_widen_add(const float* src, int rows, int cols, int64_t lds, double* dst, int64_t ldd, void* stream) {
  VLM_REQUIRE(src && dst && rows > 0 && cols > 0 && lds >= cols && ldd >= cols, VLM_ERR_INVALID_ARG,
              "vlm_widen_add: bad arguments");
  int nsm = 0;
  if (int rc = device_sm_count(&nsm)) return rc;
  const int64_t n = (int64_t)rows * cols;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)nsm * 8);
  widen_add_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(src, rows, cols, lds, dst, ldd);
  VLM_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

namespace {
// One solver context per (device, stream): a cuSOLVER handle owns a cuBLAS handle and workspace, so concurrent solves
// on different streams must not share one; the factorisation workspace is kept with it and only ever grows (a
// stream-ordered cudaMallocAsync per solve went back to the driver at every synchronisation: milliseconds of
// jitter per call, BENCH_r01 regmean.seconds_both_runs 0.066 / 0.288).  The library assumes one host thread per
// device drives these entry points at a time (the lock covers the map, not the use of a context).
struct SolveCtx {
  cusolverDnHandle_t h = nullptr;
  double* work = nullptr;
  size_t work_elems = 0;
};
std::map<std::pair<int, cudaStream_t>, SolveCtx> g_cs_ctx;

int solve_ctx(cudaStream_t st, size_t want_elems, SolveCtx* out) {
  int dev = 0;
  VLM_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_cs_mu);
  if (int rc = load_cusolver()) return rc;
  auto key = std::make_pair(dev, st);
  auto it = g_cs_ctx.find(key);
  if (it == g_cs_ctx.end()) {
    VLM_REQUIRE(g_cs_ctx.size() < 256, VLM_ERR_UNSUPPORTED, "too many distinct streams use vlm_spd_solve_right");
    SolveCtx c;
    VLM_REQUIRE(g_cs.create(&c.h) == 0, VLM_ERR_DRIVER, "cusolverDnCreate failed");
    VLM_REQUIRE(g_cs.set_stream(c.h, st) == 0, VLM_ERR_DRIVER, "cusolverDnSetStream failed");
    it = g_cs_ctx.emplace(key, c).first;
  }
  SolveCtx& c = it->second;
  // re-bind on every use: a stream that was destroyed and re-created may come back with the same handle value
  VLM_REQUIRE(g_cs.set_stream(c.h, st) == 0, VLM_ERR_DRIVER, "cusolverDnSetStream failed");
  if (c.work_elems < want_elems) {
    // the old buffer may still be in use by work queued on `st`: free it in stream order, allocate the new one now
    if (c.work) VLM_CUDA(cudaFreeAsync(c.work, st));
    c.work = nullptr;
    c.work_elems = 0;
    const size_t n = std::max<size_t>(want_elems, (size_t)1 << 16);
    VLM_CUDA(cudaMalloc(reinterpret_cast<void**>(&c.work), sizeof(double) * n));
    c.work_elems = n;
  }
  *out = c;
  return 0;
}

// potrf + potrs on `st`; info_dev[0..1] receive the two LAPACK-style status words.
int enqueue_spd_solve(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr, int* info_dev,
                      cudaStream_t st) {
  SolveCtx c;
  if (int rc = solve_ctx(st, 0, &c)) return rc;
  // Row-major symmetric S is also column-major S.  Row-major R (out_f x in_f) read column-major is
  // R^T (in_f x out_f), and S * X^T = R^T  <=>  X = R * S^{-1}: potrs leaves X row-major in r.
  const int uplo_lower = 0;  // CUBLAS_FILL_MODE_LOWER
  int lwork = 0;
  VLM_REQUIRE(g_cs.potrf_bufsize(c.h, uplo_lower, in_f, s, (int)lds, &lwork) == 0, VLM_ERR_DRIVER,
              "cusolverDnDpotrf_bufferSize failed");
  if (int rc = solve_ctx(st, (size_t)std::max(lwork, 1), &c)) return rc;
  cusolverStatus_t cs1 = g_cs.potrf(c.h, uplo_lower, in_f, s, (int)lds, c.work, lwork, info_dev);
  potrf_status_kernel<<<1, 256, 0, st>>>(s, in_f, lds, info_dev);
  VLM_CUDA(cudaGetLastError());
  cusolverStatus_t cs2 = g_cs.potrs(c.h, uplo_lower, in_f, out_f, s, (int)lds, r, (int)ldr, info_dev + 1);
  count_launch(3);
  VLM_REQUIRE(cs1 == 0 && cs2 == 0, VLM_ERR_INTERNAL, "cuSOLVER potrf/potrs status %d/%d", cs1, cs2);
  return 0;
}
}  // namespace

// General (pivoted LU) variant of vlm_spd_solve_right for a summed Gram that Cholesky rejects: the reference
// inverts with torch.inverse (LU, src/vilt/modules/vilt_module.py:432,483), which returns a result for any
// numerically non-singular matrix — e.g. a Gram sum that rounding has left slightly indefinite.  Rare path:
// allocates its pivots and synchronises `stream`.
extern "C" int vlm_lu_solve_right(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr, void* stream) {
  VLM_REQUIRE(s && r && in_f > 0 && out_f > 0 && lds >= in_f && ldr >= in_f, VLM_ERR_INVALID_ARG,
              "vlm_lu_solve_right: bad arguments");
  auto st = static_cast<cudaStream_t>(stream);
  SolveCtx c;
  if (int rc = solve_ctx(st, 0, &c)) return rc;
  int lwork = 0;
  VLM_REQUIRE(g_cs.getrf_bufsize(c.h, in_f, in_f, s, (int)lds, &lwork) == 0, VLM_ERR_DRIVER,
              "cusolverDnDgetrf_bufferSize failed");
  if (int rc = solve_ctx(st, (size_t)std::max(lwork, 1), &c)) return rc;
  int* ipiv = nullptr;
  VLM_CUDA(cudaMalloc(reinterpret_cast<void**>(&ipiv), sizeof(int) * ((size_t)in_f + 2)));
  int* info = ipiv + in_f;
  // S symmetric: its row-major storage is also its column-major storage; S * X^T = R^T as in the Cholesky path
  cusolverStatus_t cs1 = g_cs.getrf(c.h, in_f, in_f, s, (int)lds, c.work, ipiv, info);
  cusolverStatus_t cs2 = g_cs.getrs(c.h, 0 /* CUBLAS_OP_N */, in_f, out_f, s, (int)lds, ipiv, r, (int)ldr, info + 1);
  count_launch(2);
  int info_host[2] = {0, 0};
  cudaError_t e = cudaMemcpyAsync(info_host, info, sizeof(info_host), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(ipiv);
  if (e != cudaSuccess) return fail((int)e, "vlm_lu_solve_right: %s", cudaGetErrorString(e));
  VLM_REQUIRE(cs1 == 0 && cs2 == 0, VLM_ERR_INTERNAL, "cuSOLVER getrf/getrs status %d/%d", cs1, cs2);
  VLM_REQUIRE(info_host[0] == 0, VLM_ERR_NOT_SPD, "summed Gram is singular (zero pivot %d in the LU factorisation)",
              info_host[0]);
  VLM_REQUIRE(info_host[1] == 0, VLM_ERR_INTERNAL, "cusolverDnDgetrs info %d", info_host[1]);
  return 0;
}

extern "C" int vlm_spd_solve_right_async(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr,
                                         int* info_dev, void* stream) {
  VLM_REQUIRE(s && r && info_dev && in_f > 0 && out_f > 0 && lds >= in_f && ldr >= in_f, VLM_ERR_INVALID_ARG,
              "vlm_spd_solve_right_async: bad arguments");
  return enqueue_spd_solve(s, in_f, lds, r, out_f, ldr, info_dev, static_cast<cudaStream_t>(stream));
}

extern "C" int vlm_spd_solve_right(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr,
                                   void* stream) {
  VLM_REQUIRE(s && r && in_f > 0 && out_f > 0 && lds >= in_f && ldr >= in_f, VLM_ERR_INVALID_ARG,
              "vlm_spd_solve_right: bad arguments");
  auto st = static_cast<cudaStream_t>(stream);
  int* info = nullptr;
  VLM_CUDA(cudaMalloc(reinterpret_cast<void**>(&info), sizeof(int) * 2));
  const int rc = enqueue_spd_solve(s, in_f, lds, r, out_f, ldr, info, st);
  int info_host[2] = {0, 0};
  cudaError_t e = cudaSuccess;
  if (rc == 0) {
    e = cudaMemcpyAsync(info_host, info, sizeof(info_host), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  cudaFree(info);
  if (rc != 0) return rc;
  if (e != cudaSuccess) return fail((int)e, "vlm_spd_solve_right: %s", cudaGetErrorString(e));
  VLM_REQUIRE(info_host[0] == 0, VLM_ERR_NOT_SPD,
              "summed Gram is not positive definite (leading minor %d); calibrate with more rows than "
              "features or use scaling_for_non_diag < 1",
              info_host[0]);
  VLM_REQUIRE(info_host[1] == 0, VLM_ERR_INTERNAL, "cusolverDnDpotrs info %d", info_host[1]);
  return 0;
}
