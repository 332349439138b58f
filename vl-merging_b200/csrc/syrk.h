// syrk.h — declarations shared by the SYRK translation units.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/vlmerge.h"

namespace vlm {

// One unit of work of the tcgen05 SYRK kernel: output tile rows [col_a, col_a+128), columns
// [col_b, col_b+128*w) of G, accumulated over row chunks [k0, k1) of X (chunk = BK rows).
struct SyrkSeg {
  int32_t col_a, col_b, w, k0, k1;
};

// Rows of X are processed in panels small enough to stay in L2 while every tile re-reads them: one chunk
// (BK rows) of all d columns is always d * 128 bytes, and a panel is ~40 MB of X (VLM_SYRK_PANEL_MB), at
// least 32 chunks.  VLM_SYRK_PANEL_CHUNKS overrides the result (experiments).
inline int64_t syrk_panel_chunks(int d) {
  if (const char* e = getenv("VLM_SYRK_PANEL_CHUNKS")) return std::max(1, atoi(e));
  double mb = 40.0;
  if (const char* e = getenv("VLM_SYRK_PANEL_MB")) mb = std::max(1.0, atof(e));
  return std::max<int64_t>(32, (int64_t)(mb * 1e6 / (128.0 * d)));
}

void build_syrk_schedule(int64_t kc, int d, int nsm, std::vector<SyrkSeg>* segs, std::vector<int>* off);

int syrk_tc_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                   cudaStream_t stream);
// One unit of work of a CLUSTER (CTA-pair kernels): super-tile (sa, sb) in 256-column units, row chunks [k0, k1).
struct PairSeg {
  int32_t sa, sb, k0, k1;
};
// seg_cap: chunks per accumulation (0: the default 128, or $VLM_SYRK_SEG_CHUNKS); min_piece: shortest K piece a
// left-over tile is cut into (0: 64 chunks for long sweeps, 8 for short ones)
void build_pair_schedule(int64_t kc, int d, int nclusters_max, std::vector<PairSeg>* segs, std::vector<int>* off,
                         int64_t seg_cap = 0, int64_t min_piece = 0);
// exact Gram on the integer tensor cores (syrk_i8.cuh): fp32 activations -> four int8 digit planes -> fp64 Gram
size_t syrk_i8x4_scratch_bytes(int64_t rows, int d);
int syrk_i8x4_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, void* scratch,
                     double* g, int64_t ldg, cudaStream_t stream);

void build_syrk_i8_schedule_host(int64_t kc, int d, int nsm, std::vector<int32_t>* flat, std::vector<int>* off);

// CTA-pair kernel (syrk_pair.cu + syrk_2sm.cuh: one tcgen05.mma.cta_group::2 stream per pair); needs whole 128-byte
// column groups
bool syrk_pair_supported(int dtype, int d, int64_t ldx);
// seg_rows > 0: X is rows/seg_rows row segments of seg_rows rows, seg_stride elements apart (0: contiguous rows)
int syrk_pair_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                    float* g, int64_t ldg, cudaStream_t stream);
// fp32 -> [2][rows][d] {hi, lo} TF32 planes (the VLM_TF32X2 operand of the pair kernel, syrk_2sm.cuh)
int tf32_split_launch(const float* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, float* out,
                      cudaStream_t stream);
// several independent problems (same dtype) in one grid; every problem must satisfy syrk_pair_supported
int syrk_pair_batch_launch(const vlm_syrk_problem* probs, int n, int dtype, cudaStream_t stream);
void build_syrk_pair_schedule_host(int64_t kc, int d, int nsm, std::vector<int32_t>* flat, std::vector<int>* off);
int syrk_simt_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                     cudaStream_t stream);

}  // namespace vlm
