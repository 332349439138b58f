// syrk.h — declarations shared by the SYRK translation units.
#pragma once
#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/vlmerge.h"

namespace vlm {

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

// CTA-pair kernel (syrk_pair.cu + syrk_2sm.cuh: one tcgen05.mma.cta_group::2 stream per pair).  The one statement of
// what it takes: whole 128-byte column groups, x and g 16-byte aligned, row pitch and segment stride multiples of
// 16 bytes, ldg % 4 == 0.  Every other Gram goes to the CUDA-core kernel (syrk_simt_launch).
bool syrk_pair_supported(int dtype, const void* x, int d, int64_t ldx, int64_t seg_stride, const float* g, int64_t ldg);
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
