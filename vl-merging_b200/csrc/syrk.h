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

// ---- deterministic mode (vlm_set_deterministic; syrk_det.cu) ---------------------------------------------------------
// The calling thread's mode, read by every Gram launch.  In it no two CTAs add into the same G element: every
// (tile, K range) partial lands in its own te x te slot of a per-call workspace (slot i at element offset i * te * te,
// row pitch te), and one reduction launch then forms G_tile += ((s0 + s1) + s2) + ... over each tile's slots.
bool deterministic_mode();
// One upper tile of one Gram: slots [slot_begin, slot_end) summed in that order into G rows row0.., columns col0..
// (entries inside d only).  mode 0: the whole tile; 1: a 256 x 256 diagonal tile of the CTA-pair kernels, whose block
// below the diagonal (local rows >= 128, columns < 128) is never formed; 2: only c >= r (the CUDA-core kernel).
struct DetItem {
  int32_t pid, d, row0, col0, mode, slot_begin, slot_end, pad;
};
struct DetGram {  // G of problem pid in a grouped launch
  void* g;
  int64_t ldg;
};
// Stream-ordered workspace: slot_bytes of slots, then (when items is not NULL) a copy of *items.  Free with cudaFreeAsync.
int det_workspace(size_t slot_bytes, const std::vector<DetItem>* items, cudaStream_t stream, void** ws, DetItem** d_items);
// The reduction launch.  f64: slots and G are fp64, else fp32.  grams NULL: every item adds into g1 / ldg1.
int det_reduce_launch(const DetItem* d_items, int nitems, int te, bool f64, const void* ws, void* g1, int64_t ldg1,
                      const DetGram* grams, cudaStream_t stream);

}  // namespace vlm
