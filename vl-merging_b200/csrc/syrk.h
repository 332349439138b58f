// syrk.h — declarations shared by the SYRK translation units.
#pragma once
#include <cstdint>
#include <functional>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/vlmerge.h"

namespace vlm {

// exact Gram on the integer tensor cores (syrk_i8.cuh): fp32 activations -> four int8 digit planes -> fp64 Gram
size_t syrk_i8x4_scratch_bytes(int64_t rows, int d);
int syrk_i8x4_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, void* scratch,
                     double* g, int64_t ldg, cudaStream_t stream);

// CTA-pair kernel (syrk_pair.cu + syrk_2sm.cuh: one tcgen05.mma.cta_group::2 stream per pair).  The one statement of
// what it takes: whole 128-byte column groups, x and g 16-byte aligned, row pitch and segment stride multiples of
// 16 bytes, ldg % 4 == 0.  Every other Gram goes to the CUDA-core kernel (syrk_simt_launch).
bool syrk_pair_supported(int dtype, const void* x, int d, int64_t ldx, int64_t seg_stride, const float* g, int64_t ldg);
// seg_rows > 0: X is rows/seg_rows >= 2 row segments of seg_rows rows, seg_stride elements apart (0: contiguous rows;
// never for VLM_TF32X2).  The segmentation arrives normalised (api.cu), here and in syrk_pair_batch_launch.
int syrk_pair_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                    float* g, int64_t ldg, cudaStream_t stream);
// fp32 -> [2][rows][d] {hi, lo} TF32 planes (the VLM_TF32X2 operand of the pair kernel, syrk_2sm.cuh)
int tf32_split_launch(const float* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride, float* out,
                      cudaStream_t stream);
// several independent problems (same dtype) in one grid; every problem must satisfy syrk_pair_supported
int syrk_pair_batch_launch(const vlm_syrk_problem* probs, int n, int dtype, cudaStream_t stream);
// Host view of the schedule of a single (int8: int8x4) launch of kc chunks for the CPU tests: segments as
// {super_row, super_col | phase << 16, k0, k1}, cluster c's at off[c] .. off[c + 1]
void syrk_schedule_host(int64_t kc, int d, int nsm, bool int8, std::vector<int32_t>* flat, std::vector<int>* off);
int syrk_simt_launch(const void* x, int dtype, int64_t rows, int d, int64_t ldx, float* g, int64_t ldg,
                     cudaStream_t stream);
// A row-major fp32 (f64: fp64) matrix of rows x cols, row pitch `pitch` elements, as a 2-D TMA tensor in the box and
// swizzle of the CTA-pair kernels' epilogue slabs (128 bytes of columns x 128 rows, SWIZZLE_128B): G, and the slot
// workspace of the deterministic mode
int encode_matrix_map(CUtensorMap* tm, bool f64, void* ptr, int64_t rows, int64_t cols, int64_t pitch);

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
// What the reduction adds: nitems tiles at d_items (device memory) into g / ldg, or with grams (grouped launches) into
// the G of each item's problem
struct DetReduce {
  const DetItem* d_items;
  int nitems;
  void* g;
  int64_t ldg;
  const DetGram* grams;
};
// The launch sequence of the deterministic mode.  It allocates a stream-ordered workspace of nslots te x te slots (fp64
// when f64, else fp32), followed by a copy of *items when `items` is not NULL (the reduction then reads those);
// describes the slots to TMA in *slot_map (encode_matrix_map, te columns) when slot_map is not NULL; calls
// launch(workspace); enqueues the reduction; and frees the workspace on every return path.
int det_launch(int nslots, int te, bool f64, const std::vector<DetItem>* items, DetReduce red, CUtensorMap* slot_map,
               cudaStream_t stream, const std::function<int(void*)>& launch);
// det_launch for a kernel over a regular grid: the upper te x te tiles of a d x d Gram, numbered row-major over the
// upper triangle; tile t writes the `pieces` slots t * pieces .. + pieces, which the reduction adds in `mode` (DetItem)
int det_grid_launch(int d, int te, int pieces, int mode, bool f64, void* g, int64_t ldg, cudaStream_t stream,
                    const std::function<int(void*)>& launch);

}  // namespace vlm
