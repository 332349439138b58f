/*
 * vlmerge.h — C ABI of libvlmerge.so, the B200 (sm_100a) merge hot path of ylsung/vl-merging.
 *
 * The reference has no FFI layer: its operator boundary is (1) a PyTorch forward hook and
 * (2) three state_dict -> state_dict methods (SURVEY.md §8b).  Each entry point below replaces
 * the arithmetic of one reference call site; the Python shim in vl-merging_b200/ binds them with
 * ctypes and mirrors the reference's hook / merge-method signatures on top.
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = vlm_status, >0 = cudaError_t.  Nothing throws.
 *     vlm_last_error() returns a thread-local message for the last non-zero return.
 *   - all pointers are DEVICE pointers unless the name ends in _host.  The library borrows them
 *     for the duration of the call (work is enqueued on `stream`, a cudaStream_t passed as void*;
 *     NULL = legacy default stream) and never frees or retains them.
 *   - matrices are row-major with leading dimension in ELEMENTS.
 *   - there is no CPU path: without a CUDA device every compute entry point fails.
 */
#ifndef VLMERGE_H_
#define VLMERGE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLM_ABI_VERSION 3

typedef enum {
  VLM_OK = 0,
  VLM_ERR_INVALID_ARG = -1,   /* null pointer, negative size, bad enum */
  VLM_ERR_ALIGNMENT = -2,     /* pointer / leading dimension not usable by the requested path */
  VLM_ERR_UNSUPPORTED = -3,   /* e.g. device is not sm_100 */
  VLM_ERR_DRIVER = -4,        /* cuTensorMapEncodeTiled / cuSOLVER symbol lookup failed */
  VLM_ERR_NOT_SPD = -5,       /* Cholesky failed: summed Gram is singular / not positive definite */
  VLM_ERR_INTERNAL = -6
} vlm_status;

typedef enum {
  VLM_F32 = 0, VLM_BF16 = 1, VLM_F16 = 2, VLM_F64 = 3,
  VLM_TF32X2 = 4   /* Gram input only: the {hi, lo} TF32 planes written by vlm_tf32_split */
} vlm_dtype;

/* ---- library ------------------------------------------------------------------------------- */
int         vlm_version(void);          /* VLM_ABI_VERSION */
const char* vlm_last_error(void);       /* thread-local, never NULL */
/* number of kernels this library has launched in the calling process (bench.py gpu_launches) */
uint64_t    vlm_launch_count(void);

/* ---- (a) Gram accumulation -----------------------------------------------------------------
 * Replaces hook_gram_input, src/cache_gram_matrices.py:246-254:
 *     flatten_input = input.reshape(-1, D).to(float64); gram = flatten_input.T @ flatten_input
 *     middle_representations[name] += gram.cpu()
 * G[r][c] += sum_k X[k][r] * X[k][c]  for every c >= r (upper triangle; elements below the
 * diagonal are scratch until vlm_sym_mirror_batch).  X is the hooked activation viewed as
 * [rows, d]; any alignment and any width.  The tensor-core path (the CTA-pair kernel: f32 -> rounded to TF32 by TMA ->
 * TF32 tensor cores, bf16/f16 -> f16-kind tensor cores, fp32 accumulation in TMEM and fp32 in G) takes X when d is a
 * whole number of 128-byte column groups (d % 32 == 0 for f32, d % 64 == 0 for bf16/f16), x and g are 16-byte aligned,
 * ldx*sizeof(elem) % 16 == 0 and ldg % 4 == 0.  Everything else runs on the CUDA-core kernel of vlm_syrk_accum_simt
 * (fp32 FMA).  dtype VLM_TF32X2 has only the tensor-core path: VLM_ERR_UNSUPPORTED if d % 32 != 0, VLM_ERR_ALIGNMENT
 * if the planes or g are not aligned as above.  rows == 0 is a no-op. */
int vlm_syrk_accum(const void* x, int dtype, int64_t rows, int d, int64_t ldx,
                   float* g, int64_t ldg, void* stream);

/* Split-precision ("3xTF32") Gram input for RegMean-grade Grams.  The reference forms X^T X in fp64
 * (src/cache_gram_matrices.py:251-252) and regmean inverts the sum (src/vilt/modules/vilt_module.py:432-434,
 * :483-484); one TF32 pass carries 2^-11 of rounding noise per operand, which the inverse amplifies.
 * vlm_tf32_split writes out[0][r][c] = hi = tf32(x[r][c]) and out[1][r][c] = lo = tf32(x - hi) (out: 2*rows*d
 * floats, contiguous, 16-byte aligned; x fp32 with row pitch ldx, optionally row-segmented as in
 * vlm_syrk_accum_strided, seg_rows = 0 for plain rows).  vlm_syrk_accum / vlm_syrk_accum_batch with
 * dtype = VLM_TF32X2, x = out, ldx = d then accumulate hi'hi + hi'lo + lo'hi: three tensor-core products per
 * K step on the same TMA / tcgen05 pipeline.  Needs d % 32 == 0 (VLM_ERR_UNSUPPORTED otherwise). */
int vlm_tf32_split(const float* x, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                   float* out, void* stream);

/* Reference-precision Gram: fp64 products and fp64 accumulation into an fp64 G — the arithmetic of the reference
 * hook itself (src/cache_gram_matrices.py:251-252), on the fp64 tensor-core path (DMMA).  The tcgen05 kernels
 * above accumulate in the tensor core's truncating fp32 accumulator (~2e-5 non-uniform shrink even with exact
 * operands), which regmean's inverse (src/vilt/modules/vilt_module.py:432-434) amplifies on ill-conditioned
 * Gram sums; this entry point is the RegMean-grade mode (GramCache(precision="fp64")).  x: f32 / bf16 / f16,
 * any alignment (16-byte aligned rows take the cp.async path), optionally row-segmented (seg_rows = 0: plain
 * rows).  Upper block triangle only, like vlm_syrk_accum; vlm_sym_mirror_batch (dtype VLM_F64) mirrors it. */
int vlm_syrk_accum_f64(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                       int64_t seg_stride, double* g, int64_t ldg, void* stream);

/* The same Gram, exact, on the INTEGER tensor cores: column c is scaled by 2^(26-E_c), 2^E_c the power of two just
 * above its maximum in this call (2^(E_c-1) <= max < 2^E_c; E_c = 0 for a zero column), and every value becomes four
 * balanced int8 digits (q = rint(x * 2^(26-E_c)) = sum D_p * 128^(3-p));
 * the thirteen digit-plane products with p + q <= 4 run as tcgen05.mma kind::i8 (int32 accumulation: exact) and are
 * added to the fp64 Gram with their power-of-two scales (fp64 TMA reduce-adds).  Error: at most 2^(E_c-27) per
 * element, i.e. 2^-27 to 2^-26 of the column maximum (unbiased quantisation) + the dropped products (< 1e-9 of
 * sqrt(G_ii G_jj)) — measured 1e-10 on normal data, 3e-9 on LayerNorm outputs: RegMean-grade — at about 3.5x the cost
 * of the single TF32 pass instead of the fp64 path's 28x.  E_c is clamped below at -100 so that the float scale
 * 2^(26-E_c) stays finite: a column whose maximum is below 2^-101 is quantised with the fixed step 2^-126, an error of
 * up to 2^-127 per element, which is 2^-127 / max of the column maximum (2^-17 for a maximum of 2^-110) instead of
 * 2^-27.  x: VLM_F32 / VLM_F16 / VLM_BF16 (16-bit values are widened exactly), 16-byte aligned, ldx % 4 == 0,
 * optionally row-segmented; d % 128 == 0 (VLM_ERR_UNSUPPORTED otherwise: use vlm_syrk_accum_f64); scratch:
 * vlm_syrk_i8x4_scratch_bytes(rows, d) bytes of device memory, 16-byte aligned, borrowed for the call.  G as for
 * vlm_syrk_accum_f64, 16-byte aligned with an even ldg (TMA). */
uint64_t vlm_syrk_i8x4_scratch_bytes(int64_t rows, int d);
int vlm_syrk_accum_i8x4(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows, int64_t seg_stride,
                        void* scratch, uint64_t scratch_bytes, double* g, int64_t ldg, void* stream);

/* Several independent vlm_syrk_accum problems of the same dtype in ONE launch (e.g. the 48 small Grams of the
 * text tower of one forward, which are launch-bound one by one).  Same contract per problem; the activations
 * must stay alive and unmodified until `stream` has run the launch.  Problems outside the tensor-core condition of
 * vlm_syrk_accum (for segmented ones also seg_stride*sizeof(elem) % 16 == 0) are issued as individual launches. */
typedef struct {
  const void* x;
  int64_t     rows;        /* total rows (= number of row segments * seg_rows when segmented) */
  int64_t     ldx;
  float*      g;
  int64_t     ldg;
  int32_t     d;
  int32_t     reserved;
  int64_t     seg_rows;    /* 0: rows are one contiguous run; > 0: see vlm_syrk_accum_strided */
  int64_t     seg_stride;  /* elements between the first rows of consecutive segments */
} vlm_syrk_problem;
int vlm_syrk_accum_batch(const vlm_syrk_problem* probs_host, int n, int dtype, void* stream);

/* Row-sliced activation: X is rows/seg_rows SEGMENTS of seg_rows rows each (row pitch ldx), segment s starting
 * seg_stride elements after segment s-1 — the view `h[:, a:b]` of a (B, N, D) activation that the fused
 * vision-language route feeds to the per-modality experts (src/vilt/modules/vision_transformer.py:619-637,
 * :667-677), where the reference's `input.reshape(-1, D)` (src/cache_gram_matrices.py:250) makes a copy.
 * Here the slice is read in place through a 4-D tensor map when the tensor-core condition of vlm_syrk_accum holds and
 * seg_stride * sizeof(elem) is a multiple of 16; otherwise each segment is one vlm_syrk_accum.  rows must be a multiple
 * of seg_rows.  Otherwise the contract of vlm_syrk_accum. */
int vlm_syrk_accum_strided(const void* x, int dtype, int64_t rows, int d, int64_t ldx, int64_t seg_rows,
                           int64_t seg_stride, float* g, int64_t ldg, void* stream);

/* Same contract on CUDA cores (fp32 FMA), any alignment, whatever the shape.  Debug oracle on the device
 * (GramCache(use_simt=True)) and the kernel vlm_syrk_accum runs outside its tensor-core condition. */
int vlm_syrk_accum_simt(const void* x, int dtype, int64_t rows, int d, int64_t ldx,
                        float* g, int64_t ldg, void* stream);

/* Symmetric Gram storage.  The SYRK entry points above form only the upper triangle of G; the packed form of a Gram is
 * its row-major upper triangle, row r = columns r..d-1 at element offset r*d - r*(r-1)/2, d*(d+1)/2 values in all: the
 * on-disk container (vl-merging_b200/gramfile.py; replaces the 2.15 GB fp64 pickle of src/cache_gram_matrices.py:349
 * <-> src/vilt/modules/vilt_module.py:386 with 0.54 GB) and the exchange buffer of GramCache.all_reduce.
 * Each call below treats all its Grams in ONE launch: items[i] = {full (d x d, pitch ld), packed, d}, every item of the
 * element type `dtype` (VLM_F32 or VLM_F64) on both sides.
 *   vlm_sym_pack_upper_batch  reads the upper triangle of `full` (below the diagonal is never read) into `packed`;
 *   vlm_sym_unpack_batch      writes both triangles of `full` from `packed`;
 *   vlm_sym_mirror_batch      in place: the lower triangle of `full` from its upper one (G[c][r] = G[r][c], c > r);
 *                             `packed` is ignored and may be NULL. */
typedef struct vlm_sym_item {
  const void* full;
  void* packed;
  int32_t d;
  int32_t reserved;
  int64_t ld;
} vlm_sym_item;
int vlm_sym_pack_upper_batch(const vlm_sym_item* items, int n, int dtype, void* stream);
int vlm_sym_unpack_batch(const vlm_sym_item* items, int n, int dtype, void* stream);
int vlm_sym_mirror_batch(const vlm_sym_item* items, int n, int dtype, void* stream);

/* The exchange step of data-parallel Gram caching as ONE kernel over NVSwitch multicast memory (the reference has no
 * reduction: every DDP rank overwrites the same file, src/cache_gram_matrices.py:349).  multicast_base: the multicast
 * mapping of a symmetric allocation that holds, at the same offsets on every rank, the Grams described by `spans`.
 * The upper-triangular 32 x 32 tiles are dealt round-robin to the ranks; the owner reads a tile with
 * multimem.ld_reduce.add (the switch returns the sum over all ranks) and multimem.st's it into every rank's copy:
 * pack + all-reduce + unpack in one launch, bit-identical on all ranks; the lower triangles follow locally
 * (vlm_sym_mirror_batch).  The caller
 * brackets the launch with cross-rank barriers on `stream` (all ranks' accumulation before, all stores landed
 * after).  fp32 Grams need d and ld multiples of 4; offsets 16-byte aligned. */
typedef struct vlm_sym_span {
  uint64_t offset_bytes;
  int32_t d;
  int32_t reserved;
  int64_t ld;
} vlm_sym_span;
int vlm_sym_allreduce_multimem(void* multicast_base, const vlm_sym_span* spans, int n, int dtype, int rank, int world,
                               void* stream);

/* Host-only view of the work decomposition of vlm_syrk_accum's CTA-pair kernel for (rows, d) on a device with nsm SMs
 * (elem_bytes 4 = f32, 2 = bf16/f16): writes segments as 4 int32 each {super_row, super_col (256-column units),
 * chunk_begin, chunk_end} and ncluster+1 offsets into them.  elem_bytes 1 = the int8 digit-plane kernel
 * (vlm_syrk_accum_i8x4): 32-row chunks, the phase (0, 1, 2) in bits 16.. of super_col.  Returns the number of segments
 * (>= 0) or a vlm_status.  No CUDA calls; used by the CPU tests. */
int vlm_syrk_pair_schedule_host(int64_t rows, int d, int elem_bytes, int nsm, int32_t* segs_out, int cap,
                                int32_t* off_out, int off_cap, int* ncluster_out);

/* ---- (b) streaming merge -------------------------------------------------------------------
 * Replaces the per-tensor loops of merge_weights (src/vilt/modules/vilt_module.py:586-635),
 * sum_task_vectors (:696-744) and the simple-average branches of regmean (:436-457, :486-529).
 * One launch streams every segment once; fp32, rounding order identical to the reference:
 *   VLM_MERGE_WSUM     dst = (c0*s0) + (c1*s1) + ...            (products rounded, then added)
 *   VLM_MERGE_SEQ_LERP dst = s0; dst = dst + c_m*(s_m - dst)    m = 1..n_src-1  (s0 = central;
 *                      the reference's aliased in-place update, SURVEY.md §8 a-7)
 *   VLM_MERGE_MEAN     dst = (s0 + s1 + ...) / n_src
 */
typedef enum { VLM_MERGE_WSUM = 0, VLM_MERGE_SEQ_LERP = 1, VLM_MERGE_MEAN = 2 } vlm_merge_mode;
#define VLM_MERGE_MAX_SRC 4

typedef struct {
  float*       dst;                       /* n fp32 elements (device) */
  const float* src[VLM_MERGE_MAX_SRC];    /* n_src device pointers, n elements each */
  float        coef[VLM_MERGE_MAX_SRC];   /* per-source coefficient (unused for MEAN; coef[0] unused for SEQ_LERP) */
  uint64_t     n;
  int32_t      n_src;                     /* 1..VLM_MERGE_MAX_SRC */
  int32_t      mode;                      /* vlm_merge_mode */
} vlm_merge_seg;

typedef struct vlm_merge_plan vlm_merge_plan;
/* Upload the segment table once (host array), run it any number of times. */
int vlm_merge_plan_create(const vlm_merge_seg* segs_host, int n_seg, vlm_merge_plan** out);
int vlm_merge_plan_run(const vlm_merge_plan* plan, void* stream);
int vlm_merge_plan_destroy(vlm_merge_plan* plan);
/* algorithmic bytes one run moves: sum over segments of (n_src + 1) * n * 4 */
uint64_t vlm_merge_plan_bytes(const vlm_merge_plan* plan);

/* n copies dst_base + dst_off_bytes[i] <- src[i] (nbytes[i] each; host or device sources, cudaMemcpyDefault) enqueued
 * on `stream` in one call: stages the ~400 tensors of a host checkpoint into the merge's input arena.  Pinned sources
 * copy asynchronously; pageable ones are staged by the driver before the call returns. */
int vlm_copy_batch(void* dst_base, const uint64_t* dst_off_bytes, const void* const* src_host_or_dev,
                   const uint64_t* nbytes, int n, void* stream);

/* ---- (c) RegMean ---------------------------------------------------------------------------
 * Replaces, in regmean (src/vilt/modules/vilt_module.py:366-531):
 *   scale_G (:388-392)              Ghat = a*G + (1-a)*diag(G)
 *   summed_gram += G (:423,474)     vlm_gram_scale_accum
 *   later_weight += W.double() @ G (:424,475)   vlm_regmean_rhs
 *   matmul(later_weight, inverse(summed_gram)) (:432-434,:483-484)   vlm_spd_solve_right
 * All fp64 like the reference.  g_dtype is VLM_F64 (the reference's Gram file) or VLM_F32 (our
 * on-device Gram buffers); G must be the full symmetric matrix (after vlm_sym_mirror_batch). */
int vlm_gram_scale_accum(const void* g, int g_dtype, int d, int64_t ldg, double alpha,
                         double* out, int64_t ldo, int accumulate, void* stream);
/* acc[out_f][in_f] (+)= sum_k W[out_f][k] * Ghat[k][in_f];  W fp32 (out_f x in_f), G (in_f x in_f). */
int vlm_regmean_rhs(const float* w, int out_f, int in_f, int64_t ldw,
                    const void* g, int g_dtype, int64_t ldg, double alpha,
                    double* acc, int64_t ldacc, int accumulate, void* stream);
/* The same with the left operand W - W_base (same shape and pitch; the difference is formed in fp64).  With M experts
 * and S = sum Ghat_m:  (sum_m W_m Ghat_m) S^-1  =  W_base + (sum_{m != base} (W_m - W_base) Ghat_m) S^-1,  one GEMM
 * fewer than the reference's formula (half the flops for the two-modality layers), identical in exact arithmetic. */
int vlm_regmean_rhs_diff(const float* w, const float* w_base, int out_f, int in_f, int64_t ldw,
                         const void* g, int g_dtype, int64_t ldg, double alpha,
                         double* acc, int64_t ldacc, int accumulate, void* stream);
/* dst[rows][cols] (fp64) += src[rows][cols] (fp32): adds W_base back after the solve. */
int vlm_widen_add(const float* src, int rows, int cols, int64_t lds, double* dst, int64_t ldd, void* stream);
/* X = R * S^{-1} for SPD S (in_f x in_f, fp64, overwritten by its Cholesky factor); R (out_f x
 * in_f, fp64) is overwritten by X.  cuSOLVER potrf/potrs; off the hot path, timed separately.
 * Synchronises `stream` to read the factorisation status. */
int vlm_spd_solve_right(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr,
                        void* stream);
/* Same without the synchronisation, so that independent solves can run concurrently on several streams
 * (a Cholesky factorisation of a 768..4096-wide matrix does not fill the GPU on its own): the two status words
 * (potrf: > 0 = leading minor that is not positive definite; potrs) are written to info_dev[0..1] (device
 * memory) for the caller to read after its own synchronisation.  One cuSOLVER handle is kept per stream. */
int vlm_spd_solve_right_async(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr,
                              int* info_dev, void* stream);

/* ---- retrieval step after the merge (SURVEY.md §8f rank 2) ------------------------------------
 * Replaces, in compute_irtr_recall (src/vilt/modules/objectives.py:684-710),
 *     scores = img_cls_feats @ txt_cls_feats.t();  scores.topk(k, dim=1)  (k = 1, 5, 10)
 * and, with the operands swapped, scores.topk(k, dim=0): the ten best rows of B for every row of A, by
 * A[i] . B[j], straight from the tensor-core accumulators — the m x n score matrix (500 MB for 5,000 x 25,000) is
 * never written.  a [m, d], b [n, d]: VLM_F16 or VLM_BF16 (what the towers produce under the reference's autocast),
 * row-major, 16-byte aligned, lda / ldb multiples of 8.  Products exact, fp32 accumulation.
 * out_val / out_idx: [m][splits][10] — per row `splits` partial lists (one per range of B), each sorted descending
 * with the lower index first among equal scores, padded with -inf / -1; splits = vlm_sim_topk_splits(m, n)
 * (chosen so that few row blocks still fill the GPU).  The caller merges the partial lists. */
int vlm_sim_topk_splits(int64_t m, int64_t n);
int vlm_sim_topk(const void* a, int64_t m, int64_t lda, const void* b, int64_t n, int64_t ldb, int d, int dtype,
                 float* out_val, int32_t* out_idx, int splits, void* stream);

/* Pivoted-LU variant for a summed Gram that Cholesky rejects (VLM_ERR_NOT_SPD / potrf status > 0): the reference
 * inverts with torch.inverse (LU; src/vilt/modules/vilt_module.py:432,483), which succeeds on any numerically
 * non-singular matrix.  s must hold the FULL symmetric matrix again (potrf overwrote a triangle); both s and r are
 * overwritten.  Synchronises `stream`.  VLM_ERR_NOT_SPD here means an exactly zero pivot (singular). */
int vlm_lu_solve_right(double* s, int in_f, int64_t lds, double* r, int out_f, int64_t ldr, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VLMERGE_H_ */
