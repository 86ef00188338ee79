/*
 * agf_b200.h -- C ABI of libagf_b200.so: the sm_100a kernels behind aggforce's
 * frame-parallel statistics path.
 *
 * The reference (noegroup/aggforce) is pure Python and has no FFI; the interface each
 * entry point replaces is therefore a handful of numpy lines, cited per function as
 * <file>:<lines> relative to the reference root.  INTEGRATION.md shows the ctypes stub a
 * reference maintainer would add at each of those sites.
 *
 * Conventions
 *   - plain C, no torch / C++ types in any signature;
 *   - every pointer documented "device" is a CUDA device pointer owned by the caller,
 *     "host" is ordinary (ideally pinned) host memory; the library never frees or
 *     retains caller memory;
 *   - sizes are int64_t / int32_t, streams are passed as void* (a cudaStream_t);
 *   - functions are stream-ordered and re-entrant per (device, stream); the only global
 *     state is a thread-local error string;
 *   - return value: 0 = OK, negative = error (see AGF_E_*), message via agf_last_error();
 *   - accumulating outputs are documented "(+=)": the caller zeroes them once and may
 *     call repeatedly over frame chunks / keep partial sums per rank and all-reduce them.
 *   - dtype codes: AGF_F32 = 0, AGF_F64 = 1.
 */
#ifndef AGF_B200_H
#define AGF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGF_VERSION 100

#define AGF_F32 0
#define AGF_F64 1

#define AGF_OK 0
#define AGF_E_INVALID (-1)   /* bad argument (shape, dtype, null pointer, alignment) */
#define AGF_E_CUDA (-2)      /* a CUDA runtime call or kernel launch failed */
#define AGF_E_UNSUPPORTED (-3)
#define AGF_E_NAN (-4)       /* NaN protocol violated (result depends on NaN positions) */

int agf_version(void);
const char* agf_last_error(void);
/* Number of SMs of the current device (grid sizing / reporting). */
int agf_device_sm_count(void);

/* ------------------------------------------------------------------------------------
 * (a) linear second-moment Gram.
 * Replaces  src/aggforce/qp/qplinear.py:66-71
 *     reg_mat = matmul(qp_form(forces), con_mat);  qp_mat = matmul(reg_mat.T, reg_mat)
 * with the one-hot con_mat given as a CSR list of the sites of every reduced column
 * (src/aggforce/qp/qplinear.py:147-163).
 *
 *   forces     device, [n_frames, n_sites, 3] contiguous, dtype f32 or f64
 *   col_ptr    device int32 [n_red + 1], col_sites device int32 [col_ptr[n_red]]
 *   gram       device f64 [n_red, n_red] row-major, UPPER BLOCK-TRIANGLE (+=).  Call
 *              agf_symmetrize() once after the last chunk (and after any all-reduce).
 * FP64 tensor-core (DMMA) SYRK; inputs staged in shared memory with 1-D TMA bulk copies.
 */
int agf_gram_linear(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                    const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                    double* gram, void* stream);

/* Same contract as agf_gram_linear for n_red > 128, with a caller-provided scratch buffer: the
 * constraint-group sums are written once per frame into `workspace` (blocked f64 panels) and a
 * TMA-fed DMMA SYRK consumes them -- about 3x faster at n_red = 2600.  `workspace` is device
 * memory, 16-byte aligned; any size >= one chunk works (frames are processed in slabs), the
 * recommended size comes from agf_gram_linear_workspace_bytes (0 = the plain entry point is used).
 * Falls back to agf_gram_linear when n_red <= 128 or the workspace is NULL / too small.
 */
size_t agf_gram_linear_workspace_bytes(int32_t n_sites, int32_t n_red, int64_t n_frames);
int agf_gram_linear_ws(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                       const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                       double* gram, void* workspace, size_t workspace_bytes, void* stream);

/* Per-frame weighted Gram  P += sum_t w_t v_t v_t^T  (weighted force-map fits: reweighted or pooled
 * trajectories).  Same arguments, workspace and fallbacks as agf_gram_linear / agf_gram_linear_ws, plus
 *   frame_weights  device f64 [n_frames], one weight per frame of THIS call (frame t of `forces` reads
 *                  frame_weights[t]); the caller guarantees finite, non-negative values.  NULL = unweighted
 *                  (identical to the entry points above).
 * Runs the FP64 DMMA kernels: the group sums of frame t are multiplied by sqrt(w_t) in float64 where they
 * are staged (n_red <= 128) or packed (n_red > 128).  The int8 tensor-core Grams have no weighted form.
 */
int agf_gram_linear_weighted(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                             const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                             double* gram, const double* frame_weights, void* stream);
int agf_gram_linear_ws_weighted(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                                double* gram, void* workspace, size_t workspace_bytes,
                                const double* frame_weights, void* stream);

/* The same Gram through the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in
 * TMEM): float32 forces, n_red <= 97, constraint groups of at most 4 sites.  Group sums are scaled per
 * column by a power of two taken from a sample of the frames, rounded to 39-bit fixed point and split
 * into five signed 8-bit digits; the 15 digit-plane products with s + t <= 4 are accumulated exactly
 * in int32 and recombined in float64 (Ozaki scheme; 2e-12 relative Frobenius error on cln025, bar
 * 1e-9).  Frames holding a value outside the fixed-point range (or a non-finite one) are added in
 * float64 by a second kernel.  Accumulates into the upper triangle of gram like agf_gram_linear.
 *   max_group   largest number of sites in one reduced column
 *   slot_members  performance hint, 0 = none: byte c = largest group size among the columns
 *               4 q + c (q = 0..23), i.e. of "slot c" of the column quads a lane of the fill owns; with
 *               columns dealt to the slots by size (largest groups to slot 0) the fill runs straight-line
 *   workspace   device, agf_gram_linear_i8_workspace_bytes(...) bytes (0: shape not supported --
 *               use agf_gram_linear), 16-byte aligned
 */
size_t agf_gram_linear_i8_workspace_bytes(int32_t n_sites, int32_t n_red, int64_t n_frames);
int agf_gram_linear_i8(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                       const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                       int32_t max_group, uint32_t slot_members, double* gram, void* workspace,
                       size_t workspace_bytes, void* stream);

/* The tensor-core Gram for LARGE reduced problems (97 < n_red <= 8192, float32 forces, groups of any size):
 * the same digit scheme as agf_gram_linear_i8, tiled.  Per slab of 16 384 frames one kernel writes the five
 * digit planes of the group sums to `workspace` in the shared-memory layout of the tensor core (chunks of 32
 * frames of one xyz component, 16-column blocks: every operand plane of a tile is one contiguous span, moved
 * by 1-D TMA bulk copies), and a persistent kernel accumulates 128 x 96 tiles of the upper block-triangle
 * (tcgen05.mma kind::i8, five int32 accumulators per tile in TMEM, 4 096 contraction rows per work unit,
 * float64 recombination, atomic adds into gram).  Replaces agf_gram_linear_ws (FP64 DMMA) for float32 input:
 * same contract -- gram (+=) holds the element-wise upper triangle, call agf_symmetrize() afterwards.
 *   workspace   device, agf_gram_linear_i8t_workspace_bytes(...) bytes (0: shape not supported), 16-byte aligned
 */
size_t agf_gram_linear_i8t_workspace_bytes(int32_t n_sites, int32_t n_red, int64_t n_frames);
int agf_gram_linear_i8t(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                        const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red, double* gram,
                        void* workspace, size_t workspace_bytes, void* stream);

/* gram[j, i] = gram[i, j] for i < j (device f64 [n, n]). */
int agf_symmetrize(double* gram, int32_t n, void* stream);

/* ------------------------------------------------------------------------------------
 * (d) map application, fused with the NaN probe and the residual reduction.
 * Replaces  src/aggforce/util.py:119-124  (einsum "tfd,cf->tcd")
 *           src/aggforce/map/core.py:13-16,219-240 (NaN probe + NaN protocol)
 *           src/aggforce/agg.py:291-297 (mean(x**2), returned as a running sum)
 *
 * Dense form: the (n_cg, n_fg) matrix is passed column-compressed -- sites whose matrix
 * columns are identical share one "unique column" u (for an optimised force map these are
 * exactly the constraint groups); all-zero columns may be dropped when nan_mode == 1.
 *   points     device [n_frames, n_sites, 3], dtype in_dtype
 *   ucol_ptr   device int32 [n_ucol + 1], ucol_sites device int32 [nnz]: sites of column u
 *   umat_t     device f64 [n_ucol, n_cg] row-major: TRANSPOSE of the matrix restricted to
 *              the unique columns
 *   out        device [n_frames, n_cg, 3], dtype out_dtype
 *   sumsq      device f64 [1] (+=) sum of out**2 (values as stored), or NULL
 *   nan_mode   0: plain arithmetic (NaN propagates, 0*NaN = NaN as in numpy)
 *              1: reference NaN protocol -- NaN inputs count as 0; nan_flags[0] is set to 1
 *                 when any NaN was seen and nan_flags[1] to 1 when a result would change
 *                 beyond  atol + 1e-5*|result|  if the NaNs were -1 instead (core.py:230).
 *   nan_flags  device int32 [2] (|=), required when nan_mode == 1
 */
int agf_map_apply(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                  const int32_t* ucol_ptr, const int32_t* ucol_sites, int32_t n_ucol, int32_t nnz,
                  const double* umat_t, int32_t n_cg, void* out, int out_dtype, double* sumsq,
                  int nan_mode, double nan_atol, int32_t* nan_flags, void* stream);

/* Same contract with a caller-provided scratch buffer for maps too large for the shared-memory
 * resident kernel (n_cg > 64, e.g. 500 beads x 2600 unique columns): group sums are packed once
 * into f64 operand panels and a TMA-fed DMMA GEMM contracts them (about 8x faster than the
 * fallback at that size).  `workspace`: device memory, 256-byte aligned, size from
 * agf_map_apply_workspace_bytes (0 = not needed, the small kernel applies); frames are processed in
 * slabs, so any size >= header + packed map + one 128-frame block works.  NULL / too small =
 * agf_map_apply.
 */
size_t agf_map_apply_workspace_bytes(int in_dtype, int32_t n_sites, int32_t n_ucol, int32_t nnz,
                                     int32_t n_cg, int64_t n_frames);
int agf_map_apply_ws(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                     const int32_t* ucol_ptr, const int32_t* ucol_sites, int32_t n_ucol, int32_t nnz,
                     const double* umat_t, int32_t n_cg, void* out, int out_dtype, double* sumsq,
                     int nan_mode, double nan_atol, int32_t* nan_flags, void* workspace,
                     size_t workspace_bytes, void* stream);

/* The large dense application on the 5th-generation tensor cores (float32 input, finite weights, n_ucol <= 8192):
 * same outputs and NaN semantics as agf_map_apply_ws.  The sums of every unique column are scaled per column by
 * a power of two taken from a sample of the frames, rounded to 39-bit fixed point and split into five signed
 * 8-bit digit planes (columns = contraction dimension, K-major core matrices, one frame block x 32 columns per
 * TMA bulk copy); the weights, multiplied by the column scales, get a power-of-two scale per bead and the same
 * five digits.  A persistent kernel accumulates the 15 plane products with s + t <= 4 exactly in int32
 * (tcgen05.mma kind::i8, TMEM accumulators) per (32 frames x 128 beads) tile and recombines them in float64.
 * Frames holding a non-finite or out-of-range value are computed in float64 by a second kernel, which also
 * carries the NaN protocol (nan_mode 1: NaN counts as 0, nan_flags as for agf_map_apply).
 *   workspace   device, agf_map_apply_i8_workspace_bytes(...) bytes (0: shape not supported), 16-byte aligned
 */
size_t agf_map_apply_i8_workspace_bytes(int32_t n_sites, int32_t n_ucol, int32_t n_cg, int64_t n_frames);
int agf_map_apply_i8(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                     const int32_t* ucol_ptr, const int32_t* ucol_sites, int32_t n_ucol,
                     const double* umat_t, int32_t n_cg, void* out, int out_dtype, double* sumsq,
                     int nan_mode, double nan_atol, int32_t* nan_flags, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Sparse-row form for slice / uniform maps (a few non-zeros per bead): CSR rows
 *   row_ptr device int32 [n_cg + 1], row_sites device int32 [nnz], row_weights device f64 [nnz].
 * Only the referenced sites are read.  Same outputs / NaN semantics as agf_map_apply with
 * nan_mode 1 restricted to the referenced sites.
 */
int agf_map_apply_sparse(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                         const int32_t* row_ptr, const int32_t* row_sites, const double* row_weights,
                         int32_t n_cg, void* out, int out_dtype, double* sumsq, int nan_mode,
                         double nan_atol, int32_t* nan_flags, void* stream);

/* Slice maps: exactly one site per bead (row_sites int32 [n_cg], row_weights f64 [n_cg]) -- the
 * usual coordinate map.  Same outputs / NaN semantics; four gathers in flight per thread.
 */
int agf_map_apply_slice(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                        const int32_t* row_sites, const double* row_weights, int32_t n_cg,
                        void* out, int out_dtype, double* sumsq, int nan_mode, double nan_atol,
                        int32_t* nan_flags, void* stream);

/* Weighted residual numerator of a frame-weighted fit:  sumsq += sum_t w_t sum_e x[t, e]^2.
 *   x              device [n_frames, per_frame] contiguous (a mapped array: per_frame = 3 n_cg), f32 or f64
 *   frame_weights  device f64 [n_frames]
 *   sumsq          device f64 [1] (+=)
 * The unweighted sum comes from the `sumsq` epilogue of the agf_map_apply* kernels.
 */
int agf_weighted_sumsq(const void* x, int dtype, int64_t n_frames, int32_t per_frame,
                       const double* frame_weights, double* sumsq, void* stream);

/* ------------------------------------------------------------------------------------
 * (c) pair-distance moments for constraint detection.
 * Replaces  src/aggforce/util.py:64-70 (all-pairs displacement + norm) and
 *           src/aggforce/constraints/constfinder.py:47 (variance over frames).
 *
 * For each listed pair p = (i over `other`, j over `xyz`):  d_t = |xyz[t, j] - other[t, i]|
 * in float64;  acc[2p] += sum_t (d_t - shift[p]),  acc[2p+1] += sum_t (d_t - shift[p])^2.
 *   xyz        device [n_frames, n_sites, 3]; other: device [n_frames, n_other, 3] or NULL
 *              (NULL = same array, the reference's cross_xyz=None)
 *   pairs      device int32 [n_pairs, 2] (i, j)
 *   shift      device f64 [n_pairs] (any value near the mean distance; see agf_pair_first)
 *   acc        device f64 [n_pairs, 2] (+=)
 */
int agf_pair_moments(const void* xyz, const void* other, int dtype, int64_t n_frames,
                     int32_t n_sites, int32_t n_other, const int32_t* pairs, int64_t n_pairs,
                     const double* shift, double* acc, void* stream);

/* shift[p] = distance of pair p in frame 0 of the given arrays. */
int agf_pair_first(const void* xyz, const void* other, int dtype, int32_t n_sites,
                   int32_t n_other, const int32_t* pairs, int64_t n_pairs, double* shift,
                   void* stream);

/* All-pairs screening pass: for every (i, j) -- i < j when other == NULL, all n_other x
 * n_sites otherwise -- the sum of squared deviations of d_t from its mean over the given
 * frames, m2[i * n_sites + j] (device f64, overwritten; entries not visited hold +inf).
 * Used for exact progressive pruning: M2 over a subset of frames never exceeds M2 over
 * all frames, so a pair whose partial M2 already exceeds threshold^2 * T_total cannot be
 * a constraint.
 */
int agf_pair_screen(const void* xyz, const void* other, int dtype, int64_t n_frames,
                    int32_t n_sites, int32_t n_other, double* m2, void* stream);

/* Ordered compaction of the screened pair matrix (small systems, n_other * n_sites <= 2^18): the
 * device-side form of constfinder.py:52  nonzero(sds < threshold)  applied to the pruning bound --
 * pairs with m2 <= bound in row-major order (sharded runs: counts != NULL is a device array of the
 * n_counts per-rank frame counts and `bound` is threshold^2 -- the kernel forms
 * threshold^2 * sum(counts) itself, so the reduced screening buffer is consumed as it arrives), each with its frame-0 distance (the `shift` of agf_pair_moments) and zeroed accumulators.
 *   xyz / other   device frame 0 of the arrays passed to agf_pair_screen, [n_sites, 3] / [n_other, 3]
 *   pairs int32 [cap, 2], shift f64 [cap], acc f64 [cap, 2]   device, written for the survivors
 *   count int32 [1]  survivors, or -(survivors) when they exceed cap (then nothing else is written)
 */
int agf_pair_select(const double* m2, double bound, const double* counts, int32_t n_counts,
                    const void* xyz, const void* other, int dtype, int32_t n_sites, int32_t n_other,
                    int32_t cap,
                    int32_t* pairs, double* shift, double* acc, int32_t* count, void* stream);

/* ------------------------------------------------------------------------------------
 * (b) featurised Gram for Multifeaturize([id_feat, gb_feat]).
 * Replaces  src/aggforce/qp/featlinearmap.py:361-370 (einsum + kbt*div + reg.T @ reg) and the
 * feature generators src/aggforce/qp/featlinearmap.py:553-627 (id_feat),
 * src/aggforce/qp/jaxfeat.py:20-567 (gb_feat): features are evaluated in shared memory in
 * float64 and never written to HBM.
 *
 *   coords, forces  device [n_frames, n_sites, 3] (same dtype)
 *   grp_ptr/grp_sites  CSR label -> member sites, n_groups labels (id_feat's labels)
 *   n_channels      gb channels: n_groups, or n_groups - 1 to reproduce the reference's dropped
 *                   last channel (jaxfeat.py:115)
 *   bead_ptr/bead_sites/bead_w  CSR rows of the coordinate map (bead positions)
 *   centers         device f64 [nb] Gaussian centres (jaxfeat.py:235-236); width, clip as
 *                   jaxfeat.py:272-276; kbt multiplies the divergence (featlinearmap.py:368)
 *   gram            device f64 [n_cg, n_feat, n_feat] (+=), n_feat = n_groups + nb*n_channels,
 *                   feature order [id | channel-major gb]; UPPER block triangle: call
 *                   agf_symmetrize_batch afterwards.
 */
int agf_gram_feat(const void* coords, const void* forces, int dtype, int64_t n_frames,
                  int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                  int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                  const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                  const double* centers, int32_t nb, double width, double clip, double kbt,
                  double* gram, void* stream);

/* Same contract with a caller-provided scratch buffer (device, 16-byte aligned, size from
 * agf_gram_feat_workspace_bytes; frames are processed in slabs so any size >= one 8-frame chunk
 * works): every regression row is evaluated once, written as packed f64 operand panels and
 * contracted by a batched TMA-fed DMMA SYRK.  NULL / too small = agf_gram_feat.
 */
size_t agf_gram_feat_workspace_bytes(int32_t n_groups, int32_t n_channels, int32_t nb, int32_t n_cg,
                                     int64_t n_frames);
int agf_gram_feat_ws(const void* coords, const void* forces, int dtype, int64_t n_frames,
                     int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                     int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                     const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                     const double* centers, int32_t nb, double width, double clip, double kbt,
                     double* gram, void* workspace, size_t workspace_bytes, void* stream);

/* Per-frame weighted featurised Grams  P_c += sum_t w_t v_t v_t^T: every regression row of frame t
 * (id and gb columns, the kbt divergence term included) is multiplied by sqrt(w_t) in float64 once it
 * is complete.  Same arguments, workspace and fallbacks as agf_gram_feat / agf_gram_feat_ws, plus
 *   frame_weights  device f64 [n_frames], one finite non-negative weight per frame of this call; NULL =
 *                  unweighted.  FP64 DMMA kernels only (no weighted form of agf_gram_feat_i8).
 */
int agf_gram_feat_weighted(const void* coords, const void* forces, int dtype, int64_t n_frames,
                           int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                           int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                           const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                           const double* centers, int32_t nb, double width, double clip, double kbt,
                           double* gram, const double* frame_weights, void* stream);
int agf_gram_feat_ws_weighted(const void* coords, const void* forces, int dtype, int64_t n_frames,
                              int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                              int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                              const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                              const double* centers, int32_t nb, double width, double clip, double kbt,
                              double* gram, void* workspace, size_t workspace_bytes,
                              const double* frame_weights, void* stream);

/* The featurised Gram on the 5th-generation tensor cores (n_feat > 97; float32 or float64 input): same contract and
 * arguments as agf_gram_feat_ws.  The regression rows are evaluated in float64 exactly as there, scaled per
 * (bead, feature column) by a power of two taken from a sample of frame groups, rounded to 39-bit fixed point
 * and split into five signed 8-bit digit planes; the tiled tcgen05 int8 SYRK of agf_gram_linear_i8t runs batched
 * over the beads (128 x 96 tiles of every bead's upper block-triangle).  Frames with a non-finite or out-of-range
 * row value are added in float64 by a second kernel.
 *   workspace   device, agf_gram_feat_i8_workspace_bytes(...) bytes (0: shape not supported -- use
 *               agf_gram_feat_ws), 16-byte aligned
 */
size_t agf_gram_feat_i8_workspace_bytes(int32_t n_groups, int32_t n_channels, int32_t nb, int32_t n_cg,
                                        int64_t n_frames);
int agf_gram_feat_i8(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                     const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups,
                     int32_t n_channels, const int32_t* bead_ptr, const int32_t* bead_sites,
                     const double* bead_w, int32_t n_cg, const double* centers, int32_t nb, double width,
                     double clip, double kbt, double* gram, void* workspace, size_t workspace_bytes,
                     void* stream);

int agf_symmetrize_batch(double* gram, int32_t n, int32_t batch, void* stream);

/* ------------------------------------------------------------------------------------
 * Gaussian augmentation for joptgauss_map:  y = A x + eps,  eps ~ N(0, var I).
 * Replaces  src/aggforce/trajectory/core.py:353-390 (AugmentedTrajectory._augment) and the JAX
 * augmenter behind it, src/aggforce/trajectory/jaxgausstraj.py:232-284 (sample + autodiff
 * log-gradients; closed form as in simplegausstraj.py:108-110):
 *     out_coords = [x ; A x + eps]     out_forces = [F + kbt A^T eps / var ; -kbt eps / var]
 *   coords, forces   device [n_frames, n_sites, 3], dtype f32 or f64 (either may be NULL when
 *                    its output is NULL)
 *   bead_*           CSR rows of A (bead -> sites, weights); site_*: CSR rows of A^T
 *   noise            device [n_frames, n_cg, 3] standard normals in the array dtype, or NULL to
 *                    draw them in-kernel: Philox4x32-10 keyed by (seed, frame0 + t, bead, draw),
 *                    so any slab / rank reproduces the same noise for the same key
 *   out_coords/out_forces  device [n_frames, n_sites + n_cg, 3], same dtype, or NULL
 */
int agf_gauss_augment(const void* coords, const void* forces, int dtype, int64_t n_frames,
                      int32_t n_sites, const int32_t* bead_ptr, const int32_t* bead_sites,
                      const double* bead_w, int32_t n_cg, const int32_t* site_ptr,
                      const int32_t* site_beads, const double* site_w, double var, double kbt,
                      const void* noise, uint64_t seed, uint32_t draw, int64_t frame0,
                      void* out_coords, void* out_forces, void* stream);

/* Equality-constraint rows of one bead's feature QP for a few frames,
 * rows[s, c', f] = sum_a cmap[c', a] phi_bead[frames[s], a, f]
 * (src/aggforce/qp/featlinearmap.py:446-450).  frames: device int64 [n_sel];
 * label_of_site: device int32 [n_sites]; rows: device f64 [n_sel, n_cg, n_feat] (overwritten).
 */
int agf_feat_rows(const void* coords, int dtype, int32_t n_sites, const int64_t* frames,
                  int32_t n_sel, int32_t bead, const int32_t* label_of_site,
                  const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups,
                  int32_t n_channels, const int32_t* bead_ptr, const int32_t* bead_sites,
                  const double* bead_w, int32_t n_cg, const double* centers, int32_t nb,
                  double width, double clip, double* rows, void* stream);

/* Application of the fitted featurised map (src/aggforce/qp/featlinearmap.py:512-520 +
 * src/aggforce/map/core.py:428-430): out[t, c, :] = sum_a w[t,c,a] F[t,a,:] + trans[t,c,:] with
 * per-frame weights w = phi . coef and trans = div . coef (no kbt factor, as the reference),
 * never materialising w.  coefs: device f64 [n_cg, n_feat]; out [n_frames, n_cg, 3].
 */
int agf_feat_apply(const void* coords, const void* forces, int dtype, int64_t n_frames,
                   int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                   int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                   const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                   const double* centers, int32_t nb, double width, double clip,
                   const double* coefs, void* out, int out_dtype, double* sumsq, void* stream);

/* ------------------------------------------------------------------------------------
 * Equality-constrained QP of qp_linear_map on the device, small reduced problems (SURVEY 8f-1).
 * Replaces  src/aggforce/qp/qplinear.py:76-86 (P += l2 C'C; per bead solve_qp(P, 0, A, e_bead)):
 * all beads at once,  X = P^-1 A' (A P^-1 A')^-1,  one CTA, P in shared memory.
 *   gram      device f64 [n_red, n_red]; only the (element-wise) upper triangle is read, which is
 *             what agf_gram_linear accumulates -- no symmetrise pass needed in between
 *   diag_add  device f64 [n_red] added to the diagonal (l2 * group size) or NULL
 *   a_mat     device f64 [n_cg, n_red] equality rows (cmap C), same column order as gram
 *   x_out     device f64 [n_cg, n_red]:  x_out[c, x_index[p]] = X[p, c]   (x_index: a permutation)
 *   u_out     device f64 [n_ucol, n_cg] or NULL:  u_out[u_index[p], c] = X[p, c]  -- the `umat_t`
 *             operand of agf_map_apply, so the fitted map is applied without a host round trip
 *   status    device int32 [1], written only on failure: 1 P not positive definite, 2 Schur
 *             complement not positive definite, 3 non-finite solution, 4 equality constraints missed by
 *             more than 1e-6 (caller falls back to the host)
 * Limits: n_red <= 128, n_cg <= 32 (agf_qp_equality_small_supported).
 */
int agf_qp_equality_small(const double* gram, int32_t n_red, const double* diag_add,
                          const double* a_mat, int32_t n_cg, const int32_t* x_index, double* x_out,
                          const int32_t* u_index, double* u_out, int32_t* status, void* stream);
int agf_qp_equality_small_supported(int32_t n_red, int32_t n_cg);

/* ------------------------------------------------------------------------------------
 * Validation projections on random Gaussian force fields (SURVEY 8f-4).
 * Replaces  src/aggforce/jaxmapval.py:365-401 (sq_gaussian_energies / sq_gaussian_forces: JAX
 * autodiff of  E = sum_{i,j} exp(-((|x_j - x_i|^2 - offset)/width)^2)  over the full squared
 * distance matrix) and the per-sample loops of random_force_proj (:309-319, mscg_ip :359-360) and
 * random_residual_shift (:227-237).  All samples are evaluated in ONE pass over the frames:
 *   out[s, 0] += sum_{t,i} F[t,i,:] . G_s[t,i,:]        out[s, 1] += sum_{t,i} |G_s[t,i,:]|^2
 * with G_s the force field of offset offsets[s]  (projection = out[s,0] / n_frames;
 * residual shift = (out[s,1] - 2 out[s,0]) / (3 n_frames n_sites)).
 *   coords, forces  device [n_frames, n_sites, 3] (the MAPPED arrays), dtype f32 or f64
 *   offsets         device f64 [n_samples];  width: the (already squared, if sq_args) width
 *   out             device f64 [n_samples, 2], accumulated into (zero it first)
 */
int agf_gauss_field_moments(const void* coords, const void* forces, int dtype, int64_t n_frames,
                            int32_t n_sites, const double* offsets, int32_t n_samples,
                            double width, double* out, void* stream);

/* One force field written out: out[t, i, :] = -dE/dx_i for a single (offset, width)
 * (src/aggforce/jaxmapval.py:396-401 as called by rsqpg_forces :139).  out [n_frames, n_sites, 3].
 */
int agf_sq_gaussian_forces(const void* coords, int dtype, int64_t n_frames, int32_t n_sites,
                           double offset, double width, void* out, int out_dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * Synthetic trajectory generator for benchmarks and tests (counter-based, so any
 * frame range of any sharding reproduces the same data):  frame0 = global index of the
 * first generated frame.  See aggforce_b200/synth.py for the model.
 *   ref_pos    device f32 [n_sites, 3]; parent device int32 [n_sites] (-1 for heavy atoms)
 *   bond_len   device f32 [n_sites]
 *   coords/forces  device f32 [n_frames, n_sites, 3] (overwritten); either may be NULL
 */
int agf_synth_frames(const float* ref_pos, const int32_t* parent, const float* bond_len,
                     int32_t n_sites, int64_t frame0, int64_t n_frames, uint64_t seed,
                     float pos_sigma, float force_sigma, float h_coupling, float* coords,
                     float* forces, void* stream);

/* ------------------------------------------------------------------------------------
 * One-shot exchange of small float64 payloads between the ranks of a frame-sharded fit, over
 * NVLink peer memory (SURVEY 8e: the all-reduce of Gram / pair moments / residual sums; the
 * reference has no multi-device code).  Every rank owns one symmetric buffer of
 * agf_peer_buffer_bytes(slot_doubles) bytes, zero-initialised, that all peers have mapped;
 * peer_ptrs is a DEVICE array [world] with every rank's buffer address in this process.  One
 * kernel on `stream`: copy-in, signal / wait (release / acquire, system scope), combine.
 *   op 0: out[i] = sum_r in_r[i]   op 1: out[i] = max_r in_r[i] (NaN wins)
 *   op 2: out[r * count + i] = in_r[i] (all-gather)
 *   op 3 | (k << 8): sum for i < k, max for i >= k (residual sums and NaN flags in one message)
 *   seq   call number, the same on all ranks, starting at 1 and increasing by 1 per call
 *   error device int32 [1], set to 1 if a peer's signal never arrived (result then invalid)
 */
size_t agf_peer_buffer_bytes(int64_t slot_doubles);
int agf_peer_exchange(const uint64_t* peer_ptrs, int32_t rank, int32_t world, uint32_t seq,
                      int32_t op, const double* in, double* out, int64_t count,
                      int64_t slot_doubles, int32_t* error, void* stream);

/* ------------------------------------------------------------------------------------
 * Roofline probes (bench.py measures its denominators in the run that quotes them; no reference
 * counterpart).  agf_probe_dmma: every SM streams independent DMMA.8x8x4 tiles for `iters`
 * iterations; *flop_out = flops issued; sink: device f64 [sm_count * 8 * 256].
 * agf_probe_read: one streaming read of `bytes` bytes (16-byte aligned device buffer).
 */
int agf_probe_dmma(int32_t iters, double* sink, int64_t* flop_out, void* stream);
int agf_probe_read(const void* src, int64_t bytes, float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGF_B200_H */
