/*
 * osb200.h -- C ABI of libosb200.so, the B200 (sm_100a) sparse-3D-convolution + open-vocabulary
 * matching engine that replaces the MinkowskiEngine native backend and the driver-side torch ops on
 * OpenScene's hot path.
 *
 * What each group replaces in the reference (paths relative to the reference root):
 *   osb_coordset_* / osb_kernel_map_*   the coordinate manager inside MinkowskiEngine that
 *        `ME.SparseTensor(feat, coords)` (run/evaluate.py:284, run/distill.py:316) and every
 *        `ME.MinkowskiConvolution(..., kernel_size=k, stride=s)` (models/mink_unet.py:47-113) drive:
 *        coordinate hash, tensor-stride sets, per-offset kernel maps.
 *   osb_conv_*                          `MinkowskiConvolution.forward` / `MinkowskiConvolutionTranspose.forward`
 *        (gather -> GEMM -> scatter-add per sparse-conv layer; models/mink_unet.py:116-174) and their autograd
 *        backward (run/distill.py:333).
 *        `MinkowskiBatchNorm` (eval) / `MinkowskiReLU` / the BasicBlock residual / `ME.cat` have no entry points of their
 *        own: they are arguments of osb_conv_* (scale/shift, relu, res, src1), folded into the convolution's epilogue
 *        (models/mink_unet.py:50,114,147).
 *   osb_match_*                         `predictions[inds_reverse]`, `x/(|x|+1e-5)`, `.half() @ text_features.t()`,
 *        `torch.max(pred,1)` (run/evaluate.py:288-323).
 *   osb_voxelize_*                      `Voxelizer.voxelize` + `sparse_quantize`/`fnv_hash_vec`
 *        (dataset/voxelizer.py:97-140, dataset/voxelization_utils.py:9-22,44-137).
 *   osb_fusion_*                        the multi-view fusion loop: `PointCloudToImageMapper.compute_mapping`
 *        (scripts/feature_fusion/fusion_util.py:102-139) + the running mean of
 *        scripts/feature_fusion/scannet_openseg.py:74-108 (SURVEY.md 8f rank 2).
 *   osb_feature_remap                   the fused-feature index remap of `FusedFeatureLoader.__getitem__`
 *        (dataset/feature_loader.py:101-172) (SURVEY.md 8f rank 3).
 *   osb_confusion_* / osb_intersection_union   `confusion_matrix` (util/metric.py:9-25) and
 *        `intersectionAndUnionGPU` (util/util.py:132-145) (SURVEY.md 8f rank 4).
 *
 * Conventions
 *   - every pointer is a raw DEVICE pointer unless the name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises
 *     unless documented ("SYNC");
 *   - the CALLER allocates every output and workspace (sizes via the *_workspace_bytes queries), so
 *     memory stays in the caller's allocator; the library keeps no per-call state (the only process-wide state are the
 *     tuning knobs of osb_tuning_set, which never change results);
 *   - every function returns 0 on success, non-zero on failure; osb_last_error() returns a
 *     thread-local description; no exception crosses the ABI;
 *   - there is no CPU fallback: on a machine without an sm_100 GPU every compute entry point fails.
 */
#ifndef OSB200_H
#define OSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OSB_VERSION 100

/* ------------------------------------------------------------------ misc */
int         osb_version(void);
const char *osb_last_error(void);
/* sm count, compute capability of the current device. */
int osb_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
int64_t osb_launch_count(void);
/* SM clock in MHz measured on the device (clock64 against %globaltimer over ~20 us); *mhz_dev is a device float. */
int osb_measure_sm_mhz(float *mhz_dev, void *stream);

/* --------------------------------------------------------- coordinate sets
 * A coordinate is an int32 row (b, x, y, z).  Valid range: 0 <= b < 1024, |x|,|y|,|z| < 2^17 - 256.
 * Internally rows are kept in Morton order (b major) -- the "internal order"; `perm[r]` is the
 * caller's row of internal row r.
 *
 * Hash table: `cap` slots of 16 bytes {uint64 key, int32 row, int32 pad}, cap a power of two >= 2n.
 */
size_t osb_coordset_workspace_bytes(int64_t n);

/* Build the tensor-stride-1 set from caller-order coordinates.
 *   coords      in  int32 [n,4]
 *   coords_int  out int32 [n,4]   coordinates in internal (Morton) order
 *   perm        out int32 [n]     internal row -> caller row
 *   inv_perm    out int32 [n]     caller row  -> internal row
 *   slots       out 16B  [cap]    hash table over coords_int
 *   status_host out int32 [6]     HOST: [0] bit0 = coordinate out of range, bit1 = duplicate coordinate; [1] reserved;
 *                                 [2..5] = OR (lo, hi word) and AND (lo, hi word) of the 64-bit Morton keys
 *                                 b<<54 | interleave(x+2^17, y+2^17, z+2^17) -- sizes the occupancy grid below
 *   slots may be NULL (no hash table wanted: the caller uses an occupancy grid)
 * SYNC: waits for `stream` to deliver status_host. */
int osb_coordset_build(const int32_t *coords, int64_t n, int32_t *coords_int, int32_t *perm, int32_t *inv_perm,
                       void *slots, int64_t cap, int32_t *status_host, void *ws, size_t ws_bytes, void *stream);

/* Coarser set: unique(floor(c / new_ts) * new_ts) per batch index, Morton ordered.
 *   coords_fine   in  int32 [n,4] (internal order)
 *   new_ts        absolute tensor stride of the coarse set (any integer >= 1)
 *   coords_coarse out int32 [<=n,4]
 *   parent_of     out int32 [n]     fine row -> coarse row
 *   n_coarse_host out int64 [1]     HOST
 * SYNC. */
int osb_coordset_stride(const int32_t *coords_fine, int64_t n, int32_t new_ts, int32_t *coords_coarse,
                        int32_t *parent_of, int64_t *n_coarse_host, void *ws, size_t ws_bytes, void *stream);

/* The whole stride-2 pyramid of a U-Net encoder in one call (2 host syncs instead of 2 per level): tensor-stride-1 set
 * as osb_coordset_build, plus `n_levels` coarser sets with tensor strides 2, 4, ..., 2^n_levels.  Children are Morton
 * sorted, so parents of a power-of-two stride are already in order: no sort, level counts stay on the device.
 *   coords_lvl  out int32 [n_levels][n,4]   coarse sets, upper-bound sized (use the first n_host[l+1] rows of slab l)
 *   parent_lvl  out int32 [n_levels][n]     parent_lvl[l][r]: row of level-l row r in level l+1
 *   n_host      out int64 [n_levels+1]      HOST: rows per level;  status_host as osb_coordset_build
 * SYNC. */
int osb_coordset_pyramid(const int32_t *coords, int64_t n, int32_t n_levels, int32_t *coords_int, int32_t *perm,
                         int32_t *inv_perm, void *slots, int64_t cap, int32_t *coords_lvl, int32_t *parent_lvl,
                         int64_t *n_host, int32_t *status_host, void *ws, size_t ws_bytes, void *stream);

/* (Re)build a hash table over internal-order coordinates. */
int osb_hash_build(const int32_t *coords_int, int64_t n, void *slots, int64_t cap, void *stream);

/* Kernel map in output-stationary form: nbr[k*n_out + o] = input row at c_out[o] + delta_k*step, or -1.
 * Offsets enumerate x fastest; odd kernel sizes are centred, even ones use delta in {0..ks-1}
 * (region convention of the generalised sparse convolution; SURVEY.md 8a a6).
 *   pairs_per_k   out int32 [K] (may be NULL): number of valid pairs per offset. */
int osb_kernel_map_build(const int32_t *coords_out, int64_t n_out, const void *slots_in, int64_t cap_in,
                         int32_t ks_x, int32_t ks_y, int32_t ks_z, int32_t step, int32_t *nbr,
                         int32_t *pairs_per_k, void *stream);

/* Swap the roles of input and output: nbr_t[k*n_in + i] = o  iff  nbr[k*n_out + o] = i  (else -1). */
int osb_kernel_map_transpose(const int32_t *nbr, int64_t n_out, int32_t K, int32_t *nbr_t, int64_t n_in,
                             void *stream);

/* ----------------------------------------------------------- sparse conv
 * Generic fp32 path (CUDA cores; any channel counts).  out[o,:] = sum_k in[nbr[k][o],:] @ W[k]
 *   in   fp32 [n_in, cin] (row stride ld_in floats)     w  fp32 [K, cin, cout]
 *   out  fp32 [n_out, cout]
 *   transpose_w != 0: use W[k]^T, i.e. w is [K, cout, cin] (dgrad). */
int osb_conv_fwd_f32(const float *in, int64_t ld_in, const int32_t *nbr, int64_t n_out, int32_t K,
                     const float *w, int32_t cin, int32_t cout, int32_t transpose_w, float *out, void *stream);

/* Weight gradient: gw[k] = sum_o in[nbr[k][o],:]^T gout[o,:]   (gw fp32 [K,cin,cout], overwritten). */
int osb_conv_wgrad_f32(const float *in, const int32_t *nbr, int64_t n_out, int32_t K, const float *gout,
                       int32_t cin, int32_t cout, float *gw, void *stream);

/* Weight gradient on tensor cores (run/distill.py:333): gw[k] = sum_o x[nbr[k][o],:]^T gout[o,:] with both operands in the
 * split layout (x_split [n_in, cin], gout_split [n_out, cout]); gw fp32 [K,cin,cout] is overwritten.  Every product is the
 * full (hi+lo)(hi+lo) expansion on kind::f16 MMAs with fp32 accumulation; partial tiles are reduced in a fixed order
 * (bit-reproducible, no atomics).  ws: osb_conv_wgrad_tc_workspace_bytes(...) bytes. */
size_t osb_conv_wgrad_tc_workspace_bytes(int64_t n_out, int32_t K, int32_t cin, int32_t cout);
int osb_conv_wgrad_tc(const void *x_split, int32_t cin, int64_t n_in, const int32_t *nbr, int64_t n_out, int32_t K,
                      const void *gout_split, int32_t cout, float *gw, void *ws, size_t ws_bytes, void *stream);

/* Tensor-core path (tcgen05, bf16x3 split-fp32 operands, fp32 accumulation in TMEM).
 *
 * Activation "split" layout: a row of C channels (C % 32 == 0) is 4*C bytes; every 32-channel block is
 * one 128-byte line [bf16 hi x32 | bf16 lo x32] with hi = bf16_rn(v), lo = bf16_rn(v - hi).
 * Packed weights (osb_conv_pack_weights): per offset k, cout_pad rows of the same split layout over
 * cin, i.e. the K-major B operand.
 *
 *   src0/src1   split rows, c0 and c1 channels (src1 may be NULL with c1 = 0): the conv input is the
 *               column concatenation [src0 | src1] -- `ME.cat` without materialising it
 *   nbr         int32 [K, n_out]  (NULL with K == 1 means identity: a 1x1x1 conv)
 *   wpack       packed weights for cin = c0 + c1
 *   scale/shift fp32 [cout] or NULL: y = acc*scale + shift   (eval-mode BatchNorm folded)
 *   res         residual added before ReLU: split rows [n_out, cout] or NULL
 *   relu        != 0 applies max(y, 0)
 *   out_split   split rows [n_out, cout] or NULL
 *   out_f32     fp32 [n_out, cout] or NULL; out_row_map (int32 [n_out] or NULL) scatters fp32 rows:
 *               row o is written to out_f32[out_row_map[o]]
 *   flags       bit0: launch with programmatic stream serialization (PDL).  The kernel's prologue (barrier / TMEM
 *               set-up, loading `nbr`, scale, shift) then overlaps the tail of the previous kernel in `stream`; it
 *               waits for that kernel before touching src*, res, ws or any output.  Only legal when nbr / wpack /
 *               scale / shift were NOT produced by the immediately preceding kernel in the stream.
 */
size_t osb_conv_packed_weight_bytes(int32_t K, int32_t cin, int32_t cout);
/* Scratch osb_conv_fwd_tc needs for this shape: small problems are split over the (offset, channel-block)
 * sequence across CTAs (fp32 partials + a deterministic reduce kernel); 0 when no split is used. */
size_t osb_conv_tc_workspace_bytes(int64_t n_out, int32_t K, int32_t cin, int32_t cout);
int osb_conv_pack_weights(const float *w, int32_t K, int32_t cin, int32_t cout, int32_t transpose_w,
                          void *wpack, void *stream);
int osb_conv_fwd_tc(const void *src0, int32_t c0, int64_t n_src0, const void *src1, int32_t c1, int64_t n_src1,
                    const int32_t *nbr, int64_t n_out, int32_t K, const void *wpack, int32_t cout,
                    const float *scale, const float *shift, const void *res, int32_t relu, void *out_split,
                    float *out_f32, const int32_t *out_row_map, void *ws, size_t ws_bytes, int32_t flags, void *stream);

/* Transposed stride-2 convolution (`MinkowskiConvolutionTranspose(kernel_size=2, stride=2)`, models/mink_unet.py:79-101) as a
 * dense GEMM over the coarse rows followed by a scatter to the children: wpack = osb_conv_pack_weights of the
 * [1, cin, kvol*cout] matrix (column block k = W[k]); down_nbr = int32 [kvol, n_coarse], the kernel map of the matching
 * strided convolution (child row of parent o through offset k, -1 if absent).  out_* have one row per FINE voxel and
 * `cout` channels; every fine row is written exactly once.  scale/shift/relu/flags as osb_conv_fwd_tc. */
int osb_convtr_fwd_tc(const void *src, int32_t cin, int64_t n_coarse, const int32_t *down_nbr, int32_t kvol, const void *wpack,
                      int32_t cout, const float *scale, const float *shift, int32_t relu, void *out_split, float *out_f32,
                      int32_t flags, void *stream);


/* ----------------------------------------------------------- persistent convolution chains (conv_chain.cu)
 * Second-generation tensor-core path: ONE launch executes a list of convolution layers (`MinkowskiConvolution` /
 * `MinkowskiConvolutionTranspose` forwards of consecutive modules of models/mink_unet.py:116-174, BasicBlock included) with
 * one persistent CTA per SM, dedicated epilogue warps, a double-buffered TMEM accumulator, split-K reduced inside the
 * kernel and grid barriers between dependent layers.  Same arithmetic and the same argument meaning as osb_conv_fwd_tc.
 *
 * A layer is described by an opaque record of osb_conv_desc_bytes() bytes, filled on the HOST by osb_conv_desc_fill; the
 * launch passes the records to the kernel as launch parameters (16 layers per launch, longer lists in several launches).
 *   wtiles          osb_conv_pack_weight_tiles(w [K,cin,cout]) -- tile-major, pre-swizzled B operands
 *   cmap/cmap_cout  non-NULL: dense transposed stride-2 convolution as in osb_convtr_fwd_tc (wtiles of the [1,cin,kvol*cout]
 *                   matrix, cout = kvol*cmap_cout, cmap = the stride-2 map [kvol, n_out] of the matching strided conv)
 *   ws / ws_bytes   scratch for split-K partials, osb_conv_chain_workspace_bytes(...) bytes (0 = not split).  Consecutive
 *                   split layers without a barrier between them need different scratch
 *   barrier_before  != 0: this layer reads (src*, res) what an earlier layer of the SAME launch wrote
 *   grid_barrier    2 x uint32 in device memory, zeroed once when allocated (never reset afterwards); required when any
 *                   layer of the launch is split or asks for a barrier.  One launch at a time may use it.
 *   flags           bit0: PDL, as in osb_conv_fwd_tc */
size_t osb_conv_desc_bytes(void);
size_t osb_conv_weight_tiles_bytes(int32_t K, int32_t cin, int32_t cout);
int osb_conv_pack_weight_tiles(const float *w, int32_t K, int32_t cin, int32_t cout, int32_t transpose_w, void *wtiles,
                               void *stream);
int osb_conv_chain_grid(void);
size_t osb_conv_chain_workspace_bytes(int64_t n_out, int32_t K, int32_t cin, int32_t cout);
int osb_conv_desc_fill(void *desc_host, const void *src0, int32_t c0, const void *src1, int32_t c1, const int32_t *nbr,
                       int64_t n_out, int32_t K, const void *wtiles, int32_t cout, const float *scale, const float *shift,
                       const void *res, int32_t relu, void *out_split, float *out_f32, const int32_t *out_row_map,
                       const int32_t *cmap, int32_t cmap_cout, void *ws, size_t ws_bytes, int32_t barrier_before);
int osb_conv_chain_launch(const void *descs_host, int32_t n_layers, void *grid_barrier, int32_t flags, void *stream);

/* Process-wide tuning knobs (tile shapes, ring depths, split factors, profiling hooks).  They select between
 * equivalent schedules and never change results; unknown names fail.  Names: see csrc/conv_chain.cu, csrc/conv_tc.cu. */
int osb_tuning_set(const char *name, int64_t value);

/* Stem: fused kernel-map probe + conv for tiny cin (<= 3) and cout <= 32, fp32 FMA.  One launch replaces the
 * 5x5x5 map build (125 probes / voxel) and the 3->32 convolution of `conv0p1s1`.
 *   in  fp32 [n, cin] internal order;  w fp32 [K, cin, cout];  epilogue as osb_conv_fwd_tc. */
int osb_conv_stem_fused(const float *in, int32_t cin, const int32_t *coords, int64_t n, const void *slots,
                        int64_t cap, int32_t ks, int32_t step, const float *w, int32_t cout, const float *scale,
                        const float *shift, int32_t relu, void *out_split, float *out_f32, void *stream);

/* fp32 [n,c] <-> split rows. */
int osb_f32_to_split(const float *in, int64_t n, int32_t c, void *out_split, void *stream);
int osb_split_to_f32(const void *in_split, int64_t n, int32_t c, float *out, void *stream);

/* ------------------------------------------------------ row-wise helpers */
/* out[r,:] = in[idx[r],:]  (fp32 rows of c floats; idx int32) */
int osb_gather_rows_f32(const float *in, const int32_t *idx, int64_t n_out, int32_t c, float *out, void *stream);

/* ------------------------------------------------- open-vocabulary match
 * One pass over the voxel features per query point p (v = inds_reverse[p], or p when NULL):
 *   a = feat[v,:] (fp32 or fp16);  if normalize: a = a / (|a| + 1e-5)
 *   s = fp16( fp16(a) . text[k,:] )  with fp32 accumulation  (text fp16 [K, C] row major)
 *   scores[p,k] = s (fp16, may be NULL), label[p] = argmax_k s (first maximum), smax[p] = max_k s (may be NULL)
 * Mirrors run/evaluate.py:290-292 (distill), :294-296 (fusion), :303-310 (the two normalised products). */
int osb_match_scores(const void *feat, int32_t feat_is_f16, int64_t n_vox, int32_t c, const int64_t *inds_reverse,
                     int64_t n_pts, const void *text_f16, int32_t k_text, int32_t normalize, void *scores_f16,
                     int64_t *label, float *smax, void *stream);
/* Ensemble select + final product (run/evaluate.py:316-322):
 *   m = smax3d[p] < smax2d[p];  fe = m ? feat2d_f16[v] : fp16(feat3d[v]);  scores = fe @ text^T;  label = argmax
 *   feat_out_f16 (may be NULL) receives fe. */
int osb_match_ensemble(const float *feat3d, const void *feat2d_f16, int64_t n_vox, int32_t c,
                       const int64_t *inds_reverse, int64_t n_pts, const float *smax3d, const float *smax2d,
                       const void *text_f16, int32_t k_text, void *scores_f16, int64_t *label, void *feat_out_f16,
                       void *stream);

/* Test-time repeats (run/evaluate.py:385-425): the product of osb_match_scores (feat2_f16 == NULL) or of
 * osb_match_ensemble (feat = feat3d fp32, feat2_f16 = feat2d, sel_a = smax3d, sel_b = smax2d, normalize = 0), folded into
 * a running fp16 sum instead of being written out:
 *   h = fp16(a . text[k,:])                      the score osb_match_* returns
 *   store[p,k] = first ? h + (+0.0) : h + store[p,k]   one fp16 rounding (== torch's `pred + store` on fp16 tensors;
 *                                                     the first repeat turns -0 into +0 like `pred + 0.0`)
 *   label[p]   = first argmax_k of the ACCUMULATED store[p,:] (== `store.float().max(1)[1]`; may be NULL)
 *   store      in/out fp16 [n_pts, K]; read only when first == 0
 * Limits as the tensor-core matcher: C in {512, 768}, 1 <= K <= 480.  Without inds_reverse n_pts must equal n_vox.
 * There is no CUDA-core variant: under OSB_MATCH_SIMT=1 the call fails. */
int osb_match_accumulate(const void *feat, int32_t feat_is_f16, const void *feat2_f16, const float *sel_a, const float *sel_b,
                         int64_t n_vox, int32_t c, const int64_t *inds_reverse, int64_t n_pts, const void *text_f16,
                         int32_t k_text, int32_t normalize, void *store_f16, int32_t first, int64_t *label, void *stream);
/* Test-time repeats of class logits (run/eval_mink.py:168-216), CUDA cores, any C >= 1:
 *   x = logits[inds_reverse[p], :] (fp32 [n_vox, C]; row p when inds_reverse is NULL, then n_pts == n_vox)
 *   store[p,:] = first ? x + 0.0 : x + store[p,:]      (fp32 in/out [n_pts, C])
 *   label_cur[p] = first argmax of x (this repeat alone), label_acc[p] = first argmax of store[p,:]; either may be NULL */
int osb_logits_accumulate(const float *logits, int64_t n_vox, int32_t c, const int64_t *inds_reverse, int64_t n_pts,
                          float *store, int32_t first, int64_t *label_cur, int64_t *label_acc, void *stream);

/* Optional folded head (engine.forward_scores): rows z = [x L | x U] (fp32, row pitch ld floats) from one 1x1x1
 * convolution with the weights [L | U], W W^T = L L^T, U = W T^T  ->  score_k = fp16((x.U_k) / (|x L| + 1e-5)),
 * label = first argmax.  Same cosine scores as run/evaluate.py:305-310 without materialising the 768-d features. */
int osb_folded_head_finish(const float *z, int64_t n, int32_t ld, int32_t c_norm, int32_t k_text, void *scores_f16,
                           int64_t *label, float *smax, void *stream);

/* ------------------------------------------------------------- voxeliser
 * coords (fp32 or fp64 [n,3]) -> c = floor([p,1] . M^T[:, :3]) with M the HOST 4x4 row-major fp64 matrix,
 * c -= min(c), FNV-64 key (multiply-then-xor over uint64 words), unique by ascending key keeping the
 * FIRST occurrence (np.unique semantics).
 *   coords_vox    out int32 [<=n,3]    voxel coordinates, in ascending-key order
 *   inds          out int64 [<=n]      first-occurrence point index per voxel
 *   inds_reverse  out int64 [n]        voxel row of every point
 *   n_vox_host    out int64 [1] HOST;  min_host out fp64 [3] HOST (the subtracted minimum)
 * SYNC. */
size_t osb_voxelize_workspace_bytes(int64_t n);
int osb_voxelize(const void *coords, int32_t coords_is_f64, int64_t n, const double *matrix_host,
                 int32_t *coords_vox, int64_t *inds, int64_t *inds_reverse, int64_t *n_vox_host,
                 double *min_host, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------- occupancy grid (alternative to the hash table)
 * For a coordinate set whose coordinates are all >= 0 and < (2^nbits << log2_ts): one bit per cell of a 2^nbits cube per
 * batch index, cells in Morton order, + the first row of every 64-cell word.  Because the rows of a set are Morton
 * sorted, row(cell) = first_row[word] + popcount(bits below): a neighbour lookup is two loads from a table of a few
 * MB shared by nearby voxels instead of a probe chain.  Limits: 2 <= nbits <= 9, n_batch << (3 nbits) <= 2^27 cells.
 *   grid        osb_occgrid_bytes(nbits, n_batch) bytes (0 = not representable: use the hash)
 *   coords_int  the set in internal (Morton) order, as produced by osb_coordset_build / _pyramid
 *   status_dev  in/out int32 [1] DEVICE: bit0 set if a coordinate fell outside the grid
 * osb_kernel_map_build_grid / osb_conv_stem_fused_grid are osb_kernel_map_build / osb_conv_stem_fused with the grid of
 * the INPUT set in place of its hash table; results are identical. */
size_t osb_occgrid_bytes(int32_t nbits, int32_t n_batch);
int osb_occgrid_build(const int32_t *coords_int, int64_t n, int32_t log2_ts, int32_t nbits, int32_t n_batch, void *grid,
                      int32_t *status_dev, void *stream);
int osb_kernel_map_build_grid(const int32_t *coords_out, int64_t n_out, const void *grid, int32_t log2_ts, int32_t nbits,
                              int32_t n_batch, int32_t ks_x, int32_t ks_y, int32_t ks_z, int32_t step, int32_t *nbr,
                              int32_t *pairs_per_k, void *stream);
int osb_conv_stem_fused_grid(const float *in, int32_t cin, const int32_t *coords, int64_t n, const void *grid, int32_t log2_ts,
                             int32_t nbits, int32_t n_batch, int32_t ks, int32_t step, const float *w, int32_t cout,
                             const float *scale, const float *shift, int32_t relu, void *out_split, float *out_f32, void *stream);

/* ------------------------------------------------------------- multi-view feature fusion (8f rank 2)
 * One call handles a batch of 1..32 frames, in frame order.
 *   points   fp32 or fp64 [n,3] world coordinates
 *   w2c      fp64 [F,16]  row-major world-to-camera matrices (= inv(pose), fusion_util.py:120)
 *   intr     fp64 [F,4]   (fx, fy, cx, cy) per frame (intrinsic[0][0], [1][1], [0][2], [1][2])
 *   depth    fp64 [F,H,W] metres, or NULL (then the test is p_z > 0, fusion_util.py:134)
 *   feat     fp16 [F,H,W,C] per-pixel features (the memory the reference holds as a permuted [C,H,W] view),
 *            C % 8 == 0, C <= 1024
 *   sum      in/out fp32 [n,C]; counter in/out fp32 [n]: sum += feature, counter += 1 for every frame that sees the
 *            point, applied in frame order (bit-identical to the reference's per-frame fp32 adds).
 *            sum == NULL computes the mapping only.
 *   mapping  out int32 [F,n,3] = (row v, col u, visible) as compute_mapping returns it, or NULL
 *   ws       osb_fusion_workspace_bytes(n, F) bytes */
size_t osb_fusion_workspace_bytes(int64_t n, int32_t n_frames);
int osb_fusion_accumulate(const void *points, int32_t points_is_f64, int64_t n, const double *w2c, const double *intr,
                          const double *depth, const void *feat, int32_t n_frames, int32_t H, int32_t W, int32_t C,
                          int32_t cut_bound, double vis_thres, float *sum, float *counter, int32_t *mapping, void *ws,
                          size_t ws_bytes, void *stream);
/* feat_bank = sum / (counter == 0 ? 1e-5 : counter)   (scannet_openseg.py:104-105); feat_bank may alias sum */
int osb_fusion_finalize(const float *sum, const float *counter, int64_t n, int32_t C, float *feat_bank, void *stream);

/* ------------------------------------------------------------- segmentation metrics (8f rank 4)
 * confusion  in/out uint64 [(C+1),(C+1)], rows = prediction, columns = ground truth; points with gt == ignore_id are
 *            skipped, predictions equal to nofeat_id land in row C (util/metric.py:13-20; the caller slices [:C,:C]).
 * bad_labels in/out int32 [1]: number of labels outside the valid range (the reference would raise in reshape).
 * Labels are int32 or int64 device arrays. */
int osb_confusion_accumulate(const void *pred, const void *gt, int32_t labels_are_i64, int64_t n, int32_t num_classes,
                             int32_t ignore_id, int32_t nofeat_id, uint64_t *confusion, int32_t *bad_labels, void *stream);
/* areas in/out uint64 [3,K] = (intersection, output area, target area) with the reference's histc semantics
 * (util/util.py:132-145): where target == ignore_id the prediction is ignored too; labels outside 0..K-1 are dropped.
 * union = output + target - intersection. */
int osb_intersection_union(const void *output, const void *target, int32_t labels_are_i64, int64_t n, int32_t K,
                           int32_t ignore_id, uint64_t *areas, void *stream);

/* ------------------------------------------------------------- fused-feature remap after voxelisation (8f rank 3)
 * The fused 2-D features of a scene are stored as {feat [M,C], mask_full bool [n_pts]} with one feat row per True
 * entry of mask_full, in point order (scripts/feature_fusion/fusion_util.py:87-89).  Given the voxeliser's
 * representative point per voxel (vox_ind), produce what dataset/feature_loader.py:101-172 hands to the model:
 *   mask_vox  out uint8 [n_vox]            mask_full[vox_ind]                                  (:127)
 *   feat_out  out [<= n_vox, row_bytes]    keep_all == 0 (train): rows of the voxels with mask_vox set, in voxel
 *                                          order (:128-145); keep_all != 0 (val / test): one row per voxel, zeros
 *                                          where the voxel has no feature (:107-111,167-170)
 *   n_out_host out int64 [1] HOST          rows written
 * Rows are opaque: row_bytes = C * element size, a multiple of 16.  m_rows must equal popcount(mask_full).  SYNC. */
size_t osb_feature_remap_workspace_bytes(int64_t n_pts, int64_t n_vox);
int osb_feature_remap(const uint8_t *mask_full, int64_t n_pts, const int64_t *vox_ind, int64_t n_vox, const void *feat,
                      int64_t m_rows, int32_t row_bytes, int32_t keep_all, uint8_t *mask_vox, void *feat_out,
                      int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OSB200_H */
