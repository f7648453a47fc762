/*
 * mspl_b200.h -- C ABI of libmspl_b200.so: the B200 (sm_100a) kernels behind MSPL's multi-source
 * pseudo-label generation and its uncertainty-weighted loss.
 *
 * The reference (ShigemichiMatsuzaki/MSPL) is pure Python and has no FFI/plugin registry; its "API" for
 * this path is a set of Python callables.  Each entry point below names the reference interface it
 * replaces (file:line relative to the reference tree).  The Python mirror of those callables lives in
 * mspl_b200/ (uest_seg_multi_os.py, loss_fns/segmentation_loss.py) and binds this library with ctypes.
 *
 * Conventions
 *   - Plain pointers and sizes only; every pointer is a DEVICE pointer unless marked HOST.
 *   - The library never allocates, frees or synchronises: the caller owns all buffers and the stream.
 *   - All work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - Returns MSPL_OK (0) or a negative mspl_status; never throws, never exits.  mspl_strerror() explains.
 *   - Logits are fp32, contiguous NCHW: plane (n, c) starts at ((n * C + c) * pixels_per_image) floats.
 *   - Accumulating outputs (histograms, counters) are ADDED to; the caller zeroes them.
 *   - There is no CPU fallback anywhere in this library.
 */
#ifndef MSPL_B200_H
#define MSPL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MSPL_API __attribute__((visibility("default")))
#else
#define MSPL_API
#endif

#define MSPL_ABI_VERSION 5
#define MSPL_MAX_SOURCES 8      /* S: sources fused per call                                        */
#define MSPL_MAX_SRC_CLASSES 256 /* C_s: the reference stores the argmax as uint8 (uest_seg_multi_os.py:904) */
#define MSPL_MAX_CLASSES 8      /* K: target (greenhouse) classes; the reference has 5 (greenhouse.py:14).  Eight is what the
                                 * kernels' packed per-pixel state holds: votes in 8 x 4 bits, class counts in 8 x 8 bits, and a
                                 * K x 2048-bin confidence histogram per CTA in shared memory (64 KB at K = 8) next to the ring */
#define MSPL_RADIX_BINS 2048    /* bins of one histogram pass: linear conf bins, or 11 bits of the key */
#define MSPL_RADIX_PASSES 3     /* 11 + 11 + 10 bits of the order-preserving fp32 key               */

typedef enum mspl_status {
    MSPL_OK = 0,
    MSPL_ERR_BAD_ARG = -1,      /* null pointer, negative size, K/S/C out of range                  */
    MSPL_ERR_ALIGN = -2,        /* a pointer is not aligned for its element type                    */
    MSPL_ERR_UNSUPPORTED = -3,  /* valid request this build has no kernel for                       */
    MSPL_ERR_CUDA = -4,         /* launch failed (cudaPeekAtLastError)                              */
    MSPL_ERR_WORKSPACE = -5     /* workspace too small                                              */
} mspl_status;

/* Fusion policy of mspl_fuse_sources. */
#define MSPL_POLICY_VOTE 0      /* merge_outputs vote with threshold vote_t (reference behaviour)   */
#define MSPL_POLICY_PROB 1      /* [NEW] argmax of the averaged greenhouse-class probabilities      */

MSPL_API const char* mspl_strerror(int status);
MSPL_API int mspl_abi_version(void);
/* Name of the fused kernel variant this build dispatches to (for bench/profiling records). */
MSPL_API const char* mspl_fuse_variant(void);

/* ---- K0: get_output's device half ---------------------------------------------------------------
 * Replaces uest_seg_multi_os.py:687-691 (`softmax2d(pred + 0.5*pred_aux)` and `PixelwiseKLD(pred, pred_aux)`).
 * prob (n, c, pixels) and/or kld (n, pixels) may be NULL to skip that output. */
MSPL_API int mspl_softmax_kld(const float* main_logits, const float* aux_logits, int64_t n, int c,
                     int64_t pixels_per_image, float* prob, float* kld, void* stream);

/* ---- K1: fused multi-source pseudo-label generation ---------------------------------------------
 * Replaces the per-image loop body of generate_pseudo_label_multi_model (uest_seg_multi_os.py:897-921):
 * get_output (:669-693) -> np.argmax (:904) -> id_*_to_greenhouse gather (:907-912,
 * data_loader/segmentation/greenhouse.py:15-58) -> merge_outputs (:695-718) -> class_array (:919-921),
 * plus the KLD the reference computes and discards (:691, loss_fns/segmentation_loss.py:181-189), plus the
 * [NEW] per-pixel confidence (average over sources of transfer_output_to_greenhouse, :1334-1350) and the
 * first radix-select histogram pass of the class-balanced thresholds.
 *
 *   main_logits/aux_logits  HOST arrays of S device pointers, source s is (num_images, num_classes[s], pixels)
 *   num_classes, lut        HOST arrays; lut[s] is a HOST table of num_classes[s] bytes with values < K
 *   policy, vote_t          MSPL_POLICY_VOTE: label = lowest k with the most votes, or `ignore_label` when the
 *                           winning count < vote_t (vote_t: S//2+1 for 'half', S for 'all');
 *                           MSPL_POLICY_PROB: label = first argmax_k of F = (sum_s G_s)/S
 *   label      (num_images*pixels) u8             conf, unc   same shape f32, NULLable
 *   kld_per_source  HOST array of S device pointers (or NULL; entries may be NULL): per-source KLD maps
 *   class_hist      K u64, += number of pixels per label (the reference's class_array)
 *   conf_hist       K*MSPL_RADIX_BINS u64 or NULL, += linear histogram of conf per label (bin = min(2047, floor(conf*2048)),
 *                   the input of mspl_bracket_select), restricted to pixels with (pixel_index_in_image % ds_rate) == 0
 *   marginal_count  u64 or NULL, += pixels where, for some source, the softmax margin between the best class of its
 *                   winning target and the best class of any OTHER target is < 1e-6 (and, for MSPL_POLICY_PROB, the
 *                   top-2 margin of F): the only pixels whose label may legitimately differ from the reference's
 *                   argmax-of-softmax (a near-tie between two source classes of the same target cannot change it) */
MSPL_API int mspl_fuse_sources(int num_sources, const float* const* main_logits, const float* const* aux_logits,
                      const int* num_classes, const uint8_t* const* lut, int64_t num_images,
                      int64_t pixels_per_image, int num_target_classes, int policy, int vote_t,
                      int ignore_label, int ds_rate, uint8_t* label, float* conf, float* unc,
                      float* const* kld_per_source, unsigned long long* class_hist,
                      unsigned long long* conf_hist, unsigned long long* marginal_count, void* stream);

/* Host-only helper (no device work): the order in which K1 visits the classes of a source with label table `lut` -- sorted by
 * (target class, class index), so that the kernel tracks one running maximum per target group instead of an arg-max index.
 * row[i] = the source class visited i-th (num_classes bytes); seg[j] bit b = slot b of chunk j is the last class of its target
 * group (ceil(num_classes / chunk) bytes); *present bit k = some class maps to target k.  Returns the chunk size (classes per
 * shared-memory stage) the build uses, or a negative status. */
MSPL_API int mspl_class_order(const uint8_t* lut, int num_classes, int num_target_classes, uint8_t* row, uint8_t* seg,
                     uint32_t* present);
/* Host-only companion: what K1's per-source epilogue reads besides the order -- vote[i] = 1 << 4*(target class of the i-th target
 * group in visiting order), the amount a source adds to a pixel's packed vote counters (4 bits per target, hence
 * MSPL_MAX_SOURCES <= 15) when that group holds its largest fused logit (MSPL_MAX_CLASSES entries, unused ones 0), and *nchunk =
 * the number of class chunks the kernel's inner loop runs for this source.  Returns the number of target groups (>= 1), or a
 * negative status. */
MSPL_API int mspl_class_order_votes(const uint8_t* lut, int num_classes, int num_target_classes, uint32_t* vote, uint32_t* nchunk);
/* Host-only companion: which compiled chunk shape K1 runs for this table -- 1 + the index of the listed shape (the greenhouse
 * tables' class orders, which the kernel runs as straight-line code) whose class count, chunk count and group boundaries the
 * table's order has, or 0 for the generic chunk loop.  Negative status on bad arguments. */
MSPL_API int mspl_class_order_shape(const uint8_t* lut, int num_classes, int num_target_classes);

/* ---- K1-lowres: K1 with the network's final upsample fused in (next-row component, SURVEY.md 8f-1) ------------------
 * Same outputs and semantics as mspl_fuse_sources, but source s hands over its logits BEFORE the final
 * F.interpolate(..., size=(out_h,out_w), mode='bilinear', align_corners=True) of model/segmentation/espdnet_ue.py:301-302:
 * main_logits[s] is (num_images, C_s, main_hw[2s], main_hw[2s+1]) and aux_logits[s] is (num_images, C_s, aux_hw[2s],
 * aux_hw[2s+1]); the kernel interpolates with ATen's upsample_bilinear2d source coordinates and weights, summing the four
 * taps in one fma chain (the interpolated logit can differ from ATen's nested form in the last ulp; the parity definition of this
 * row excuses labels where the top-2 probability margin is < 1e-5).  HBM traffic falls from
 * 8*sum(C_s) to ~1.25*sum(C_s) bytes per output pixel for the x2 / x4 heads of ESPDNetUE.
 * Needs every row length (main/aux width) to be a multiple of 4 and out_h*out_w % 4 == 0; returns MSPL_ERR_UNSUPPORTED when
 * the tile's source rows do not fit in shared memory (very wide images): upsample and call mspl_fuse_sources instead.
 * Pixels whose head maxima sit more than 16 logit units above the fused maximum (heads that disagree that strongly) or whose
 * fused logits exceed +-48 take a per-pixel slow path that re-interpolates the pixel's logits from global memory and evaluates
 * the softmax directly, like mspl_fuse_sources: the 1e-5 confidence tolerance holds for any input. */
MSPL_API int mspl_fuse_sources_lowres(int num_sources, const float* const* main_logits, const float* const* aux_logits,
                             const int* num_classes, const uint8_t* const* lut, const int* main_hw, const int* aux_hw,
                             int64_t num_images, int out_h, int out_w, int num_target_classes, int policy, int vote_t,
                             int ignore_label, int ds_rate, uint8_t* label, float* conf, float* unc,
                             float* const* kld_per_source, unsigned long long* class_hist,
                             unsigned long long* conf_hist, unsigned long long* marginal_count, void* stream);

/* ---- merge_outputs on hard labels ----------------------------------------------------------------
 * Replaces merge_outputs (uest_seg_multi_os.py:695-718; duplicate eval_label.py:76-100).
 * labels is (num_sources, num_pixels) u8 with values < K. */
MSPL_API int mspl_vote_labels(const uint8_t* labels, int num_sources, int64_t num_pixels, int num_target_classes,
                     int vote_t, int ignore_label, uint8_t* merged, void* stream);

/* ---- K2/K3: class-balanced thresholds and selection ([NEW]; CBST/CRST vestiges at
 * uest_seg_multi_os.py:88-107, 216-219 -- no reference implementation) --------------------------------
 * thresh[k] = 1.0 if floor(n_k*portion)==0 else the floor(n_k*portion)-th largest conf among the pixels of class k
 * with (pixel_index_in_image % ds_rate) == 0;  final = label if (label != ignore_label && conf >= thresh[label])
 * else ignore_label.  Exact order statistics, no sort, no host synchronisation.  Two protocols:
 *
 * (1) Bracketed -- what the pipeline runs: ONE pass over (label, conf), 6 B/pixel.
 *   hist (K*MSPL_RADIX_BINS u64, zeroed) holds the LINEAR confidence histogram: bin = clamp(floor(conf*2048), 0, 2047);
 *   mspl_fuse_sources accumulates it as `conf_hist`, or call mspl_conf_hist.            [all-reduce hist over ranks]
 *   mspl_bracket_select: per class, the bin holding the j-th largest conf -> bracket[k] = {lo, hi} (2K f32), the rank left
 *     inside the bin in `state` (mspl_radix_state_bytes, zeroed), kept_count[k] = n_k, thresh[k] = 1.0 for j == 0; zeroes hist.
 *     final_hist (K u64, NULLable, needs ignore_label in [0,K)): += the final class counts of the pixels settled outright,
 *     read off the histogram instead of being counted by the classify pass (pass final_hist = NULL there): class k keeps the
 *     pixels in the bins above its bracket bin, everything else counts as ignored until mspl_cand_apply patches it.  Only
 *     valid when the histogram was accumulated with ds_rate == 1 over exactly the pixels to be classified; `local_hist`
 *     is this rank's own (pre-all-reduce) copy of it, or NULL when `hist` was never all-reduced.
 *     The ignore class is never selected, so its threshold is left unresolved: thresh[ignore_label] = +inf (with the vote
 *     policies all its pixels have conf == 0 and would all be candidates); ignore_label = -1 resolves every class, which
 *     mspl_bracket_classify accepts only in thresholds-only mode (final_label, ignore_mask, final_hist all NULL).
 *   mspl_bracket_classify: conf >= hi: kept; conf < lo: ignored; otherwise the pixel index is appended to cand_index
 *     (u32, capacity num_pixels; *cand_count u64 zeroed by the caller) and provisionally ignored.  Writes final_label /
 *     ignore_mask (either may be NULL) and += final_hist (K u64, NULLable).  num_pixels < 2^32.
 *   for pass = 0, 1, 2: mspl_cand_hist_pass (radix histogram of the candidates only); [all-reduce hist];
 *     mspl_cand_select (zeroes hist; after pass 2 thresh is final).  final_hist (K u64, NULLable): after pass 2, the number
 *     of candidates that reach the threshold moves from final_hist[ignore_label] to final_hist[k] -- read off the (all-reduced)
 *     histograms, so the patch is the global one and identical on every rank; pass final_hist = NULL to mspl_cand_apply then.
 *     A class with floor(n_k*portion) == 0 (threshold 1.0) takes part in the passes only to count its conf >= 1.0 candidates.
 *   mspl_cand_apply: candidates with conf >= thresh[label] get their label back (final_label, ignore_mask, final_hist).
 *   mspl_cand_resolve: the three candidate passes, their selects and mspl_cand_apply in ONE launch, for callers with no
 *     all-reduce to run in between (a single rank): one 8-CTA thread-block cluster per class, per-CTA candidate cache in
 *     shared memory, histograms combined over distributed shared memory.  final_hist gets this call's own patch.  Returns
 *     MSPL_ERR_UNSUPPORTED (nothing launched) when the device cannot host an 8-CTA cluster of this kernel right now (e.g. a
 *     partitioned GPU): run the three mspl_cand_hist_pass / mspl_cand_select rounds and mspl_cand_apply instead.
 *
 * (2) Generic radix -- 3 full passes over the order-preserving fp32 key (11+11+10 bits), 16 B/pixel with
 *   mspl_apply_thresholds: zero `hist` and `state`; for pass = 0, 1, 2: mspl_radix_hist_pass; [all-reduce hist];
 *   mspl_radix_select (zeroes hist).  Independent of (1); the test-suite checks that both give the same bits. */
MSPL_API size_t mspl_radix_state_bytes(int num_target_classes);
MSPL_API int mspl_conf_hist(const uint8_t* label, const float* conf, int64_t num_pixels, int64_t pixels_per_image,
                   int num_target_classes, unsigned long long* hist, int ds_rate, void* stream);
MSPL_API int mspl_bracket_select(unsigned long long* hist, int num_target_classes, double portion, int ignore_label,
                        void* state, float* bracket, float* thresh, unsigned long long* kept_count,
                        const unsigned long long* local_hist, unsigned long long* final_hist, void* stream);
MSPL_API int mspl_bracket_classify(const uint8_t* label, const float* conf, const float* bracket, int64_t num_pixels,
                          int num_target_classes, int ignore_label, uint8_t* final_label, uint8_t* ignore_mask,
                          unsigned long long* final_hist, uint32_t* cand_index, unsigned long long* cand_count,
                          void* stream);
MSPL_API int mspl_cand_hist_pass(const uint8_t* label, const float* conf, const uint32_t* cand_index,
                        const unsigned long long* cand_count, int64_t pixels_per_image, int num_target_classes,
                        int pass, const void* state, unsigned long long* hist, int ds_rate, void* stream);
MSPL_API int mspl_cand_select(unsigned long long* hist, int num_target_classes, int pass, void* state, float* thresh,
                     unsigned long long* final_hist, int ignore_label, void* stream);
MSPL_API int mspl_cand_resolve(const uint8_t* label, const float* conf, const uint32_t* cand_index,
                      const unsigned long long* cand_count, int64_t pixels_per_image, int num_target_classes,
                      int ignore_label, int ds_rate, void* state, float* thresh, uint8_t* final_label,
                      uint8_t* ignore_mask, unsigned long long* final_hist, void* stream);
MSPL_API int mspl_cand_apply(const uint8_t* label, const float* conf, const float* thresh, const uint32_t* cand_index,
                    const unsigned long long* cand_count, int num_target_classes, int ignore_label,
                    uint8_t* final_label, uint8_t* ignore_mask, unsigned long long* final_hist, void* stream);
MSPL_API int mspl_radix_hist_pass(const uint8_t* label, const float* conf, int64_t num_pixels,
                         int64_t pixels_per_image, int num_target_classes, int pass, const void* state,
                         unsigned long long* hist, int ds_rate, void* stream);
MSPL_API int mspl_radix_select(unsigned long long* hist, int num_target_classes, int pass, double portion,
                      void* state, float* thresh, unsigned long long* kept_count, void* stream);

/* ---- K3 stand-alone: thresholding / ignore mask with given thresholds ([NEW]) ----------------------------
 * final = label if (label != ignore_label && conf >= thresh[label]) else ignore_label.
 * ignore_mask (u8, 1 where final == ignore_label) and final_hist (K u64, +=) may be NULL. */
MSPL_API int mspl_apply_thresholds(const uint8_t* label, const float* conf, const float* thresh,
                          int64_t num_pixels, int num_target_classes, int ignore_label,
                          uint8_t* final_label, uint8_t* ignore_mask, unsigned long long* final_hist,
                          void* stream);

/* ---- K4: fused rectified uncertainty-weighted CE, forward + backward ------------------------------
 * Replaces the training-loss expression at uest_seg_multi_os.py:1020-1023 (trav_mask_train.py:333-338):
 *   kld = PixelwiseKLD()(pred, pred_aux); loss = criterion(pred + 0.5*pred_aux, labels, kld) * alpha + kld.mean()
 * with criterion = UncertaintyWeightedSegmentationLoss (loss_fns/segmentation_loss.py:146-175).
 *   target         (num_pixels) int64, values in [0,K); anything else contributes like a zero-weight class
 *   class_weights  K f32 (device)          norm_pixels  the divisor N of the means (global pixel count under DP)
 *   out3           3 f32: {loss, mean of w*ce*exp(-kld) (un-scaled), mean kld}
 *   d_main, d_aux  gradients of `loss * grad_scale`, or both NULL for forward only
 *   workspace      mspl_uw_ce_workspace_bytes() bytes, zeroed once by the caller; left zeroed by each call */
MSPL_API size_t mspl_uw_ce_workspace_bytes(void);
MSPL_API int mspl_uw_ce_fwd_bwd(const float* main_logits, const float* aux_logits, const int64_t* target,
                       const float* class_weights, int64_t num_images, int num_classes,
                       int64_t pixels_per_image, float alpha, double norm_pixels, float grad_scale,
                       float* out3, float* d_main, float* d_aux, void* workspace, size_t workspace_bytes,
                       void* stream);
/* The same with the target given as uint8 class indices -- the format the label maps are generated, stored and
 * written to PNG in (uest_seg_multi_os.py:929-931), 1 byte per pixel instead of the 8 that torch's gather needs
 * (loss_fns/segmentation_loss.py:160-166): 81 instead of 88 algorithmic bytes per pixel.  Values >= K (e.g. 255)
 * contribute like a zero-weight class. */
MSPL_API int mspl_uw_ce_fwd_bwd_u8(const float* main_logits, const float* aux_logits, const uint8_t* target,
                          const float* class_weights, int64_t num_images, int num_classes,
                          int64_t pixels_per_image, float alpha, double norm_pixels, float grad_scale,
                          float* out3, float* d_main, float* d_aux, void* workspace, size_t workspace_bytes,
                          void* stream);
/* One training step's worth of the path in one launch: the loss above plus the counts MIOU.get_iou(pred, labels) makes of the
 * very same tensors straight after it (uest_seg_multi_os.py:1032, utilities/metrics/segmentation_miou.py:13-44):
 * pred = first-max argmax of main_logits, both sides cast to uint8 and shifted by one, pixels with shifted target 0 dropped.
 *   target      int64 (target_is_u8 == 0) or uint8 class indices
 *   iou_counts  3*K u64, += : [K intersection | K prediction | K mask] pixel counts (the metric's num_classes = K);
 *               NULL = loss only.  area_union = prediction + mask - intersection (+1e-6 on the host, :41). */
MSPL_API int mspl_uw_ce_step(const float* main_logits, const float* aux_logits, const void* target, int target_is_u8,
                    const float* class_weights, int64_t num_images, int num_classes, int64_t pixels_per_image,
                    float alpha, double norm_pixels, float grad_scale, float* out3, float* d_main, float* d_aux,
                    unsigned long long* iou_counts, void* workspace, size_t workspace_bytes, void* stream);
/* K4-lowres (next-row component, SURVEY.md 8f-1): the same loss on the tensors ESPDNetUE hands to its closing
 * F.interpolate(..., size=(out_h,out_w), mode='bilinear', align_corners=True) calls (model/segmentation/espdnet_ue.py:301-302):
 * main_lowres (num_images, K, main_h, main_w), aux_lowres (num_images, K, aux_h, aux_w), target (num_images, out_h, out_w).
 * The interpolation (ATen's upsample_bilinear2d arithmetic) and its transpose run inside the kernel; d_main_lowres /
 * d_aux_lowres receive the gradients w.r.t. the PRE-upsample tensors (both NULL = forward only); they are reproducible bit
 * for bit for row scale factors up to x4 at widths up to 480, to rounding beyond (fp32 adds of three tile shares).  Upsampling only
 * (source sizes <= output size); MSPL_ERR_UNSUPPORTED when one output row of gradients does not fit in shared memory. */
MSPL_API int mspl_uw_ce_lowres_fwd_bwd(const float* main_lowres, const float* aux_lowres, const int64_t* target,
                              const float* class_weights, int64_t num_images, int num_classes, int main_h, int main_w,
                              int aux_h, int aux_w, int out_h, int out_w, float alpha, double norm_pixels,
                              float grad_scale, float* out3, float* d_main_lowres, float* d_aux_lowres,
                              void* workspace, size_t workspace_bytes, void* stream);
MSPL_API int mspl_uw_ce_lowres_fwd_bwd_u8(const float* main_lowres, const float* aux_lowres, const uint8_t* target,
                                 const float* class_weights, int64_t num_images, int num_classes, int main_h, int main_w,
                                 int aux_h, int aux_w, int out_h, int out_w, float alpha, double norm_pixels,
                                 float grad_scale, float* out3, float* d_main_lowres, float* d_aux_lowres,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* In-place x *= *scale unless *scale == 1 (device scalar); lets autograd apply an upstream gradient
 * without a host sync. */
MSPL_API int mspl_scale_inplace(float* x, int64_t count, const float* scale, void* stream);

/* ---- Generic (un-fused) forms behind the reference's two nn.Modules -------------------------------- */
/* PixelwiseKLD.forward (loss_fns/segmentation_loss.py:181-189) and its vector-Jacobian product. */
MSPL_API int mspl_kld_fwd(const float* dist1, const float* dist2, int64_t n, int c, int64_t pixels_per_image,
                 float* kld, void* stream);
MSPL_API int mspl_kld_bwd(const float* dist1, const float* dist2, const float* grad_kld, int64_t n, int c,
                 int64_t pixels_per_image, float* grad1, float* grad2, void* stream);
/* UncertaintyWeightedSegmentationLoss.forward (loss_fns/segmentation_loss.py:155-175) and its backward.
 * loss is one f32; grad_loss is a device scalar; d_u may be NULL. Workspace as for mspl_uw_ce_fwd_bwd. */
MSPL_API int mspl_uw_loss_fwd(const float* pred, const int64_t* target, const float* u_weight,
                     const float* class_weights, int64_t n, int num_classes, int64_t pixels_per_image,
                     double norm_pixels, float* loss, void* workspace, size_t workspace_bytes, void* stream);
MSPL_API int mspl_uw_loss_bwd(const float* pred, const int64_t* target, const float* u_weight,
                     const float* class_weights, const float* grad_loss, int64_t n, int num_classes,
                     int64_t pixels_per_image, double norm_pixels, float* d_pred, float* d_u, void* stream);

/* ---- GPU MIOU.get_iou (next-row component, SURVEY.md 8f) ----------------------------------------------
 * Replaces MIOU.get_iou (utilities/metrics/segmentation_miou.py:13-44; call sites uest_seg_multi_os.py:1032, 1198,
 * eval_label.py:201), which moves pred/target to the CPU and runs torch.histc three times.
 * counts: 3*num_classes u64, += [area_inter | area_pred | area_mask]; area_union = pred + mask - inter + 1e-6 on the host.
 * Semantics are the reference's: uint8 casts, the "+1 so that 255 is 0" shift, pixels with shifted target 0 dropped,
 * class ids >= num_classes not counted.  num_classes <= 255. */
MSPL_API int mspl_miou_from_logits(const float* logits, const int64_t* target, int64_t n, int c, int64_t pixels_per_image,
                          int num_classes, unsigned long long* counts, void* stream);
MSPL_API int mspl_miou_from_labels(const void* pred, int pred_is_int64, const int64_t* target, int64_t num_pixels,
                          int num_classes, unsigned long long* counts, void* stream);

/* ---- NIDLoss (next-row component, SURVEY.md 8f-4) ---------------------------------------------------------
 * Replaces NIDLoss.forward + SoftArgMax (loss_fns/segmentation_loss.py:54-144; call site uest_seg_multi_os.py:1027-1030):
 * loss = (NID(grey camera image, soft-argmax label) - 0.95) * 20 from soft joint / marginal histograms, in one pass over the
 * pixels instead of image_bins sequential sigmoid-window passes and a (K x num_pixel)(num_pixel x C) product.
 *   camera (batch, 3, pixels) f32, label (batch, num_classes, pixels) f32 logits; image_bins <= 32, label_bins <= 8
 *   workspace: mspl_nid_workspace_bytes(), zeroed once by the caller; state: mspl_nid_state_bytes(), written by the forward
 *   (its first float is the loss) and read by the backward; d_label gets d(loss * *grad_loss)/d(label) (the camera image
 *   receives no gradient, as in the reference's use). */
MSPL_API size_t mspl_nid_workspace_bytes(void);
MSPL_API size_t mspl_nid_state_bytes(void);
MSPL_API int mspl_nid_fwd(const float* camera, const float* label, int64_t batch, int num_classes, int64_t pixels_per_image,
                 int image_bins, int label_bins, float bw_camera, float bw_label, void* workspace, size_t workspace_bytes,
                 void* state, void* stream);
MSPL_API int mspl_nid_bwd(const float* camera, const float* label, const float* grad_loss, int64_t batch, int num_classes,
                 int64_t pixels_per_image, int image_bins, int label_bins, float bw_camera, float bw_label, const void* state,
                 float* d_label, void* stream);

/* ---- in-training visualisation maps (next-row component, SURVEY.md 8f-4) ----------------------------------
 * Replaces the device half of in_training_visualization_img (utilities/utils.py:76-133; call sites uest_seg_multi_os.py:1060-1066,
 * 1211-1215): predictions = argmax_c(main + 0.5*aux) (first maximal index; aux may be NULL: argmax of main), kld =
 * PixelwiseKLD(main, aux), kld_max_key (u32, zeroed by the caller) = order-preserving key of max(kld) over the batch;
 * mspl_kld_heatmap then writes -kld / max(kld) + 1 (IEEE division, :92) without the reference's host round trip, and
 * mspl_label_colors is LongTensorToRGBPIL (:188-237) for a batch: labels (n, pixels) int64 -> rgb (n, 3, pixels) u8 through a
 * HOST table of num_colors (<= 256) RGB triples; labels outside the table give black. */
MSPL_API int mspl_prediction_maps(const float* main_logits, const float* aux_logits, int64_t n, int c, int64_t pixels_per_image,
                         int64_t* labels, float* kld, unsigned int* kld_max_key, void* stream);
MSPL_API int mspl_kld_heatmap(const float* kld, int64_t count, const unsigned int* kld_max_key, float* heat, void* stream);
MSPL_API int mspl_label_colors(const int64_t* labels, int64_t n, int64_t pixels_per_image, const uint8_t* colors_rgb,
                      int num_colors, uint8_t* rgb, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSPL_B200_H */
