/*
 * tiseg_b200.h — C ABI of libtiseg_b200.so: the sm_100a (B200) implementation of the test-time
 * instance pipeline (post-process + evaluation) of clownrat6/Tissue-Image-Segmentation (`tiseg`).
 *
 * This is the drop-in boundary.  Every entry point is batched over N independent tiles
 * ([N, H, W] C-contiguous arrays, row pitch W), stream-ordered on the context's CUDA stream, and
 * takes plain pointers and sizes.  A pointer may be a DEVICE pointer (zero-copy, asynchronous,
 * nothing is synchronised) or a HOST pointer (numpy buffer: the library stages it host<->device
 * on the context stream and synchronises before returning) — detected per pointer with
 * cudaPointerGetAttributes.  There is NO CPU implementation behind any of them: without a CUDA
 * device tiseg_create fails and nothing else can be called.
 *
 * Each function names the reference code (file:line under the reference repository) it replaces.
 * All return TISEG_OK (0) or an error code; tiseg_last_error() gives the message (thread-local).
 *
 * Errors that only a kernel can detect (an instance id outside [0, max(H*W+1, 65536))) are raised on the device.
 * A call with a host output synchronises anyway and reports them itself; a call with device outputs only returns
 * before execution, and the error is reported by the next call on the context that synchronises (any call with a
 * host output, or tiseg_synchronize).  No call decides anything on the host in the middle of its kernels, except
 * tiseg_reconstruction_erosion_u8 / tiseg_postproc_dist_lambda_typed with lamb > 0 (iteration to a fixed point).
 */
#ifndef TISEG_B200_H
#define TISEG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TISEG_OK 0
#define TISEG_ERR_CUDA 1   /* a CUDA runtime call or kernel launch failed                     */
#define TISEG_ERR_ARG 2    /* bad argument (null pointer, non-positive size, unknown option)  */
#define TISEG_ERR_NOGPU 3  /* no CUDA device: there is no CPU fallback                        */
#define TISEG_ERR_LIMIT 4  /* a data-dependent limit was exceeded (instance id out of range)  */

/* Element type of the network outputs (logits, distance / HV / foreground maps, direction and point heads) handed to
 * the entries whose second argument is `dtype`: tiseg_softmax_argmax_typed, tiseg_softmax_argmax_tta_typed,
 * tiseg_tta_mean_typed, tiseg_postproc_dist_lambda_typed, tiseg_postproc_hover_ex, tiseg_cdnet_refine_typed,
 * tiseg_mtcdnet_refine_typed, tiseg_cdnet_refine_tta_typed and tiseg_mtcdnet_refine_tta_typed.  All network inputs of one call share it.  Half-precision inputs are converted to fp32 as
 * they are loaded and the arithmetic after the load is the fp32 path's, so a call fed fp16 / bf16 returns the bits the
 * same call returns for the fp32 upcast of its inputs, at half the input bytes (a host buffer crosses PCIe at 2 B per
 * element).  Outputs keep their types: probabilities and means stay fp32.  Another code returns TISEG_ERR_ARG. */
#define TISEG_DTYPE_F32 0
#define TISEG_DTYPE_F16 1
#define TISEG_DTYPE_BF16 2

typedef struct tiseg_ctx tiseg_ctx;

/* ---- context -------------------------------------------------------------------------------- */
int tiseg_create(tiseg_ctx** out, int device);
int tiseg_destroy(tiseg_ctx* ctx);
/* run on an existing cudaStream_t (e.g. torch's current stream; NULL = the legacy default stream).
 * A fresh context owns a private non-blocking stream until this is called. */
int tiseg_set_stream(tiseg_ctx* ctx, void* cuda_stream);
int tiseg_synchronize(tiseg_ctx* ctx);
const char* tiseg_last_error(void);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
long long tiseg_launch_count(tiseg_ctx* ctx);
int tiseg_version(void);
/* hash of the source tree (csrc/, this header, compiler flags) the library was built from; the Python loader compares it
 * with the sources next to it and refuses a stale binary */
const char* tiseg_build_hash(void);
/* optional per-kernel CUDA-event timing (bench.py's roofline leg): enable, run, then read one
 * "kernel_name launches total_ms" line per kernel (aggregated and reset). */
int tiseg_timing_enable(tiseg_ctx* ctx, int on);
int tiseg_timing_report(tiseg_ctx* ctx, char* buf, int cap);

/* ---- A1: softmax / TTA mean / argmax ---------------------------------------------------------
 * tiseg/models/segmentors/base.py:321-339 (F.softmax per TTA variant, sum/len, resize == identity
 * at ori_hw) followed by `sem_logit.argmax(dim=1)` (unet.py:62, dist.py:266, hovernet.py:271).
 * logits [N, T, C, H, W] of element type `dtype` (TISEG_DTYPE_*); prob [N, C, H, W] fp32 or NULL; cls [N, H, W] uint8
 * or NULL (first maximum wins, like torch.argmax). */
int tiseg_softmax_argmax_typed(tiseg_ctx* ctx, int dtype, const void* logits, int N, int T, int C, int H, int W,
                               float* prob, uint8_t* cls);

/* ---- the step before A1, fused: window stitch + TTA reverse + softmax + mean + argmax -------------------------
 * Replaces split_inference's canvas (base.py:255-295), reverse_tta_transform (base.py:365-381) and the softmax /
 * mean / argmax of A1 with ONE pass that reads each logit once from the tensors the network produced.
 * logits: per tile, the T variants back to back; variant t was computed on tta_transform(img, rotate_degrees[t],
 * flips[t]) (flips: 0 none, 1 horizontal, 2 vertical, 3 diagonal) and is either the whole [C, Ht, Wt] output
 * (window = 0; (Ht, Wt) = (W, H) for 90/270 degrees) or its windows [My*Mx, C, window, window] in the row-major
 * order split_inference visits them.  tiseg_tta_input_elems gives the elements per tile.  H, W: the original image. */
long long tiseg_tta_input_elems(int T, int C, int H, int W, const int* rotate_degrees, int window, int overlap);
int tiseg_softmax_argmax_tta_typed(tiseg_ctx* ctx, int dtype, const void* logits, int N, int T, int C, int H, int W,
                                   const int* rotate_degrees, const int* flips, int window, int overlap,
                                   float* prob, uint8_t* cls);

/* The plain (no softmax) TTA mean of a regression head with the same stitch + reverse-transform indexing:
 * `sum(dist_logit_list) / len(dist_logit_list)` of dist.py:398-410; hovernet.py:406 keeps variant 0 only (T = 1).
 * maps laid out like the logits of tiseg_softmax_argmax_tta_typed; mean_out [N, C, H, W]. */
int tiseg_tta_mean_typed(tiseg_ctx* ctx, int dtype, const void* maps, int N, int T, int C, int H, int W,
                         const int* rotate_degrees, const int* flips, int window, int overlap, float* mean_out);

/* ---- A5 / A6 / A15: connected-component labelling ---------------------------------------------
 * skimage.measure.label(img, background=bg, connectivity=conn) (unet.py:85, dist.py:107,123,
 * multi_task_unet.py:101, inst_metrics.py:12-13,142-143) and scipy.ndimage.label (hovernet.py:296,358;
 * conn=1).  Equal-valued neighbouring non-background pixels are connected; conn 1 = 4-neighbourhood,
 * 2 = 8-neighbourhood; ids 1..K in raster order of each component's first pixel.  Because the ids are
 * canonical, this is also re_instance (datasets/utils/instance_semantic.py:5-15) composed with the
 * label call inside every metric.  img / out [N,H,W] int32; count [N] int32 (K per tile) or NULL. */
int tiseg_label(tiseg_ctx* ctx, const int32_t* img, int N, int H, int W, int32_t background,
                int connectivity, int32_t* out, int32_t* count);
/* same on a uint8 image (masks, class maps) */
int tiseg_label_u8(tiseg_ctx* ctx, const uint8_t* img, int N, int H, int W, int32_t background,
                   int connectivity, int32_t* out, int32_t* count);
/* re_instance alone (instance_semantic.py:5-15): sorted unique non-zero ids -> 1..K, order-preserving */
int tiseg_re_instance(tiseg_ctx* ctx, const int32_t* img, int N, int H, int W, int32_t* out, int32_t* count);

/* ---- A3: scipy.ndimage.binary_fill_holes (unet.py:83, hovernet.py:355, multi_task_unet.py:95) ---
 * mask / out [N,H,W] uint8 (non-zero = foreground; out is 0/1). */
int tiseg_fill_holes(tiseg_ctx* ctx, const uint8_t* mask, int N, int H, int W, uint8_t* out);

/* ---- A4: skimage.morphology.remove_small_objects ------------------------------------------------
 * bool input (unet.py:84): components of `connectivity` (1 -> 4-neighbourhood), size < min_size zeroed. */
int tiseg_remove_small_objects(tiseg_ctx* ctx, const uint8_t* mask, int N, int H, int W, int min_size,
                               int connectivity, uint8_t* out);
/* int input (hovernet.py:297,359): the values are the component ids; ids with count < min_size zeroed. */
int tiseg_remove_small_labels(tiseg_ctx* ctx, const int32_t* lab, int N, int H, int W, int min_size,
                              int32_t* out);

/* ---- A7: skimage.morphology.dilation / erosion on label images (unet.py:86, dist.py:88-94) -------
 * footprint 0 = disk(radius) {x^2+y^2<=r^2}, 1 = square(2*radius+1); out-of-image taps ignored
 * (== ndimage 'reflect' for these symmetric footprints).  radius <= 3. */
int tiseg_dilate_labels(tiseg_ctx* ctx, const int32_t* lab, int N, int H, int W, int footprint,
                        int radius, int32_t* out);
int tiseg_erode_labels(tiseg_ctx* ctx, const int32_t* lab, int N, int H, int W, int footprint,
                       int radius, int32_t* out);

/* ---- A2: UNet-family postprocess ----------------------------------------------------------------
 * unet.py:71-93, micronet.py:185-207 (radius 1); cunet.py:70-93, cdnet.py:96-119, fullnet.py:190-213,
 * cmicronet.py:186-209 (radius 3, edge_id = num_classes zeroed IN PLACE in `cls`); dcan.py:193-217.
 * cls [N,H,W] uint8 class map (argmax output; mutated when edge_id >= 0); for each class id present,
 * ascending: fill holes -> remove_small_objects(5) -> label -> dilation(disk(radius)) -> overwrite.
 * sem_out [N,H,W] uint8, inst_out [N,H,W] int32. max_class = largest class id that can occur (<= 63);
 * edge_id < 0 = none; kill (NULL or [N,H,W] uint8) = DCAN's contour map: cls[kill > 0] = 0 in place
 * (dcan.py:196). */
int tiseg_postproc_unet(tiseg_ctx* ctx, uint8_t* cls, int N, int H, int W, int max_class, int radius,
                        int edge_id, const uint8_t* kill, uint8_t* sem_out, int32_t* inst_out);

/* ---- A10: skimage.segmentation.watershed(image, markers, mask) -----------------------------------
 * connectivity 1, compactness 0, no lines (dist.py:124, hovernet.py:361).  Ordered (value, age) flood,
 * 4-neighbours visited up/left/right/down, label-at-push; seeds ordered by (value, flat index).
 * image [N,H,W] uint8 / fp64; markers int32; mask uint8 (NULL = all); out int32. */
int tiseg_watershed_u8(tiseg_ctx* ctx, const uint8_t* image, const int32_t* markers, const uint8_t* mask,
                       int N, int H, int W, int32_t* out);
int tiseg_watershed_f64(tiseg_ctx* ctx, const double* image, const int32_t* markers, const uint8_t* mask,
                        int N, int H, int W, int32_t* out);

/* ---- A8: DIST postprocess (dist.py:275-284 -> dynamic_watershed_alias :114-129) ---------------------
 * dist [N,H,W] raw distance-head output of element type `dtype` (TISEG_DTYPE_*), read once, by the step that truncates
 * it to levels; inst_out [N,H,W] int32 (the reference returns int64 with the same values).  Optional debug outputs
 * (NULL to skip): markers int32, ws int32 (raw flood).  lamb is the paper's p1 ("lamb" of dynamic_watershed_alias,
 * dist.py:114; the reference's test path passes 0.0, dist.py:281): markers and flood levels come from
 * Hrecons = reconstruction_by_erosion(min(255, I + lamb), I).  lamb > 0 runs an iterative reconstruction that
 * synchronises with the host between sweeps. */
int tiseg_postproc_dist_lambda_typed(tiseg_ctx* ctx, int dtype, const void* dist, int N, int H, int W, int lamb,
                                     int32_t* inst_out, int32_t* markers_out, int32_t* ws_out);

/* ---- A9: skimage.morphology.reconstruction(seed, mask, method='erosion') on uint8 images, 3x3 footprint
 * (dist.py:56).  seed is clamped from below by mask.  Synchronises with the host between sweeps. */
int tiseg_reconstruction_erosion_u8(tiseg_ctx* ctx, const uint8_t* seed, const uint8_t* mask, int N, int H, int W,
                                    uint8_t* out);

/* ---- A11: HoVer-Net post-process (hovernet.py:283-365, hover_post_proc(fore_map, hv_map, fx, scale_factor)) ----
 * fore_map [N,H,W] (softmax channel 1 of the foreground head), hv_map [N,H,W,2] HWC (horizontal, vertical) as the
 * reference passes them after permute(0,2,3,1), both of element type `dtype` (TISEG_DTYPE_*); with scale_factor 2 the
 * resize reads them and the chain after it runs on fp32.  scale_factor: 1 (the MoNuSeg / CoNSeP configs) or 2 (the
 * CoNIC config: cv2.resize x2 bilinear in, the whole chain at 2H x 2W, INTER_NEAREST back).
 * inst_out [N,H,W] int32.  Optional debug outputs (NULL to skip), at the SCALED size [N, sH, sW]: blb uint8,
 * dist fp64 (the flooded image), marker int32.
 * fx is given as the two integers the reference derives from it: ksize = int(20 * fx + 1), the Sobel kernel
 * size (odd, 1..31: the sizes cv2.Sobel accepts; ksize 1 is the 3-tap derivative without smoothing), and
 * obj_size = ceil(10 * fx^2), the size below which a marker is dropped (>= 0; 0 and 1 drop none); the reference's
 * default fx = 1 is ksize 21, obj_size 10.  The blb mask keeps its fixed min_size 10, as in the reference.
 * TISEG_ERR_ARG for an even or out-of-range ksize, a negative obj_size or a scale_factor other than 1 or 2. */
int tiseg_postproc_hover_ex(tiseg_ctx* ctx, int dtype, const void* fore_map, const void* hv_map, int N, int H, int W,
                            int scale_factor, int ksize, int obj_size, int32_t* inst_out, uint8_t* blb_out,
                            double* dist_out, int32_t* marker_out);

/* ---- A12: CDNet direction-guided refinement ----------------------------------------------------------------
 * generate_direction_differential_map(dir_map, 9) (tiseg/models/utils/direct_diff_map.py:95-167):
 * dir_map [N,H,W] uint8 (0 = background, 1..8 directions) -> dd [N,H,W] fp32 in {0, 0.5, 1}. */
int tiseg_ddm(tiseg_ctx* ctx, const uint8_t* dir_map, int N, int H, int W, float* dd);
/* The tail of CDNet.inference after the CNN (cdnet.py:183-217) including _ddm_enhencement (:354-367):
 * sem_logits [N,T,C,H,W], dir_logits [N,T,D=9,H,W], point_logits [N,T,1,H,W] raw head outputs of the T TTA
 * variants, of element type `dtype` (TISEG_DTYPE_*).  Outputs (any may be NULL): sem_prob_out [N,C,H,W] refined fp32
 * probabilities, cls_out [N,H,W] their argmax, dir_map_out [N,H,W] direction map of variant 0, dd_out [N,H,W] mean
 * DDM. */
int tiseg_cdnet_refine_typed(tiseg_ctx* ctx, int dtype, const void* sem_logits, const void* dir_logits,
                             const void* point_logits, int N, int T, int C, int D, int H, int W, int if_ddm,
                             float* sem_prob_out, uint8_t* cls_out, uint8_t* dir_map_out, float* dd_out);

/* _ddm_enhencement alone, IN PLACE on sem_prob [N,C,H,W]: mode 0 = CDNet (cdnet.py:354-367), mode 1 = MultiTaskCDNet
 * (multi_task_cdnet.py:548-564).  dd [N,H,W] mean DDM, point [N,H,W] TTA-mean point map (channel 0 of point_logit). */
int tiseg_ddm_enhance(tiseg_ctx* ctx, float* sem_prob, const float* dd, const float* point, int N, int C, int H, int W, int mode);
/* The tail of MultiTaskCDNet.inference after the CNN (multi_task_cdnet.py:262-330; D == 9: use_regression = False;
 * D == 1: use_regression = True, dir_logits [N,T,1,H,W] is the angle head in radians and every variant's direction map
 * is 1 + the class of the clamped angle with eight angles, 0 on the background of the mean tc map, :304-315): softmax +
 * TTA mean of the three-class (tc) and semantic heads, TTA mean of the point head, per variant dir[:,0] *= tc[:,0] ->
 * argmax -> DDM, mean DDM, its own _ddm_enhencement (:548-564) on the tc probabilities.  tc_logits [N,T,Ctc,H,W],
 * sem_logits [N,T,Csem,H,W], dir_logits [N,T,9,H,W], point_logits [N,T,1,H,W], the four heads of element type `dtype`
 * (TISEG_DTYPE_*).  Outputs (any may be NULL): tc_prob_out [N,Ctc,H,W] refined, tc_cls_out / sem_cls_out [N,H,W] the
 * argmax maps postprocess consumes (:209-213), sem_prob_out [N,Csem,H,W], dir_map_out [N,H,W] direction map of
 * variant 0, dd_out [N,H,W]. */
int tiseg_mtcdnet_refine_typed(tiseg_ctx* ctx, int dtype, const void* tc_logits, const void* sem_logits,
                               const void* dir_logits, const void* point_logits, int N, int T, int Ctc, int Csem, int D,
                               int H, int W, int if_ddm, float* tc_prob_out, uint8_t* tc_cls_out, float* sem_prob_out,
                               uint8_t* sem_cls_out, uint8_t* dir_map_out, float* dd_out);

/* The same two tails fed the RAW outputs of the TTA variants, with the window stitch (base.py:255-295) and
 * reverse_tta_transform (base.py:365-381) fused into the loads, like tiseg_softmax_argmax_tta_typed: every head is laid
 * out like its logits (per tile, the T <= 16 variants back to back, whole transformed images when window == 0, else
 * their windows in the order split_inference visits them), tiseg_tta_input_elems(T, that head's channels, H, W, ...)
 * elements per tile.  H, W: the original image.  The semantic / three-class heads are averaged by the softmax TTA kernel;
 * the direction, angle (D == 1) and point heads are staged through shared memory one 32 x 32 tile at a time, so every
 * head element is read once, coalesced for all eight transforms.  Outputs and arguments otherwise as the entries above,
 * and equal to them (bit for bit) on the reverse-transformed, stitched heads; dir_map_out is variant 0's map in the
 * original orientation. */
int tiseg_cdnet_refine_tta_typed(tiseg_ctx* ctx, int dtype, const void* sem, const void* dir, const void* point, int N,
                                 int T, int C, int D, int H, int W, const int* rotate_degrees, const int* flips,
                                 int window, int overlap, int if_ddm, float* sem_prob_out, uint8_t* cls_out,
                                 uint8_t* dir_map_out, float* dd_out);
int tiseg_mtcdnet_refine_tta_typed(tiseg_ctx* ctx, int dtype, const void* tc, const void* sem, const void* dir,
                                   const void* point, int N, int T, int Ctc, int Csem, int D, int H, int W,
                                   const int* rotate_degrees, const int* flips, int window, int overlap, int if_ddm,
                                   float* tc_prob_out, uint8_t* tc_cls_out, float* sem_prob_out, uint8_t* sem_cls_out,
                                   uint8_t* dir_map_out, float* dd_out);

/* ---- A13: align_foreground (tiseg/models/utils/postprocess.py:123-155) -----------------------------------
 * Ordered multi-source BFS growing the labels of `pred` into `foreground` (8-neighbourhood, first claimant
 * wins, at most time-1 rounds).  pred [N,H,W] int32 is modified in place; foreground uint8. */
int tiseg_align_foreground(tiseg_ctx* ctx, int32_t* pred, const uint8_t* foreground, int N, int H, int W, int time);

/* Multi-task postprocess (multi_task_unet.py:84-106, multi_task_cunet.py:86-108, multi_task_cdnet.py:222-243):
 * sem canvas = per class remove_small_objects(5) then binary_fill_holes; instances = measure.label(inner,
 * connectivity=1) with the edge class (edge_id, < 0 = none) zeroed, grown by align_foreground(., canvas>0, time).
 * inner / sem uint8; canvas_out uint8; inst_out int32. */
int tiseg_postproc_multitask(tiseg_ctx* ctx, const uint8_t* inner, const uint8_t* sem, int N, int H, int W,
                             int max_class, int edge_id, int time, uint8_t* canvas_out, int32_t* inst_out);

/* ---- A16 / A17: pre_eval_bin_aji + pre_eval_bin_pq (inst_metrics.py:10-92, 138-229) ---------------
 * pred / gt [N,H,W] int32 instance maps with arbitrary ids (the relabelling the reference does with
 * re_instance + measure.label is done inside).  aji [N,2] fp64 = (overall_inter, overall_union);
 * pq [N,4] fp64 = (tp, fp, fn, iou_sum).  Either output may be NULL.  match_iou is pre_eval_bin_pq's (reference
 * default 0.5; a pair matches when iou > match_iou, inst_metrics.py:197-203); it must be >= 0.5 (the Hungarian branch
 * for match_iou < 0.5 is reached by no caller of the reference and is not built). */
int tiseg_pair_metrics_bin_iou(tiseg_ctx* ctx, const int32_t* pred, const int32_t* gt, int N, int H, int W, double match_iou,
                               double* aji, double* pq);
/* the same with the ground truth shipped as uint16 (ids below 65536: every dataset the reference converts,
 * tools/convert_dataset/*.py): half the host-to-device bytes of the largest evaluation input */
int tiseg_pair_metrics_bin_u16gt(tiseg_ctx* ctx, const int32_t* pred, const uint16_t* gt, int N, int H, int W, double match_iou,
                                 double* aji, double* pq);

/* ---- A18: CoNIC multi-class evaluation (conic.py:165-188) -----------------------------------------------
 * assign_sem_class_to_insts (datasets/utils/instance_semantic.py:68-93) on both sides, then pre_eval_aji /
 * pre_eval_pq (inst_metrics.py:95-135, 232-280), and optionally the binary records, from ONE pair table.
 * *_inst int32 (ids < max(H*W+1, 65536)), *_sem uint8, C = number of classes incl. background.
 * aji [N,C,2], pq [N,C,4] fp64 with slot 0 = the reference's class-0 slot (dropped by reduce_zero_label);
 * bin_aji [N,2], bin_pq [N,4] as tiseg_pair_metrics_bin_iou with match_iou 0.5.  Any output may be NULL. */
int tiseg_pair_metrics_multiclass(tiseg_ctx* ctx, const int32_t* pred_inst, const uint8_t* pred_sem,
                                  const int32_t* gt_inst, const uint8_t* gt_sem, int N, int H, int W, int C,
                                  double* aji, double* pq, double* bin_aji, double* bin_pq);
/* the same with the ground-truth instance map as uint16 (ids below 65536), read as it is by every kernel of the ground-truth
 * side (equality planes, largest id, class histogram, component classes): 3 B/px of ground truth (instances + classes)
 * instead of 5.  The results are those of the int32 upcast, bit for bit; the prediction stays int32. */
int tiseg_pair_metrics_multiclass_u16gt(tiseg_ctx* ctx, const int32_t* pred_inst, const uint8_t* pred_sem,
                                        const uint16_t* gt_inst, const uint8_t* gt_sem, int N, int H, int W, int C,
                                        double* aji, double* pq, double* bin_aji, double* bin_pq);

/* assign_sem_class_to_insts (datasets/utils/instance_semantic.py:68-93) as a table: table_out [N, VM] uint8 with
 * VM = max(H*W + 1, 65536); entry v = class of instance id v (first argmax over the classes >= 1 of its pixel counts,
 * 0 if it has no non-background pixel; id 0 is class 0), 255 = the id does not occur. */
int tiseg_assign_sem_class(tiseg_ctx* ctx, const int32_t* inst, const uint8_t* sem, int N, int H, int W, int C,
                           uint8_t* table_out);
/* the same for a uint16 instance map (read as it is; the table is that of the int32 upcast) */
int tiseg_assign_sem_class_u16(tiseg_ctx* ctx, const uint16_t* inst, const uint8_t* sem, int N, int H, int W, int C,
                               uint8_t* table_out);

/* ---- A19: pre_eval_all_semantic_metric (sem_metrics.py:16-53) --------------------------------------
 * pred / gt [N,H,W] uint8; counts [N, 5, C] int64 = TP, FP, FN, Pred, GT per class (TN derived on the
 * host as N_valid - (TP+FP+FN)); valid [N] int64 = pixels with gt != ignore_index. */
int tiseg_sem_counts(tiseg_ctx* ctx, const uint8_t* pred, const uint8_t* gt, int N, int H, int W, int C,
                     int ignore_index, int64_t* counts, int64_t* valid);

/* ---- mudslide_watershed(seg, dir_graph, fore) (models/utils/postprocess.py:158-181 with get_graph_degree :12-28 and
 * prepare :31-120; exported by the reference, enabled by no shipped config).  seg / fore [N,H,W] uint8 masks,
 * dir_graph [N,H,W] uint8 direction labels 0..8, MODIFIED IN PLACE as the reference does (small direction regions
 * cleared, directions filled in by the ordered pass).  pred_out, boundary_out uint8 masks. */
int tiseg_mudslide_watershed(tiseg_ctx* ctx, const uint8_t* seg, uint8_t* dir_graph, const uint8_t* fore, int N, int H,
                             int W, uint8_t* pred_out, uint8_t* boundary_out);

/* ---- A14: distance transforms (label generation: datasets/ops/distance_map.py:93, direction_map.py:167,179,
 * unet_map.py:72, utils/direction_calculation.py:164; losses/surface_loss.py:7) -------------------------------
 * mask [N,H,W] uint8 (non-zero = object).  edt: fp64 Euclidean distance to the nearest zero pixel
 * (scipy.ndimage.distance_transform_edt, bit-identical: sqrt of the exact integer squared distance);
 * cdt: int32 chessboard distance (scipy.ndimage.distance_transform_cdt, default metric; -1 when a tile has no zero). */
int tiseg_distance_transform_edt(tiseg_ctx* ctx, const uint8_t* mask, int N, int H, int W, double* out);
int tiseg_distance_transform_cdt(tiseg_ctx* ctx, const uint8_t* mask, int N, int H, int W, int32_t* out);

/* ---- train-time label generation (SURVEY §8f rank 4) -----------------------------------------------------------
 * gen_instance_hv_map (datasets/ops/hv_map.py:18-97): inst [N,H,W] int32 -> hv_out [N,H,W,2] fp32 (x map, y map).
 * The per-instance chessboard distance of DistanceLabelMake.__call__ (datasets/ops/distance_map.py:59-110), on an
 * instance map already passed through its _fix_inst: dist_out [N,H,W] fp32, divided by the instance maximum when
 * inst_norm != 0.  Instance ids must be < max(H*W+1, 65536) (deferred error otherwise). */
int tiseg_gen_hv_map(tiseg_ctx* ctx, const int32_t* inst, int N, int H, int W, float* hv_out);
/* gen_instance_hv_map of a uint16 instance map, read as it is: hv_out is that of the int32 upcast, bit for bit */
int tiseg_gen_hv_map_u16(tiseg_ctx* ctx, const uint16_t* inst, int N, int H, int W, float* hv_out);
int tiseg_instance_distance_map(tiseg_ctx* ctx, const int32_t* inst, int N, int H, int W, int inst_norm, float* dist_out);
/* _fix_inst, the first step of every label maker (distance_map.py:41-57, bound_map.py:18-33, unet_map.py:36-51,
 * direction_map.py:17-32): per id drop the 4-connected pieces under 5 px, split into 8-connected pieces, renumber
 * 1..K in (id, raster order of the piece) order. */
int tiseg_fix_inst(tiseg_ctx* ctx, const int32_t* inst, int N, int H, int W, int32_t* out);
/* _fix_inst of a uint16 instance map: both labellings read the ids at 2 B/px; out is int32 and equals that of the int32
 * upcast */
int tiseg_fix_inst_u16(tiseg_ctx* ctx, const uint16_t* inst, int N, int H, int W, int32_t* out);
/* BoundLabelMake.__call__ after _fix_inst (bound_map.py:62-88): sem_out = sem with unlabelled pixels zeroed (may be
 * NULL), sem_w_bound_out = sem_out with edge_id on dilation(diamond(radius_dilate)) & ~erosion(diamond(radius_erode))
 * of every instance. */
int tiseg_bound_label(tiseg_ctx* ctx, const uint8_t* sem, const int32_t* inst, int N, int H, int W, int edge_id,
                      int radius_dilate, int radius_erode, uint8_t* sem_out, uint8_t* sem_w_bound_out);

/* UNetLabelMake after _fix_inst (unet_map.py:53-98, 111-119 with wc = None): inner_out = every instance eroded by
 * diamond(1) (_remove_1px_boundary); wmap_out [N,H,W] fp64 = 1 + w0 * exp(-((d1 + d2) / sigma)^2 / 2) on the pixels
 * outside the eroded instances, d1 / d2 = Euclidean distance to the nearest / second nearest eroded instance (1
 * everywhere when fewer than two instances remain). */
int tiseg_unet_weight_map(tiseg_ctx* ctx, const int32_t* inst, int N, int H, int W, double w0, double sigma,
                          int32_t* inner_out, double* wmap_out);

/* DirectionLabelMake.__call__ after _fix_inst, to_center = True (datasets/ops/direction_map.py:36-193; the per-pixel
 * centerness search of datasets/utils/center_calculation.py:8-54, the 11x11 gradient of gradient_calculation.py:8-50, the
 * angle binning of direction_calculation.py:60-121) on a batch of fixed instance maps:
 *   dist_out  [N,H,W] fp32  sqrt(1 - d(centre) / (max d + 1e-7)) * 10 inside the instances     (data['dist_gt'])
 *   point_out [N,H,W] fp32  gaussian_filter(255 at the centres, sigma) with the given kernel    (data['point_gt'])
 *   dir_out   [N,H,W] u8    0 = background, 1 + direction class (num_angles classes)            (data['dir_gt'])
 *   reg_dir_out [N,H,W] fp32 angle of the gradient in [0, 2 pi)                                 (data['reg_dir_gt'])
 *   weight_out [N,H,W] fp32 dilation(ddm(dir) * (10 - dist), disk(1)) * 2 + 1; NULL unless num_angles == 8
 * gauss_weights: HOST array of 2 * gauss_radius + 1 doubles (scipy's _gaussian_kernel1d(sigma, 0, radius)).
 * Centres, dist_out and point_out follow the reference bit for bit; the gradient is a float32 sum whose order in the
 * reference is torch's convolution backend's, so angles (and classes on a bin edge) agree to float tolerance. */
int tiseg_direction_labels(tiseg_ctx* ctx, const int32_t* inst, int N, int H, int W, int num_angles,
                           const double* gauss_weights, int gauss_radius, float* dist_out, float* point_out,
                           uint8_t* dir_out, float* reg_dir_out, float* weight_out);

#ifdef __cplusplus
}
#endif
#endif
