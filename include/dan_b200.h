/*
 * dan_b200 -- C ABI of the Blackwell-native (sm_100a) anchor hot path of HiKapok/DAN.
 *
 * This is the drop-in boundary.  Everything the reference reaches for this path
 * through TensorFlow graph ops and the `SmallMiningMatch` custom op
 * (cpp/ExtraLib/build/libextra_lib.so, loaded by utility/custom_op.py:33-48) is
 * exposed here as plain `extern "C"` functions taking device pointers, sizes and
 * a cudaStream_t (passed as void*).  No C++ types, no exceptions, no torch types.
 *
 * Conventions
 *   - every function returns 0 on success or a negative DAN_ERR_* code; the
 *     message is available from dan_last_error() (thread local);
 *   - the caller owns every buffer; the library only touches the caller-provided
 *     workspace (size from the matching dan_*_workspace_bytes());
 *   - all pointers are DEVICE pointers unless the name starts with `h_`;
 *   - `stream` is a cudaStream_t; work is enqueued, never synchronised, so every
 *     call is CUDA-graph capturable;
 *   - boxes are fp32 [ymin, xmin, ymax, xmax]; the +1 (inclusive pixel) convention
 *     of utility/anchor_manipulator.py is used everywhere except inside NMS
 *     (tf.image.non_max_suppression has no +1);
 *   - the library is stateless and re-entrant across host threads / streams
 *     (the reference op is called concurrently from 36-48 queue threads,
 *     train_sfd.py:37-39); two concurrent calls must not share a workspace.
 *
 * Reference citations are relative to /root/reference.
 */
#ifndef DAN_B200_H_
#define DAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAN_B200_VERSION 100

#define DAN_OK 0
#define DAN_ERR_INVALID_ARGUMENT (-1) /* mirrors errors::InvalidArgument of the TF op */
#define DAN_ERR_WORKSPACE (-2)        /* workspace missing or too small                */
#define DAN_ERR_CUDA (-3)             /* a CUDA runtime call / launch failed           */
#define DAN_ERR_UNSUPPORTED (-4)      /* size beyond what the kernels were built for   */

#define DAN_MAX_LAYERS 16
#define DAN_MAX_DEPTH_TOTAL 128
#define DAN_MAX_GRIDS 8 /* levels a dan_encode_params layout hint can describe */

/* matcher selection for dan_encode_batch */
#define DAN_MATCH_DUAL 0   /* do_dual_max_match, utility/anchor_manipulator.py:54-105 */
#define DAN_MATCH_MINING 1 /* SmallMiningMatch,  cpp/ExtraLib/small_mining_match.cc   */

/* element type of the predictions of the *_typed entry points.  fp16 and bf16 values
 * are widened to fp32 as they are loaded (exact), and all arithmetic after the load is
 * the fp32 path's: the results are bit-identical to the fp32 call on the widened
 * predictions.  Outputs are always fp32. */
#define DAN_DTYPE_F32 0
#define DAN_DTYPE_F16 1
#define DAN_DTYPE_BF16 2

int dan_version(void);
const char* dan_last_error(void);
/* 1 when a CUDA device of compute capability 10.x is visible, else 0 (no error set). */
int dan_device_ok(void);

/* ------------------------------------------------------------------------- *
 * (a2-a5) anchors: AnchorEncoder.get_all_anchors
 *         utility/anchor_manipulator.py:163-198 (per layer), :213-273 (all)
 * ------------------------------------------------------------------------- */
typedef struct dan_pyramid {
  int32_t num_layers;
  int32_t image_h, image_w;
  int32_t layer_h[DAN_MAX_LAYERS], layer_w[DAN_MAX_LAYERS];
  int32_t depth[DAN_MAX_LAYERS];        /* anchors per cell (get_anchors_width_height) */
  int32_t clip[DAN_MAX_LAYERS];         /* should_clips                                */
  float stride[DAN_MAX_LAYERS];         /* feat_strides                                */
  float offset_h[DAN_MAX_LAYERS], offset_w[DAN_MAX_LAYERS];
  float border[DAN_MAX_LAYERS];         /* allowed_borders                             */
  /* per-layer anchor heights / widths, concatenated in layer order (sum depth)        */
  float anchor_h[DAN_MAX_DEPTH_TOTAL], anchor_w[DAN_MAX_DEPTH_TOTAL];
} dan_pyramid;

/* total anchors; <0 on invalid pyramid */
int64_t dan_anchor_count(const dan_pyramid* h_pyr);

/* out_*: fp32 [N]; out_inside_mask: uint8 [N] (may be NULL). */
int dan_generate_anchors(const dan_pyramid* h_pyr, float* out_ymin, float* out_xmin, float* out_ymax,
                         float* out_xmax, uint8_t* out_inside_mask, void* stream);

/* ------------------------------------------------------------------------- *
 * (a6) iou_matrix: utility/anchor_manipulator.py:24-52, materialised [N, M].
 *      inside_mask may be NULL (then no mask multiply, like iou_matrix itself).
 * ------------------------------------------------------------------------- */
int dan_iou_matrix(const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax,
                   const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes,
                   int32_t num_gt, float* out_overlaps, void* stream);

/* intersection(), anchor_manipulator.py:29-43, materialised [N, M] (no mask). */
int dan_intersection_matrix(const float* a_ymin, const float* a_xmin, const float* a_ymax,
                            const float* a_xmax, int32_t num_anchors, const float* gt_boxes,
                            int32_t num_gt, float* out_inter, void* stream);

/* ------------------------------------------------------------------------- *
 * (a8) the SmallMiningMatch op on a dense overlaps matrix -- the literal
 *      replacement of REGISTER_OP("SmallMiningMatch") small_mining_match.cc:31-54.
 *      overlaps: fp32 [N, M] row major, every element in [0, 1] (op doc :42-43).
 *      Attribute checks are those of the op constructor (:292-305).
 * ------------------------------------------------------------------------- */
size_t dan_match_workspace_bytes(int32_t num_anchors, int32_t num_gt);
int dan_small_mining_match(const float* overlaps, int32_t num_anchors, int32_t num_gt,
                           float negative_low_thres, float negative_high_thres, float positive_thres,
                           int32_t min_match, float stop_positive_thres, int32_t* out_match_indices,
                           float* out_match_scores, void* workspace, size_t workspace_bytes,
                           void* stream);

/* (a7) do_dual_max_match on a dense overlaps matrix, anchor_manipulator.py:54-105.
 *      out_match_indices is int64 like tf.argmax. */
int dan_dual_max_match(const float* overlaps, int32_t num_anchors, int32_t num_gt, float low_thres,
                       float high_thres, int32_t ignore_between, int32_t gt_max_first,
                       int64_t* out_match_indices, float* out_match_scores, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- *
 * (a9/a10) batched fused encode: IoU + match + encode, no [N,M] matrix in HBM.
 *   encode_anchors    anchor_manipulator.py:275-326  (pa_scale = 0)
 *   encode_pa_anchors anchor_manipulator.py:328-387  (pa_scale = scale > 0)
 * One call encodes `batch` images that share one anchor set; image b owns GT rows
 * [gt_offsets[b], gt_offsets[b+1]) of gt_boxes (CSR).  An image with no GT gets
 * the reference's dummy box [0,0,1,1] (:286).
 * ------------------------------------------------------------------------- */
typedef struct dan_encode_params {
  int32_t matcher;          /* DAN_MATCH_DUAL | DAN_MATCH_MINING                         */
  float ignore_threshold;   /* dual: low_thres; mining: negative_high_thres              */
  float positive_threshold; /* dual: high_thres; mining: positive_thres                  */
  float prior_scaling[4];
  float pa_scale;           /* 0: encode_anchors; >0: encode_pa_anchors with this scale  */
  int32_t debug;            /* debug=True: targets carry the raw anchors (:319-320)      */
  /* mining attributes (small_mining_match.cc:33-37); the reference call site
   * anchor_manipulator.py:291 uses (0., ignore, positive, 6, 0.3) */
  float negative_low_thres;
  int32_t min_match;
  float stop_positive_thres;
  /* dual options (anchor_manipulator.py:54) */
  int32_t ignore_between;
  int32_t gt_max_first;
  /* optional LAYOUT HINT (performance only; the results do not depend on it).  The
   * encode entry points take the anchors as flat arrays, as the reference does
   * (anchor_manipulator.py:275).  When a pyramid level is a row-major grid with ONE
   * anchor per cell (get_all_anchors order, :213-273), say so here and the kernels
   * give every warp an 8 x 4 tile of cells instead of a 32 x 1 strip, whose bounding
   * box meets ~28 % fewer ground-truth boxes at 640^2.  Requirements per grid:
   * grid_start % 32 == 0, grid_w % 8 == 0, grid_h % 4 == 0, grids ascending and
   * inside [0, num_anchors).  num_grids = 0: no hint. */
  int32_t num_grids;
  int32_t grid_start[DAN_MAX_GRIDS]; /* index of the level's first anchor */
  int32_t grid_w[DAN_MAX_GRIDS];     /* cells per row                     */
  int32_t grid_h[DAN_MAX_GRIDS];     /* rows                              */
} dan_encode_params;

size_t dan_encode_workspace_bytes(int32_t num_anchors, int32_t batch, int32_t total_gt);

/* out_targets [B,N,4] f32; out_labels [B,N] int64 (1 pos, 0 neg, -1 ignore);
 * out_scores [B,N] f32; out_matched_gt [B,N,4] f32 (may be NULL);
 * out_match [B,N] int32 (may be NULL): >=0 GT index within the image, -1, -2.  */
int dan_encode_batch(const dan_encode_params* h_params, const float* a_ymin, const float* a_xmin,
                     const float* a_ymax, const float* a_xmax, const uint8_t* inside_mask,
                     int32_t num_anchors, const float* gt_boxes, const int32_t* gt_offsets,
                     int32_t batch, int32_t total_gt, float* out_targets, int64_t* out_labels,
                     float* out_scores, float* out_matched_gt, int32_t* out_match, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Profiling variant (bench.py roofline): same work, but records CUDA events on `stream`
 * around each launch, synchronises, and writes the duration in ms of pass 1 (column
 * maxima), pass 2 (match + encode + all outputs) and pass 3 (mining compensation;
 * 0 for the dual matcher) to h_pass_ms[3] (HOST pointer).  Not graph capturable. */
int dan_encode_batch_profile(const dan_encode_params* h_params, const float* a_ymin,
                             const float* a_xmin, const float* a_ymax, const float* a_xmax,
                             const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes,
                             const int32_t* gt_offsets, int32_t batch, int32_t total_gt,
                             float* out_targets, int64_t* out_labels, float* out_scores,
                             float* out_matched_gt, int32_t* out_match, void* workspace,
                             size_t workspace_bytes, void* stream, float* h_pass_ms);

/* ------------------------------------------------------------------------- *
 * (a11) decode_anchors / batch_decode_anchors, anchor_manipulator.py:389-424.
 *       pred [B,N,4] (cy,cx,h,w offsets) -> out [B,N,4] boxes.
 * ------------------------------------------------------------------------- */
int dan_decode_batch(const float* pred, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                     const float* a_xmax, int32_t num_anchors, int32_t batch,
                     const float* h_prior_scaling, float* out_boxes, void* stream);
/* The same with pred of element type pred_dtype (DAN_DTYPE_*): 16-byte aligned for
 * fp32, 8-byte aligned (one row per anchor) for fp16 / bf16.  out_boxes is fp32. */
int dan_decode_batch_typed(int32_t pred_dtype, const void* pred, const float* a_ymin,
                           const float* a_xmin, const float* a_ymax, const float* a_xmax,
                           int32_t num_anchors, int32_t batch, const float* h_prior_scaling,
                           float* out_boxes, void* stream);

/* ------------------------------------------------------------------------- *
 * (a12-a18) utility/bbox_util.py helpers, one kernel each (elementwise).
 * ------------------------------------------------------------------------- */
/* tf.nn.softmax over the last axis (bbox_util.py:105), rows x classes. */
int dan_softmax(const float* logits, int64_t rows, int32_t num_classes, float* out, void* stream);
/* select_bboxes :24-36 for one class column: out_boxes = boxes*m, out_scores = s*m. */
int dan_select_bboxes(const float* scores, int32_t num_classes, int32_t class_ind, const float* boxes,
                      int64_t n, float select_threshold, float* out_boxes, float* out_scores,
                      void* stream);
/* clip_bboxes :38-48 on an AoS [n,4] tensor (in place allowed). */
int dan_clip_bboxes(const float* boxes, int64_t n, float height, float width, float* out_boxes,
                    void* stream);
/* filter_bboxes :50-59 ; min_size_plus_1 = fp32(min_size + 1.) */
int dan_filter_bboxes(const float* scores, const float* boxes, int64_t n, float min_size_plus_1,
                      float* out_scores, float* out_boxes, void* stream);
/* bbox_point2center :92-96 (mode 0) / bbox_center2point :98-101 (mode 1) /
 * areas() anchor_manipulator.py:24-27 (mode 2: area written to column 0, rest 0) */
int dan_bbox_convert(const float* boxes, int64_t n, int32_t mode, float* out_boxes, void* stream);

/* sort_bboxes :61-72 = tf.nn.top_k(sorted) + gather + zero pad to keep_topk.
 * Descending score, equal scores -> lower index first.  out_* have keep_topk rows;
 * out_index (int32, may be NULL) is -1 in the padding. */
size_t dan_sort_workspace_bytes(int64_t n, int32_t keep_topk);
int dan_sort_bboxes(const float* scores, const float* boxes, int64_t n, int32_t keep_topk,
                    float* out_scores, float* out_boxes, int32_t* out_index, void* workspace,
                    size_t workspace_bytes, void* stream);

/* nms_bboxes :75-78 / nms_bboxes_with_padding :80-90 = tf.image.non_max_suppression
 * (greedy, IoU without +1, strict >, area<=0 never suppresses) + gather + zero pad
 * to nms_topk.  Input need not be sorted; equal scores keep input order (documented
 * tie policy).  out_count: int32 [1] number of selected boxes; out_keep int32
 * [nms_topk] selected input indices (-1 padded; may be NULL). */
size_t dan_nms_workspace_bytes(int64_t n, int32_t nms_topk);
int dan_nms_bboxes(const float* scores, const float* boxes, int64_t n, int32_t nms_topk,
                   float nms_threshold, float* out_scores, float* out_boxes, int32_t* out_keep,
                   int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- *
 * (a17) batched fused parse_by_class, bbox_util.py:103-119:
 *   softmax -> select(threshold) -> [decode] -> clip -> min-size filter ->
 *   per-class top-k (block radix select + sort) -> greedy NMS against the kept
 *   list -> zero pad.
 * cls_pred [B,N,C] logits.  Exactly one of `loc_pred` ([B,N,4] offsets, decoded
 * in-kernel against the anchors like decode_anchors) or `boxes_pred` ([B,N,4]
 * already decoded boxes, what parse_by_class literally takes) must be non-NULL.
 * HOST-RESIDENT GEOMETRY: `loc_pred` / `boxes_pred` may also point to page-locked
 * host memory that is mapped for the device (cudaHostAlloc, cudaHostRegister; with
 * unified addressing that is every pinned allocation).  Only the rows of anchors
 * whose score passes `select_threshold` are ever read (~3 % for a detector's
 * output), so the kernels fetch exactly those rows over PCIe, once (the decoded box
 * is kept in the workspace), and the other rows never leave the host: 16 of the
 * 24 bytes per anchor of a host-side caller's input are not transferred at all.
 * `cls_pred` is read in full and must be device memory.  Pageable host memory is
 * refused with DAN_ERR_INVALID_ARGUMENT.
 * fp16 / bf16 predictions: dan_postprocess_batch_typed (section (e) below).
 * ------------------------------------------------------------------------- */
typedef struct dan_postprocess_params {
  int32_t num_classes;
  int32_t image_h, image_w;
  float select_threshold; /* must be >= 0 */
  float min_size;
  int32_t keep_topk;
  int32_t nms_topk;
  float nms_threshold;
  float prior_scaling[4];
} dan_postprocess_params;

size_t dan_postprocess_workspace_bytes(int32_t num_anchors, int32_t batch, int32_t num_classes,
                                       int32_t keep_topk);

/* Outputs are indexed [b][c-1] for classes c = 1..C-1:
 *   out_boxes  [B, C-1, nms_topk, 4] f32, zero padded
 *   out_scores [B, C-1, nms_topk]    f32, zero padded
 *   out_counts [B, C-1]              int32  number of REAL (score>0) detections kept
 *   out_anchor_index [B, C-1, nms_topk] int32 (may be NULL): anchor index of each
 *       kept detection, -1 in the padding
 *   out_keep_pos [B, C-1, nms_topk] int32 (may be NULL): what
 *       tf.image.non_max_suppression returns inside nms_bboxes_with_padding, i.e.
 *       positions in the top-k sorted list (zero-score filler rows included),
 *       -1 beyond the number selected. */
int dan_postprocess_batch(const dan_postprocess_params* h_params, const float* cls_pred,
                          const float* loc_pred, const float* boxes_pred, const float* a_ymin,
                          const float* a_xmin, const float* a_ymax, const float* a_xmax,
                          int32_t num_anchors, int32_t batch, float* out_boxes, float* out_scores,
                          int32_t* out_counts, int32_t* out_anchor_index, int32_t* out_keep_pos,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Profiling variant: durations in ms of the filter kernel and of the top-k/sort +
 * NMS kernel written to h_kernel_ms[2] (HOST pointer).
 * Synchronises; not graph capturable. */
int dan_postprocess_batch_profile(const dan_postprocess_params* h_params, const float* cls_pred,
                                  const float* loc_pred, const float* boxes_pred,
                                  const float* a_ymin, const float* a_xmin, const float* a_ymax,
                                  const float* a_xmax, int32_t num_anchors, int32_t batch,
                                  float* out_boxes, float* out_scores, int32_t* out_counts,
                                  int32_t* out_anchor_index, int32_t* out_keep_pos, void* workspace,
                                  size_t workspace_bytes, void* stream, float* h_kernel_ms);

/* ------------------------------------------------------------------------- *
 * (f3, SURVEY.md 8f) per-image hard-negative mining, the step after encode on the
 * training side: mining_hard_neg, train_dan.py:286-324 (inline copy
 * train_sfd.py:349-384) and mining_hard_neg_across_batch, train_dan.py:247-284.
 *   cls_pred [rows*row_len, num_logits] logits; cls_targets [rows*row_len] int64
 *   (the labels dan_encode_batch writes: 1 positive, 0 negative, -1 ignore);
 *   loc_pred / loc_targets [rows*row_len, 4].
 * rows = batch and row_len = anchors for the per-image rule; rows = 1 and
 * row_len = batch*anchors with strict_greater = 1 for the across-batch rule.
 * at_least_one: the tf.maximum(., 1) of train_dan.py:302 (0 for train_sfd.py).
 * Outputs: out_final_mask [rows*row_len] (train_dan.py:316), out_n_neg_select
 * [rows] int32 (:301-302), out_score_at_k [rows] (:311; NaN where n_neg_select < 1,
 * which the reference cannot index), and the four boolean_mask results (:319-322)
 * compacted in order into caller buffers of capacity rows*row_len rows, their
 * lengths in out_counts[2] = {selected rows, positive rows}.
 * ------------------------------------------------------------------------- */
size_t dan_hard_negative_workspace_bytes(int32_t rows, int64_t row_len);
int dan_hard_negative_mining(const float* cls_pred, int32_t num_logits, const int64_t* cls_targets,
                             const float* loc_pred, const float* loc_targets, int32_t rows,
                             int64_t row_len, float negative_ratio, int32_t num_classes,
                             int32_t at_least_one, int32_t strict_greater, uint8_t* out_final_mask,
                             int32_t* out_n_neg_select, float* out_score_at_k, float* out_cls_pred,
                             int64_t* out_cls_targets, float* out_loc_pred, float* out_loc_targets,
                             int32_t* out_counts, void* workspace, size_t workspace_bytes,
                             void* stream);

/* ------------------------------------------------------------------------- *
 * (f1, SURVEY.md 8f) DynamicAnchorRouting, EVALUATION branch
 * (cpp/ExtraLib/dynamic_anchor_routing.cc:328-408; op definition :31-59; called once
 * per pyramid layer and image on /cpu:0 by eval_dan.py:383-391).  One call handles
 * all layers of all images of a batch; a single layer with batch 1 is the op itself.
 *   anchors    [B, N, 4] decoded stage-1 boxes (ymin, xmin, ymax, xmax)
 *   gt_targets [B, N, 4] stage-2 offsets (cy, cx, h, w) already divided by the
 *                        prior scaling (eval_dan.py:384)
 *   labels     [B, N]    stage-2 probability;  mask_in [B, N] int32 (stage-1 score > thres)
 * with N = sum over layers of feat_height*feat_width*anchor_depth, anchors ordered
 * layer by layer, (y, x, depth) inside a layer.
 *   mask_out [B, N] int32 in {0, 1};  decode_out [B, N, 4] the stage-2 boxes.
 * The op's attrs `thres` / `ignore_thres` and inputs img_height / img_width are not
 * used by the evaluation branch.  The training branch draws from an unseeded
 * std::random_device and is not provided.
 * ------------------------------------------------------------------------- */
typedef struct dan_routing_layers {
  int32_t num_layers;
  int32_t feat_height[DAN_MAX_LAYERS];
  int32_t feat_width[DAN_MAX_LAYERS];
  int32_t anchor_depth[DAN_MAX_LAYERS];
  int32_t feat_strides[DAN_MAX_LAYERS];
} dan_routing_layers;

size_t dan_routing_workspace_bytes(int64_t num_anchors, int32_t batch);
int dan_dynamic_anchor_routing_eval(const dan_routing_layers* h_layers, const float* anchors,
                                    const float* gt_targets, const float* labels,
                                    const int32_t* mask_in, int64_t num_anchors, int32_t batch,
                                    int32_t* mask_out, float* decode_out, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- *
 * (f2, SURVEY.md 8f) the evaluation merge of the reference's scripts.
 * dan_detect_face_select: detect_face after net.run (eval_sfd.py:101-112 =
 *   eval_dan.py:101-118): bboxes [n,4] (ymin,xmin,ymax,xmax) / shrink -> rows
 *   (xmin, ymin, xmax, ymax, score), the top min(n-1, top) by descending score
 *   (top = int(1.5 * max_per_image) = 1125); equal scores: higher index first.
 *   out_det [top,5] zero padded, out_index [top] (-1 padded, may be NULL), out_count [1].
 * dan_detect_face_batch: the whole detect_face chain of the evaluation scripts
 *   (softmax :279, decode_anchors :283, detect_face :95-114) for B images from the
 *   head's raw outputs: cls_pred [B,N,2] logits, loc_pred [B,N,4] offsets (cy,cx,h,w),
 *   one dtype for both (DAN_DTYPE_*), and the N anchors.  Every image gets
 *   k = max(min(N - 1, top), 0) rows, which the caller knows without a host read:
 *   out_det [B,top,5] (xmin, ymin, xmax, ymax, score) zero padded, out_index [B,top]
 *   anchor index (-1 padded, may be NULL).  Bit-identical to dan_softmax column 1 ->
 *   dan_decode_batch -> dan_detect_face_select per image; fp16 / bf16 predictions give
 *   the results of the fp32 call on the widened values.  Only the k rows are decoded;
 *   nothing N-sized but one 8-byte key per anchor reaches memory.  top in [1, 8192],
 *   N < 2^31, loc_pred rows 16-byte (fp32) / 8-byte (fp16, bf16) aligned; cls_pred
 *   needs no alignment beyond its element type.  batch == 0 enqueues nothing.
 * dan_bbox_vote: bbox_vote (eval_sfd.py:170-210 = eval_dan.py:201-241), batched:
 *   det [B, capacity, 5] rows (xmin, ymin, xmax, ymax, score), counts [B] valid rows
 *   per image (NULL = capacity); out_det [B, max_per_image, 5] zero padded,
 *   out_count [B]; optional out_order / out_assign [B, capacity]: sorted position ->
 *   input row / head position (-2 = head deleted alone), for inspection.
 *   capacity <= 8192.  A stack of P passes (scales, flips) of 1.5 * max_per_image
 *   rows each has 1125 P rows at the default 750: the recipe's 4 to 10 passes per
 *   image give up to 11 250, so dan_bbox_vote_ws is the entry point for stacks.
 * dan_bbox_vote_ws: dan_bbox_vote with the same arguments and results for
 *   capacity <= 1048576 (2^20) rows per image; larger capacities are refused with
 *   DAN_ERR_UNSUPPORTED.  capacity <= 8192 runs the same kernel as dan_bbox_vote and
 *   needs no workspace (dan_bbox_vote_workspace_bytes returns 0, workspace may be
 *   NULL).  Above 8192 the detections of each image are sorted and merged in the
 *   workspace (16-byte aligned, at least dan_bbox_vote_workspace_bytes(batch,
 *   capacity) bytes, else DAN_ERR_WORKSPACE); the results are the same bits.  The
 *   path is chosen from capacity alone.  Every check happens before anything is
 *   enqueued; nothing synchronises, and the call can be captured in a CUDA graph.
 * dan_bbox_vote_workspace_bytes: bytes for capacity in (8192, 2^20], else 0.
 * ------------------------------------------------------------------------- */
size_t dan_detect_face_workspace_bytes(int64_t n);
int dan_detect_face_select(const float* bboxes, const float* scores, int64_t n, float shrink,
                           int32_t top, float* out_det, int32_t* out_index, int32_t* out_count,
                           void* workspace, size_t workspace_bytes, void* stream);
size_t dan_detect_face_batch_workspace_bytes(int64_t num_anchors, int32_t batch);
int dan_detect_face_batch(int32_t pred_dtype, const void* cls_pred, const void* loc_pred,
                          const float* a_ymin, const float* a_xmin, const float* a_ymax,
                          const float* a_xmax, int64_t num_anchors, int32_t batch,
                          const float* h_prior_scaling, float shrink, int32_t top,
                          float* out_det, int32_t* out_index, void* workspace,
                          size_t workspace_bytes, void* stream);
int dan_bbox_vote(const float* det, const int32_t* counts, int32_t batch, int32_t capacity,
                  float nms_threshold, int32_t max_per_image, float* out_det, int32_t* out_count,
                  int32_t* out_order, int32_t* out_assign, void* stream);
size_t dan_bbox_vote_workspace_bytes(int32_t batch, int32_t capacity);
int dan_bbox_vote_ws(const float* det, const int32_t* counts, int32_t batch, int32_t capacity,
                     float nms_threshold, int32_t max_per_image, float* out_det,
                     int32_t* out_count, int32_t* out_order, int32_t* out_assign,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- *
 * (f4, SURVEY.md 8f) input hand-off: the deterministic tail of the training
 * preprocessing between the sampled patch and encode_anchors, for a batch:
 * mirror (sfd_preprocessing.py:482-493, the coin flip is an input), rescale to the
 * net input (:529-533), small-face filter `h > 6 & w > 3` (:544-550), and the
 * keep_input rule that drops images left without boxes (dataset_common.py:178,186).
 *   gt_boxes [total_gt,4] (ymin,xmin,ymax,xmax) in patch pixels, gt_offsets [B+1],
 *   patch_hw [B,2] (height, width of the patch), mirror [B] uint8 or NULL.
 * Outputs: the CSR batch dan_encode_batch consumes: out_gt_boxes [total_gt,4]
 * capacity, out_gt_offsets [B+1] capacity, out_image_index [B] (source image of
 * each kept image), out_counts[2] = {kept images, kept boxes}.
 * ------------------------------------------------------------------------- */
int dan_gt_handoff(const float* gt_boxes, const int32_t* gt_offsets, const float* patch_hw,
                   const uint8_t* mirror, int32_t batch, int32_t total_gt, float target_height,
                   float target_width, float min_height, float min_width, float* out_gt_boxes,
                   int32_t* out_gt_offsets, int32_t* out_image_index, int32_t* out_counts,
                   void* stream);

/* ------------------------------------------------------------------------- *
 * (e) multi-GPU: the one exchange step of the path.  Images are sharded per rank
 * with no data-path collective (the reference's analogue is the batch split of
 * tf_replicate_model_fn.py:458-501, which has no collective at all); the
 * variable-length detections of all ranks are exchanged as fixed-capacity slabs
 * (counts | boxes | scores, written in place by dan_postprocess_batch) with ONE
 * ncclAllGather enqueued on `stream`, i.e. on the device timeline right after the
 * NMS kernel and capturable in the step's CUDA graph (SURVEY.md 8b, 8e).
 *   dan_nccl_load       bind NCCL at run time (NULL / "" = the libnccl.so.2 the
 *                       process already uses, e.g. PyTorch's); optional, the other
 *                       calls bind on first use.
 *   dan_comm_unique_id  ncclGetUniqueId -> 128 bytes (rank 0; ship them to the
 *                       other ranks by any means).
 *   dan_comm_init       ncclCommInitRank on the CURRENT device -> opaque comm
 *                       (dan_comm_init_ctas: ncclCommInitRankConfig with maxCTAs = max_ctas,
 *                       0 = NCCL's default).
 *   dan_gather_detections  recv_slabs [world, slab_bytes] <- send_slab [slab_bytes]
 *                       of every rank, rank order.
 * ------------------------------------------------------------------------- */
/* The same exchange WITHOUT a collective kernel: the ranks of one node map each other's receive buffers (CUDA IPC over
 * NVLink) and the NMS kernel stores every slab row it writes into all of them as well - the transfer is the tail of
 * the compute kernel, no CTA waits for another rank.  The last CTA of the launch then writes the rank's step number into
 * its flag slot of every destination; dan_wait_detections enqueues a one-warp kernel that returns when the flags of all
 * ranks have reached this rank's own step number (one-sided: reusing a receive buffer before every reader is done
 * with it is the caller's business, e.g. by rotating buffers).
 *   dan_peer_alloc   cudaMalloc'ed, zeroed buffer + its 64-byte IPC handle; dan_peer_open maps a handle of ANOTHER
 *                    process; dan_peer_close / dan_peer_free undo them.
 *   dan_peer_exchange  num_destinations (<= DAN_MAX_PEERS); delta_bytes[q]: what to add to an address inside this rank's
 *                    slab (out_counts / out_boxes / out_scores must all lie in it) to reach its copy in destination q
 *                    (a multiple of 16); flag[q]: this rank's int32 flag inside destination q; state: two zeroed int32
 *                    device words owned by this rank (CTAs done, step number). */
#define DAN_MAX_PEERS 16
typedef struct dan_peer_exchange {
  int32_t num_destinations;
  int64_t delta_bytes[DAN_MAX_PEERS];
  int32_t* flag[DAN_MAX_PEERS];
  int32_t* state;
} dan_peer_exchange;
int dan_peer_alloc(size_t bytes, void** out_ptr, void* out_handle64);
int dan_peer_open(const void* handle64, void** out_ptr);
int dan_peer_close(void* ptr);
int dan_peer_free(void* ptr);
int dan_postprocess_batch_peers(const dan_postprocess_params* h_params, const float* cls_pred,
                                const float* loc_pred, const float* boxes_pred, const float* a_ymin,
                                const float* a_xmin, const float* a_ymax, const float* a_xmax,
                                int32_t num_anchors, int32_t batch, float* out_boxes, float* out_scores,
                                int32_t* out_counts, int32_t* out_anchor_index, int32_t* out_keep_pos,
                                void* workspace, size_t workspace_bytes,
                                const dan_peer_exchange* h_peers, void* stream);

/* dan_postprocess_batch / _peers / _profile with the element type of the predictions as
 * an argument (DAN_DTYPE_*, one type for cls_pred and loc_pred / boxes_pred).  A detection
 * head run under autocast hands over fp16 / bf16 predictions without a conversion pass,
 * and a host-side caller sends half the bytes.  Outputs, the workspace and
 * dan_postprocess_workspace_bytes are those of the fp32 call.
 *   alignment: fp32 as dan_postprocess_batch; fp16 / bf16 loc_pred / boxes_pred 8-byte
 *       aligned (one 8-byte row per anchor).  Two classes run fused into the NMS kernel
 *       when cls_pred is aligned to one anchor's two logits (8 bytes fp32, 4 bytes
 *       fp16 / bf16), else through the separate filter kernel.
 *   host-resident geometry works as for fp32: the 8-byte rows are read in place and the
 *       decoded fp32 boxes are kept in the workspace.  cls_pred must be device memory.
 *   h_peers: NULL = no exchange (else as dan_postprocess_batch_peers).
 *   h_kernel_ms: NULL = enqueue only (graph capturable); non-NULL = the synchronising
 *       semantics of dan_postprocess_batch_profile.
 *   h_peers and h_kernel_ms both non-NULL, or an unknown pred_dtype:
 *       DAN_ERR_INVALID_ARGUMENT before anything is enqueued. */
int dan_postprocess_batch_typed(const dan_postprocess_params* h_params, int32_t pred_dtype,
                                const void* cls_pred, const void* loc_pred, const void* boxes_pred,
                                const float* a_ymin, const float* a_xmin, const float* a_ymax,
                                const float* a_xmax, int32_t num_anchors, int32_t batch,
                                float* out_boxes, float* out_scores, int32_t* out_counts,
                                int32_t* out_anchor_index, int32_t* out_keep_pos, void* workspace,
                                size_t workspace_bytes, const dan_peer_exchange* h_peers,
                                void* stream, float* h_kernel_ms);
int dan_wait_detections(const int32_t* flags, const int32_t* state, int32_t world_size, void* stream);

int dan_nccl_load(const char* path);
int dan_nccl_version(void);
int dan_comm_unique_id(void* out_id128);
int dan_comm_init(const void* id128, int32_t rank, int32_t world_size, void** out_comm);
int dan_comm_init_ctas(const void* id128, int32_t rank, int32_t world_size, int32_t max_ctas,
                       void** out_comm);
int dan_comm_destroy(void* comm);
int dan_gather_detections(void* comm, const void* send_slab, void* recv_slabs, size_t slab_bytes,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DAN_B200_H_ */
