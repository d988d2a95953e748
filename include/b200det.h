/* b200det.h — C ABI of libb200det.so: the B200 (sm_100a) detection post-network hot path.
 *
 * Drop-in boundary for tfwcn/tensorflow2-machine-vision.  The reference has no FFI/plugin layer
 * (grep for load_op_library / ctypes / dlpack: 0 hits), so each entry point replaces one Python
 * function of the reference's L2 utilities; the citation beside each declaration names it
 * (paths relative to AIServer/ai_api/ai_models/).  INTEGRATION.md shows the ctypes/DLPack stub a
 * maintainer adds on the reference side.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer unless the name ends in _host; fp32, NHWC, C-contiguous;
 *   - the caller owns every buffer (inputs, outputs, workspace); nothing is allocated or freed here;
 *   - `stream` is a cudaStream_t passed as void*; calls enqueue work and return without synchronising;
 *   - return 0 on success, negative on error (B200_ERR_*), message via b200_last_error() (thread-local);
 *   - no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef B200DET_H_
#define B200DET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DET_VERSION 200

#define B200_OK 0
#define B200_ERR_BAD_ARG (-1)
#define B200_ERR_WORKSPACE (-2)
#define B200_ERR_CUDA (-3)
#define B200_ERR_UNSUPPORTED (-4)

/* Pairwise metric selector.  Two families exist in the reference and both are reproduced bit-for-bit:
 * YOLO (utils/tf_iou_utils.py:5-65, boxes x1,y1,x2,y2) and EfficientDet (efficientnet/utils/iou.py:26-100,
 * boxes y1,x1,y2,x2, NaN-free). */
enum {
  B200_METRIC_YOLO_IOU = 0,
  B200_METRIC_YOLO_DIOU = 1, /* iou - (u/c)^0.6, tf_iou_utils.py:50 */
  B200_METRIC_YOLO_CIOU = 2, /* iou - (u/c + alpha*v), tf_iou_utils.py:55-61 */
  B200_METRIC_EFF_IOU = 3,
  B200_METRIC_EFF_GIOU = 4,
  B200_METRIC_EFF_DIOU = 5,
  B200_METRIC_EFF_CIOU = 6,
  B200_METRIC_COUNT = 7
};

/* NMS survivor predicate. */
enum {
  B200_NMS_AGNOSTIC = 0, /* survivor iff metric < thr (NaN drops): GetIOUNMS tiu:98, get_nms enms:51 */
  B200_NMS_BY_CLASS = 1  /* suppressed iff metric >= thr and same class (NaN stays): GetIOUNMSByClasses tiu:146 */
};

const char* b200_last_error(void);
int b200_version(void);
/* 0 if a CUDA device is usable, else B200_ERR_CUDA (the library has no CPU path). */
int b200_device_ok(void);

/* Device-wide hint for the DRAM->L2 fetch granularity (32, 64 or 128 bytes; cudaLimitMaxL2FetchGranularity).
 * Optional: the sector-sparse loss kernels read less DRAM with 32; nothing depends on it for correctness. */
int b200_set_l2_fetch_granularity(int bytes);
int b200_get_l2_fetch_granularity(void);

/* detmath self-test hook: out[i] = f(x[i]) evaluated on the device with csrc/detmath.h. */
enum {
  B200_DM_EXP = 0, B200_DM_SIGMOID = 1, B200_DM_LOG = 2, B200_DM_LOG1P = 3, B200_DM_ATAN = 4,
  B200_DM_POW06 = 5, B200_DM_POW15 = 6, B200_DM_BCE = 7 /* bce_with_logits(label=y, logit=x) */, B200_DM_COUNT = 8
};
int b200_detmath_eval(int op, const float* x, const float* y, float* out, size_t n, void* stream);

/* GetIOU (utils/tf_iou_utils.py:5-65) / get_iou (efficientnet/utils/iou.py:26-100).
 * pairwise: out[n1,n2] = metric(b1[i], b2[j]);  elementwise: out[n] = metric(b1[i], b2[i]). */
int b200_pairwise_iou(const float* b1, int n1, const float* b2, int n2, int metric, float* out, void* stream);
int b200_elementwise_iou(const float* b1, const float* b2, size_t n, int metric, float* out, void* stream);

/* _get_v (efficientnet/utils/iou.py:5-24): the aspect-ratio term of the EfficientDet CIoU and the hand-written gradient
 * its tf.custom_gradient returns for the second box's (height, width) given an upstream dv.  Elementwise over n; v_out or
 * the gradient outputs may be NULL. */
int b200_ciou_v_grad(const float* b1_height, const float* b1_width, const float* b2_height, const float* b2_width,
                     const float* dv, size_t n, float* v_out, float* grad_height_out, float* grad_width_out, void* stream);

/* GetIOUNMS tiu:67-108, GetIOUNMSByClasses tiu:110-157, get_nms enms:5-61 — batched over segments.
 * boxes [total,4] (16-byte aligned), scores [total], classes [total] int32 or NULL, order_id [total] or NULL
 * (unique ids giving the tie order; NULL = position), seg_offsets [num_segments+1] int32 (device).
 * out_idx [num_segments, max_out]: positions local to the segment, in emit order; out_count [num_segments].
 * use_score_thr != 0 stops at the first top score < score_thr (enms:44).  max_out <= 4096. */
int b200_nms(const float* boxes, const float* scores, const int32_t* classes, const uint32_t* order_id,
             const int32_t* seg_offsets, int num_segments, int metric, int mode, float iou_thr,
             int use_score_thr, float score_thr, int max_out, int32_t* out_idx, int32_t* out_count, void* stream);

/* GetNMSBoxes (utils/tf_yolo_utils.py:169-269) for a batch, B==1 semantics per image:
 * GetBoxes decode (:129-167), strict thresholds conf > conf_thr and max_c sigmoid(cls) > score_thr (:191-192),
 * score = max_c sigmoid(cls), class_id = argmax (:199-203), per-class NMS capped at max_out (:255-261; the
 * reference hard-codes 500), gather (:262-266).
 * heads[l]: device (B,H_l,W_l,A*(5+C)), 16-byte aligned; hw = {H0,W0,H1,W1,H2,W2}; anchors_wh_host [3][A][2]
 * pixels (layer 0 = coarsest head); image_wh_host [2]; metric in YOLO_IOU/DIOU/CIOU.
 * Outputs are padded to max_out rows per image, `out_count[B]` gives the valid rows:
 *   out_boxes [B,max_out,4] x1,y1,x2,y2 normalised; out_class_id [B,max_out] int32; out_score [B,max_out];
 *   out_classes [B,max_out,C] (may be NULL); out_conf [B,max_out];
 *   out_sel_idx [B,max_out] position in the reference's compacted candidate list (may be NULL);
 *   out_sel_anchor [B,max_out] flat anchor index level-major/h/w/a (may be NULL). */
size_t b200_yolo_decode_nms_workspace_bytes(const int32_t hw[6], int B, int A, int max_out);
int b200_yolo_decode_nms(const float* const heads[3], const int32_t hw[6], int B, int A, int C,
                         const float* anchors_wh_host, const float* image_wh_host, float conf_thr, float score_thr,
                         float iou_thr, int metric, int max_out, float* out_boxes, int32_t* out_class_id,
                         float* out_score, float* out_classes, float* out_conf, int32_t* out_sel_idx,
                         int32_t* out_sel_anchor, int32_t* out_count, void* workspace, size_t workspace_bytes,
                         void* stream);

/* GetBoxes (utils/tf_yolo_utils.py:129-167) without the final boolean_mask: dense decode of one level.
 * head (B,H,W,A*(5+C)); anchors_wh_norm_dev [A][2] = anchors/image_wh (device); outputs for all B*H*W*A
 * anchors in row-major order: boxes [N,4], conf [N], classes [N,C] (sigmoid), valid [N] (x2>x1 && y2>y1). */
int b200_yolo_decode_dense(const float* head, int B, int H, int W, int A, int C, const float* anchors_wh_norm_dev,
                           float* boxes, float* conf, float* classes, unsigned char* valid, void* stream);

/* GetLoss (utils/tf_yolo_utils.py:6-127) / Yolov4Loss.call (losses/yolo_loss.py:85-159).
 * y_true[l]: (B,H_l,W_l,A,5+C) dense targets (xy,wh normalised, obj, one-hot); y_pred[l]: (B,H_l,W_l,A*(5+C)) logits.
 * anchors_wh_host [3][A][2] pixels, layer 0 = coarsest head; metric selects the ignore-mask IoU (iou|diou|ciou);
 * variant 0 = tf_yolo_utils.GetLoss (+1e-8 in the log, raw_xy multiplied by obj), 1 = Yolov4Loss / unit-test copy.
 * batch_divisor: the batch size the sums are divided by (pass the GLOBAL batch when sharding images over ranks;
 * the 12 partial terms are then summed across ranks by one all-reduce).
 * out_parts [3][4] = per level {xy, wh, obj, cls} / batch_divisor (may be NULL); out_loss: scalar;
 * out_ignore [B, anchors_per_image] (may be NULL): the ignore mask float(best_iou < thr) of tyu:94 as bytes,
 * anchors in level-major / h / w / a order — not returned by the reference, exposed for parity checks. */
enum { B200_YOLO_LOSS_TF_YOLO_UTILS = 0, B200_YOLO_LOSS_KERAS_YOLO3 = 1 };
size_t b200_yolo_loss_workspace_bytes(const int32_t hw[6], int B, int A);
int b200_yolo_loss(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B, int A,
                   int C, const float* anchors_wh_host, const float* image_wh_host, float iou_thresh, int metric,
                   int variant, float batch_divisor, float* out_parts, float* out_loss, unsigned char* out_ignore,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Measurement hook: b200_yolo_loss restricted to a subset of its four launches (bit 0 object scan, 1 GT preparation,
 * 2 ignore mask + object terms, 3 finalize); the workspace carries the state, stages must be issued in order. */
int b200_yolo_loss_stages(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B, int A,
                          int C, const float* anchors_wh_host, const float* image_wh_host, float iou_thresh, int metric,
                          int variant, float batch_divisor, float* out_parts, float* out_loss, void* workspace,
                          size_t workspace_bytes, int stages, void* stream);

/* GetLoss forward + analytic backward (SURVEY §8f N1; tf.GradientTape differentiates GetLoss in train_step,
 * yolo_v4/model.py:318-338): out_grad[l] (B,H_l,W_l,A*(5+C)) = d loss / d y_pred[l] for an upstream gradient of 1
 * (d/dt_xy = obj*scale*(sigmoid(t)-raw_xy)/B, d/dt_wh = obj*scale*(t-raw_wh)/B, d/dconf = (sigmoid(p)-obj)*
 * (obj+(1-obj)*ignore)/B, d/dcls = obj*(sigmoid(c)-t_cls)/B; no gradient through targets or the ignore mask).
 * Same workspace size as b200_yolo_loss. */
int b200_yolo_loss_grad(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B, int A,
                        int C, const float* anchors_wh_host, const float* image_wh_host, float iou_thresh, int metric,
                        int variant, float batch_divisor, float* out_parts, float* out_loss, float* const out_grad[3],
                        void* workspace, size_t workspace_bytes, void* stream);

/* Sparse-target fusion (SURVEY §8f N3; an API extension, no reference signature): DataGenerator.GetTargets
 * (datasets/coco_dataset.py:185-285) followed by GetLoss (utils/tf_yolo_utils.py:6-127) without materialising the
 * dense y_true.  boxes [total,4] pixel corners x1,y1,x2,y2 / classes [total] / offsets [B+1] as for
 * b200_yolo_assign_targets; assign_anchors_wh_host = the anchors GetTargets compares against (cds:209-217),
 * anchors_wh_host = the anchors of the loss.  Same result as assign + b200_yolo_loss up to fp64 summation order;
 * out_ignore as in b200_yolo_loss.  The backward is b200_yolo_loss_from_boxes_grad. */
size_t b200_yolo_loss_from_boxes_workspace_bytes(const int32_t hw[6], int B, int A, int total_boxes);
int b200_yolo_loss_from_boxes(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                              const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                              int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                              float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                              float* out_loss, unsigned char* out_ignore, void* workspace, size_t workspace_bytes,
                              void* stream);

/* b200_yolo_loss_from_boxes forward + the analytic backward of b200_yolo_loss_grad, still without a dense y_true:
 * out_grad[l] (B,H_l,W_l,A*(5+C)), 16-byte aligned, = d loss / d y_pred[l] for an upstream gradient of 1, bit-identical
 * to b200_yolo_loss_grad on the targets b200_yolo_assign_targets writes from the same boxes.  Same workspace size as
 * b200_yolo_loss_from_boxes.  Data parallel: each rank passes its own images with batch_divisor = the global batch; the
 * gradients need no exchange, out_parts go through any all-reduce + b200_yolo_loss_combine for the global loss. */
int b200_yolo_loss_from_boxes_grad(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                                   const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                                   int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                   float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                                   float* out_loss, float* const out_grad[3], void* workspace, size_t workspace_bytes,
                                   void* stream);

/* DataGenerator.GetTargets (datasets/coco_dataset.py:185-285), batched: boxes [total,4] pixel corners
 * x1,y1,x2,y2, classes [total] int32, offsets [B+1] int32 (all device).  targets[l]: (B,H_l,W_l,A,5+C), zeroed
 * here when zero_fill != 0.  Boxes whose cell falls outside the grid are skipped (tf.scatter_nd would raise). */
int b200_yolo_assign_targets(const float* boxes, const int32_t* classes, const int32_t* offsets, int B,
                             int total_boxes, const float* anchors_wh_host, int A, const float* image_wh_host, int C,
                             const int32_t hw[6], float* const targets[3], int zero_fill, void* stream);
int b200_fill_zero(float* dst, size_t n, void* stream);
/* Sparse reset for a target buffer that is reused step after step (the reference allocates fresh tf.zeros per image,
 * cds:265-276): zeroes exactly the records b200_yolo_assign_targets touched for the previous ground-truth set
 * (prev_boxes / prev_offsets, same layout), leaving an all-zero buffer without the dense re-fill. */
int b200_yolo_reset_targets(const float* prev_boxes, const int32_t* prev_offsets, int B, int total_boxes,
                            const float* anchors_wh_host, int A, const float* image_wh_host, int C,
                            const int32_t hw[6], float* const targets[3], void* stream);

/* tf.boolean_mask (row-major order preserved): flags[n] bytes -> pos[n] = exclusive prefix of the flags, *total =
 * number of set flags (device int).  gather_rows copies the flagged rows of src [n,row_floats] to dst[pos[i]].
 * Used by GetBoxes (tyu:163-166) and GetGroudTruth. */
size_t b200_row_positions_workspace_bytes(long long n);
int b200_row_positions(const unsigned char* flags, long long n, int* pos, int* total, void* workspace,
                       size_t workspace_bytes, void* stream);
int b200_gather_rows(const float* src, int row_floats, const unsigned char* flags, const int* pos, long long n,
                     float* dst, void* stream);
/* GetGroudTruth (yolo_v4/model.py:380-395) before the boolean_mask: for every record of a dense target
 * y (…,5+C): rows[i] = [x-w/2, y-h/2, x+w/2, y+h/2, argmax(classes)], flags[i] = (conf != 0). */
int b200_yolo_ground_truth_rows(const float* y, long long n_records, int C, float* rows, unsigned char* flags,
                                void* stream);

/* Get_mAP_one (utils/mAP.py:114-125; SURVEY §8f N2), batched: gt [total_gt,5] x1,y1,x2,y2,class; pred [total_pred,6]
 * x1,y1,x2,y2,class,score (fp32, as test_step concatenates them); offsets [num_images+1] int32; out [num_images] fp64.
 * max_*_per_image are upper bounds used to size shared memory.  fp64 arithmetic like the NumPy original. */
int b200_map_per_image(const float* gt, const int32_t* gt_offsets, const float* pred, const int32_t* pred_offsets,
                       int num_images, int max_gt_per_image, int max_pred_per_image, int class_num, double thresh,
                       double* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * EfficientDet (efficientnet/utils/anchors.py, iou.py, nms.py; losses/focal_loss.py, box_loss.py;
 * efficientnet/efficientdet_net_train.py:41-52).  Levels are described by hw = {H0,W0,H1,W1,...} and A anchors
 * per location; anchors are rebuilt in-kernel from a device table of b200_effdet_table_floats() floats laid out
 * per level as [yc(H) | xc(W) | hy(A) | hx(A)]: row/column centres tf.range(stride/2, size, stride) and half
 * extents anchor_scale*stride*2^(octave/num_scales)*aspect/2 (anc:58-71; aspect[1] scales x, aspect[0] scales y),
 * a = octave*len(aspects)+aspect_index.  The host computes the table (see INTEGRATION.md). */
size_t b200_effdet_table_floats(int num_levels, const int32_t* hw, int A);
/* Anchors._generate_boxes anc:46-84 for one level: out (H,W,A,4) y1,x1,y2,x2 pixels. */
int b200_effdet_anchors(int num_levels, const int32_t* hw, int A, const float* table_dev, int level, float* out,
                        void* stream);
/* convert_outputs_boxes / _boxes_decoder anc:141-158,245-274: rel[l] (B,H,W,A,4) ty,tx,th,tw -> out[l] y1,x1,y2,x2. */
int b200_effdet_decode(int num_levels, const int32_t* hw, int A, const float* table_dev, int B,
                       const float* const rel[], float* const out[], void* stream);
/* convert_outputs_one anc:161-202 for images [first_image, first_image+num_images) of a batch of B:
 * per anchor argmax/max over the C class logits, background (id 0) dropped, class-agnostic get_nms (enms:5-61)
 * on the raw max logits with score_thr (reference: max_out 200, iou_thr 0.5, score_thr 1e-4, diou), sigmoid of the
 * survivors' scores.  boxes[l] (B,H,W,A,4) decoded, classes[l] (B,H,W,A,C) logits.  Outputs padded to max_out rows:
 * out_boxes [n,max_out,4], out_class_id [n,max_out] int64, out_score [n,max_out], out_sel_idx (position in the
 * reference's concatenated candidate list, may be NULL), out_sel_anchor (flat anchor index, may be NULL),
 * out_count [n]. */
size_t b200_effdet_postprocess_workspace_bytes(int num_levels, const int32_t* hw, int A, int num_images, int max_out);
int b200_effdet_postprocess(int num_levels, const int32_t* hw, int A, int C, int B, int first_image, int num_images,
                            const float* const boxes[], const float* const classes[], int max_out, float iou_thr,
                            float score_thr, int metric, float* out_boxes, long long* out_class_id, float* out_score,
                            int32_t* out_sel_idx, int32_t* out_sel_anchor, int32_t* out_count, void* workspace,
                            size_t workspace_bytes, void* stream);
/* Anchors.generate_targets anc:91-138 + _boxes_encoder anc:219-243, batched: gt_boxes [total,4] y1,x1,y2,x2,
 * gt_classes [total] int32, gt_offsets [B+1].  Per level: out_boxes (B,H,W,A,4), out_onehot (B,H,W,A,C),
 * out_mask (B,H,W,A,1) bytes.  Anchor -> best GT (first max IoU), mask = max >= iou_thr; unmatched anchors get
 * one-hot class 0 and zero box targets.  An image without GT yields all-unmatched (the reference would raise). */
int b200_effdet_assign_targets(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                               const float* gt_boxes, const int32_t* gt_classes, const int32_t* gt_offsets,
                               float iou_thr, float* const out_boxes[], float* const out_onehot[],
                               unsigned char* const out_mask[], void* stream);
/* Sparse-target mode (SURVEY §8f N3; an API extension): out_class (B,H,W,A) int32 holds the class id whose one-hot row
 * b200_effdet_assign_targets would write (0 = background for unmatched anchors); everything else is identical. */
int b200_effdet_assign_targets_indexed(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                       const float* gt_boxes, const int32_t* gt_classes, const int32_t* gt_offsets,
                                       float iou_thr, float* const out_boxes[], int32_t* const out_class[],
                                       unsigned char* const out_mask[], void* stream);
/* FocalLoss.call focal_loss.py:26-52, elementwise: out = alpha_factor*modulating*ce/normalizer. */
int b200_focal_elementwise(const float* y_true, const float* y_pred, size_t n, float normalizer, float alpha,
                           float gamma, float label_smoothing, float* out, void* stream);
/* _get_loss edt:41-52 in two steps so a data-parallel caller can all-reduce in between:
 * partial_sums -> sums_out[2L+1] (device fp64): [0,L) sum of alpha*mod*ce per level, [L,2L) sum of masked Huber
 * per level, [2L] number of positive anchors.  anchors_per_level[l] = B*H*W*A of this call; a level may omit its
 * class half or its box half (NULL pointers) for stand-alone FocalLoss / BoxLoss.
 * finalize: num_pos = sums[2L]+1; box_l = huber_l/(4 num_pos); focal_l = focal_l/num_pos/numel_l (numel_l = GLOBAL
 * element count of level l's class tensor, host array); out_parts [L][2] = {box_l, focal_l} (may be NULL);
 * out_loss = sum_l (50 box_l + focal_l); out_num_positives may be NULL. */
size_t b200_focal_box_workspace_bytes(int num_levels, const unsigned long long* anchors_per_level, int C);
int b200_focal_box_partial_sums(int num_levels, const unsigned long long* anchors_per_level, int C,
                                const float* const true_boxes[], const float* const true_classes[],
                                const unsigned char* const true_masks[], const float* const pred_boxes[],
                                const float* const pred_classes[], float alpha, float gamma, float delta,
                                float label_smoothing, double* sums_out, void* workspace, size_t workspace_bytes,
                                void* stream);
/* Same sums with the class targets given as class ids (b200_effdet_assign_targets_indexed): the one-hot rows are
 * rebuilt on the fly, so the class half reads the logits only (ids outside [0,C) = all-zero row, as tf.one_hot). */
int b200_focal_box_partial_sums_indexed(int num_levels, const unsigned long long* anchors_per_level, int C,
                                        const float* const true_boxes[], const int32_t* const true_class_index[],
                                        const unsigned char* const true_masks[], const float* const pred_boxes[],
                                        const float* const pred_classes[], float alpha, float gamma, float delta,
                                        float label_smoothing, double* sums_out, void* workspace, size_t workspace_bytes,
                                        void* stream);
int b200_focal_box_finalize(int num_levels, const double* sums, const double* numel_per_level_host, float* out_parts,
                            float* out_loss, float* out_num_positives, void* stream);
/* Backward of _get_loss (SURVEY §8f N1): grad_classes[l] = d loss / d pred_classes[l], grad_boxes[l] = d loss /
 * d pred_boxes[l] for an upstream gradient of 1 (entries / arrays may be NULL).  `sums` as produced by
 * b200_focal_box_partial_sums (after the all-reduce when data-parallel); num_positives is a constant of the targets. */
int b200_focal_box_grad(int num_levels, const unsigned long long* anchors_per_level, int C,
                        const float* const true_boxes[], const float* const true_classes[],
                        const float* const pred_boxes[], const float* const pred_classes[], float alpha, float gamma,
                        float delta, float label_smoothing, const double* sums, const double* numel_per_level_host,
                        float* const grad_boxes[], float* const grad_classes[], void* stream);
/* The same with sparse class targets: true_class_index[l] (B,H,W,A) int32 class ids as
 * b200_effdet_assign_targets_indexed writes them (classes_num >= 4). */
int b200_focal_box_grad_indexed(int num_levels, const unsigned long long* anchors_per_level, int C,
                                const float* const true_boxes[], const int32_t* const true_class_index[],
                                const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                                float gamma, float delta, float label_smoothing, const double* sums,
                                const double* numel_per_level_host, float* const grad_boxes[],
                                float* const grad_classes[], void* stream);

/* generate_targets + _get_loss and its backward from box lists (SURVEY §8f N3 + N1; an API extension): no dense targets.
 * gt_boxes [total,4] y1,x1,y2,x2 (16-byte aligned), gt_classes [total] int32, gt_offsets [B+1] as for
 * b200_effdet_assign_targets.  Two stages, because num_pos scales every gradient and depends only on boxes and anchors:
 *   _match: the matched GT row of every anchor (generate_targets' IoU, tie rule and iou_thr) into the workspace; zeroes
 *     sums[2L+1] and sets sums[2L] = this call's matched anchors;
 *   _grad: one pass over the heads: sums[0..2L) as b200_focal_box_partial_sums writes them (sums[2L] unchanged) and, when
 *     the arrays are given, grad_boxes[l] / grad_classes[l] = d loss / d pred_*[l] for an upstream gradient of 1 with
 *     num_pos = sums[2L] + 1 — bit-identical to b200_focal_box_grad on the targets b200_effdet_assign_targets writes.
 *     NULL grad arrays give the loss terms only.  classes_num < 4 returns B200_ERR_UNSUPPORTED.
 * Then b200_focal_box_finalize(sums, numel_per_level_host) gives the loss.  Both stages take the same workspace
 * (b200_effdet_loss_from_boxes_workspace_bytes, 256-byte aligned; its size does not depend on the device).
 * Data parallel, on every rank: _match; all-reduce sums[2L]; _grad with the GLOBAL numel; all-reduce sums[0..2L);
 * b200_focal_box_finalize.  Not b200_focal_box_finalize_dp: sums[2L] is already global and would be added `world` times. */
size_t b200_effdet_loss_from_boxes_workspace_bytes(int num_levels, const int32_t* hw, int A, int B);
int b200_effdet_loss_from_boxes_match(int num_levels, const int32_t* hw, int A, const float* table_dev, int B,
                                      const float* gt_boxes, const int32_t* gt_offsets, int total_boxes, float iou_thr,
                                      double* sums, void* workspace, size_t workspace_bytes, void* stream);
int b200_effdet_loss_from_boxes_grad(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                     const float* gt_boxes, const int32_t* gt_classes, int total_boxes,
                                     const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                                     float gamma, float delta, float label_smoothing, const double* numel_per_level_host,
                                     double* sums, float* const grad_boxes[], float* const grad_classes[], void* workspace,
                                     size_t workspace_bytes, void* stream);

/* Serving-path box post-processing (SURVEY §8f N4; views/object_detection.py:70-85): boxes [B,max_rows,4] normalised
 * x1,y1,x2,y2 on the letterboxed image (image_size = (w,h) of the network input, padding = (top,bottom,left,right) of
 * opencvProportionalResize, image_size_old = (w,h) of the original image; host int32) -> pixel boxes on the original
 * image, clipped, rows with width or height <= 2 dropped, truncated to int32.  counts [B] (device, may be NULL = all
 * rows).  out_boxes [B,max_rows,4] kept rows first, out_index [B,max_rows] their source rows, out_count [B].
 * fp32 step by step (NumPy 1.x casting of the reference's era). */
int b200_unletterbox_boxes(const float* boxes, const int32_t* counts, int B, int max_rows, const int32_t image_size[2],
                           const int32_t padding[4], const int32_t image_size_old[2], int32_t* out_boxes,
                           int32_t* out_index, int32_t* out_count, void* stream);

/* Serving-path image pre-processing (SURVEY §8f N4): ImageHelper.opencvProportionalResize (utils/image_helper.py:293-325,
 * bg_mode = BORDER_CONSTANT) and, when out_f32 is given, the colour swap and float conversion `predict` applies to its
 * result (views/object_detection.py:50-62).  img [height,width,3] uint8 (device, or pinned host memory); the image is
 * resized proportionally with OpenCV's INTER_AREA arithmetic (bit-exact for 8-bit images, DESIGN.md §2) to fit
 * out_width x out_height and centred on bg_color.  out_u8 [out_height,out_width,3] (optional): the letterboxed image in
 * the input's channel order; out_f32 [out_height,out_width,3] (optional): the same with the channels reversed, / 255.
 * padding_out (host) = top,bottom,left,right as the reference returns them; resized_wh_out (host, optional) = size of
 * the image inside the border.  An input smaller than the target in either direction takes, as in OpenCV, the 8-bit
 * bilinear fallback of INTER_AREA (also bit-exact).  channels != 3 returns B200_ERR_UNSUPPORTED. */
int b200_letterbox_image(const uint8_t* img, int height, int width, int channels, int out_width, int out_height,
                         const uint8_t bg_color[3], uint8_t* out_u8, float* out_f32, int32_t padding_out[4],
                         int32_t resized_wh_out[2], void* stream);

/* b200_letterbox_image for N frames of any sizes in one launch per 84 frames (a longer batch is split): slot i of
 * out_u8 / out_f32 [N,out_height,out_width,3] is bit for bit what b200_letterbox_image gives for frame i alone.
 * imgs (host array of N pointers) [hw[2i], hw[2i+1], 3] uint8 frames in device or pinned host memory; hw (host) [N,2]
 * height,width; padding_out (host) [N,4]; resized_wh_out (host, optional) [N,2]; geometry_out (device, optional) [N,6]
 * top,bottom,left,right,width,height of every frame, written by the kernel (what b200_unletterbox_boxes_batch reads).
 * The per-frame plans travel in the kernel arguments (no workspace, no copy), so the call can be captured in a CUDA
 * graph; a replay letterboxes frames of the captured sizes.  Every frame is checked before anything is launched: an
 * invalid frame (empty resize, bad size, null pointer, channels != 3) fails the call and the message names its index.
 * N == 0 does nothing. */
int b200_letterbox_batch(int N, const uint8_t* const imgs[], const int32_t* hw, int channels, int out_width,
                         int out_height, const uint8_t bg_color[3], uint8_t* out_u8, float* out_f32, int32_t* padding_out,
                         int32_t* resized_wh_out, int32_t* geometry_out, void* stream);

/* b200_unletterbox_boxes with per-image geometry (device [B,6]: padding top,bottom,left,right, then old_w, old_h, as
 * b200_letterbox_batch writes it): frames of different sizes mapped back in one launch, same arithmetic. */
int b200_unletterbox_boxes_batch(const float* boxes, const int32_t* counts, int B, int max_rows, const int32_t image_size[2],
                                 const int32_t* geometry, int32_t* out_boxes, int32_t* out_index, int32_t* out_count,
                                 void* stream);

/* test_step of EfficientDetNetTrain (efficientnet/efficientdet_net_train.py:135-169) in ONE pass over the heads: focal +
 * Huber partial sums (:141-151; sums_out [2L+1] fp64 as b200_focal_box_partial_sums writes them -> b200_focal_box_finalize
 * / _dp), convert_outputs_boxes (:153, out_decoded[l] (B,H,W,A,4), entries may be NULL) and convert_outputs_one for every
 * image (:156-157; outputs as b200_effdet_postprocess).  The class logits are read once instead of twice.  true_classes
 * are the dense one-hot targets.  b200_effdet_decode_postprocess is the same stream without targets (anchors.py:141-202).
 * Workspace: b200_effdet_eval_workspace_bytes (256-byte aligned). */
size_t b200_effdet_eval_workspace_bytes(int num_levels, const int32_t* hw, int A, int num_images, int max_out);
int b200_effdet_eval_step(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                          const float* const true_boxes[], const float* const true_classes[],
                          const unsigned char* const true_masks[], const float* const pred_boxes[],
                          const float* const pred_classes[], float alpha, float gamma, float delta, float label_smoothing,
                          double* sums_out, float* const out_decoded[], int max_out, float iou_thr, float score_thr,
                          int metric, float* out_boxes, long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                          int32_t* out_sel_anchor, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream);
int b200_effdet_decode_postprocess(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                   const float* const pred_boxes[], const float* const pred_classes[],
                                   float* const out_decoded[], int max_out, float iou_thr, float score_thr, int metric,
                                   float* out_boxes, long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                                   int32_t* out_sel_anchor, int32_t* out_count, void* workspace, size_t workspace_bytes,
                                   void* stream);

/* ---- the collective of the path (SURVEY §8b b200_allreduce_loss, §8e) ------------------------------------------
 * Data parallel over images: the only inter-GPU traffic is the sum of a handful of per-GPU partial loss terms (YOLO:
 * 12 floats; EfficientDet: 2L+1 doubles).  The reference's only collective site is the MirroredStrategy reduce of
 * facenet/facenet_model.py:297,318-322 (strategy.reduce(SUM, per_replica_losses)); its YOLO / EfficientDet train
 * steps are single-replica.  Two transports, both stream-ordered and CUDA-graph capturable:
 *
 * (1) peer mailboxes over NVLink (one process per GPU, CUDA IPC).  Each rank creates a mailbox, hands the 64-byte
 *     handle to its peers by any host channel (torch.distributed, MPI, a file), and maps theirs.  The *_dp entry
 *     points below then do the exchange INSIDE their finalize kernel (peer stores + release/acquire flags, sum in rank
 *     order: identical bits on every rank, no separate collective launch).  mailboxes[r] = rank r's mailbox as mapped
 *     in this process (own one included), world <= 8, n <= 32 values.  A peer that never arrives is reported through
 *     b200_peer_mailbox_status(errors) after 20 s instead of hanging the GPU. */
size_t b200_peer_mailbox_bytes(void);
int b200_peer_mailbox_create(void** mailbox_out, void* ipc_handle_out /* 64 bytes, may be NULL */);
int b200_peer_mailbox_open(const void* ipc_handle /* 64 bytes */, void** mapped_out);
int b200_peer_mailbox_close(void* mapped);
int b200_peer_mailbox_destroy(void* mailbox);
int b200_peer_mailbox_status(const void* own_mailbox, unsigned long long* epoch_out, unsigned int* errors_out); /* synchronous */
/* stand-alone exchange (one warp): values[n] <- sum over ranks, in place */
int b200_allreduce_loss_peer(float* partials, int n, int rank, int world, void* const mailboxes[], void* stream);
int b200_allreduce_sums_peer(double* sums, int n, int rank, int world, void* const mailboxes[], void* stream);
/* protocol self-test on one device: `world` CTAs of one grid play the ranks; out [world, rounds, n] */
int b200_peer_exchange_selftest(int world, int rounds, int n, void* workspace, size_t workspace_bytes, float* out, void* stream);
/* GetLoss / GetLossFromBoxes on one rank's images with the exchange fused into the finalize kernel: batch divisor =
 * global_batch, out_parts / out_loss = the GLOBAL values on every rank (tyu:120-125 order of additions). */
int b200_yolo_loss_dp(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B, int A,
                      int C, const float* anchors_wh_host, const float* image_wh_host, float iou_thresh, int metric,
                      int variant, float global_batch, float* out_parts, float* out_loss, void* workspace,
                      size_t workspace_bytes, int rank, int world, void* const mailboxes[], void* stream);
/* The exchange split in two halves so that the wait can be hidden: b200_yolo_loss_dp_publish ends with the publish half
 * (peer stores, no wait; out_parts / out_loss = this rank's own terms); b200_yolo_loss_collect_peer — on any stream ordered
 * behind it, e.g. a second stream running under the next step — waits for the peers' flags in the local mailbox, sums in
 * rank order and writes the global parts [12] (may be NULL) and loss.  Rule: the publish of step f must be ordered after
 * this rank's own collect of step f-2 (four slot sets; see csrc/exchange.cuh), i.e. one collect may run under the next step. */
int b200_yolo_loss_dp_publish(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B, int A,
                              int C, const float* anchors_wh_host, const float* image_wh_host, float iou_thresh, int metric,
                              int variant, float global_batch, float* out_parts, float* out_loss, void* workspace,
                              size_t workspace_bytes, int rank, int world, void* const mailboxes[], void* stream);
int b200_yolo_loss_collect_peer(float* out_parts, float* out_loss, int rank, int world, void* const mailboxes[], void* stream);
int b200_yolo_loss_from_boxes_dp(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                                 const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                                 int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                 float iou_thresh, int metric, int variant, float global_batch, float* out_parts,
                                 float* out_loss, void* workspace, size_t workspace_bytes, int rank, int world,
                                 void* const mailboxes[], void* stream);
/* _get_loss (edt:41-52) data parallel: sums = this rank's b200_focal_box_partial_sums on entry, the global sums on
 * return; numel_per_level_host = GLOBAL element counts. */
int b200_focal_box_finalize_dp(int num_levels, double* sums, const double* numel_per_level_host, float* out_parts,
                               float* out_loss, float* out_num_positives, int rank, int world, void* const mailboxes[],
                               void* stream);

/* (2) NCCL.  `comm` is an ncclComm_t (passed as void*): the caller's own, or one made by b200_nccl_comm_init from a
 *     128-byte ncclUniqueId that rank 0 obtains with b200_nccl_unique_id and broadcasts.  libnccl.so.2 is opened with
 *     dlopen on first use (env B200_NCCL_LIB overrides the name); ncclAllReduce(sum) in place on `stream`. */
int b200_nccl_unique_id(void* id128_out);
int b200_nccl_comm_init(void** comm_out, int world, int rank, const void* id128);
int b200_nccl_comm_destroy(void* comm);
int b200_allreduce_loss(void* comm /* ncclComm_t */, float* partials, int n, void* stream);
int b200_allreduce_sums(void* comm /* ncclComm_t */, double* sums, int n, void* stream);
/* loss = sum_l ((xy_l + wh_l) + obj_l) + cls_l from the 12 all-reduced terms, the reference's order (tyu:120-125). */
int b200_yolo_loss_combine(const float* parts, float* out_loss, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200DET_H_ */
