/*
 * ysb_postproc.h -- C ABI of the B200-native detection post-processing engine
 * (libysb_postproc.so, built from yoloseries_b200/csrc by yoloseries_b200/build.py).
 *
 * Drop-in boundary for the per-image hot path of yl-jiang/YOLOSeries.  The reference has
 * no FFI of its own (it is pure Python + numba); the interfaces each entry point stands
 * behind are the Python call signatures listed in SURVEY.md section 8b:
 *
 *   ysb_decode            XEvaluator.do_inference          trainer/eval_yolov5.py:181-209, eval_yolov7.py:123-151,
 *                                                          eval_yolox.py:123-150, eval_yolov8.py:75-102,
 *                                                          eval_retinanet.py:59-75 (+22-57,185-200), eval_fcos.py:125-161
 *   ysb_filter_candidates head of XEvaluator.numba_nms     trainer/eval_yolov5.py:265-286 (and the same block in every
 *                         (mask, cls*obj, max/argmax)      eval_*.py; operators per family in SURVEY.md 8a-2)
 *   ysb_select_nms        class offset + utils.numba_nms   trainer/eval_yolov5.py:293-316, utils/nms.py:10-27,
 *                         + max_det + postprocess_bbox     utils/bbox_tools.py:12-35
 *   ysb_postprocess       XEvaluator.__call__ minus model  trainer/eval_yolov5.py:30-42
 *   ysb_postprocess_tta   the same with hyp['use_tta']     trainer/eval_yolov5.py:30-42 + 152-179 (test_time_augmentation)
 *   ysb_decode_into       one pass of test_time_augmentation (decode + scale/flip undo + concat slot)
 *   ysb_elementwise_iou_backward  autograd of the three      loss/yolov5_loss.py:110, yolov7_loss.py:130, yolov8_loss.py:306
 *   ysb_pairwise_iou_backward     autograd of utils.gpu_iou  loss/yolox_loss.py:133, loss/yolov7_loss.py:312
 *   ysb_soft_nms          utils.gpu_*_soft_nms             utils/nms.py:68-140
 *   ysb_undo_letterbox    box half of preds_postprocess    val_yolov5.py:166-172
 *   ysb_wbf, ysb_wbf_collect  weighted_fusion_bbox / do_wfb   utils/weighted_fusion_bbox.py:41-96, trainer/eval_yolov5.py:44-92
 *   ysb_map_iou           utils.mAP.iou                    utils/mAP.py:18-42
 *   ysb_compute_tp        mAP_v2.compute_tp                utils/mAP.py:70-100
 *   ysb_match_tp, ysb_match_compact  the same on the post-processors' own row blocks, + the per-run concatenation
 *   ysb_nms               utils.numba_nms / utils.gpu_nms  utils/nms.py:10-27 / 30-65
 *   ysb_pairwise_iou      utils.numba_iou / utils.gpu_iou  utils/bbox_tools.py:12-35 / 164-190
 *   ysb_elementwise_iou   utils.gpu_Giou/gpu_DIoU/gpu_CIoU utils/bbox_tools.py:193-339
 *
 * Conventions: extern "C"; plain pointers and sizes; every pointer named d_* is a DEVICE
 * pointer owned by the caller; all work is enqueued on the caller's cudaStream_t (passed
 * as void*) and nothing synchronises the host; no hidden allocation (workspace sizes come
 * from the *_workspace_bytes queries); return value is a ysb_status (0 = ok, < 0 = error,
 * never an abort/exception).  There is no CPU fallback: without a CUDA device every
 * compute entry point returns YSB_ERR_CUDA.
 */
#ifndef YSB_POSTPROC_H_
#define YSB_POSTPROC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YSB_ABI_VERSION 6
#define YSB_MAX_LEVELS 8
#define YSB_MAX_ANCHORS 9
#define YSB_MAX_PASSES 4             /* test-time-augmentation passes merged by ysb_postprocess_tta */
#define YSB_MAX_DET_LIMIT 1024      /* max_det upper bound (kept list lives in shared memory) */
/* Sort-key layouts (ysb_filter_candidates): up to 1024 classes the key has 22 candidate bits and 10 class bits; from
 * 1025 to YSB_MAX_CLASSES classes it has 21 candidate bits and 11 class bits, so those calls accept at most
 * YSB_MAX_CANDIDATES_WIDE candidates per image (summed over the passes of a TTA call).  Libraries before 2048-class
 * support refuse num_classes > 1024 with YSB_ERR_LIMIT. */
#define YSB_MAX_CANDIDATES 4194303       /* candidate index must fit 22 bits of the sort key (num_classes <= 1024) */
#define YSB_MAX_CANDIDATES_WIDE 2097151  /* 21 bits: the limit when num_classes > 1024 */
#define YSB_MAX_CLASSES 2048             /* class id must fit 11 bits of the wide sort key */
#define YSB_MAX_PEERS 16            /* ranks (GPUs of one NVLink domain) in a detection gather */
#define YSB_IPC_HANDLE_BYTES 64     /* sizeof(cudaIpcMemHandle_t) */
#define YSB_CNT_ABSENT (-2)         /* gathered count of an image a rank did not have in a partial step */

typedef enum ysb_status {
    YSB_OK = 0,
    YSB_ERR_BAD_ARG = -1,          /* null pointer, negative size, unknown enum value */
    YSB_ERR_UNSUPPORTED = -2,      /* valid request this build does not implement (multi_label for RetinaNet, where the
                                      reference's own branch is broken) */
    YSB_ERR_WORKSPACE = -3,        /* workspace smaller than *_workspace_bytes() */
    YSB_ERR_CUDA = -4,             /* a CUDA call failed; see ysb_last_cuda_error() */
    YSB_ERR_LIMIT = -5             /* N, num_classes or max_det beyond the limits above */
} ysb_status;

typedef enum ysb_family {
    YSB_YOLOV5 = 0,        /* heads: L x (b, A*(5+C), H, W)                       trainer/eval_yolov5.py */
    YSB_YOLOV7 = 1,        /* heads: L x (b, A, H, W, 5+C)                        trainer/eval_yolov7.py */
    YSB_YOLOX = 2,         /* heads: L x (b, A, 5+C, H, W)                        trainer/eval_yolox.py */
    YSB_YOLOV8 = 3,        /* heads: L x (b, 4*bins + C, H, W)                    trainer/eval_yolov8.py */
    YSB_RETINANET = 4,     /* heads: reg (b, N, 4), cls (b, N, C)                 trainer/eval_retinanet.py */
    YSB_RETINANET_EXP = 5, /* heads: reg (b, N, 5), cls (b, N, C)                 trainer/eval_retinanet_experiment.py */
    YSB_FCOS = 6           /* heads: L x cls (b,C,H,W), L x reg (b,4,H,W), L x ctr (b,1,H,W)  trainer/eval_fcos.py */
} ysb_family;

/* Element type of the raw head tensors.  16-bit heads are widened to float32 right after every load (exact): all
 * arithmetic and every output stay float32, bit-identical to a float32 call on the widened heads. */
typedef enum ysb_dtype {
    YSB_F32 = 0,
    YSB_F16 = 1,   /* IEEE binary16 (torch.float16) */
    YSB_BF16 = 2,  /* bfloat16 (torch.bfloat16) */
    YSB_F64 = 3    /* float64: ground truth of ysb_match_step only (heads refuse it) */
} ysb_dtype;

/* What d_heads point to.  RAW_HEADS_NHWC (added in ABI version 6 without a layout change of ysb_params; an older library
 * refuses it with YSB_ERR_BAD_ARG) is raw heads in channels-last memory, as a model run with
 * torch.channels_last emits them.  The logical shapes are those of enum ysb_family, the memory is:
 *   YOLOv5 level (b, H, W, A*(5+C));  YOLOX level (b, H, W, A, 5+C) (the (b, A, 5+C, H, W) view of a channels-last conv);
 *   YOLOv8 level (b, H, W, 4*bins + C);  FCOS cls (b, H, W, C), reg (b, H, W, 4), ctr (b, H, W, 1).
 * Results (rows, det_idx, counts, decoded rows) are bit-identical to RAW_HEADS on the same values.  YOLOv7 and RetinaNet
 * heads already are rows: kind 2 returns YSB_ERR_BAD_ARG for them.  A candidate's channels form one row that the filter
 * kernel stages in shared memory: rows wider than that tile allows (5+C, 4*bins+C or C above ~450) return YSB_ERR_LIMIT.
 * Every entry point that takes raw heads accepts it, with every head_dtype; the passes of one TTA call share one kind. */
typedef enum ysb_input_kind {
    YSB_INPUT_RAW_HEADS = 0,      /* raw model outputs (contiguous NCHW); decode is fused into the filter/NMS kernels */
    YSB_INPUT_DECODED_ROWS = 1,   /* the (b, N, C') tensor do_inference returns; heads[0] points at it */
    YSB_INPUT_RAW_HEADS_NHWC = 2  /* raw model outputs in channels-last memory (above) */
} ysb_input_kind;

/* IoU flavours.  NUMBA_F64MIX is the live path (utils/bbox_tools.py:12-35: float32 sides/areas,
 * float64 product/denominator/quotient, no clamp, NaN for 0/0); the others are the float32 torch
 * routines behind gpu_nms (utils/bbox_tools.py:164-339). */
typedef enum ysb_iou_kind {
    YSB_IOU_NUMBA_F64MIX = 0,
    YSB_IOU_F32 = 1,
    YSB_GIOU = 2,
    YSB_DIOU = 3,
    YSB_CIOU = 4
} ysb_iou_kind;

typedef enum ysb_cmp { YSB_CMP_GE = 0 /* numba_nms: iou >= thr */, YSB_CMP_GT = 1 /* gpu_nms: iou > thr */ } ysb_cmp;

/* One description of "which heads, which thresholds".  Plain data, passed by pointer, copied by the callee. */
typedef struct ysb_params {
    int32_t family;            /* ysb_family */
    int32_t input_kind;        /* ysb_input_kind */
    int32_t batch;             /* images in this call */
    int32_t num_classes;       /* C */
    int32_t img_h, img_w;      /* network input size (letterboxed pixels) */
    int32_t num_levels;        /* L (RetinaNet: 5 pyramid levels 3..7) */
    int32_t level_h[YSB_MAX_LEVELS];
    int32_t level_w[YSB_MAX_LEVELS];
    float level_stride[YSB_MAX_LEVELS];
    int32_t anchors_per_cell;  /* A: 3 (v5/v7), num_anchors (YOLOX), 9 (RetinaNet), 1 otherwise */
    /* v5/v7: anchor[l][a] = {w/stride, h/stride, 0, 0} as float32 (eval_yolov5.py:192);
     * RetinaNet: the 9 base anchors {x1,y1,x2,y2} of level l (utils/anchor.py:176-191). */
    float anchor[YSB_MAX_LEVELS][YSB_MAX_ANCHORS][4];
    float reg_scale[4];        /* RetinaNet tar_box_scale_factor (eval_retinanet.py:36-39) */
    int32_t dfl_bins;          /* YOLOv8 'reg' (16) */
    /* thresholds: float32 because numpy compares float32 arrays with Python floats in float32 */
    float conf_thr;            /* conf_threshold */
    float cls_thr;             /* cls_threshold */
    float pre_nms_thr;         /* FCOS pre_nms_thresh */
    double iou_thr;            /* iou_threshold, compared in float64 (utils/nms.py:22) */
    int32_t max_det;           /* max_predictions_per_img */
    int32_t class_aware;       /* hyp['agnostic'] (sic): add cls*4096 to the boxes before NMS */
    int32_t multi_label;       /* hyp['mutil_label'] (sic): one record per (candidate, class) above cls_thr */
    int32_t postprocess_bbox;  /* hyp['postprocess_bbox'] */
    float min_box_wh;          /* min_prediction_box_wh (v7 / FCOS remove_small_boxes) */
    int32_t pre_nms_topk;      /* FCOS pre_nms_topk */
    int32_t thresh_with_ctr;   /* FCOS thresh_with_ctr */
    int32_t decoded_rows;      /* DECODED_ROWS input only: rows per image when it is not the family's own N
                                  (e.g. the concatenation of three TTA passes, eval_yolov5.py:152-179); 0 = N */
    /* Test-time-augmentation undo of ONE pass (test_time_augmentation, eval_yolov5.py:152-179, eval_yolov8.py:40-73,
     * eval_retinanet.py:148-182, eval_fcos.py:90-123), applied to the four box columns right after the decode, RAW_HEADS
     * input only:  box /= tta_scale (float32 division; 0 or 1 = off), then for tta_flip == 2 (picture flipped along h)
     * cy = tta_img_h - cy   or   (y1, y2) = (tta_img_h - y2, tta_img_h - y1);  tta_flip == 3 (along w) likewise with x and
     * tta_img_w.  tta_img_h/w are the size of the UN-augmented input (img_h/img_w above describe the padded pass). */
    float tta_scale;
    int32_t tta_flip;          /* 0 none, 2, 3: the reference's flip_axis values */
    int32_t tta_img_h, tta_img_w;
    /* Optional letterbox undo fused into the row write of ysb_select_nms / ysb_postprocess(_tta) (the first consumer of
     * the kept rows, val_yolov5.py:166-172 preds_postprocess): DEVICE pointer to (batch, 5) float32
     * {scale, pad_top, pad_left, org_h, org_w}, or NULL = rows stay in network-input pixels (the reference's evaluator
     * output).  Same arithmetic as ysb_undo_letterbox; applied after NMS, the postprocess_bbox count filter and
     * remove_small_boxes, which all see the un-mapped boxes exactly like the reference. */
    const float *d_letterbox;
    /* ysb_dtype of every tensor in d_heads (RAW_HEADS input; one type per call, every TTA pass the same).  0 = float32,
     * so a zero-filled struct keeps the float32 behaviour.  DECODED_ROWS input is float32 only: another value there, an
     * unknown value or passes of different types return YSB_ERR_BAD_ARG. */
    int32_t head_dtype;
} ysb_params;

int ysb_abi_version(void);
const char *ysb_status_string(int status);
/* cudaError_t of the last failing CUDA call made by this library on the calling thread (0 if none). */
int ysb_last_cuda_error(void);

/* N = candidates per image and the row width C' of the decoded tensor for these params. */
int ysb_num_candidates(const ysb_params *p, int64_t *n_out, int32_t *row_width_out);

/* do_inference: raw heads -> d_decoded (batch, N, C') float32, reference row layout per family. */
int ysb_decode(const ysb_params *p, const void *const *d_heads, int num_heads, float *d_decoded, void *stream);

/* The same decode written into a larger tensor: d_decoded is (batch, rows_total, C') and this pass fills rows
 * [row_offset, row_offset + N) of every image -- with the tta_* undo of the params applied, three calls build the merged
 * tensor of test_time_augmentation (eval_yolov5.py:179, torch.cat(aug_preds, dim=1)) without an intermediate copy. */
int ysb_decode_into(const ysb_params *p, const void *const *d_heads, int num_heads, float *d_decoded, int64_t rows_total,
                    int64_t row_offset, void *stream);

/* Filter + class pick + compaction.  d_keys: (batch, key_capacity) uint64 sort keys
 *   key = score_bits << 32 | (YSB_MAX_CANDIDATES - cand) << 10 | (1023 - cls)         num_classes <= 1024
 *   key = score_bits << 32 | (YSB_MAX_CANDIDATES_WIDE - cand) << 11 | (2047 - cls)   num_classes 1025..2048
 * so that "descending key" == (score desc, candidate asc, class asc), the order numba_nms visits boxes.
 * d_counts: (batch, 4) int32 = {survivors M, pre-mask passes (FCOS top-k), max score bits, ~min score bits};
 * zero-filled by this call before the kernels run.  key_capacity >= N (N*C with multi_label). */
int ysb_filter_candidates(const ysb_params *p, const void *const *d_heads, int num_heads, uint64_t *d_keys,
                          int64_t key_capacity, int32_t *d_counts, void *stream);

/* Top-k selection + sort + greedy class-aware NMS (early exit at max_det) + postprocess_bbox count filter
 * (+ RetinaNet merge, + remove_small_boxes) for every image.
 *   d_dets   (batch, max_det, 6) float32 rows [x1, y1, x2, y2, score, cls], NMS keep order
 *   d_det_idx(batch, max_det) int32 original candidate index of every row (may be NULL)
 *   d_det_cnt(batch) int32 number of rows; -1 where the reference returns None */
int ysb_select_nms(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                   int64_t key_capacity, const int32_t *d_counts, float *d_dets, int32_t *d_det_idx,
                   int32_t *d_det_cnt, void *stream);

/* Whole path = ysb_filter_candidates + ysb_select_nms with the intermediates in d_workspace. */
int ysb_postprocess_workspace_bytes(const ysb_params *p, size_t *bytes_out);
int ysb_postprocess(const ysb_params *p, const void *const *d_heads, int num_heads, void *d_workspace,
                    size_t workspace_bytes, float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, void *stream);

/* XEvaluator.__call__ with hyp['use_tta'] (eval_yolov5.py:30-42 + 152-179) minus the model forwards: num_passes
 * parameter sets (same family / thresholds / batch, own geometry and tta_* undo each) and their raw heads, concatenated in
 * d_heads (heads_per_pass[i] pointers for pass i).  Candidate index space = the concatenation of the passes in order, as
 * in the reference's merged tensor; the merged (b, sum N_i, C') tensor is never materialised: every pass runs the filter
 * kernel on its own heads appending to one key list per image, and ONE selection/NMS kernel decodes the boxes of the
 * candidates it visits from the pass they belong to.  Outputs as ysb_select_nms (d_det_idx = merged candidate index). */
int ysb_postprocess_tta_workspace_bytes(const ysb_params *passes, int num_passes, size_t *bytes_out);
int ysb_postprocess_tta(const ysb_params *passes, int num_passes, const void *const *d_heads, const int32_t *heads_per_pass,
                        void *d_workspace, size_t workspace_bytes, float *d_dets, int32_t *d_det_idx,
                        int32_t *d_det_cnt, void *stream);
/* The two halves of ysb_postprocess_tta, for callers that own their key buffers (the pass list follows the same rules).
 * d_keys (batch, key_capacity) uint64, d_counts (batch, 4) int32 as in ysb_filter_candidates; key_capacity >= the summed
 * key slots of the passes (N_i each, N_i*C with multi_label), else YSB_ERR_WORKSPACE.  ysb_filter_candidates_tta runs
 * the filter kernel of every pass, all appending to one key list per image; it zero-fills d_counts before the first
 * pass.  ysb_select_nms_tta: outputs as ysb_postprocess_tta.  ysb_select_nms_tta_gather: the same, its rows and counts
 * stored into every rank's slot like ysb_select_nms_gather (g->batch and g->max_det must match the passes; d_det_idx
 * stays local, may be NULL).  Every refusal returns before any CUDA call. */
int ysb_filter_candidates_tta(const ysb_params *passes, int num_passes, const void *const *d_heads,
                              const int32_t *heads_per_pass, uint64_t *d_keys, int64_t key_capacity, int32_t *d_counts,
                              void *stream);
int ysb_select_nms_tta(const ysb_params *passes, int num_passes, const void *const *d_heads, const int32_t *heads_per_pass,
                       const uint64_t *d_keys, int64_t key_capacity, const int32_t *d_counts, float *d_dets,
                       int32_t *d_det_idx, int32_t *d_det_cnt, void *stream);

/* Greedy NMS over one explicit box/score array (utils.numba_nms / utils.gpu_nms).
 *   d_boxes (m,4) float32, d_scores (m) float32 >= 0 (zero scores are never kept, utils/nms.py:16)
 *   max_keep: stop after this many keeps (<= 0: run to exhaustion like the reference)
 *   d_keep (min(m, max_keep or m)) int32, d_keep_cnt (1) int32 */
int ysb_nms_workspace_bytes(int64_t m, size_t *bytes_out);
int ysb_nms(const float *d_boxes, const float *d_scores, int64_t m, double iou_thr, int cmp, int iou_kind,
            int64_t max_keep, void *d_workspace, size_t workspace_bytes, int32_t *d_keep, int32_t *d_keep_cnt,
            void *stream);

/* Backward of ysb_elementwise_iou for the loss-side callers that differentiate through gpu_CIoU (loss/yolov5_loss.py:110,
 * loss/yolov7_loss.py:130, loss/yolov8_loss.py:306, loss/loss.py:109) / gpu_Giou / gpu_DIoU: given d_grad_out (n2) it
 * writes dL/d_b2 (n2,4) and dL/d_b1 (n1,4; summed over the rows when n1 == 1).  Either gradient pointer may be NULL.
 * torch's sub-gradient conventions (ties of max/min split evenly, clamp passes the gradient on its bounds, alpha of CIoU
 * constant).  float32 throughout. */
int ysb_elementwise_iou_backward(const float *d_b1, int64_t n1, const float *d_b2, int64_t n2, int iou_kind,
                                 const float *d_grad_out, float *d_grad_b1, float *d_grad_b2, void *stream);

/* Backward of the float32 pairwise IoU (ysb_pairwise_iou with YSB_IOU_F32 = utils.gpu_iou, utils/bbox_tools.py:164-190):
 * the label assignment of loss/yolox_loss.py:133 and loss/yolov7_loss.py:312 calls gpu_iou(tar_box, pred_box) with grad
 * enabled (`torch.no_grad()` at yolox_loss.py:92 is a bare statement, not a decorator), so patching utils.gpu_iou needs it.
 * d_grad_out (n, m) -> dL/d_b1 (n,4) = sum over columns, dL/d_b2 (m,4) = sum over rows (float64 accumulation, float32
 * results).  Either gradient pointer may be NULL.  All box / gradient pointers 16-byte aligned. */
int ysb_pairwise_iou_backward(const float *d_b1, int64_t n, const float *d_b2, int64_t m, const float *d_grad_out,
                              float *d_grad_b1, float *d_grad_b2, void *stream);

/* Weighted-box-fusion (hyp['wfb'], utils/weighted_fusion_bbox.py:63-96 + update_fusion_bbox :41-60; caller
 * trainer/eval_yolov5.py:44-92 do_wfb, identical in eval_yolov7.py / eval_yolox.py).
 * ysb_wbf: d_rows (batch, stride, row_width) float32 rows (x1, y1, x2, y2, score, label, weight[, position]); image i
 * holds d_counts[i] <= stride rows.  row_width 8: column 7 carries, as uint32 bits, the row's position in the reference's
 * stacked list (rows may then be stored in any order); row_width 7: storage order is that position.  Per image and label
 * (ascending), boxes are visited by descending score (equal scores: the later row first -- argsort()[::-1] of a stable
 * sort; numpy's default sort is only stable up to 16 elements, unpinned beyond); a box joins every cluster whose fused
 * box it meets with cpu_iou >= iou_thr (float32 box area, float64 otherwise, utils/bbox_tools.py:63-84), else it founds
 * one; fused box = mean over members of box*score/sum(score) -- i.e. the score-weighted mean divided by the member
 * count AGAIN, the reference's arithmetic, kept --, fused score = sum(score*weight)/sum(weight).  float64; cluster sums
 * are kept incrementally (the reference re-sums every cluster after every box: values agree to ~1e-15 relative).
 * Outputs, all (batch, stride[, .]): d_order int32 = row visited at every sorted position; the clusters of a label occupy
 * consecutive slots from the label's first sorted position: d_members int32 = member count (0 = no cluster in this
 * slot), d_fusion float64 (.., 6) = (x1, y1, x2, y2, score, label).  d_pairs (pair_capacity, 2) int32 + d_pair_count (1)
 * uint64, both optional: (cluster slot, sorted position) of every membership as indices into the flattened
 * (batch * stride) arrays, unordered; the count may exceed the
 * capacity (call again with more).  d_status (batch) int32: 1 = the best box of some label does not meet itself
 * (degenerate box; the reference raises IndexError there).
 * ysb_wbf_collect: do_wfb's per-pass filter on the decoded (batch, rows, 5 + C) tensor of all passes (xywh, obj, C class
 * scores; pass q owns pass_rows[q] consecutive rows and weight pass_weights[q], HOST arrays): obj > skip_thr, conf =
 * cls * obj, best class with conf > skip_thr (multi_label: every class above it), xywh -> xyxy -> d_records
 * (batch, capacity, 8) rows as above with positions, d_counts (batch).  Survivors beyond capacity are counted, not stored. */
int ysb_wbf_workspace_bytes(int batch, int64_t stride, size_t *bytes_out);
int ysb_wbf(const float *d_rows, int row_width, const int32_t *d_counts, int batch, int64_t stride, double iou_thr,
            void *d_workspace, size_t workspace_bytes, int32_t *d_order, double *d_fusion, int32_t *d_members,
            int32_t *d_pairs, int64_t pair_capacity, uint64_t *d_pair_count, int32_t *d_status, void *stream);
int ysb_wbf_collect(const float *d_decoded, int batch, int64_t rows, int row_width, int num_classes, float skip_thr,
                    int multi_label, const int64_t *pass_rows, const float *pass_weights, int num_passes,
                    float *d_records, int32_t *d_counts, int64_t capacity, void *stream);

/* Self-test of the arithmetic the parity claims rest on: the sigmoid's reciprocal is spelled out (MUFU.RCP + one FMA
 * Newton step) instead of calling __frcp_rn; this compares the two for every float in [1, +inf] on the device.
 * d_mismatches (2) uint64: {values where the guarded routine differs, values where the branch-free batch variant differs
 * or mis-flags its out-of-range case}.  Both must come back 0. */
int ysb_selftest_reciprocal(uint64_t *d_mismatches, void *stream);

/* Tuning / test hook: CTA flavour of the selection + NMS kernel.  0 (default): chosen per call from the batch size and the
 * family (csrc/nms_kernel.cu, launch_any); 512 / 1024: forced (512 only applies while max_det <= 320).  Both flavours give
 * bit-identical results (tests/test_gpu_edge.py::test_nms_cta_flavours_agree_with_the_oracle).  Process-wide, not
 * thread-safe: meant for A/B measurements and tests.  No reference counterpart. */
int ysb_set_nms_cta_threads(int threads);

/* mAP hand-off (the consumer of the kept rows, val_yolov5.py:388 -> utils/mAP.py).
 * ysb_map_iou: utils/mAP.py:18-42 `iou(box1, box2)` -- rows of row_w1 / row_w2 values whose first four are
 * (x1, y1, x2, y2); float32 or float64 (is_f64) in, the same type out, (n, m);  inter / clip(a1 + a2 - inter, 1e-6, 1e7).
 * ysb_compute_tp: utils/mAP.py:70-100 `mAP_v2.compute_tp(gt, pred)` for a batch of images in one launch.  d_gt: all
 * images' ground-truth rows (x1, y1, x2, y2, cls) concatenated, d_pred: all kept rows (x1, y1, x2, y2, score, cls)
 * concatenated, *_offsets (batch + 1) int64 row offsets on the device.  iou_thresholds: 10 HOST doubles
 * (np.linspace(0.5, 0.95, 10)).  d_tp (total_pred, 10) uint8 <- the reference's bool matrix: pairs with
 * iou >= thr[0] and equal label are ranked by IoU, every prediction keeps its best ground-truth box, every ground-truth
 * box then keeps the LOWEST-index prediction that chose it (the reference's second np.unique runs over a list ordered
 * by prediction index), and tp[j, t] = iou >= thr[t] in float64.  Equal IoUs for one prediction: the larger ground-truth
 * index wins (argsort()[::-1] of a stable sort; numpy's default sort is only stable up to 16 elements -- unpinned beyond).
 * Workspace: one int32 per ground-truth row. */
int ysb_map_iou(const void *d_box1, int64_t n, int row_w1, const void *d_box2, int64_t m, int row_w2, int is_f64,
                void *d_out, void *stream);
int ysb_compute_tp_workspace_bytes(int64_t total_gt, size_t *bytes_out);
int ysb_compute_tp(const void *d_gt, const int64_t *d_gt_offsets, int64_t total_gt, const void *d_pred,
                   const int64_t *d_pred_offsets, int64_t total_pred, int batch, int is_f64, const double *iou_thresholds,
                   void *d_workspace, size_t workspace_bytes, uint8_t *d_tp, void *stream);

/* The same matching on the rows where the post-processors keep them: a (world, batch, max_det, 6) float32 block (the
 * rows of DetectionBuffers with world = 1, or one gather slot, ysb_gather_slot_views / ysb_gather_strides) and its
 * (world, batch) counts, against padded ground truth.  Image k = rank * batch + i; one step = one such block.
 *   count c >= 0: c rows;  -1 (the reference's None): no rows, the image's ground truth still counts as targets;
 *   YSB_CNT_ABSENT: the image is not part of the step (partial gather steps): skipped, its tp rows are left untouched.
 * Ground truth rows (x1, y1, x2, y2, cls) are gt_dtype, one type per call: YSB_F32 matches in float32, YSB_F64 in
 * float64 with the float32 rows widened exactly -- what ysb_compute_tp computes on the promoted arrays.  Counts above
 * max_gt (or max_det) are clamped to it. */
typedef struct ysb_match_step {
    int32_t world, batch, max_det, max_gt;
    const float *d_rows;         /* rank r's (batch, max_det, 6) rows start r * rows_rank_bytes after d_rows */
    int64_t rows_rank_bytes;     /* >= batch * max_det * 24 */
    const int32_t *d_cnt;        /* rank r's (batch) counts start r * cnt_rank_bytes after d_cnt */
    int64_t cnt_rank_bytes;      /* >= batch * 4 */
    const void *d_gt;            /* (world, batch, max_gt, 5) gt_dtype, dense */
    const int32_t *d_gt_cnt;     /* (world, batch) int32, dense: ground-truth rows of every image */
    int32_t gt_dtype;            /* YSB_F32 or YSB_F64 */
} ysb_match_step;

/* ysb_match_tp: d_tp (world, batch, max_det, 10) uint8 <- for every present image, ysb_compute_tp of its ground truth
 * and its rows, bit for bit, aligned with the rows (rows past the count are not written).  iou_thresholds: 10 HOST
 * doubles.  One launch, one CTA per image.  Workspace: one int32 per ground-truth slot (world * batch * max_gt).
 * ysb_match_compact: appends the step's present images, in image order, to the caller's run-long arrays: per kept
 * row d_conf[p] = score, d_pred_cls[p] = class (float32) and d_tp_out[p] (10 uint8, from d_tp of ysb_match_tp); per
 * ground-truth row d_target_cls[g] = class (float64).  d_acc_in = {rows, targets} appended so far (int64, device), read;
 * d_acc_out (another 2 int64) <- d_acc_in + the step's rows and targets: feed it to the next step as d_acc_in.  Rows
 * or targets beyond the capacities are counted in d_acc_out but not written.  The result is the concatenation of
 * mAP_v2.compute_tp over the images in order, the arrays the AP integration consumes.
 * Both refuse, before any CUDA call: null pointers, negative sizes, world < 1 or > YSB_MAX_PEERS, strides smaller than
 * a rank's rows / counts, max_det > YSB_MAX_DET_LIMIT (YSB_ERR_LIMIT), an unknown gt_dtype, d_acc_in == d_acc_out. */
int ysb_match_tp_workspace_bytes(const ysb_match_step *step, size_t *bytes_out);
int ysb_match_tp(const ysb_match_step *step, const double *iou_thresholds, void *d_workspace, size_t workspace_bytes,
                 uint8_t *d_tp, void *stream);
int ysb_match_compact(const ysb_match_step *step, const uint8_t *d_tp, const int64_t *d_acc_in, int64_t *d_acc_out,
                      float *d_conf, float *d_pred_cls, uint8_t *d_tp_out, int64_t row_capacity, double *d_target_cls,
                      int64_t target_capacity, void *stream);

/* Soft-NMS (utils/nms.py:68-140; no caller in the reference, float32 GIoU/DIoU/CIoU flavours only -- 'iou' is broken
 * there).  Repeats: pick the first arg-max, record processed[idx] = its current score, decay every score whose IoU with
 * it exceeds iou_thr by (1 - iou) (mode 0, linear) or exp(-iou^2 / sigma) (mode 1, exponential), until no score is > 0.
 * d_processed (m) float32 receives the recorded scores (0 where never picked); the caller thresholds them.
 * Workspace: m floats.  The loop is capped at max(64, 104*sigma + 2) * m + 1024 picks: in exponential mode a picked box
 * only decays itself by exp(-1/sigma), so the reference loops until float32 underflow (~104*sigma picks per box), and it
 * never terminates when a self-IoU does not exceed the threshold. */
int ysb_soft_nms(const float *d_boxes, const float *d_scores, int64_t m, float iou_thr, int iou_kind, int mode,
                 float sigma, void *d_workspace, size_t workspace_bytes, float *d_processed, void *stream);

/* "Next" row after the path (val_yolov5.py:140-179, preds_postprocess): undo the letterbox on the kept rows in place.
 * d_info (batch, 5) float32 = {scale, pad_top, pad_left, org_h, org_w}:  x = clamp((x - pad_left) / scale, 1, org_w - 1),
 * y = clamp((y - pad_top) / scale, 1, org_h - 1), float32, one rounding per operation. */
int ysb_undo_letterbox(float *d_dets, const int32_t *d_det_cnt, int batch, int max_det, const float *d_info, void *stream);

/* ---- multi-GPU: all-gather of the kept detections fused into the NMS kernel (SURVEY.md 8b item 6, 8e) ----------------
 * Images shard over the ranks (one process per GPU); the only exchange on the path is the final all-gather of every
 * rank's fixed-stride rows (batch, max_det, 6) + counts (batch) for mAP evaluation.  The reference has no such step (its
 * val sampler is not rank-sliced, dataset/data_sampler.py:185-192; the closest is the unused pickle-over-gloo all_gather
 * of utils/dist.py:176-211).  Here there is NO collective launch: every rank owns one symmetric receive buffer that its
 * peers map over NVLink (CUDA IPC), and the NMS kernel's ordered row write stores each row straight into every peer's
 * slot, followed by one system-scope arrival count per image.  Slots = batches in flight per rank.
 *
 *   buffer layout (identical on every rank, zero-initialised):
 *     rows    [slots][world][batch][max_det][6] f32     cnt  [slots][world][batch] i32
 *     arrived [slots][world] u32  (images of peer r that have landed in this slot, cumulative)
 *     ack     [slots][world] u32  (peer r has finished reading use u of MY slot region: I may overwrite it)
 *     use     [slots] u32 (completed uses of the slot, local)      err [1] u32 (a spin timed out, local)
 *   per step and slot, all on the caller's stream:
 *     ysb_gather_begin       zero the filter counters, tell every peer "I have consumed the previous use of this slot"
 *                            (a remote store per peer, no waiting)
 *     ysb_filter_candidates, ysb_select_nms_gather  (or, for test-time augmentation, ysb_filter_candidates_tta and
 *                            ysb_select_nms_tta_gather)  (each image's CTA waits for the peers' acks of this slot -- sent a
 *                            whole filter + NMS pass earlier -- then rows + counts -> every peer's slot, then arrival counts)
 *     ysb_gather_wait        wait until the rows of every rank have landed in MY slot
 *   Every rank must run the same sequence of (slot) steps.  Spins are bounded (~20 s); a timeout sets `err`, which
 *   ysb_gather_error reads back (host sync).
 *   Partial steps (the tail of a dataset that is not a multiple of world * batch): a rank that holds n < g->batch images
 *   in a step calls ysb_select_nms_gather_partial (or ysb_select_nms_tta_gather_partial) with a plan of batch n, 0
 *   included, in place of the strict entry; the rest of its step is unchanged.  The NMS kernel runs for images [0, n)
 *   (no launch for n = 0), then one small kernel waits for every peer's ack of the slot, stores YSB_CNT_ABSENT into
 *   every rank's count words of images [n, g->batch) and adds g->batch - n to the arrival counters, so every rank still
 *   arrives with g->batch images per step and ysb_gather_wait works unchanged.  Rows of absent images are unspecified. */
typedef struct ysb_gather {
    int32_t world, rank, slots, batch, max_det;
    void *d_buf[YSB_MAX_PEERS];   /* d_buf[rank] = own buffer (ysb_gather_alloc), the others = ysb_gather_open mappings */
} ysb_gather;

int ysb_gather_buffer_bytes(int world, int slots, int batch, int max_det, size_t *bytes_out);
/* cudaMalloc + zero fill on the current device; handle_out (YSB_IPC_HANDLE_BYTES) is what the peers pass to _open. */
int ysb_gather_alloc(size_t bytes, void **d_buf_out, unsigned char *handle_out);
int ysb_gather_open(const unsigned char *handle, void **d_peer_buf_out);
int ysb_gather_close(void *d_peer_buf);
int ysb_gather_free(void *d_buf);
/* pointers into the OWN buffer: rows (world, batch, max_det, 6) f32 and counts (world, batch) i32 of one slot */
int ysb_gather_slot_views(const ysb_gather *g, int slot, float **d_rows_out, int32_t **d_cnt_out);
/* the per-rank regions inside a slot are padded to 256 bytes: rank r's rows start r * rows_rank_bytes after d_rows_out */
int ysb_gather_strides(const ysb_gather *g, int64_t *rows_rank_bytes, int64_t *cnt_rank_bytes);
int ysb_gather_begin(const ysb_gather *g, int slot, int32_t *d_counts, int64_t n_counts, void *stream);
/* ysb_select_nms whose rows/counts go to every rank's slot (d_det_idx stays local, may be NULL). */
int ysb_select_nms_gather(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                          int64_t key_capacity, const int32_t *d_counts, const ysb_gather *g, int slot,
                          int32_t *d_det_idx, void *stream);
/* ysb_select_nms_tta whose rows/counts go to every rank's slot (declared here because it needs ysb_gather). */
int ysb_select_nms_tta_gather(const ysb_params *passes, int num_passes, const void *const *d_heads,
                              const int32_t *heads_per_pass, const uint64_t *d_keys, int64_t key_capacity,
                              const int32_t *d_counts, const ysb_gather *g, int slot, int32_t *d_det_idx, void *stream);
/* Partial steps: the arguments of ysb_select_nms_gather / ysb_select_nms_tta_gather, but the plan may hold
 * 0 <= batch <= g->batch images (max_det must still match); images [batch, g->batch) of this rank read YSB_CNT_ABSENT in
 * every rank's slot.  Every refusal returns before any CUDA call. */
int ysb_select_nms_gather_partial(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                                  int64_t key_capacity, const int32_t *d_counts, const ysb_gather *g, int slot,
                                  int32_t *d_det_idx, void *stream);
int ysb_select_nms_tta_gather_partial(const ysb_params *passes, int num_passes, const void *const *d_heads,
                                      const int32_t *heads_per_pass, const uint64_t *d_keys, int64_t key_capacity,
                                      const int32_t *d_counts, const ysb_gather *g, int slot, int32_t *d_det_idx,
                                      void *stream);
int ysb_gather_wait(const ysb_gather *g, int slot, void *stream);
int ysb_gather_error(const ysb_gather *g, uint32_t *err_out);

/* (n,4) x (m,4) -> (n,m).  kind NUMBA_F64MIX writes float64 (numba_iou), F32 writes float32 (gpu_iou). */
int ysb_pairwise_iou(const float *d_b1, int64_t n, const float *d_b2, int64_t m, int iou_kind, void *d_out,
                     void *stream);
/* Row-wise GIoU / DIoU / CIoU with the reference's (1|n,4) x (n,4) broadcasting -> (n) float32. */
int ysb_elementwise_iou(const float *d_b1, int64_t n1, const float *d_b2, int64_t n2, int iou_kind, float *d_out,
                        void *stream);

#ifdef __cplusplus
}
#endif
#endif /* YSB_POSTPROC_H_ */
