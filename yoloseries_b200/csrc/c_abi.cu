// c_abi.cu -- extern "C" entry points of libysb_postproc.so (see include/ysb_postproc.h).
//
// Translates the caller's plain ysb_params + head pointers into the device Plan (geometry + the per-family filter
// operators of SURVEY.md 8a-2), validates limits, and enqueues the kernels on the caller's stream.  No allocation,
// no host synchronisation, no exceptions across the boundary.
#include <cstdio>
#include <cstring>

#include "ysb_internal.cuh"

namespace ysb {
// dtype: ysb_dtype of the heads the Plan points at
cudaError_t launch_filter(const Plan &P, int vec, uint64_t *d_keys, int64_t key_cap, int32_t *d_counts, cudaStream_t stream,
                          bool zero_counts, int dtype);
cudaError_t launch_select_nms(const Plan &P, const uint64_t *d_keys, int64_t key_cap, const int32_t *d_counts,
                              float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, cudaStream_t stream,
                              const GatherSink *sink, int dtype);
bool make_gather_sink(const ysb_gather *g, int slot, GatherSink *out);
bool gather_valid(const ysb_gather *g, int slot);
cudaError_t launch_gather_begin(const ysb_gather *g, int slot, int32_t *d_counts, int64_t n_counts, cudaStream_t stream);
cudaError_t launch_gather_wait(const ysb_gather *g, int slot, cudaStream_t stream);
cudaError_t launch_gather_absent(const GatherSink &sink, int first, int batch, cudaStream_t stream);
cudaError_t launch_select_nms_tta(const Plan &P, const ExtraPasses &X, const uint64_t *d_keys, int64_t key_cap,
                                  const int32_t *d_counts, float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt,
                                  cudaStream_t stream, const GatherSink *sink, int dtype);
cudaError_t launch_decode(const Plan &P, float *d_out, int64_t rows_total, int64_t row_offset, cudaStream_t stream,
                          int dtype);
cudaError_t launch_array_nms(const float *d_boxes, const float *d_scores, int64_t m, double iou_thr, int cmp, int iou_kind,
                             int64_t max_keep, void *ws, int32_t *d_keep, int32_t *d_keep_cnt, cudaStream_t stream);
size_t array_nms_workspace_bytes(int64_t m);
cudaError_t launch_pairwise_iou(const float *b1, int64_t n, const float *b2, int64_t m, int kind, void *out, cudaStream_t stream);
cudaError_t launch_elementwise_iou(const float *b1, int64_t n1, const float *b2, int64_t n2, int kind, float *out,
                                   cudaStream_t stream);

#ifdef YSB_K2_TIMING
cudaError_t debug_k2_timing(long long *host_out);
#endif
void debug_set_nms_threads(int t);

cudaError_t launch_elementwise_iou_backward(const float *b1, int64_t n1, const float *b2, int64_t n2, int kind,
                                            const float *grad_out, float *g1, float *g2, cudaStream_t stream);
size_t wbf_workspace_bytes(int batch, int64_t stride);
cudaError_t launch_wbf(const float *rows, int row_w, const int32_t *counts, int batch, int64_t stride, double thr, void *ws,
                       int32_t *order, double *fusion, int32_t *members, int32_t *pairs, long long pair_cap,
                       unsigned long long *pair_count, int32_t *status, cudaStream_t stream);
cudaError_t launch_wbf_collect(const float *decoded, int batch, int64_t rows, int row_w, int C, float thr, int multi,
                               const int64_t *pass_rows, const float *pass_weights, int n_pass, float *rec, int32_t *counts,
                               int64_t cap, cudaStream_t stream);
cudaError_t launch_selftest_reciprocal(unsigned long long *d_mismatches, cudaStream_t stream);
cudaError_t launch_map_iou(const void *b1, int64_t n, int w1, const void *b2, int64_t m, int w2, int f64, void *out,
                           cudaStream_t stream);
cudaError_t launch_compute_tp(const void *gt, const int64_t *gt_off, const void *pred, const int64_t *pred_off, int batch,
                              int f64, const double *thr10, int32_t *first_pred, uint8_t *tp, cudaStream_t stream);
cudaError_t launch_match_tp(const ysb_match_step &s, const double *thr10, int32_t *first_pred, uint8_t *tp,
                            cudaStream_t stream);
cudaError_t launch_match_compact(const ysb_match_step &s, const uint8_t *tp, const int64_t *acc_in, int64_t *acc_out,
                                 float *conf, float *pred_cls, uint8_t *tp_out, int64_t row_cap, double *target_cls,
                                 int64_t target_cap, cudaStream_t stream);
cudaError_t launch_pairwise_iou_backward(const float *b1, int64_t n, const float *b2, int64_t m, const float *grad_out,
                                         float *g1, float *g2, cudaStream_t stream);
cudaError_t launch_soft_nms(const float *boxes, const float *scores, int64_t m, float thr, int kind, int mode, float sigma,
                            void *ws, float *processed, cudaStream_t stream);
cudaError_t launch_undo_letterbox(float *dets, const int32_t *cnt, int batch, int max_det, const float *info, cudaStream_t stream);

static thread_local int g_last_cuda_error = 0;

static int cuda_status(cudaError_t e)
{
    if (e == cudaSuccess) return YSB_OK;
    g_last_cuda_error = static_cast<int>(e);
    return YSB_ERR_CUDA;
}

// key slots per image: one per candidate, or one per (candidate, class) with mutil_label
static int64_t key_slots(const Plan &P) { return static_cast<int64_t>(P.N) * (P.multi_label ? P.C : 1); }

struct Built {
    Plan plan;
    int vec;  // 4-element vector loads possible for the planes kernel
    int heads_expected;
    int dtype;  // ysb_dtype of the heads
};

static size_t dtype_bytes(int dtype) { return dtype == YSB_F32 ? 4 : 2; }

// candidates per image (summed over TTA passes) the sort key of a call with this many classes can index
static int64_t max_candidates(int num_classes)
{
    return wide_keys(num_classes) ? YSB_MAX_CANDIDATES_WIDE : YSB_MAX_CANDIDATES;
}

static int expected_heads(const ysb_params *p)
{
    if (p->input_kind == YSB_INPUT_DECODED_ROWS) return 1;
    switch (p->family) {
    case YSB_RETINANET:
    case YSB_RETINANET_EXP: return 2;
    case YSB_FCOS: return 3 * p->num_levels;
    default: return p->num_levels;
    }
}

// Fills everything except pointers when d_heads == nullptr (used by the size queries).
static int build_plan(const ysb_params *p, const void *const *d_heads, int num_heads, Built *out)
{
    if (!p || !out) return YSB_ERR_BAD_ARG;
    if (p->family < YSB_YOLOV5 || p->family > YSB_FCOS) return YSB_ERR_BAD_ARG;
    if (p->input_kind != YSB_INPUT_RAW_HEADS && p->input_kind != YSB_INPUT_DECODED_ROWS &&
        p->input_kind != YSB_INPUT_RAW_HEADS_NHWC)
        return YSB_ERR_BAD_ARG;
    // channels-last memory is a layout of the planes families only (YOLOv7 / RetinaNet heads already are rows)
    const bool nhwc = p->input_kind == YSB_INPUT_RAW_HEADS_NHWC;
    if (nhwc && p->family != YSB_YOLOV5 && p->family != YSB_YOLOX && p->family != YSB_YOLOV8 && p->family != YSB_FCOS)
        return YSB_ERR_BAD_ARG;
    if (p->head_dtype != YSB_F32 && p->head_dtype != YSB_F16 && p->head_dtype != YSB_BF16) return YSB_ERR_BAD_ARG;
    if (p->head_dtype != YSB_F32 && p->input_kind == YSB_INPUT_DECODED_ROWS) return YSB_ERR_BAD_ARG;  // decoded rows: float32
    if (p->batch < 0 || p->num_classes <= 0 || p->num_levels <= 0 || p->num_levels > YSB_MAX_LEVELS) return YSB_ERR_BAD_ARG;
    if (p->anchors_per_cell <= 0 || p->anchors_per_cell > YSB_MAX_ANCHORS) return YSB_ERR_BAD_ARG;
    if (p->num_classes > YSB_MAX_CLASSES) return YSB_ERR_LIMIT;
    if (p->max_det <= 0 || p->max_det > YSB_MAX_DET_LIMIT) return YSB_ERR_LIMIT;
    // the reference's multi-label branch is broken for RetinaNet (nonzero(as_tuple=True) on an ndarray, SURVEY 8a-2)
    if (p->multi_label && (p->family == YSB_RETINANET || p->family == YSB_RETINANET_EXP)) return YSB_ERR_UNSUPPORTED;
    const int C = p->num_classes;
    const int A = p->anchors_per_cell;
    const int L = p->num_levels;
    Plan &P = out->plan;
    std::memset(&P, 0, sizeof(P));
    P.family = p->family;
    P.input_kind = nhwc ? YSB_INPUT_RAW_HEADS : p->input_kind;   // NHWC heads take every raw-head branch (layout below)
    P.batch = p->batch;
    P.C = C;
    P.A = A;
    P.L = L;
    P.img_h = p->img_h;
    P.img_w = p->img_w;
    P.dfl_bins = p->dfl_bins;
    std::memcpy(P.anchor, p->anchor, sizeof(P.anchor));
    std::memcpy(P.reg_scale, p->reg_scale, sizeof(P.reg_scale));
    P.conf_thr = p->conf_thr;
    P.cls_thr = p->cls_thr;
    P.pre_thr = p->pre_nms_thr;
    P.iou_thr = p->iou_thr;
    P.max_det = p->max_det;
    P.class_aware = p->class_aware != 0;
    P.postprocess_bbox = p->postprocess_bbox != 0;
    P.window_hi = 3000;
    P.min_box_wh = p->min_box_wh;
    P.pre_nms_topk = p->pre_nms_topk;
    P.obj_col = -1;
    P.multi_label = p->multi_label != 0;
    P.multi_strict = p->family == YSB_FCOS;  // eval_fcos.py:247 uses '>', the other families '>='
    // test-time-augmentation undo of this pass (raw heads only: decoded rows already carry it)
    if (p->tta_flip != 0 && p->tta_flip != 2 && p->tta_flip != 3) return YSB_ERR_BAD_ARG;
    if (p->tta_scale < 0.0f || p->tta_scale != p->tta_scale) return YSB_ERR_BAD_ARG;
    P.tta_on = (p->tta_scale != 0.0f && p->tta_scale != 1.0f) || p->tta_flip != 0;
    if (P.tta_on && P.input_kind != YSB_INPUT_RAW_HEADS) return YSB_ERR_BAD_ARG;
    P.tta_div = p->tta_scale == 0.0f ? 1.0f : p->tta_scale;
    P.tta_flip = p->tta_flip;
    P.tta_h = static_cast<float>(p->tta_img_h);
    P.tta_w = static_cast<float>(p->tta_img_w);
    P.letterbox = p->d_letterbox;

    int64_t n = 0;
    for (int l = 0; l < L; ++l) {
        if (p->level_h[l] <= 0 || p->level_w[l] <= 0) return YSB_ERR_BAD_ARG;
        LevelDesc &lv = P.lv[l];
        lv.h = p->level_h[l];
        lv.w = p->level_w[l];
        lv.hw = lv.h * lv.w;
        lv.stride = p->level_stride[l];
        lv.cand_off = static_cast<int>(n);
        n += static_cast<int64_t>(A) * lv.hw;
        if (n > max_candidates(C)) return YSB_ERR_LIMIT;
    }
    if (p->input_kind == YSB_INPUT_DECODED_ROWS && p->decoded_rows > 0) n = p->decoded_rows;
    if (p->decoded_rows < 0 || n > max_candidates(C)) return YSB_ERR_LIMIT;
    P.N = static_cast<int>(n);

    // ---- per-family operators and layouts (SURVEY.md 8a-1, 8a-2) ---------------------------------------------
    switch (p->family) {
    case YSB_YOLOV5:
    case YSB_YOLOX:
        P.layout = LAYOUT_PLANES;
        P.cls_nch = 5 + C; P.cls_ch = 5; P.obj_nch = 5 + C; P.obj_ch = 4; P.obj_src = 0;
        P.row_w = 5 + C; P.box_col = 0; P.obj_col = 4; P.cls_col = 5; P.box_is_xywh = 1;
        P.use_obj = 1;
        P.pre_kind = p->family == YSB_YOLOV5 ? PRE_OBJ : PRE_OBJ_X_MAX;     // eval_yolov5.py:266 / eval_yolox.py:206-207
        P.post_strict = p->family == YSB_YOLOV5;                             // eval_yolov5.py:285 '>' / eval_yolox.py:227 '>='
        break;
    case YSB_YOLOV7:
        P.layout = LAYOUT_ROWS;
        P.row_w_in = 5 + C; P.cls_col_in = 5; P.obj_col_in = 4; P.obj_src = 0;
        P.row_w = 5 + C; P.box_col = 0; P.obj_col = 4; P.cls_col = 5; P.box_is_xywh = 1;
        P.use_obj = 1; P.pre_kind = PRE_OBJ_X_MAX; P.post_strict = 0;       // eval_yolov7.py:220-221,240
        P.small_box_filter = 1; P.none_when_empty = 1;                        // eval_yolov7.py:272-280
        break;
    case YSB_YOLOV8:
        if (p->dfl_bins <= 0 || p->dfl_bins > 64) return YSB_ERR_BAD_ARG;
        P.layout = LAYOUT_PLANES;
        P.cls_nch = 4 * p->dfl_bins + C; P.cls_ch = 4 * p->dfl_bins; P.obj_src = 0;
        P.row_w = 4 + C; P.box_col = 0; P.cls_col = 4; P.box_is_xywh = 0;
        P.use_obj = 0; P.pre_kind = PRE_MAXCLS; P.post_strict = 0;           // eval_yolov8.py:175,195
        break;
    case YSB_RETINANET:
    case YSB_RETINANET_EXP: {
        const bool ex = p->family == YSB_RETINANET_EXP;
        P.layout = LAYOUT_ROWS;
        P.row_w_in = C; P.cls_col_in = 0; P.obj_col_in = -1; P.obj_src = ex ? 1 : 0;
        P.reg_row_w = ex ? 5 : 4;
        P.row_w = C + (ex ? 5 : 4); P.cls_col = 0; P.box_col = C; P.obj_col = ex ? C + 4 : -1; P.box_is_xywh = 0;
        P.use_obj = ex; P.pre_kind = ex ? PRE_OBJ : PRE_NONE; P.post_strict = 1;  // eval_retinanet.py:324 / _experiment.py:320,329
        P.merge_boxes = 1;                                                         // eval_retinanet.py:349
        break;
    }
    case YSB_FCOS:
        P.layout = LAYOUT_PLANES;
        P.cls_nch = C; P.cls_ch = 0; P.obj_nch = 1; P.obj_ch = 0; P.obj_src = 2;
        P.row_w = 5 + C; P.box_col = 0; P.obj_col = 4; P.cls_col = 5; P.box_is_xywh = 0;
        P.use_obj = p->thresh_with_ctr != 0; P.pre_kind = PRE_ANY_GT; P.post_strict = 1;  // eval_fcos.py:242-243,252,269
        P.topk_sqrt = 1; P.window_hi = 301;                                     // eval_fcos.py:272-281,288
        P.small_box_filter = 1; P.none_when_empty = 1;                          // eval_fcos.py:298-305
        if (P.pre_nms_topk <= 0) return YSB_ERR_BAD_ARG;
        break;
    default: return YSB_ERR_BAD_ARG;
    }
    if (nhwc) {
        // channels-last planes-family heads: a level is one (H*W*A, K) row matrix per image, K = the channels of one
        // anchor; the filter kernel scans it like YOLOv7's rows (cls_nch / obj_nch stay: head_elem addresses the rest)
        P.layout = LAYOUT_ROWS_NHWC;
        P.row_w_in = P.cls_nch;
        P.cls_col_in = P.cls_ch;
        P.obj_col_in = (p->family == YSB_YOLOV5 || p->family == YSB_YOLOX) ? P.obj_ch : -1;   // FCOS: ctr tensor (obj_src 2)
    }
    if (p->input_kind == YSB_INPUT_DECODED_ROWS) {
        // the (b, N, C') tensor: one rows segment, objectness (if any) inside the row
        P.layout = LAYOUT_ROWS;
        P.row_w_in = P.row_w; P.cls_col_in = P.cls_col; P.obj_col_in = P.obj_col;
        if (P.obj_src != 0 && P.use_obj) P.obj_src = 0;
        if (p->family == YSB_FCOS) P.obj_src = 0;
    }

    // channels-last heads: the filter kernel stages a tile of 128 rows in shared memory (filter_kernels.cu, k_filter_rows);
    // rows wider than ~450 floats would not fit the 227 KB a CTA can opt into.  Other rows inputs that wide (YOLOv7,
    // RetinaNet, decoded rows) run k_filter_rows_wide, which reads its rows straight from global memory.
    if (nhwc && !rows_fit_tile(P.row_w_in)) return YSB_ERR_LIMIT;

    out->heads_expected = expected_heads(p);
    out->dtype = p->head_dtype;
    const size_t esize = dtype_bytes(p->head_dtype);
    out->vec = 1;
    if (P.layout == LAYOUT_PLANES) {
        // a unit of 4 positions is one 16-byte (float32) or 8-byte (16-bit) load: plane starts stay aligned to it when
        // the tensor base is and H*W % 4 == 0
        bool aligned = true;
        if (d_heads)
            for (int i = 0; i < num_heads; ++i)
                aligned = aligned && ((reinterpret_cast<uintptr_t>(d_heads[i]) & (4 * esize - 1)) == 0);
        int n4 = 0, units = 0;
        for (int l = 0; l < L; ++l) {
            P.lv[l].vec = (aligned && P.lv[l].hw % 4 == 0) ? 4 : 1;  // e.g. FCOS' 5x5 level falls back to scalar units
            n4 += P.lv[l].vec == 4;
            P.lv[l].unit_off = units;
            units += A * (P.lv[l].hw / P.lv[l].vec);
        }
        out->vec = n4 == L ? 4 : (n4 > 0 ? 3 : 1);  // 4: all levels vectorised, 3: mixed, 1: none
        P.units_per_img = units;
    } else if (p->input_kind == YSB_INPUT_DECODED_ROWS) {
        P.L = 1;
        P.lv[0].cand_off = 0;
        P.lv[0].unit_off = 0;
        P.lv[0].img_rows = P.N;
        P.units_per_img = (P.N + 127) / 128;
    } else {
        int tiles = 0;
        for (int l = 0; l < L; ++l) {
            const int rows_l = A * P.lv[l].hw;
            P.lv[l].unit_off = tiles;
            P.lv[l].img_rows = (p->family == YSB_YOLOV7 || nhwc) ? rows_l : P.N;
            tiles += (rows_l + 127) / 128;
        }
        P.units_per_img = tiles;
    }

    if (!d_heads) return YSB_OK;
    if (num_heads != out->heads_expected) return YSB_ERR_BAD_ARG;
    for (int i = 0; i < num_heads; ++i)
        if (!d_heads[i] && P.batch > 0) return YSB_ERR_BAD_ARG;
    if (p->input_kind == YSB_INPUT_DECODED_ROWS) {
        P.lv[0].p0 = static_cast<const float *>(d_heads[0]);
        return YSB_OK;
    }
    switch (p->family) {
    case YSB_RETINANET:
    case YSB_RETINANET_EXP:
        for (int l = 0; l < L; ++l) {
            // (the Plan's pointers are typed float; the kernels reinterpret them as the head element type)
            P.lv[l].p0 = reinterpret_cast<const float *>(static_cast<const char *>(d_heads[1]) +
                                                         static_cast<size_t>(P.lv[l].cand_off) * C * esize);
            P.lv[l].p1 = static_cast<const float *>(d_heads[0]);
        }
        break;
    case YSB_FCOS:
        for (int l = 0; l < L; ++l) {
            P.lv[l].p0 = static_cast<const float *>(d_heads[l]);
            P.lv[l].p1 = static_cast<const float *>(d_heads[L + l]);
            P.lv[l].p2 = static_cast<const float *>(d_heads[2 * L + l]);
        }
        break;
    default:
        for (int l = 0; l < L; ++l) P.lv[l].p0 = static_cast<const float *>(d_heads[l]);
        break;
    }
    return YSB_OK;
}

}  // namespace ysb

using namespace ysb;

extern "C" {

int ysb_abi_version(void) { return YSB_ABI_VERSION; }

const char *ysb_status_string(int status)
{
    switch (status) {
    case YSB_OK: return "ok";
    case YSB_ERR_BAD_ARG: return "bad argument";
    case YSB_ERR_UNSUPPORTED: return "unsupported request";
    case YSB_ERR_WORKSPACE: return "workspace too small";
    case YSB_ERR_CUDA: return "CUDA error (see ysb_last_cuda_error)";
    case YSB_ERR_LIMIT: return "size beyond the engine limits";
    default: return "unknown status";
    }
}

int ysb_last_cuda_error(void) { return g_last_cuda_error; }

int ysb_num_candidates(const ysb_params *p, int64_t *n_out, int32_t *row_width_out)
{
    Built b;
    const int st = build_plan(p, nullptr, 0, &b);
    if (st != YSB_OK) return st;
    if (n_out) *n_out = b.plan.N;
    if (row_width_out) *row_width_out = b.plan.row_w;
    return YSB_OK;
}

int ysb_decode(const ysb_params *p, const void *const *d_heads, int num_heads, float *d_decoded, void *stream)
{
    if (!d_heads || !d_decoded) return YSB_ERR_BAD_ARG;
    if (p && p->input_kind != YSB_INPUT_RAW_HEADS && p->input_kind != YSB_INPUT_RAW_HEADS_NHWC) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    return cuda_status(launch_decode(b.plan, d_decoded, b.plan.N, 0, static_cast<cudaStream_t>(stream), b.dtype));
}

int ysb_decode_into(const ysb_params *p, const void *const *d_heads, int num_heads, float *d_decoded, int64_t rows_total,
                    int64_t row_offset, void *stream)
{
    if (!d_heads || !d_decoded) return YSB_ERR_BAD_ARG;
    if (p && p->input_kind != YSB_INPUT_RAW_HEADS && p->input_kind != YSB_INPUT_RAW_HEADS_NHWC) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    if (row_offset < 0 || rows_total < row_offset + b.plan.N) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_decode(b.plan, d_decoded, rows_total, row_offset, static_cast<cudaStream_t>(stream), b.dtype));
}

int ysb_filter_candidates(const ysb_params *p, const void *const *d_heads, int num_heads, uint64_t *d_keys,
                          int64_t key_capacity, int32_t *d_counts, void *stream)
{
    if (!d_heads || !d_keys || !d_counts) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    if (key_capacity < key_slots(b.plan)) return YSB_ERR_WORKSPACE;
    return cuda_status(launch_filter(b.plan, b.vec, d_keys, key_capacity, d_counts, static_cast<cudaStream_t>(stream), true,
                                     b.dtype));
}

int ysb_select_nms(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                   int64_t key_capacity, const int32_t *d_counts, float *d_dets, int32_t *d_det_idx,
                   int32_t *d_det_cnt, void *stream)
{
    if (!d_heads || !d_keys || !d_counts || !d_dets || !d_det_cnt) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    if (key_capacity < key_slots(b.plan)) return YSB_ERR_WORKSPACE;
    return cuda_status(launch_select_nms(b.plan, d_keys, key_capacity, d_counts, d_dets, d_det_idx, d_det_cnt,
                                         static_cast<cudaStream_t>(stream), nullptr, b.dtype));
}

// ---- multi-GPU detection gather (gather_kernels.cu) ------------------------------------------------------------------
int ysb_gather_buffer_bytes(int world, int slots, int batch, int max_det, size_t *bytes_out)
{
    if (!bytes_out || world < 1 || world > YSB_MAX_PEERS || slots < 1 || batch < 0 || max_det <= 0) return YSB_ERR_BAD_ARG;
    if (max_det > YSB_MAX_DET_LIMIT) return YSB_ERR_LIMIT;
    *bytes_out = gather_layout(world, slots, batch, max_det).total;
    return YSB_OK;
}

int ysb_gather_alloc(size_t bytes, void **d_buf_out, unsigned char *handle_out)
{
    if (!d_buf_out || bytes == 0) return YSB_ERR_BAD_ARG;
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return cuda_status(e);
    e = cudaMemset(p, 0, bytes);
    if (e == cudaSuccess && handle_out) {
        cudaIpcMemHandle_t h;
        static_assert(sizeof(h) == YSB_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
        e = cudaIpcGetMemHandle(&h, p);
        if (e == cudaSuccess) std::memcpy(handle_out, &h, sizeof(h));
    }
    if (e != cudaSuccess) {
        cudaFree(p);
        return cuda_status(e);
    }
    *d_buf_out = p;
    return YSB_OK;
}

int ysb_gather_open(const unsigned char *handle, void **d_peer_buf_out)
{
    if (!handle || !d_peer_buf_out) return YSB_ERR_BAD_ARG;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return cuda_status(e);
    *d_peer_buf_out = p;
    return YSB_OK;
}

int ysb_gather_close(void *d_peer_buf)
{
    if (!d_peer_buf) return YSB_ERR_BAD_ARG;
    return cuda_status(cudaIpcCloseMemHandle(d_peer_buf));
}

int ysb_gather_free(void *d_buf)
{
    if (!d_buf) return YSB_ERR_BAD_ARG;
    return cuda_status(cudaFree(d_buf));
}

int ysb_gather_slot_views(const ysb_gather *g, int slot, float **d_rows_out, int32_t **d_cnt_out)
{
    if (!gather_valid(g, slot)) return YSB_ERR_BAD_ARG;
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    unsigned char *mine = static_cast<unsigned char *>(g->d_buf[g->rank]);
    // the per-rank regions are contiguous only when their padded sizes equal the raw sizes; report the padded strides
    // through the layout: rows of rank r start at rows_out + r * rows_rank bytes (ysb_gather_buffer_bytes documents it)
    if (d_rows_out) *d_rows_out = reinterpret_cast<float *>(mine + L.rows + L.rows_slot * slot);
    if (d_cnt_out) *d_cnt_out = reinterpret_cast<int32_t *>(mine + L.cnt + L.cnt_slot * slot);
    return YSB_OK;
}

int ysb_gather_strides(const ysb_gather *g, int64_t *rows_rank_bytes, int64_t *cnt_rank_bytes)
{
    if (!gather_valid(g, 0)) return YSB_ERR_BAD_ARG;
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    if (rows_rank_bytes) *rows_rank_bytes = static_cast<int64_t>(L.rows_rank);
    if (cnt_rank_bytes) *cnt_rank_bytes = static_cast<int64_t>(L.cnt_rank);
    return YSB_OK;
}

int ysb_gather_begin(const ysb_gather *g, int slot, int32_t *d_counts, int64_t n_counts, void *stream)
{
    if (!gather_valid(g, slot) || n_counts < 0) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_gather_begin(g, slot, d_counts, n_counts, static_cast<cudaStream_t>(stream)));
}

// The plan's images against the gather's: a full step has exactly g->batch of them, a partial step 0..g->batch.
static bool gather_matches(const ysb_gather *g, const Plan &P, bool partial)
{
    return (partial ? P.batch <= g->batch : P.batch == g->batch) && P.max_det == g->max_det;
}

// The NMS kernel for the plan's images (none for a plan of 0), then, for a partial step, the absent marks and arrival
// counts of images [plan batch, g->batch).
static int nms_gather(const Plan &P, const ExtraPasses *X, const uint64_t *d_keys, int64_t key_capacity,
                      const int32_t *d_counts, const GatherSink &sink, int g_batch, int32_t *d_det_idx, int dtype,
                      cudaStream_t s)
{
    const int e = cuda_status(X ? launch_select_nms_tta(P, *X, d_keys, key_capacity, d_counts, nullptr, d_det_idx, nullptr, s,
                                                        &sink, dtype)
                                : launch_select_nms(P, d_keys, key_capacity, d_counts, nullptr, d_det_idx, nullptr, s, &sink,
                                                    dtype));
    if (e != YSB_OK) return e;
    return cuda_status(launch_gather_absent(sink, P.batch, g_batch, s));
}

static int select_nms_gather(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                             int64_t key_capacity, const int32_t *d_counts, const ysb_gather *g, int slot,
                             int32_t *d_det_idx, void *stream, bool partial)
{
    if (!d_heads || !d_keys || !d_counts) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    if (key_capacity < key_slots(b.plan)) return YSB_ERR_WORKSPACE;
    GatherSink sink;
    if (!make_gather_sink(g, slot, &sink)) return YSB_ERR_BAD_ARG;
    if (!gather_matches(g, b.plan, partial)) return YSB_ERR_BAD_ARG;
    return nms_gather(b.plan, nullptr, d_keys, key_capacity, d_counts, sink, g->batch, d_det_idx, b.dtype,
                      static_cast<cudaStream_t>(stream));
}

int ysb_select_nms_gather(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                          int64_t key_capacity, const int32_t *d_counts, const ysb_gather *g, int slot,
                          int32_t *d_det_idx, void *stream)
{
    return select_nms_gather(p, d_heads, num_heads, d_keys, key_capacity, d_counts, g, slot, d_det_idx, stream, false);
}

int ysb_select_nms_gather_partial(const ysb_params *p, const void *const *d_heads, int num_heads, const uint64_t *d_keys,
                                  int64_t key_capacity, const int32_t *d_counts, const ysb_gather *g, int slot,
                                  int32_t *d_det_idx, void *stream)
{
    return select_nms_gather(p, d_heads, num_heads, d_keys, key_capacity, d_counts, g, slot, d_det_idx, stream, true);
}

int ysb_gather_wait(const ysb_gather *g, int slot, void *stream)
{
    if (!gather_valid(g, slot)) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_gather_wait(g, slot, static_cast<cudaStream_t>(stream)));
}

int ysb_gather_error(const ysb_gather *g, uint32_t *err_out)
{
    if (!gather_valid(g, 0) || !err_out) return YSB_ERR_BAD_ARG;
    const GatherLayout L = gather_layout(g->world, g->slots, g->batch, g->max_det);
    return cuda_status(cudaMemcpy(err_out, static_cast<unsigned char *>(g->d_buf[g->rank]) + L.err, sizeof(uint32_t),
                                  cudaMemcpyDeviceToHost));
}

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

int ysb_postprocess_workspace_bytes(const ysb_params *p, size_t *bytes_out)
{
    if (!bytes_out) return YSB_ERR_BAD_ARG;
    Built b;
    const int st = build_plan(p, nullptr, 0, &b);
    if (st != YSB_OK) return st;
    *bytes_out = align256(sizeof(uint64_t) * static_cast<size_t>(key_slots(b.plan)) * b.plan.batch) +
                 align256(sizeof(int32_t) * 4 * static_cast<size_t>(b.plan.batch)) + 256;
    return YSB_OK;
}

int ysb_postprocess(const ysb_params *p, const void *const *d_heads, int num_heads, void *d_workspace,
                    size_t workspace_bytes, float *d_dets, int32_t *d_det_idx, int32_t *d_det_cnt, void *stream)
{
    if (!d_heads || !d_workspace || !d_dets || !d_det_cnt) return YSB_ERR_BAD_ARG;
    Built b;
    int st = build_plan(p, d_heads, num_heads, &b);
    if (st != YSB_OK) return st;
    size_t need = 0;
    st = ysb_postprocess_workspace_bytes(p, &need);
    if (st != YSB_OK) return st;
    if (workspace_bytes < need) return YSB_ERR_WORKSPACE;
    uintptr_t base = (reinterpret_cast<uintptr_t>(d_workspace) + 255) & ~static_cast<uintptr_t>(255);
    uint64_t *d_keys = reinterpret_cast<uint64_t *>(base);
    const int64_t slots = key_slots(b.plan);
    int32_t *d_counts = reinterpret_cast<int32_t *>(base + align256(sizeof(uint64_t) * static_cast<size_t>(slots) * b.plan.batch));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    st = cuda_status(launch_filter(b.plan, b.vec, d_keys, slots, d_counts, s, true, b.dtype));
    if (st != YSB_OK) return st;
    return cuda_status(launch_select_nms(b.plan, d_keys, slots, d_counts, d_dets, d_det_idx, d_det_cnt, s, nullptr, b.dtype));
}

// ---- test-time augmentation: several passes, one merged candidate space -------------------------------------------
struct BuiltPasses {
    Built b[YSB_MAX_PASSES];
    int64_t base[YSB_MAX_PASSES + 1];  // merged candidate index of candidate 0 of every pass; [n] = total
    int64_t slots;                     // key slots per image over all passes
};

static int build_passes(const ysb_params *passes, int num_passes, const void *const *d_heads, const int32_t *heads_per_pass,
                        BuiltPasses *out)
{
    if (!passes || !out || num_passes < 1 || num_passes > YSB_MAX_PASSES) return YSB_ERR_BAD_ARG;
    if (d_heads && !heads_per_pass) return YSB_ERR_BAD_ARG;
    int64_t base = 0, slots = 0;
    int head0 = 0;
    for (int i = 0; i < num_passes; ++i) {
        const ysb_params *p = passes + i;
        if (p->input_kind != YSB_INPUT_RAW_HEADS && p->input_kind != YSB_INPUT_RAW_HEADS_NHWC) return YSB_ERR_BAD_ARG;
        // one evaluator, one hyp: everything but the geometry and the undo must agree with pass 0 (one head layout too)
        const ysb_params *q = passes;
        if (p->family != q->family || p->batch != q->batch || p->num_classes != q->num_classes ||
            p->conf_thr != q->conf_thr || p->cls_thr != q->cls_thr || p->pre_nms_thr != q->pre_nms_thr ||
            p->iou_thr != q->iou_thr || p->max_det != q->max_det || p->class_aware != q->class_aware ||
            p->multi_label != q->multi_label || p->postprocess_bbox != q->postprocess_bbox ||
            p->min_box_wh != q->min_box_wh || p->pre_nms_topk != q->pre_nms_topk ||
            p->thresh_with_ctr != q->thresh_with_ctr || p->head_dtype != q->head_dtype || p->input_kind != q->input_kind)
            return YSB_ERR_BAD_ARG;
        const int nh = d_heads ? heads_per_pass[i] : 0;
        const int st = build_plan(p, d_heads ? d_heads + head0 : nullptr, nh, &out->b[i]);
        if (st != YSB_OK) return st;
        head0 += nh;
        out->base[i] = base;
        out->b[i].plan.cand_base = static_cast<int>(base);
        base += out->b[i].plan.N;
        slots += key_slots(out->b[i].plan);
        if (base > max_candidates(p->num_classes)) return YSB_ERR_LIMIT;
    }
    out->base[num_passes] = base;
    out->slots = slots;
    return YSB_OK;
}

int ysb_postprocess_tta_workspace_bytes(const ysb_params *passes, int num_passes, size_t *bytes_out)
{
    if (!bytes_out) return YSB_ERR_BAD_ARG;
    BuiltPasses bp;
    const int st = build_passes(passes, num_passes, nullptr, nullptr, &bp);
    if (st != YSB_OK) return st;
    const size_t batch = static_cast<size_t>(bp.b[0].plan.batch);
    *bytes_out = align256(sizeof(uint64_t) * static_cast<size_t>(bp.slots) * batch) + align256(sizeof(int32_t) * 4 * batch) + 256;
    return YSB_OK;
}

// Passes 1..n-1 as the selection/NMS kernel takes them (pass 0 is its own Plan).
static ExtraPasses extra_passes(const BuiltPasses &bp, int num_passes)
{
    ExtraPasses X;
    std::memset(&X, 0, sizeof(X));
    X.n = num_passes - 1;
    for (int i = 1; i < num_passes; ++i) {
        X.base[i - 1] = static_cast<int>(bp.base[i]);
        X.p[i - 1] = bp.b[i].plan;
    }
    return X;
}

int ysb_filter_candidates_tta(const ysb_params *passes, int num_passes, const void *const *d_heads,
                              const int32_t *heads_per_pass, uint64_t *d_keys, int64_t key_capacity, int32_t *d_counts,
                              void *stream)
{
    if (!d_heads || !heads_per_pass || !d_keys || !d_counts) return YSB_ERR_BAD_ARG;
    BuiltPasses bp;
    const int st = build_passes(passes, num_passes, d_heads, heads_per_pass, &bp);
    if (st != YSB_OK) return st;
    if (key_capacity < bp.slots) return YSB_ERR_WORKSPACE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // every pass appends its survivors to the same per-image key list (the counters are zeroed by the first pass only)
    for (int i = 0; i < num_passes; ++i) {
        const int e = cuda_status(launch_filter(bp.b[i].plan, bp.b[i].vec, d_keys, key_capacity, d_counts, s, i == 0,
                                                bp.b[i].dtype));
        if (e != YSB_OK) return e;
    }
    return YSB_OK;
}

int ysb_select_nms_tta(const ysb_params *passes, int num_passes, const void *const *d_heads, const int32_t *heads_per_pass,
                       const uint64_t *d_keys, int64_t key_capacity, const int32_t *d_counts, float *d_dets,
                       int32_t *d_det_idx, int32_t *d_det_cnt, void *stream)
{
    if (!d_heads || !heads_per_pass || !d_keys || !d_counts || !d_dets || !d_det_cnt) return YSB_ERR_BAD_ARG;
    BuiltPasses bp;
    const int st = build_passes(passes, num_passes, d_heads, heads_per_pass, &bp);
    if (st != YSB_OK) return st;
    if (key_capacity < bp.slots) return YSB_ERR_WORKSPACE;
    const ExtraPasses X = extra_passes(bp, num_passes);
    return cuda_status(launch_select_nms_tta(bp.b[0].plan, X, d_keys, key_capacity, d_counts, d_dets, d_det_idx, d_det_cnt,
                                             static_cast<cudaStream_t>(stream), nullptr, bp.b[0].dtype));
}

static int select_nms_tta_gather(const ysb_params *passes, int num_passes, const void *const *d_heads,
                                 const int32_t *heads_per_pass, const uint64_t *d_keys, int64_t key_capacity,
                                 const int32_t *d_counts, const ysb_gather *g, int slot, int32_t *d_det_idx, void *stream,
                                 bool partial)
{
    if (!d_heads || !heads_per_pass || !d_keys || !d_counts) return YSB_ERR_BAD_ARG;
    BuiltPasses bp;
    const int st = build_passes(passes, num_passes, d_heads, heads_per_pass, &bp);
    if (st != YSB_OK) return st;
    if (key_capacity < bp.slots) return YSB_ERR_WORKSPACE;
    GatherSink sink;
    if (!make_gather_sink(g, slot, &sink)) return YSB_ERR_BAD_ARG;
    if (!gather_matches(g, bp.b[0].plan, partial)) return YSB_ERR_BAD_ARG;
    const ExtraPasses X = extra_passes(bp, num_passes);
    return nms_gather(bp.b[0].plan, &X, d_keys, key_capacity, d_counts, sink, g->batch, d_det_idx, bp.b[0].dtype,
                      static_cast<cudaStream_t>(stream));
}

int ysb_select_nms_tta_gather(const ysb_params *passes, int num_passes, const void *const *d_heads,
                              const int32_t *heads_per_pass, const uint64_t *d_keys, int64_t key_capacity,
                              const int32_t *d_counts, const ysb_gather *g, int slot, int32_t *d_det_idx, void *stream)
{
    return select_nms_tta_gather(passes, num_passes, d_heads, heads_per_pass, d_keys, key_capacity, d_counts, g, slot,
                                 d_det_idx, stream, false);
}

int ysb_select_nms_tta_gather_partial(const ysb_params *passes, int num_passes, const void *const *d_heads,
                                      const int32_t *heads_per_pass, const uint64_t *d_keys, int64_t key_capacity,
                                      const int32_t *d_counts, const ysb_gather *g, int slot, int32_t *d_det_idx,
                                      void *stream)
{
    return select_nms_tta_gather(passes, num_passes, d_heads, heads_per_pass, d_keys, key_capacity, d_counts, g, slot,
                                 d_det_idx, stream, true);
}

int ysb_postprocess_tta(const ysb_params *passes, int num_passes, const void *const *d_heads, const int32_t *heads_per_pass,
                        void *d_workspace, size_t workspace_bytes, float *d_dets, int32_t *d_det_idx,
                        int32_t *d_det_cnt, void *stream)
{
    if (!d_heads || !heads_per_pass || !d_workspace || !d_dets || !d_det_cnt) return YSB_ERR_BAD_ARG;
    BuiltPasses bp;
    const int st = build_passes(passes, num_passes, d_heads, heads_per_pass, &bp);
    if (st != YSB_OK) return st;
    const size_t batch = static_cast<size_t>(bp.b[0].plan.batch);
    const size_t need = align256(sizeof(uint64_t) * static_cast<size_t>(bp.slots) * batch) + align256(sizeof(int32_t) * 4 * batch) + 256;
    if (workspace_bytes < need) return YSB_ERR_WORKSPACE;
    uintptr_t base = (reinterpret_cast<uintptr_t>(d_workspace) + 255) & ~static_cast<uintptr_t>(255);
    uint64_t *d_keys = reinterpret_cast<uint64_t *>(base);
    int32_t *d_counts = reinterpret_cast<int32_t *>(base + align256(sizeof(uint64_t) * static_cast<size_t>(bp.slots) * batch));
    const int e = ysb_filter_candidates_tta(passes, num_passes, d_heads, heads_per_pass, d_keys, bp.slots, d_counts, stream);
    if (e != YSB_OK) return e;
    return ysb_select_nms_tta(passes, num_passes, d_heads, heads_per_pass, d_keys, bp.slots, d_counts, d_dets, d_det_idx,
                              d_det_cnt, stream);
}

int ysb_nms_workspace_bytes(int64_t m, size_t *bytes_out)
{
    if (!bytes_out || m < 0) return YSB_ERR_BAD_ARG;
    if (m > YSB_MAX_CANDIDATES) return YSB_ERR_LIMIT;
    *bytes_out = array_nms_workspace_bytes(m);
    return YSB_OK;
}

int ysb_nms(const float *d_boxes, const float *d_scores, int64_t m, double iou_thr, int cmp, int iou_kind,
            int64_t max_keep, void *d_workspace, size_t workspace_bytes, int32_t *d_keep, int32_t *d_keep_cnt,
            void *stream)
{
    if (m < 0 || !d_keep_cnt || (m > 0 && (!d_boxes || !d_scores || !d_keep || !d_workspace))) return YSB_ERR_BAD_ARG;
    if (reinterpret_cast<uintptr_t>(d_boxes) & 15u) return YSB_ERR_BAD_ARG;  // boxes are read as float4
    if (cmp != YSB_CMP_GE && cmp != YSB_CMP_GT) return YSB_ERR_BAD_ARG;
    if (iou_kind < YSB_IOU_NUMBA_F64MIX || iou_kind > YSB_CIOU) return YSB_ERR_BAD_ARG;
    if (m > YSB_MAX_CANDIDATES) return YSB_ERR_LIMIT;
    if (workspace_bytes < array_nms_workspace_bytes(m)) return YSB_ERR_WORKSPACE;
    return cuda_status(launch_array_nms(d_boxes, d_scores, m, iou_thr, cmp, iou_kind, max_keep, d_workspace, d_keep,
                                        d_keep_cnt, static_cast<cudaStream_t>(stream)));
}

int ysb_elementwise_iou_backward(const float *d_b1, int64_t n1, const float *d_b2, int64_t n2, int iou_kind,
                                 const float *d_grad_out, float *d_grad_b1, float *d_grad_b2, void *stream)
{
    if (n1 < 0 || n2 < 0 || (n2 > 0 && (!d_b1 || !d_b2 || !d_grad_out))) return YSB_ERR_BAD_ARG;
    if (n1 != n2 && n1 != 1) return YSB_ERR_BAD_ARG;
    if (iou_kind != YSB_GIOU && iou_kind != YSB_DIOU && iou_kind != YSB_CIOU) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_elementwise_iou_backward(d_b1, n1, d_b2, n2, iou_kind, d_grad_out, d_grad_b1, d_grad_b2,
                                                       static_cast<cudaStream_t>(stream)));
}

int ysb_pairwise_iou_backward(const float *d_b1, int64_t n, const float *d_b2, int64_t m, const float *d_grad_out,
                              float *d_grad_b1, float *d_grad_b2, void *stream)
{
    if (n < 0 || m < 0) return YSB_ERR_BAD_ARG;
    if (n > 0 && m > 0 && (!d_b1 || !d_b2 || !d_grad_out)) return YSB_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(d_b1) | reinterpret_cast<uintptr_t>(d_b2) | reinterpret_cast<uintptr_t>(d_grad_b1) |
         reinterpret_cast<uintptr_t>(d_grad_b2)) & 15u)
        return YSB_ERR_BAD_ARG;  // boxes and gradients move as float4
    if (n > 0x7fffffffll) return YSB_ERR_LIMIT;
    return cuda_status(launch_pairwise_iou_backward(d_b1, n, d_b2, m, d_grad_out, d_grad_b1, d_grad_b2,
                                                    static_cast<cudaStream_t>(stream)));
}

int ysb_wbf_workspace_bytes(int batch, int64_t stride, size_t *bytes_out)
{
    if (batch < 0 || stride < 0 || !bytes_out) return YSB_ERR_BAD_ARG;
    *bytes_out = wbf_workspace_bytes(batch, stride);
    return YSB_OK;
}

int ysb_wbf(const float *d_rows, int row_width, const int32_t *d_counts, int batch, int64_t stride, double iou_thr,
            void *d_workspace, size_t workspace_bytes, int32_t *d_order, double *d_fusion, int32_t *d_members,
            int32_t *d_pairs, int64_t pair_capacity, uint64_t *d_pair_count, int32_t *d_status, void *stream)
{
    if (batch < 0 || stride < 0 || (row_width != 7 && row_width != 8)) return YSB_ERR_BAD_ARG;
    if (batch == 0 || stride == 0) return YSB_OK;
    if (!d_rows || !d_counts || !d_workspace || !d_order || !d_fusion || !d_members || !d_status) return YSB_ERR_BAD_ARG;
    if ((d_pairs != nullptr) != (d_pair_count != nullptr) || pair_capacity < 0) return YSB_ERR_BAD_ARG;
    if (!(iou_thr == iou_thr)) return YSB_ERR_BAD_ARG;
    if (stride > 0x7fffffffll / 32 || batch > 65535 || static_cast<int64_t>(batch) * stride > 0x7fffffffll)
        return YSB_ERR_LIMIT;
    if (workspace_bytes < wbf_workspace_bytes(batch, stride)) return YSB_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(d_workspace) & 15u) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_wbf(d_rows, row_width, d_counts, batch, stride, iou_thr, d_workspace, d_order, d_fusion,
                                  d_members, d_pairs, pair_capacity, reinterpret_cast<unsigned long long *>(d_pair_count),
                                  d_status, static_cast<cudaStream_t>(stream)));
}

int ysb_wbf_collect(const float *d_decoded, int batch, int64_t rows, int row_width, int num_classes, float skip_thr,
                    int multi_label, const int64_t *pass_rows, const float *pass_weights, int num_passes,
                    float *d_records, int32_t *d_counts, int64_t capacity, void *stream)
{
    if (batch < 0 || rows < 0 || num_classes < 1 || row_width != 5 + num_classes) return YSB_ERR_BAD_ARG;
    if (num_passes < 1 || num_passes > YSB_MAX_PASSES || !pass_rows || !pass_weights || !d_counts) return YSB_ERR_BAD_ARG;
    int64_t total = 0;
    for (int q = 0; q < num_passes; ++q) {
        if (pass_rows[q] < 0) return YSB_ERR_BAD_ARG;
        total += pass_rows[q];
    }
    if (total != rows) return YSB_ERR_BAD_ARG;
    if (batch > 0 && rows > 0 && (!d_decoded || !d_records || capacity < 1)) return YSB_ERR_BAD_ARG;
    if (batch > 65535 || rows * (multi_label ? num_classes : 1) > 0xffffffffll) return YSB_ERR_LIMIT;
    return cuda_status(launch_wbf_collect(d_decoded, batch, rows, row_width, num_classes, skip_thr, multi_label != 0,
                                          pass_rows, pass_weights, num_passes, d_records, d_counts, capacity,
                                          static_cast<cudaStream_t>(stream)));
}

int ysb_selftest_reciprocal(uint64_t *d_mismatches, void *stream)
{
    if (!d_mismatches) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_selftest_reciprocal(reinterpret_cast<unsigned long long *>(d_mismatches),
                                                  static_cast<cudaStream_t>(stream)));
}

int ysb_map_iou(const void *d_box1, int64_t n, int row_w1, const void *d_box2, int64_t m, int row_w2, int is_f64,
                void *d_out, void *stream)
{
    if (n < 0 || m < 0 || row_w1 < 4 || row_w2 < 4) return YSB_ERR_BAD_ARG;
    if (n > 0 && m > 0 && (!d_box1 || !d_box2 || !d_out)) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_map_iou(d_box1, n, row_w1, d_box2, m, row_w2, is_f64 != 0, d_out,
                                      static_cast<cudaStream_t>(stream)));
}

int ysb_compute_tp_workspace_bytes(int64_t total_gt, size_t *bytes_out)
{
    if (total_gt < 0 || !bytes_out) return YSB_ERR_BAD_ARG;
    *bytes_out = sizeof(int32_t) * static_cast<size_t>(total_gt > 0 ? total_gt : 1);
    return YSB_OK;
}

int ysb_compute_tp(const void *d_gt, const int64_t *d_gt_offsets, int64_t total_gt, const void *d_pred,
                   const int64_t *d_pred_offsets, int64_t total_pred, int batch, int is_f64, const double *iou_thresholds,
                   void *d_workspace, size_t workspace_bytes, uint8_t *d_tp, void *stream)
{
    if (batch < 0 || total_gt < 0 || total_pred < 0 || !iou_thresholds) return YSB_ERR_BAD_ARG;
    if (batch > 0 && (!d_gt_offsets || !d_pred_offsets)) return YSB_ERR_BAD_ARG;
    if ((total_gt > 0 && !d_gt) || (total_pred > 0 && (!d_pred || !d_tp))) return YSB_ERR_BAD_ARG;
    if (total_gt > 0x7fffffffll || total_pred > 0x7fffffffll / 10) return YSB_ERR_LIMIT;
    if (total_gt > 0 && (!d_workspace || workspace_bytes < sizeof(int32_t) * static_cast<size_t>(total_gt)))
        return YSB_ERR_WORKSPACE;
    for (int t = 0; t < 10; ++t)
        if (!(iou_thresholds[t] == iou_thresholds[t])) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_compute_tp(d_gt, d_gt_offsets, d_pred, d_pred_offsets, batch, is_f64 != 0, iou_thresholds,
                                         static_cast<int32_t *>(d_workspace), d_tp, static_cast<cudaStream_t>(stream)));
}

// The block description of a match step; every refusal of ysb_match_tp / ysb_match_compact except their own pointers.
static int match_step_status(const ysb_match_step *s)
{
    if (!s) return YSB_ERR_BAD_ARG;
    if (s->world < 1 || s->world > YSB_MAX_PEERS || s->batch < 0 || s->max_det < 0 || s->max_gt < 0) return YSB_ERR_BAD_ARG;
    if (s->gt_dtype != YSB_F32 && s->gt_dtype != YSB_F64) return YSB_ERR_BAD_ARG;
    if (s->max_det > YSB_MAX_DET_LIMIT) return YSB_ERR_LIMIT;
    if (static_cast<int64_t>(s->world) * s->batch * s->max_gt > 0x7fffffffll) return YSB_ERR_LIMIT;   // first_pred index
    if (s->batch == 0) return YSB_OK;
    if (!s->d_rows || !s->d_cnt || !s->d_gt_cnt || (s->max_gt > 0 && !s->d_gt)) return YSB_ERR_BAD_ARG;
    if (s->rows_rank_bytes < static_cast<int64_t>(s->batch) * s->max_det * 6 * static_cast<int64_t>(sizeof(float)) ||
        s->cnt_rank_bytes < static_cast<int64_t>(s->batch) * static_cast<int64_t>(sizeof(int32_t)))
        return YSB_ERR_BAD_ARG;
    return YSB_OK;
}

static size_t match_workspace_bytes(const ysb_match_step *s)
{
    const size_t slots = static_cast<size_t>(s->world) * static_cast<size_t>(s->batch) * static_cast<size_t>(s->max_gt);
    return sizeof(int32_t) * (slots > 0 ? slots : 1);
}

int ysb_match_tp_workspace_bytes(const ysb_match_step *step, size_t *bytes_out)
{
    const int st = match_step_status(step);
    if (st != YSB_OK) return st;
    if (!bytes_out) return YSB_ERR_BAD_ARG;
    *bytes_out = match_workspace_bytes(step);
    return YSB_OK;
}

int ysb_match_tp(const ysb_match_step *step, const double *iou_thresholds, void *d_workspace, size_t workspace_bytes,
                 uint8_t *d_tp, void *stream)
{
    const int st = match_step_status(step);
    if (st != YSB_OK) return st;
    if (!iou_thresholds) return YSB_ERR_BAD_ARG;
    for (int t = 0; t < 10; ++t)
        if (!(iou_thresholds[t] == iou_thresholds[t])) return YSB_ERR_BAD_ARG;
    if (step->batch == 0) return YSB_OK;
    if (!d_tp) return YSB_ERR_BAD_ARG;
    if (!d_workspace || workspace_bytes < match_workspace_bytes(step)) return YSB_ERR_WORKSPACE;
    return cuda_status(launch_match_tp(*step, iou_thresholds, static_cast<int32_t *>(d_workspace), d_tp,
                                       static_cast<cudaStream_t>(stream)));
}

int ysb_match_compact(const ysb_match_step *step, const uint8_t *d_tp, const int64_t *d_acc_in, int64_t *d_acc_out,
                      float *d_conf, float *d_pred_cls, uint8_t *d_tp_out, int64_t row_capacity, double *d_target_cls,
                      int64_t target_capacity, void *stream)
{
    const int st = match_step_status(step);
    if (st != YSB_OK) return st;
    if (!d_acc_in || !d_acc_out || d_acc_in == d_acc_out || row_capacity < 0 || target_capacity < 0) return YSB_ERR_BAD_ARG;
    if (step->batch > 0 && (!d_tp || !d_conf || !d_pred_cls || !d_tp_out || !d_target_cls)) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_match_compact(*step, d_tp, d_acc_in, d_acc_out, d_conf, d_pred_cls, d_tp_out, row_capacity,
                                            d_target_cls, target_capacity, static_cast<cudaStream_t>(stream)));
}

int ysb_soft_nms(const float *d_boxes, const float *d_scores, int64_t m, float iou_thr, int iou_kind, int mode,
                 float sigma, void *d_workspace, size_t workspace_bytes, float *d_processed, void *stream)
{
    if (m < 0 || (m > 0 && (!d_boxes || !d_scores || !d_workspace || !d_processed))) return YSB_ERR_BAD_ARG;
    if (reinterpret_cast<uintptr_t>(d_boxes) & 15u) return YSB_ERR_BAD_ARG;  // boxes are read as float4
    if (iou_kind != YSB_GIOU && iou_kind != YSB_DIOU && iou_kind != YSB_CIOU && iou_kind != YSB_IOU_F32) return YSB_ERR_BAD_ARG;
    if (mode != 0 && mode != 1) return YSB_ERR_BAD_ARG;
    if (mode == 1 && !(sigma > 0.0f)) return YSB_ERR_BAD_ARG;
    if (m > YSB_MAX_CANDIDATES) return YSB_ERR_LIMIT;
    if (workspace_bytes < sizeof(float) * static_cast<size_t>(m)) return YSB_ERR_WORKSPACE;
    return cuda_status(launch_soft_nms(d_boxes, d_scores, m, iou_thr, iou_kind, mode, sigma, d_workspace, d_processed,
                                       static_cast<cudaStream_t>(stream)));
}

int ysb_undo_letterbox(float *d_dets, const int32_t *d_det_cnt, int batch, int max_det, const float *d_info, void *stream)
{
    if (batch < 0 || max_det <= 0 || (batch > 0 && (!d_dets || !d_det_cnt || !d_info))) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_undo_letterbox(d_dets, d_det_cnt, batch, max_det, d_info, static_cast<cudaStream_t>(stream)));
}

int ysb_pairwise_iou(const float *d_b1, int64_t n, const float *d_b2, int64_t m, int iou_kind, void *d_out, void *stream)
{
    if (n < 0 || m < 0 || (n > 0 && m > 0 && (!d_b1 || !d_b2 || !d_out))) return YSB_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(d_b1) | reinterpret_cast<uintptr_t>(d_b2)) & 15u) return YSB_ERR_BAD_ARG;  // float4 loads
    if (iou_kind != YSB_IOU_NUMBA_F64MIX && iou_kind != YSB_IOU_F32) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_pairwise_iou(d_b1, n, d_b2, m, iou_kind, d_out, static_cast<cudaStream_t>(stream)));
}

int ysb_elementwise_iou(const float *d_b1, int64_t n1, const float *d_b2, int64_t n2, int iou_kind, float *d_out,
                        void *stream)
{
    if (n1 < 0 || n2 < 0 || (n2 > 0 && (!d_b1 || !d_b2 || !d_out))) return YSB_ERR_BAD_ARG;
    if (iou_kind != YSB_GIOU && iou_kind != YSB_DIOU && iou_kind != YSB_CIOU) return YSB_ERR_BAD_ARG;
    if (!(n1 == n2 || n1 == 1)) return YSB_ERR_BAD_ARG;
    return cuda_status(launch_elementwise_iou(d_b1, n1, d_b2, n2, iou_kind, d_out, static_cast<cudaStream_t>(stream)));
}

int ysb_set_nms_cta_threads(int threads)
{
    if (threads != 0 && threads != 512 && threads != 1024) return YSB_ERR_BAD_ARG;
    ysb::debug_set_nms_threads(threads);
    return YSB_OK;
}

#ifdef YSB_K2_TIMING
int ysb_debug_k2_timing(long long *host_out) { return cuda_status(ysb::debug_k2_timing(host_out)); }
#endif

}  // extern "C"
