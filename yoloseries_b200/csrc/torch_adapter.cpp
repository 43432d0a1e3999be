// torch_adapter.cpp -- the thin PyTorch C++ extension over the C ABI (include/ysb_postproc.h).
//
// BASELINE.json's north star: utils/nms.py, the IoU routines of utils/bbox_tools.py and the decode step of
// trainer/eval_*.py "become a thin PyTorch C++ extension over a C-ABI that calls hand-written sm_100a CUDA kernels".
// This file is that extension: TORCH_LIBRARY(ysb, ...) operators that
//   * check device / dtype / contiguity / alignment of every tensor (the C ABI only sees bare pointers),
//   * switch to the tensors' device and pick up torch's CURRENT stream on it,
//   * take outputs from torch's caching allocator,
//   * translate ysb_status into the exception the reference's callers expect (ValueError for bad arguments and limits,
//     NotImplementedError for the reference branches that do not run, RuntimeError for CUDA failures),
// and contain no arithmetic.  Built without nvcc (host C++ only) into yoloseries_b200/_lib/libysb_torch.so and linked
// against libysb_postproc.so; yoloseries_b200/_ops.py loads it with torch.ops.load_library.
//
// ysb_params travels as a CPU uint8 tensor holding the struct's bytes (the Python side owns a ctypes mirror of the
// struct and shares its memory): plain data in, no second description of the thresholds to keep in sync.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include <cstring>
#include <vector>

#include "ysb_postproc.h"

namespace {

void check_status(int status, const char *what)
{
    if (status == YSB_OK) return;
    const std::string msg = std::string(what) + ": " + ysb_status_string(status);
    if (status == YSB_ERR_BAD_ARG || status == YSB_ERR_LIMIT) TORCH_CHECK_VALUE(false, msg);
    if (status == YSB_ERR_UNSUPPORTED) TORCH_CHECK_NOT_IMPLEMENTED(false, msg);
    if (status == YSB_ERR_CUDA) TORCH_CHECK(false, msg, " [cudaError ", ysb_last_cuda_error(), "]");
    TORCH_CHECK(false, msg);
}

const ysb_params *params_of(const at::Tensor &blob)
{
    TORCH_CHECK_VALUE(blob.device().is_cpu() && blob.scalar_type() == at::kByte && blob.is_contiguous() &&
                          blob.numel() == static_cast<int64_t>(sizeof(ysb_params)),
                      "params: expected a contiguous CPU uint8 tensor of sizeof(ysb_params) = ", sizeof(ysb_params), " bytes");
    return reinterpret_cast<const ysb_params *>(blob.data_ptr());
}

void check_cuda(const at::Tensor &t, at::ScalarType dtype, const c10::Device &dev, const char *name, bool contiguous = true)
{
    TORCH_CHECK_VALUE(t.is_cuda(), name, ": expected a CUDA tensor (yoloseries_b200 has no CPU fallback)");
    TORCH_CHECK_VALUE(t.device() == dev, name, ": on ", t.device(), ", the other tensors are on ", dev);
    TORCH_CHECK_VALUE(t.scalar_type() == dtype, name, ": expected ", dtype, ", got ", t.scalar_type());
    if (contiguous) TORCH_CHECK_VALUE(t.is_contiguous(), name, ": expected a contiguous tensor");
}

// heads -> array of device pointers; every head of one dtype, on one device (their strides: check_head_layout, once the
// params say which layout the heads have)
std::vector<const void *> head_pointers(const at::TensorList &heads, c10::Device &dev)
{
    TORCH_CHECK_VALUE(!heads.empty(), "heads: no tensors");
    dev = heads[0].device();
    std::vector<const void *> p;
    p.reserve(heads.size());
    for (const auto &h : heads) {
        check_cuda(h, heads[0].scalar_type(), dev, "heads", false);
        p.push_back(h.data_ptr());
    }
    return p;
}

// A channels-last head of the family (include/ysb_postproc.h, YSB_INPUT_RAW_HEADS_NHWC): (b, K, H, W) stored as
// (b, H, W, K), or YOLOX' (b, A, K, H, W) view of a channels-last (b, A*K, H, W).  Strides of size-1 dims do not matter.
bool is_channels_last_head(const at::Tensor &t, int family)
{
    std::vector<int64_t> want;
    const auto s = t.sizes();
    if ((family == YSB_YOLOV5 || family == YSB_YOLOV8 || family == YSB_FCOS) && t.dim() == 4)
        want = {s[2] * s[3] * s[1], 1, s[3] * s[1], s[1]};
    else if (family == YSB_YOLOX && t.dim() == 5)
        want = {s[3] * s[4] * s[1] * s[2], s[2], 1, s[4] * s[1] * s[2], s[1] * s[2]};
    else
        return false;
    for (int64_t d = 0; d < t.dim(); ++d)
        if (s[d] != 1 && t.stride(d) != want[d]) return false;
    return true;
}

// the heads' memory is the layout the params announce: channels-last for YSB_INPUT_RAW_HEADS_NHWC, contiguous otherwise
void check_head_layout(const at::TensorList &heads, const ysb_params *p)
{
    for (const auto &h : heads) {
        if (p->input_kind == YSB_INPUT_RAW_HEADS_NHWC) {
            // (a message of string literals only: an exception message that streams tensor sizes crashed the process here)
            TORCH_CHECK_VALUE(is_channels_last_head(h, p->family),
                              "heads: expected channels-last heads of the params' family (params.input_kind)");
        } else {
            TORCH_CHECK_VALUE(h.is_contiguous(), "heads: expected a contiguous tensor");
        }
    }
}

// the heads' dtype is the one the params announce (ysb_params.head_dtype: float32, float16 or bfloat16)
void check_head_dtype(const at::TensorList &heads, const ysb_params *p)
{
    at::ScalarType want = at::kFloat;
    switch (p->head_dtype) {
    case YSB_F32: break;
    case YSB_F16: want = at::kHalf; break;
    case YSB_BF16: want = at::kBFloat16; break;
    default: TORCH_CHECK_VALUE(false, "params: unknown head_dtype ", p->head_dtype);
    }
    TORCH_CHECK_VALUE(heads[0].scalar_type() == want, "heads: expected ", want, " (params.head_dtype), got ",
                      heads[0].scalar_type());
}

void *current_stream(const c10::Device &dev) { return at::cuda::getCurrentCUDAStream(dev.index()).stream(); }

// ---- the hot path -------------------------------------------------------------------------------------------------------
void postprocess(at::TensorList heads, const at::Tensor &params, at::Tensor workspace, at::Tensor dets, at::Tensor det_idx,
                 at::Tensor det_cnt)
{
    c10::Device dev(c10::kCUDA, 0);
    const auto ptrs = head_pointers(heads, dev);
    const ysb_params *p = params_of(params);
    check_head_dtype(heads, p);
    check_head_layout(heads, p);
    check_cuda(workspace, at::kByte, dev, "workspace");
    check_cuda(dets, at::kFloat, dev, "dets");
    check_cuda(det_idx, at::kInt, dev, "det_idx");
    check_cuda(det_cnt, at::kInt, dev, "det_cnt");
    TORCH_CHECK_VALUE(dets.numel() >= static_cast<int64_t>(p->batch) * p->max_det * 6 &&
                          det_idx.numel() >= static_cast<int64_t>(p->batch) * p->max_det && det_cnt.numel() >= p->batch,
                      "output buffers smaller than (batch, max_det, 6) / (batch, max_det) / (batch)");
    c10::cuda::CUDAGuard guard(dev);
    check_status(ysb_postprocess(p, ptrs.data(), static_cast<int>(ptrs.size()), workspace.data_ptr(),
                                 static_cast<size_t>(workspace.numel()), dets.data_ptr<float>(), det_idx.data_ptr<int32_t>(),
                                 det_cnt.data_ptr<int32_t>(), current_stream(dev)),
                 "ysb_postprocess");
}

void filter_candidates(at::TensorList heads, const at::Tensor &params, at::Tensor keys, at::Tensor counts)
{
    c10::Device dev(c10::kCUDA, 0);
    const auto ptrs = head_pointers(heads, dev);
    const ysb_params *p = params_of(params);
    check_head_dtype(heads, p);
    check_head_layout(heads, p);
    check_cuda(keys, at::kLong, dev, "keys");
    check_cuda(counts, at::kInt, dev, "counts");
    TORCH_CHECK_VALUE(keys.dim() == 2 && keys.size(0) == p->batch && counts.numel() >= 4 * static_cast<int64_t>(p->batch),
                      "keys must be (batch, capacity) int64, counts (batch, 4) int32");
    c10::cuda::CUDAGuard guard(dev);
    check_status(ysb_filter_candidates(p, ptrs.data(), static_cast<int>(ptrs.size()),
                                       reinterpret_cast<uint64_t *>(keys.data_ptr<int64_t>()), keys.size(1),
                                       counts.data_ptr<int32_t>(), current_stream(dev)),
                 "ysb_filter_candidates");
}

void select_nms(at::TensorList heads, const at::Tensor &params, const at::Tensor &keys, const at::Tensor &counts,
                at::Tensor dets, at::Tensor det_idx, at::Tensor det_cnt)
{
    c10::Device dev(c10::kCUDA, 0);
    const auto ptrs = head_pointers(heads, dev);
    const ysb_params *p = params_of(params);
    check_head_dtype(heads, p);
    check_head_layout(heads, p);
    check_cuda(keys, at::kLong, dev, "keys");
    check_cuda(counts, at::kInt, dev, "counts");
    check_cuda(dets, at::kFloat, dev, "dets");
    check_cuda(det_idx, at::kInt, dev, "det_idx");
    check_cuda(det_cnt, at::kInt, dev, "det_cnt");
    TORCH_CHECK_VALUE(keys.dim() == 2 && keys.size(0) == p->batch, "keys must be (batch, capacity) int64");
    TORCH_CHECK_VALUE(dets.numel() >= static_cast<int64_t>(p->batch) * p->max_det * 6 &&
                          det_idx.numel() >= static_cast<int64_t>(p->batch) * p->max_det && det_cnt.numel() >= p->batch,
                      "output buffers smaller than (batch, max_det, 6) / (batch, max_det) / (batch)");
    c10::cuda::CUDAGuard guard(dev);
    check_status(ysb_select_nms(p, ptrs.data(), static_cast<int>(ptrs.size()),
                                reinterpret_cast<const uint64_t *>(keys.data_ptr<int64_t>()), keys.size(1),
                                counts.data_ptr<int32_t>(), dets.data_ptr<float>(), det_idx.data_ptr<int32_t>(),
                                det_cnt.data_ptr<int32_t>(), current_stream(dev)),
                 "ysb_select_nms");
}

// do_inference: raw heads -> a fresh (batch, N, C') tensor
at::Tensor decode(at::TensorList heads, const at::Tensor &params)
{
    c10::Device dev(c10::kCUDA, 0);
    const auto ptrs = head_pointers(heads, dev);
    const ysb_params *p = params_of(params);
    check_head_dtype(heads, p);
    check_head_layout(heads, p);
    int64_t n = 0;
    int32_t row_w = 0;
    check_status(ysb_num_candidates(p, &n, &row_w), "ysb_num_candidates");
    c10::cuda::CUDAGuard guard(dev);
    at::Tensor out = at::empty({p->batch, n, row_w}, at::TensorOptions().dtype(at::kFloat).device(dev));
    check_status(ysb_decode(p, ptrs.data(), static_cast<int>(ptrs.size()), out.data_ptr<float>(), current_stream(dev)),
                 "ysb_decode");
    return out;
}

// one pass of test_time_augmentation written into its slot of the merged tensor
void decode_into(at::TensorList heads, const at::Tensor &params, at::Tensor merged, int64_t row_offset)
{
    c10::Device dev(c10::kCUDA, 0);
    const auto ptrs = head_pointers(heads, dev);
    const ysb_params *p = params_of(params);
    check_head_dtype(heads, p);
    check_head_layout(heads, p);
    check_cuda(merged, at::kFloat, dev, "merged");
    TORCH_CHECK_VALUE(merged.dim() == 3 && merged.size(0) == p->batch, "merged must be (batch, rows_total, C')");
    c10::cuda::CUDAGuard guard(dev);
    check_status(ysb_decode_into(p, ptrs.data(), static_cast<int>(ptrs.size()), merged.data_ptr<float>(), merged.size(1),
                                 row_offset, current_stream(dev)),
                 "ysb_decode_into");
}

// ---- utils.numba_nms / utils.gpu_nms -------------------------------------------------------------------------------------
// returns (keep (cap,) int32, count (1,) int32); the caller slices keep[:count] (the one host sync of the call)
std::tuple<at::Tensor, at::Tensor> nms(const at::Tensor &boxes, const at::Tensor &scores, double iou_thr, int64_t cmp,
                                       int64_t iou_kind, int64_t max_keep)
{
    const c10::Device dev = boxes.device();
    check_cuda(boxes, at::kFloat, dev, "boxes");
    check_cuda(scores, at::kFloat, dev, "scores");
    TORCH_CHECK_VALUE(boxes.dim() == 2 && boxes.size(1) == 4 && scores.numel() == boxes.size(0),
                      "boxes must be (M, 4), scores (M,)");
    const int64_t m = boxes.size(0);
    c10::cuda::CUDAGuard guard(dev);
    size_t ws_bytes = 0;
    check_status(ysb_nms_workspace_bytes(m, &ws_bytes), "ysb_nms_workspace_bytes");
    at::Tensor ws = at::empty({static_cast<int64_t>(ws_bytes > 0 ? ws_bytes : 1)}, at::TensorOptions().dtype(at::kByte).device(dev));
    const int64_t cap = max_keep <= 0 ? m : std::min(m, max_keep);
    at::Tensor keep = at::empty({std::max<int64_t>(cap, 1)}, at::TensorOptions().dtype(at::kInt).device(dev));
    at::Tensor count = at::zeros({1}, at::TensorOptions().dtype(at::kInt).device(dev));
    check_status(ysb_nms(boxes.data_ptr<float>(), scores.data_ptr<float>(), m, iou_thr, static_cast<int>(cmp),
                         static_cast<int>(iou_kind), max_keep, ws.data_ptr(), static_cast<size_t>(ws.numel()),
                         keep.data_ptr<int32_t>(), count.data_ptr<int32_t>(), current_stream(dev)),
                 "ysb_nms");
    return {keep, count};
}

// ---- IoU family ---------------------------------------------------------------------------------------------------------
at::Tensor pairwise_iou(const at::Tensor &b1, const at::Tensor &b2, int64_t kind)
{
    const c10::Device dev = b1.device();
    check_cuda(b1, at::kFloat, dev, "bbox1");
    check_cuda(b2, at::kFloat, dev, "bbox2");
    TORCH_CHECK_VALUE(b1.dim() == 2 && b1.size(1) == 4 && b2.dim() == 2 && b2.size(1) == 4, "boxes must be (N, 4) and (M, 4)");
    c10::cuda::CUDAGuard guard(dev);
    at::Tensor out = at::empty({b1.size(0), b2.size(0)},
                               at::TensorOptions().dtype(kind == YSB_IOU_NUMBA_F64MIX ? at::kDouble : at::kFloat).device(dev));
    check_status(ysb_pairwise_iou(b1.data_ptr<float>(), b1.size(0), b2.data_ptr<float>(), b2.size(0), static_cast<int>(kind),
                                  out.data_ptr(), current_stream(dev)),
                 "ysb_pairwise_iou");
    return out;
}

std::tuple<at::Tensor, at::Tensor> pairwise_iou_backward(const at::Tensor &b1, const at::Tensor &b2, const at::Tensor &grad_out,
                                                         bool need1, bool need2)
{
    const c10::Device dev = b1.device();
    check_cuda(b1, at::kFloat, dev, "bbox1");
    check_cuda(b2, at::kFloat, dev, "bbox2");
    check_cuda(grad_out, at::kFloat, dev, "grad_out");
    TORCH_CHECK_VALUE(grad_out.numel() == b1.size(0) * b2.size(0), "grad_out must be (N, M)");
    c10::cuda::CUDAGuard guard(dev);
    at::Tensor g1 = need1 ? at::empty_like(b1) : at::Tensor();
    at::Tensor g2 = need2 ? at::empty_like(b2) : at::Tensor();
    check_status(ysb_pairwise_iou_backward(b1.data_ptr<float>(), b1.size(0), b2.data_ptr<float>(), b2.size(0),
                                           grad_out.data_ptr<float>(), need1 ? g1.data_ptr<float>() : nullptr,
                                           need2 ? g2.data_ptr<float>() : nullptr, current_stream(dev)),
                 "ysb_pairwise_iou_backward");
    return {g1, g2};
}

at::Tensor elementwise_iou(const at::Tensor &b1, const at::Tensor &b2, int64_t kind)
{
    const c10::Device dev = b2.device();
    check_cuda(b1, at::kFloat, dev, "bbox1");
    check_cuda(b2, at::kFloat, dev, "bbox2");
    TORCH_CHECK_VALUE(b1.dim() == 2 && b1.size(1) == 4 && b2.dim() == 2 && b2.size(1) == 4, "boxes must be (N|1, 4) and (N, 4)");
    c10::cuda::CUDAGuard guard(dev);
    at::Tensor out = at::empty({b2.size(0)}, at::TensorOptions().dtype(at::kFloat).device(dev));
    check_status(ysb_elementwise_iou(b1.data_ptr<float>(), b1.size(0), b2.data_ptr<float>(), b2.size(0), static_cast<int>(kind),
                                     out.data_ptr<float>(), current_stream(dev)),
                 "ysb_elementwise_iou");
    return out;
}

std::tuple<at::Tensor, at::Tensor> elementwise_iou_backward(const at::Tensor &b1, const at::Tensor &b2, int64_t kind,
                                                            const at::Tensor &grad_out, bool need1, bool need2)
{
    const c10::Device dev = b2.device();
    check_cuda(b1, at::kFloat, dev, "bbox1");
    check_cuda(b2, at::kFloat, dev, "bbox2");
    check_cuda(grad_out, at::kFloat, dev, "grad_out");
    TORCH_CHECK_VALUE(grad_out.numel() == b2.size(0), "grad_out must be (N,)");
    c10::cuda::CUDAGuard guard(dev);
    at::Tensor g1 = need1 ? at::empty_like(b1) : at::Tensor();
    at::Tensor g2 = need2 ? at::empty_like(b2) : at::Tensor();
    check_status(ysb_elementwise_iou_backward(b1.data_ptr<float>(), b1.size(0), b2.data_ptr<float>(), b2.size(0),
                                              static_cast<int>(kind), grad_out.data_ptr<float>(),
                                              need1 ? g1.data_ptr<float>() : nullptr, need2 ? g2.data_ptr<float>() : nullptr,
                                              current_stream(dev)),
                 "ysb_elementwise_iou_backward");
    return {g1, g2};
}

// ---- mAP hand-off on the post-processors' row blocks (ysb_match_tp, ysb_match_compact) -----------------------------------
// rows (world, batch, max_det, 6) float32 whose ranks may lie any distance apart (a gather slot), dense within a rank;
// counts (world, batch) int32 likewise; ground truth (world, batch, max_gt, 5) float32 / float64 and its counts dense.
ysb_match_step match_step(const at::Tensor &rows, const at::Tensor &cnt, const at::Tensor &gt, const at::Tensor &gt_cnt)
{
    const c10::Device dev = rows.device();
    check_cuda(rows, at::kFloat, dev, "rows", false);
    check_cuda(cnt, at::kInt, dev, "counts", false);
    TORCH_CHECK_VALUE(gt.is_cuda() && gt.device() == dev && gt.is_contiguous() &&
                          (gt.scalar_type() == at::kFloat || gt.scalar_type() == at::kDouble),
                      "gt: expected a contiguous float32 or float64 CUDA tensor on the rows' device");
    check_cuda(gt_cnt, at::kInt, dev, "gt_counts");
    TORCH_CHECK_VALUE(rows.dim() == 4 && rows.size(3) == 6, "rows must be (world, batch, max_det, 6)");
    const int64_t W = rows.size(0), B = rows.size(1), D = rows.size(2);
    TORCH_CHECK_VALUE((B == 0 || D == 0 || (rows.stride(3) == 1 && rows.stride(2) == 6 && rows.stride(1) == D * 6)) &&
                          (W == 1 || rows.stride(0) >= B * D * 6),
                      "rows: every rank's (batch, max_det, 6) rows must be dense");
    TORCH_CHECK_VALUE(cnt.dim() == 2 && cnt.size(0) == W && cnt.size(1) == B && (B <= 1 || cnt.stride(1) == 1) &&
                          (W == 1 || cnt.stride(0) >= B),
                      "counts must be (world, batch) with every rank's counts dense");
    TORCH_CHECK_VALUE(gt.dim() == 4 && gt.size(0) == W && gt.size(1) == B && gt.size(3) == 5,
                      "gt must be (world, batch, max_gt, 5)");
    TORCH_CHECK_VALUE(gt_cnt.dim() == 2 && gt_cnt.size(0) == W && gt_cnt.size(1) == B, "gt_counts must be (world, batch)");
    ysb_match_step s{};
    s.world = static_cast<int32_t>(W);
    s.batch = static_cast<int32_t>(B);
    s.max_det = static_cast<int32_t>(D);
    s.max_gt = static_cast<int32_t>(gt.size(2));
    s.d_rows = rows.data_ptr<float>();
    s.rows_rank_bytes = (W == 1 ? B * D * 6 : rows.stride(0)) * static_cast<int64_t>(sizeof(float));
    s.d_cnt = cnt.data_ptr<int32_t>();
    s.cnt_rank_bytes = (W == 1 ? B : cnt.stride(0)) * static_cast<int64_t>(sizeof(int32_t));
    s.d_gt = gt.data_ptr();
    s.d_gt_cnt = gt_cnt.data_ptr<int32_t>();
    s.gt_dtype = gt.scalar_type() == at::kDouble ? YSB_F64 : YSB_F32;
    return s;
}

void match_tp(const at::Tensor &rows, const at::Tensor &cnt, const at::Tensor &gt, const at::Tensor &gt_cnt,
              at::ArrayRef<double> iou_thr, at::Tensor tp)
{
    const ysb_match_step s = match_step(rows, cnt, gt, gt_cnt);
    const c10::Device dev = rows.device();
    check_cuda(tp, at::kByte, dev, "tp");
    TORCH_CHECK_VALUE(tp.dim() == 4 && tp.size(0) == s.world && tp.size(1) == s.batch && tp.size(2) == s.max_det &&
                          tp.size(3) == 10,
                      "tp must be (world, batch, max_det, 10) uint8");
    TORCH_CHECK_VALUE(iou_thr.size() == 10, "iou_thr must hold 10 thresholds");
    c10::cuda::CUDAGuard guard(dev);
    size_t ws_bytes = 0;
    check_status(ysb_match_tp_workspace_bytes(&s, &ws_bytes), "ysb_match_tp_workspace_bytes");
    at::Tensor ws = at::empty({static_cast<int64_t>(ws_bytes)}, at::TensorOptions().dtype(at::kByte).device(dev));
    check_status(ysb_match_tp(&s, iou_thr.data(), ws.data_ptr(), ws_bytes, tp.data_ptr<uint8_t>(), current_stream(dev)),
                 "ysb_match_tp");
}

void match_compact(const at::Tensor &rows, const at::Tensor &cnt, const at::Tensor &gt, const at::Tensor &gt_cnt,
                   const at::Tensor &tp, const at::Tensor &acc_in, at::Tensor acc_out, at::Tensor conf, at::Tensor pred_cls,
                   at::Tensor tp_out, at::Tensor target_cls)
{
    const ysb_match_step s = match_step(rows, cnt, gt, gt_cnt);
    const c10::Device dev = rows.device();
    check_cuda(tp, at::kByte, dev, "tp");
    TORCH_CHECK_VALUE(tp.numel() == static_cast<int64_t>(s.world) * s.batch * s.max_det * 10,
                      "tp must be (world, batch, max_det, 10) uint8");
    check_cuda(acc_in, at::kLong, dev, "acc_in");
    check_cuda(acc_out, at::kLong, dev, "acc_out");
    TORCH_CHECK_VALUE(acc_in.numel() == 2 && acc_out.numel() == 2, "acc_in / acc_out must hold 2 int64 each");
    check_cuda(conf, at::kFloat, dev, "conf");
    check_cuda(pred_cls, at::kFloat, dev, "pred_cls");
    check_cuda(tp_out, at::kByte, dev, "tp_out");
    check_cuda(target_cls, at::kDouble, dev, "target_cls");
    const int64_t cap = conf.numel();
    TORCH_CHECK_VALUE(pred_cls.numel() == cap && tp_out.numel() == cap * 10,
                      "conf, pred_cls (P,) and tp_out (P, 10) must share one capacity");
    c10::cuda::CUDAGuard guard(dev);
    check_status(ysb_match_compact(&s, tp.data_ptr<uint8_t>(), acc_in.data_ptr<int64_t>(), acc_out.data_ptr<int64_t>(),
                                   conf.data_ptr<float>(), pred_cls.data_ptr<float>(), tp_out.data_ptr<uint8_t>(), cap,
                                   target_cls.data_ptr<double>(), target_cls.numel(), current_stream(dev)),
                 "ysb_match_compact");
}

int64_t abi_version() { return ysb_abi_version(); }
int64_t params_bytes() { return static_cast<int64_t>(sizeof(ysb_params)); }

}  // namespace

TORCH_LIBRARY(ysb, m)
{
    m.def("postprocess(Tensor[] heads, Tensor params, Tensor(a!) workspace, Tensor(b!) dets, Tensor(c!) det_idx, "
          "Tensor(d!) det_cnt) -> ()", &postprocess);
    m.def("filter_candidates(Tensor[] heads, Tensor params, Tensor(a!) keys, Tensor(b!) counts) -> ()", &filter_candidates);
    m.def("select_nms(Tensor[] heads, Tensor params, Tensor keys, Tensor counts, Tensor(a!) dets, Tensor(b!) det_idx, "
          "Tensor(c!) det_cnt) -> ()", &select_nms);
    m.def("decode(Tensor[] heads, Tensor params) -> Tensor", &decode);
    m.def("decode_into(Tensor[] heads, Tensor params, Tensor(a!) merged, int row_offset) -> ()", &decode_into);
    m.def("nms(Tensor boxes, Tensor scores, float iou_thr, int cmp, int iou_kind, int max_keep) -> (Tensor, Tensor)", &nms);
    m.def("pairwise_iou(Tensor bbox1, Tensor bbox2, int kind) -> Tensor", &pairwise_iou);
    m.def("pairwise_iou_backward(Tensor bbox1, Tensor bbox2, Tensor grad_out, bool need1, bool need2) -> (Tensor, Tensor)",
          &pairwise_iou_backward);
    m.def("elementwise_iou(Tensor bbox1, Tensor bbox2, int kind) -> Tensor", &elementwise_iou);
    m.def("elementwise_iou_backward(Tensor bbox1, Tensor bbox2, int kind, Tensor grad_out, bool need1, bool need2) -> "
          "(Tensor, Tensor)", &elementwise_iou_backward);
    m.def("match_tp(Tensor rows, Tensor counts, Tensor gt, Tensor gt_counts, float[] iou_thr, Tensor(a!) tp) -> ()",
          &match_tp);
    m.def("match_compact(Tensor rows, Tensor counts, Tensor gt, Tensor gt_counts, Tensor tp, Tensor acc_in, "
          "Tensor(a!) acc_out, Tensor(b!) conf, Tensor(c!) pred_cls, Tensor(d!) tp_out, Tensor(e!) target_cls) -> ()",
          &match_compact);
    m.def("abi_version() -> int", &abi_version);
    m.def("params_bytes() -> int", &params_bytes);
}
