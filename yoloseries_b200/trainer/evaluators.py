"""Drop-in mirrors of the reference evaluators (trainer/eval_*.py): same constructors, same methods, same outputs.

    YOLOV5Evaluator(yolo, anchors, hyp, compute_metric=False)      trainer/eval_yolov5.py:10-42
    YOLOV7Evaluator(yolo, anchors, hyp, compute_metric=False)      trainer/eval_yolov7.py
    YOLOXEvaluator(yolo, hyp, compute_metric=False)                trainer/eval_yolox.py:11-41
    YOLOV8Evaluator(yolo, hyp, compute_metric=False)               trainer/eval_yolov8.py:11-38
    RetinaNetEvaluator(model, hyp, compute_metric=False)           trainer/eval_retinanet.py:9-20
    RetinaNetEvaluatorExperiment(model, hyp, compute_metric=False) trainer/eval_retinanet_experiment.py
    FCOSEvaluator(model, hyp, compute_metric=False)                trainer/eval_fcos.py:12-38

``__call__(inputs)`` returns ``list[Tensor(K,6) | None]`` -- CPU float32 rows [xmin, ymin, xmax, ymax, score, cls] in NMS
keep order, ``None`` where the reference returns ``None`` (SURVEY.md 8a-4.3).  Without TTA the model's raw heads go
straight into the fused CUDA path (no (b, N, C') tensor is ever written); contiguous float16 / bfloat16 heads (hyp['half'])
are read as they are, with results bit-identical to their float32 widening.  ``do_inference`` / ``numba_nms`` remain
available separately with the reference's signatures.  Everything heavy runs in libysb_postproc.so; there is no CPU path.
"""
import numpy as np
import torch
import torch.nn.functional as F

from ..engine import PostProcessor, native_heads

__all__ = ["YOLOV5Evaluator", "YOLOV7Evaluator", "YOLOXEvaluator", "YOLOV8Evaluator", "RetinaNetEvaluator",
           "RetinaNetEvaluatorExperiment", "FCOSEvaluator"]


class _Evaluator:
    family = None

    def _setup(self, model, hyp, compute_metric, anchors=None):
        self.hyp = hyp
        self.device = hyp["device"]
        self.num_class = hyp["num_class"]
        self.use_tta = hyp["use_tta"]
        self._model = model
        self.anchors = anchors
        pre = "compute_metric_" if compute_metric else ""
        self.iou_threshold = hyp[pre + "iou_threshold"]
        self.cls_threshold = hyp[pre + "cls_threshold"]
        if (pre + "conf_threshold") in hyp:
            self.conf_threshold = hyp[pre + "conf_threshold"]
        self._pp = PostProcessor(self.family, hyp, anchors=anchors, compute_metric=compute_metric)

    def _native(self, heads):
        """The model's outputs as the engine reads them: contiguous or channels-last heads of one 16/32-bit float type are
        passed through unchanged; anything else (and channels-last rows wider than the filter kernel's tile) is converted
        by normalise_heads."""
        return native_heads(heads, self.family, self.num_class, self.hyp.get("reg", 16))

    # ---- reference API -------------------------------------------------------------------------------------------
    @torch.no_grad()
    def __call__(self, inputs, info=None):
        """``info`` (extension, default None = the reference's behaviour): the per-image letterbox dicts val_*.py hands to
        preds_postprocess; when given, the undo is fused into the NMS kernel's row write and the rows come back in
        original-picture pixels."""
        if self.use_tta:
            if self.hyp.get("wfb", False):
                _, independent = self.test_time_augmentation(inputs)
                return self.do_wfb(independent)
            # three model forwards, then ONE fused call: no decoded or merged tensor is written (ysb_postprocess_tta)
            out = self._pp.run_tta(self._tta_passes(inputs), (inputs.size(2), inputs.size(3)), info=info)
            return self._pp.to_list(out)
        heads = self._native(self._model(inputs))
        out = self._pp.run(heads, inputs.size(2), inputs.size(3), info=info)
        return self._pp.to_list(out)

    @torch.no_grad()
    def do_inference(self, inputs):
        """model forward + decode -> (b, N, C') float32 on the heads' device (one CUDA kernel, ysb_decode)."""
        heads = self._native(self._model(inputs))
        return self._pp.decode(heads, inputs.size(2), inputs.size(3))

    def numba_nms(self, preds_out):
        """(b, N, C') decoded tensor -> list[ndarray(K,6) float32 | None] (the reference's CPU numba path, on the GPU)."""
        if isinstance(preds_out, np.ndarray):
            preds_out = torch.from_numpy(preds_out)
        preds = preds_out.detach().to(torch.float32)
        if preds.device.type != "cuda":
            preds = preds.cuda()
        preds = preds.contiguous()
        h, w = self.hyp["input_img_size"]
        out = self._pp.run(preds, int(h), int(w), decoded=True)
        return self._pp.to_list(out, as_numpy=True)

    def do_wfb(self, preds_out):
        """trainer/eval_yolov5.py:44-92 (the same method in eval_yolov7.py / eval_yolox.py): weighted-box-fusion of the
        per-pass decoded tensors [(b, X, 5+C), (b, Y, 5+C), ...] -> list over images of the reference's nesting
        ``[[fused (6,) float64 arrays of label 0], [... label 1], ...]`` or None for an image without survivors.
        Filter (ysb_wbf_collect) and fusion (ysb_wbf) run on the device for the whole batch at once.

        RetinaNet / FCOS: the reference's do_wfb indexes ``[cls..., box]`` columns its own do_inference does not produce
        and appends None inside the pass loop (eval_fcos.py:40-90, eval_retinanet.py:77-130) -- not mirrored."""
        import ctypes

        from .. import _lib
        from ..utils.weighted_fusion_bbox import fuse_batch
        if self.family not in ("yolov5", "yolov7", "yolox"):
            raise NotImplementedError(f"do_wfb of {self.family}: the reference's own method does not match its decode layout")
        weights = self.hyp.get("wfb_weights", [1.0 for _ in range(len(preds_out))])
        preds = [p.detach().to(torch.float32) for p in preds_out]
        preds = [p if p.device.type == "cuda" else p.cuda() for p in preds]
        dev = preds[0].device
        merged = preds[0].contiguous() if len(preds) == 1 else torch.cat(preds, dim=1).contiguous()
        batch, rows, row_w = merged.shape
        C = int(self.num_class)
        multi = bool(self.hyp["mutil_label"])
        cap = rows * (C if multi else 1)
        rec = torch.empty((batch, max(cap, 1), 8), dtype=torch.float32, device=dev)
        counts = torch.empty((max(batch, 1),), dtype=torch.int32, device=dev)
        n = len(preds)
        pass_rows = (ctypes.c_int64 * n)(*[int(p.shape[1]) for p in preds])
        pass_w = (ctypes.c_float * n)(*[float(weights[i]) for i in range(n)])
        with torch.cuda.device(dev):
            _lib.check(_lib.load().ysb_wbf_collect(
                merged.data_ptr(), batch, rows, row_w, C, float(self.hyp["wfb_skip_box_threshold"]), int(multi), pass_rows,
                pass_w, n, rec.data_ptr(), counts.data_ptr(), cap,
                ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "ysb_wbf_collect")
            kmax = int(counts[:batch].max().item()) if batch else 0
            if kmax == 0:
                return [None] * batch
            # the fusion works on the occupied part of every image's record list
            fused = fuse_batch(rec[:, :kmax].contiguous(), counts[:batch], float(self.hyp["wfb_iou_threshold"]), 8)
        out = []
        for item in fused:
            if item is None:
                out.append(None)
                continue
            fus = item[0]
            out.append([[fus[k].copy() for k in np.nonzero(fus[:, 5] == lab)[0]] for lab in np.unique(fus[:, 5])])
        return out

    def do_nms(self, preds_out):
        """Dead code in the reference (no caller; raises IndexError for iou_type='iou', SURVEY.md fact 3).  Mirrored
        with the live path's semantics, returning tensors."""
        return [torch.from_numpy(x) if x is not None else None for x in self.numba_nms(preds_out)]

    # ---- TTA (SURVEY.md 8f rank 2) -------------------------------------------------------------------------------
    def _tta_passes(self, inputs):
        """The three augmented forwards of test_time_augmentation (trainer/eval_yolov5.py:158-168): scale 1 / 0.83 / 0.67,
        flip none / along h / along w.  Returns [(raw heads, pass_h, pass_w, scale, flip_axis), ...]."""
        passes = []
        for s, f in zip([1, 0.83, 0.67], [None, 2, 3]):
            img = inputs.flip(dims=(f,)) if f else inputs
            img = self.scale_img(img, s)
            passes.append((self._native(self._model(img)), img.size(2), img.size(3), s, f))
        return passes

    def test_time_augmentation(self, inputs):
        """trainer/eval_yolov5.py:152-179 (xywh rows; xyxy rows: eval_yolov8.py:40-73, eval_retinanet.py:148-182,
        eval_fcos.py:90-123) -> (merged (b, sum N_i, C'), [per-pass tensors]).  Each pass is decoded, divided by its
        scale and un-flipped by one ysb_decode_into launch writing straight into its slot of the merged tensor; the
        per-pass tensors are views of it."""
        merged, views = self._pp.decode_tta(self._tta_passes(inputs), (inputs.size(2), inputs.size(3)))
        return merged, views

    @staticmethod
    def scale_img(img, scale_factor):
        """trainer/eval_yolov5.py:211-227 (identical in every evaluator)."""
        if scale_factor == 1.0:
            return img
        h, w = img.shape[2], img.shape[3]
        new_h, new_w = int(scale_factor * h), int(scale_factor * w)
        img = F.interpolate(img, size=(new_h, new_w), align_corners=False, mode="bilinear")
        out_h, out_w = int(np.ceil(h / 32) * 32), int(np.ceil(w / 32) * 32)
        return F.pad(img, [0, out_w - new_w, 0, out_h - new_h], value=0.447)


class YOLOV5Evaluator(_Evaluator):
    family = "yolov5"

    def __init__(self, yolo, anchors, hyp, compute_metric=False):
        self.yolo = yolo
        self.anchor_num = anchors.size(1)
        self.num_stage = len(anchors)
        self.ds_scales = [8, 16, 32]
        self.inp_h, self.inp_w = hyp["input_img_size"]
        self._setup(yolo, hyp, compute_metric, anchors)


class YOLOV7Evaluator(_Evaluator):
    family = "yolov7"

    def __init__(self, yolo, anchors, hyp, compute_metric=False):
        self.yolo = yolo
        self.anchor_num = anchors.size(1)
        self.num_stage = len(anchors)
        self.ds_scales = [8, 16, 32]
        self.inp_h, self.inp_w = hyp["input_img_size"]
        self._setup(yolo, hyp, compute_metric, anchors)


class YOLOXEvaluator(_Evaluator):
    family = "yolox"

    def __init__(self, yolo, hyp, compute_metric=False):
        self.yolo = yolo
        self.num_stage = hyp.get("num_stage", 3)
        self.ds_scales = [8, 16, 32]
        self.inp_h, self.inp_w = hyp["input_img_size"]
        self._setup(yolo, hyp, compute_metric)


class YOLOV8Evaluator(_Evaluator):
    family = "yolov8"

    def __init__(self, yolo, hyp, compute_metric=False):
        self.yolo = yolo
        self.inp_h, self.inp_w = hyp["input_img_size"]
        self.reg = hyp["reg"]
        self._setup(yolo, hyp, compute_metric)


class RetinaNetEvaluator(_Evaluator):
    family = "retinanet"

    def __init__(self, model, hyp, compute_metric=False):
        self.model = model
        self.enable_tta = hyp["use_tta"]
        self.iou_loss_scale = hyp["tar_box_scale_factor"]
        self._setup(model, hyp, compute_metric)

    def numba_nms(self, preds_out):
        # the reference evaluator has no hyp['input_img_size'] dependency: anchors follow the image size, and the
        # decoded tensor carries no geometry, so only its row count matters here
        if isinstance(preds_out, np.ndarray):
            preds_out = torch.from_numpy(preds_out)
        preds = preds_out.detach().to(torch.float32)
        if preds.device.type != "cuda":
            preds = preds.cuda()
        h, w = self.hyp.get("input_img_size", (640, 640))
        out = self._pp.run(preds.contiguous(), int(h), int(w), decoded=True)
        return self._pp.to_list(out, as_numpy=True)


class RetinaNetEvaluatorExperiment(RetinaNetEvaluator):
    family = "retinanet_exp"


class FCOSEvaluator(_Evaluator):
    family = "fcos"

    def __init__(self, model, hyp, compute_metric=False):
        self.model = model
        self.ds_scales = [8, 16, 32, 64, 128]
        self.inp_h, self.inp_w = hyp["input_img_size"]
        self._setup(model, hyp, compute_metric)
