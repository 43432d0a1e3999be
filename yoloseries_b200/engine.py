"""Host-side engine: turns (family, hyp, head tensors) into ysb_params + device buffers and calls the C ABI.

PyTorch is plumbing here (device memory, current stream, pinned host buffers); all compute happens in
libysb_postproc.so.  Nothing in this module computes on the CPU and nothing falls back to torch ops.
"""
import ctypes
from collections import OrderedDict

import numpy as np
import torch

from . import _lib, _ops
from ._lib import YsbParams

# element types the raw heads may have (ysb_dtype): 16-bit heads are read as they are and widened on the device
HEAD_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}

# families whose raw heads the engine also reads in channels-last memory (include/ysb_postproc.h, YSB_INPUT_RAW_HEADS_NHWC)
NHWC_FAMILIES = ("yolov5", "yolox", "yolov8", "fcos")
# A channels-last head is read as rows of one anchor's channels (5+C, 4*reg+C or C values); the filter kernel stages 128 of
# them in shared memory, at most 227 KB: 128 * (width | 1) * 4 bytes (csrc/c_abi.cu), i.e. rows of up to 453 values.
NHWC_MAX_ROW_WIDTH = 453

# strides fixed by the reference evaluators (self.ds_scales), trainer/eval_yolov5.py:21, eval_yolov7.py, eval_fcos.py:18
_FIXED_STRIDES = {"yolov5": (8, 16, 32), "yolov7": (8, 16, 32), "fcos": (8, 16, 32, 64, 128)}


def retinanet_base_anchors(size):
    """The 9 base anchors of one pyramid level, float32, ratio-major (utils/anchor.py:176-191).

    Every step is a single correctly-rounded float32 operation (mul, div, sqrt, sub), so this numpy restatement is
    bit-identical to the torch code of the reference; the device kernel adds the per-cell shift analytically.
    """
    f = np.float32
    scales = np.array([1, 2 ** (1 / 3), 2 ** (2 / 3)], dtype=f)
    ratios = np.array([0.5, 1, 2], dtype=f)
    side = f(size) * np.tile(scales, 3)
    areas = side * side
    rr = np.repeat(ratios, 3)
    w = np.sqrt(areas / rr)
    h = w * rr
    out = np.zeros((9, 4), dtype=f)
    out[:, 0] = f(0) - w / f(2)
    out[:, 1] = f(0) - h / f(2)
    out[:, 2] = w - w / f(2)
    out[:, 3] = h - h / f(2)
    return out


def flatten_heads(family, heads):
    """Head tensors in the order the C ABI expects (include/ysb_postproc.h, enum ysb_family)."""
    if family in ("retinanet", "retinanet_exp"):
        reg, cls = heads
        return [reg, cls]
    if family == "fcos":
        cls_l, reg_l, ctr_l = heads
        return list(cls_l) + list(reg_l) + list(ctr_l)
    if isinstance(heads, (dict, OrderedDict)):
        return list(heads.values())
    return list(heads)


def normalise_heads(heads):
    """Model outputs as the engine needs them: float32 and contiguous, same nesting.  A no-op (no copy) for what the
    reference's models emit by default; half-precision or permuted-view outputs are converted like the reference's own
    ``.float()`` / ``.contiguous()`` calls (trainer/eval_yolov5.py:194, 265)."""
    if isinstance(heads, torch.Tensor):
        if heads.dtype == torch.float32 and heads.is_contiguous():
            return heads
        return heads.detach().to(torch.float32).contiguous()
    if isinstance(heads, (dict, OrderedDict)):
        return type(heads)((k, normalise_heads(v)) for k, v in heads.items())
    return type(heads)(normalise_heads(v) for v in heads)


def _leaves(heads):
    if isinstance(heads, torch.Tensor):
        return [heads]
    if isinstance(heads, (dict, OrderedDict)):
        heads = heads.values()
    return [t for v in heads for t in _leaves(v)]


def nhwc_row_width(family, num_class, dfl_bins=16):
    """Values per row of a channels-last head of ``family``: the channels of one anchor (FCOS: of the cls tensor)."""
    C = int(num_class)
    return {"yolov5": 5 + C, "yolox": 5 + C, "yolov8": 4 * int(dfl_bins) + C, "fcos": C}[family]


def _channels_last_strides(family, t):
    """The strides ``t`` has when it is a channels-last head of ``family`` (None: no such pattern for its rank)."""
    if family in ("yolov5", "yolov8", "fcos") and t.dim() == 4:   # (b, K, H, W) stored as (b, H, W, K)
        _, K, H, W = t.shape
        return (H * W * K, 1, W * K, K)
    if family == "yolox" and t.dim() == 5:                         # (b, A, K, H, W) view of a channels-last (b, A*K, H, W)
        _, A, K, H, W = t.shape
        return (H * W * A * K, K, 1, W * A * K, A * K)
    return None


def is_channels_last_head(family, t):
    """True when ``t`` has the channels-last memory of a ``family`` head; the strides of size-1 dims do not matter (a
    1-channel ctr or a 1x1 level qualifies)."""
    want = _channels_last_strides(family, t)
    return want is not None and all(n == 1 or s == w for n, s, w in zip(t.shape, t.stride(), want))


def head_layout(family, flat):
    """Input kind of a flat head list: INPUT_RAW_HEADS when every tensor is contiguous (checked first, so a list that
    fits both patterns is NCHW), INPUT_RAW_HEADS_NHWC when every tensor is a channels-last head of ``family`` (YOLOv5,
    YOLOX, YOLOv8, FCOS).  Anything else -- views of other strides, or levels of different layouts -- raises ValueError."""
    if all(t.is_contiguous() for t in flat):
        return _lib.INPUT_RAW_HEADS
    if family in NHWC_FAMILIES and all(is_channels_last_head(family, t) for t in flat):
        return _lib.INPUT_RAW_HEADS_NHWC
    cl = f"; or all channels-last ({', '.join(NHWC_FAMILIES)})" if family in NHWC_FAMILIES else ""
    raise ValueError(f"head tensors must be contiguous float32, float16 or bfloat16{cl}, got strides "
                     f"{[tuple(t.stride()) for t in flat]} for shapes {[tuple(t.shape) for t in flat]}")


def native_heads(heads, family=None, num_class=None, dfl_bins=16):
    """Model outputs as the engine takes them: unchanged when every tensor is contiguous and all share one of float32,
    float16 or bfloat16 (16-bit heads are read natively, no conversion pass); anything else goes through
    normalise_heads.  With ``family`` (and ``num_class``, ``dfl_bins`` for YOLOv8), heads that are all channels-last
    (a model run with torch.channels_last) are passed through unchanged too, unless their rows are wider than
    NHWC_MAX_ROW_WIDTH."""
    leaves = _leaves(heads)
    if leaves and leaves[0].dtype in HEAD_DTYPES and all(t.dtype == leaves[0].dtype for t in leaves):
        if all(t.is_contiguous() for t in leaves):
            return heads
        if family in NHWC_FAMILIES and all(is_channels_last_head(family, t) for t in leaves):
            if num_class is None:
                raise ValueError("native_heads: num_class is required with a family")
            if nhwc_row_width(family, num_class, dfl_bins) <= NHWC_MAX_ROW_WIDTH:
                return heads
    return normalise_heads(heads)


def _level_shapes(family, flat, num_class):
    if family in ("yolov5", "yolox", "yolov8"):
        return [(t.shape[-2], t.shape[-1]) for t in flat]
    if family == "yolov7":
        return [(t.shape[2], t.shape[3]) for t in flat]
    if family == "fcos":
        n = len(flat) // 3
        return [(t.shape[2], t.shape[3]) for t in flat[:n]]
    raise ValueError(family)


def make_params(family, hyp, batch, img_h, img_w, level_shapes=None, anchors=None, input_kind=_lib.INPUT_RAW_HEADS,
                compute_metric=False, num_anchors=None, decoded_rows=0, tta=None, head_dtype=torch.float32):
    """Build ``ysb_params`` from the reference's flat ``hyp`` dict (SURVEY.md section 5 lists the keys).

    ``tta`` = (scale, flip_axis, org_h, org_w) describes one test-time-augmentation pass (trainer/eval_yolov5.py:152-179):
    the boxes decoded from this pass's heads are divided by ``scale`` and un-flipped (axis 2 or 3) against the size of
    the un-augmented input.  ``head_dtype``: element type of the raw heads, torch.float32 / float16 / bfloat16."""
    if head_dtype not in HEAD_DTYPES:
        raise ValueError(f"head_dtype must be one of {sorted(map(str, HEAD_DTYPES))}, got {head_dtype}")
    p = YsbParams()
    p.head_dtype = HEAD_DTYPES[head_dtype]
    p.family = _lib.FAMILY_IDS[family]
    p.input_kind = input_kind
    p.batch = int(batch)
    p.num_classes = int(hyp["num_class"])
    p.img_h, p.img_w = int(img_h), int(img_w)
    pre = "compute_metric_" if compute_metric else ""
    p.iou_thr = float(hyp[pre + "iou_threshold"])
    p.cls_thr = float(hyp[pre + "cls_threshold"])
    p.conf_thr = float(hyp.get(pre + "conf_threshold", 0.0))
    p.pre_nms_thr = float(hyp.get("pre_nms_thresh", 0.0))
    p.max_det = int(hyp["max_predictions_per_img"])
    p.class_aware = int(bool(hyp["agnostic"]))
    p.multi_label = int(bool(hyp["mutil_label"]))
    p.postprocess_bbox = int(bool(hyp["postprocess_bbox"]))
    p.min_box_wh = float(hyp.get("min_prediction_box_wh", 0))
    p.pre_nms_topk = int(hyp.get("pre_nms_topk", 1000))
    p.thresh_with_ctr = int(bool(hyp.get("thresh_with_ctr", True)))
    p.dfl_bins = int(hyp.get("reg", 16))
    p.decoded_rows = int(decoded_rows)
    if tta is not None:
        p.tta_scale = float(tta[0])
        p.tta_flip = int(tta[1] or 0)
        p.tta_img_h, p.tta_img_w = int(tta[2]), int(tta[3])
    scale = hyp.get("tar_box_scale_factor", [0.1, 0.1, 0.2, 0.2])
    for i in range(4):
        p.reg_scale[i] = float(scale[i])
    if family in ("retinanet", "retinanet_exp"):
        levels = (3, 4, 5, 6, 7)
        p.num_levels = len(levels)
        p.anchors_per_cell = 9
        for i, lvl in enumerate(levels):
            p.level_h[i] = (img_h - 1) // 2 ** lvl + 1
            p.level_w[i] = (img_w - 1) // 2 ** lvl + 1
            p.level_stride[i] = float(2 ** lvl)
            base = retinanet_base_anchors(2 ** (lvl + 2))
            for a in range(9):
                for c in range(4):
                    p.anchor[i][a][c] = float(base[a, c])
        return p
    if level_shapes is None:
        raise ValueError("level_shapes is required for grid families")
    p.num_levels = len(level_shapes)
    for i, (h, w) in enumerate(level_shapes):
        p.level_h[i], p.level_w[i] = int(h), int(w)
        if family == "fcos":
            # level_i_stride = self.inp_h / fm_h with inp_h from hyp['input_img_size'], not from the actual input
            # (trainer/eval_fcos.py:17,137): mirrored, so an input of another size decodes like the reference does
            p.level_stride[i] = float(int(hyp.get("input_img_size", (img_h, img_w))[0]) / h)
        elif family in _FIXED_STRIDES:
            p.level_stride[i] = float(_FIXED_STRIDES[family][i])
        else:
            p.level_stride[i] = float(img_h / h)  # eval_yolox.py:144, eval_yolov8.py:91
    if family in ("yolov5", "yolov7"):
        if anchors is None:
            raise ValueError("anchors (L, A, 2) are required for yolov5 / yolov7")
        anc = torch.as_tensor(anchors).detach().cpu()
        p.anchors_per_cell = int(anc.shape[1])
        for i in range(anc.shape[0]):
            # (self.anchors[i] / self.ds_scales[i]).type_as(inputs): true divide, then float32 (eval_yolov5.py:192)
            stage = (anc[i] / _FIXED_STRIDES[family][i]).to(torch.float32)
            for a in range(anc.shape[1]):
                p.anchor[i][a][0] = float(stage[a, 0])
                p.anchor[i][a][1] = float(stage[a, 1])
    elif family == "yolox":
        p.anchors_per_cell = int(num_anchors or hyp.get("num_anchors", 1))
    else:
        p.anchors_per_cell = 1
    return p


def letterbox_table(info):
    """list of the reference's per-image info dicts -> (b, 5) rows {scale, pad_top, pad_left, org_h, org_w}."""
    return [[float(d["scale"]), float(d["pad_top"]), float(d["pad_left"]), float(d["org_shape"][0]),
             float(d["org_shape"][1])] for d in info]


def letterbox_rows(info, batch):
    """letterbox_table(info); raises ValueError unless there is one dict per image of a ``batch``-image batch."""
    if len(info) != batch:
        raise ValueError(f"need one info dict per image: {len(info)} != {batch}")
    return letterbox_table(info)


class LetterboxStaging:
    """One pipeline lane's letterbox table: the (batch, 5) float32 device table the NMS kernel's row write reads, and the
    pinned staging buffer it is copied from with cudaMemcpyAsync on the lane's stream, so an upload never makes the host
    wait for the lane's earlier work.  Construct it under the lane's stream; the table's address never changes (CUDA
    graphs capture it, and may capture the copy as well)."""

    def __init__(self, batch, device):
        self.table = torch.empty((batch, 5), dtype=torch.float32, device=device)
        self.host = torch.empty((batch, 5), dtype=torch.float32, pin_memory=True)
        self._host_np = self.host.numpy()

    def stage(self, rows, after):
        """Write ``rows`` (letterbox_rows, up to ``batch`` of them) into the first rows of the staging buffer; returns the
        table's address.  ``after``: an event
        recorded after the previous copy out of the buffer (None: there was none).  That copy may still be queued behind
        the lane's earlier work -- in a detection gather, behind the flow control that waits for the peers -- and
        overwriting the buffer before it ran would map that earlier batch with these rows."""
        if after is not None:
            after.synchronize()
        self._host_np[:len(rows)] = rows   # float32, rounded to nearest like torch.tensor(rows, dtype=torch.float32)
        return self.table.data_ptr()

    def enqueue_copy(self):
        """The copy of the staged rows into the table on the current stream (capturable into a CUDA graph)."""
        self.table.copy_(self.host, non_blocking=True)


# ---- mAP hand-off: ground truth matched against the kept rows where they are (ysb_match_tp) -----------------------------
MATCH_DTYPES = (np.float32, np.float64)   # ground-truth element types the match kernel reads (one per step)


def _target_array(t, i):
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    if a.size == 0:
        return a.reshape(0, 5)
    if a.ndim != 2 or a.shape[1] != 5:
        raise ValueError(f"targets[{i}]: expected an (n, 5) array (x1, y1, x2, y2, cls), got shape {a.shape}")
    if a.dtype not in MATCH_DTYPES:
        raise ValueError(f"targets[{i}]: expected float32 or float64, got {a.dtype}")
    return a


def pack_targets(targets, positions, images, capacity):
    """Host half of ``match``: one (n_i, 5) ground-truth array or tensor per image of a step, in ``result()`` order, ->
    (arrays, dtype, max_n): image ``positions[i]`` of the step's ``images`` (rank * batch + image) receives
    ``targets[i]``.  dtype is the step's one element type (float32 or float64; empty arrays take any), max_n its largest
    count (at least 1), the padded stride of the block the kernel reads.  Raises ValueError for a wrong count of arrays,
    a wrong shape or dtype, mixed dtypes, or more than ``capacity`` rows in one image."""
    if len(targets) != len(positions):
        raise ValueError(f"need one target array per image of the step: {len(targets)} != {len(positions)}")
    arrs = [_target_array(t, i) for i, t in enumerate(targets)]
    for i, a in enumerate(arrs):
        if a.shape[0] > capacity:
            raise ValueError(f"targets[{i}] has {a.shape[0]} boxes, more than the processor's max_targets = {capacity}")
    dtypes = {a.dtype for a in arrs if a.shape[0]}
    if len(dtypes) > 1:
        raise ValueError(f"every target array of a step must have one dtype, got {sorted(map(str, dtypes))}")
    if any(not 0 <= k < images for k in positions):
        raise ValueError(f"image positions outside 0..{images - 1}")
    dtype = np.dtype(dtypes.pop() if dtypes else np.float32)
    max_n = max([1] + [a.shape[0] for a in arrs])
    return arrs, dtype, max_n


class TargetStaging:
    """The padded ground truth of one lane's ``match``: a pinned host buffer and a device buffer holding the (images)
    int32 counts followed by the (images, max_n, 5) rows, uploaded with one cudaMemcpyAsync on the current stream (the
    lane's), so the upload never makes the host wait for the lane's earlier work.  Both grow (powers of two) to the
    largest step seen; a step's max_n is its largest count, so a COCO step uploads tens of KB."""

    def __init__(self, images, device):
        self.images, self.device = int(images), torch.device(device)
        self._cnt_bytes = (4 * self.images + 15) // 16 * 16
        self._host = self._dev = None
        self._copied = None   # event after the last copy out of the pinned buffer

    def stage(self, arrs, positions, dtype, max_n):
        """Fill the buffer and enqueue its upload; returns device views (gt (images, max_n, 5), counts (images,))."""
        nbytes = self._cnt_bytes + self.images * max_n * 5 * dtype.itemsize
        if self._copied is not None:
            self._copied.synchronize()   # the previous upload may still be queued behind the lane's earlier work
        if self._host is None or self._host.numel() < nbytes:
            size = 1 << max(12, (nbytes - 1).bit_length())
            self._host = torch.empty(size, dtype=torch.uint8, pin_memory=True)
            self._dev = torch.empty(size, dtype=torch.uint8, device=self.device)
        raw = self._host.numpy()
        cnt = raw[:4 * self.images].view(np.int32)
        cnt[:] = 0
        vals = raw[self._cnt_bytes:nbytes].view(dtype).reshape(self.images, max_n, 5)
        for k, a in zip(positions, arrs):
            cnt[k] = a.shape[0]
            vals[k, :a.shape[0]] = a
        self._dev[:nbytes].copy_(self._host[:nbytes], non_blocking=True)
        self._copied = torch.cuda.Event()
        self._copied.record(torch.cuda.current_stream(self.device))
        gt = self._dev[self._cnt_bytes:nbytes].view(torch.float64 if dtype == np.float64 else torch.float32)
        return gt.view(self.images, max_n, 5), self._dev[:4 * self.images].view(torch.int32)


class Matches:
    """What ``match`` enqueued for one step, all device tensors ordered on ``stream`` (the lane's): the step's rows
    (world, batch, max_det, 6) and counts (world, batch) as the processor keeps them, the staged ground truth
    (world, batch, max_n, 5) and its counts, and ``tp`` (world, batch, max_det, 10) uint8 -- the reference's bool matrix
    of every present image, aligned with its rows (world = 1 for PostProcessor and PipelinedPostProcessor).  Valid until
    the lane's buffers are reused, like the ticket.  MatchStats.add appends it to a run's arrays."""

    def __init__(self, rows, cnt, gt, gt_cnt, tp, stream, n_targets):
        self.rows, self.cnt, self.gt, self.gt_cnt, self.tp = rows, cnt, gt, gt_cnt, tp
        self.stream, self.n_targets = stream, n_targets

    def to_list(self):
        """Host copy: list over the step's present images in ``result()`` order of (K, 10) bool arrays (K = 0 for the
        reference's None).  Synchronises the lane."""
        self.stream.synchronize()
        cnt = self.cnt.cpu().reshape(-1).tolist()
        tp = self.tp.cpu().numpy().reshape(len(cnt), self.tp.shape[2], 10).astype(bool)
        return [tp[k, :max(c, 0)] for k, c in enumerate(cnt) if c != _lib.YSB_CNT_ABSENT]


class StepMatcher:
    """The device state of ``match`` for one output buffer (a PostProcessor entry, a pipeline lane, a gather slot):
    the ground-truth staging and the tp rows.  Construct and run it under the buffer's stream."""

    def __init__(self, world, batch, max_det, capacity, device):
        self.world, self.batch, self.capacity = int(world), int(batch), int(capacity)
        self.staging = TargetStaging(self.world * self.batch, device)
        self.tp = torch.empty((self.world, self.batch, int(max_det), 10), dtype=torch.uint8, device=device)

    def run(self, rows, cnt, targets, positions, iou_thr=None):
        from .utils.mAP import IOU_THRESHOLDS
        thr = [float(v) for v in np.asarray(IOU_THRESHOLDS if iou_thr is None else iou_thr, dtype=np.float64).reshape(-1)]
        if len(thr) != 10:
            raise ValueError("iou_thr must hold 10 thresholds (np.linspace(0.5, 0.95, 10) in the reference)")
        arrs, dtype, max_n = pack_targets(targets, positions, self.world * self.batch, self.capacity)
        gt, gt_cnt = self.staging.stage(arrs, positions, dtype, max_n)
        gt, gt_cnt = gt.view(self.world, self.batch, max_n, 5), gt_cnt.view(self.world, self.batch)
        _ops.load().match_tp(rows, cnt, gt, gt_cnt, thr, self.tp)
        return Matches(rows, cnt, gt, gt_cnt, self.tp, torch.cuda.current_stream(self.tp.device),
                       sum(a.shape[0] for a in arrs))


def check_max_targets(max_targets):
    if int(max_targets) < 1:
        raise ValueError(f"max_targets must be at least 1, got {max_targets}")
    return int(max_targets)


class DetectionList(list):
    """The evaluator's output list (CPU rows, the reference's contract) that also remembers the device rows it was read
    from, so that preds_postprocess can map them without staging them back to the GPU."""
    device_rows = None    # (b, max_det, 6) float32 CUDA tensor (a private copy, not the reused output buffer)
    device_cnt = None     # (b,) int32 CUDA tensor


def preds_postprocess(outputs, info):
    """val_yolov5.py:164-177 for an evaluator's output list: list[Tensor(K,6) | None] -> list[ndarray(K,6) | None].

    (The image half of the reference's method -- un-padding and resizing the input picture for drawing -- is
    visualisation and stays with the caller.)  When ``outputs`` is the DetectionList an evaluator mirror returned, the
    rows are still on the device: ysb_undo_letterbox runs on them and only the mapped rows come back.  Any other list is
    staged to the device first.  (Callers that pass ``info`` to the evaluator get the undo fused into the NMS kernel's
    row write and need neither.)
    """
    if len(outputs) != len(info):
        raise ValueError(f"need one info dict per image: {len(info)} != {len(outputs)}")
    if not outputs:
        return []
    if not torch.cuda.is_available():
        raise RuntimeError("yoloseries_b200 needs a CUDA device: the engine has no CPU fallback")
    lib = _lib.load()
    if isinstance(outputs, DetectionList) and outputs.device_rows is not None:
        dets, dcnt = outputs.device_rows.clone(), outputs.device_cnt
        dev = dets.device
        cnt = [(-1 if o is None else int(o.shape[0])) for o in outputs]
        kmax = dets.shape[1]
    else:
        dev = torch.device("cuda", torch.cuda.current_device())
        kmax = max([1] + [int(o.shape[0]) for o in outputs if o is not None])
        host = torch.zeros((len(outputs), kmax, 6), dtype=torch.float32)
        cnt = [(-1 if o is None else int(o.shape[0])) for o in outputs]
        for i, o in enumerate(outputs):
            if o is not None and o.shape[0]:
                host[i, : o.shape[0]] = torch.as_tensor(o, dtype=torch.float32).reshape(-1, 6)
        dets, dcnt = host.to(dev), torch.tensor(cnt, dtype=torch.int32).to(dev)
    table = torch.tensor(letterbox_table(info), dtype=torch.float32).to(dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ysb_undo_letterbox(dets.data_ptr(), dcnt.data_ptr(), len(outputs), kmax, table.data_ptr(),
                                          ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "ysb_undo_letterbox")
    back = dets[:, : max(max(cnt), 1)].cpu().numpy()
    return [None if c < 0 else back[i, :c].copy() for i, c in enumerate(cnt)]


def validate_heads(family, flat, num_class, anchors=None, dfl_bins=16, decoded_row_w=None):
    """Full shape check of the head tensors against the family's layout (include/ysb_postproc.h, enum ysb_family).  The C
    ABI receives bare pointers, so this is the only place a wrong channel count / batch / level count can be caught; the
    reference raises a reshape error in the same situations (e.g. trainer/eval_yolov5.py:194)."""
    C = int(num_class)

    def bad(msg):
        raise ValueError(f"{family} heads: {msg}")
    if not flat:
        bad("no tensors")
    if not 1 <= C <= _lib.YSB_MAX_CLASSES:
        bad(f"num_class {C} is outside 1..{_lib.YSB_MAX_CLASSES} (YSB_MAX_CLASSES)")
    b = flat[0].shape[0]
    for i, t in enumerate(flat):
        if t.dtype not in HEAD_DTYPES or (decoded_row_w is not None and not t.is_contiguous()):
            raise ValueError(f"head tensors must be contiguous float32, float16 or bfloat16, got {t.dtype}")
        if t.dtype != flat[0].dtype:
            raise ValueError(f"head tensors must share one dtype (contiguous float32, float16 or bfloat16), got "
                             f"{flat[0].dtype} and {t.dtype}")
        if t.dim() < 2 or t.shape[0] != b:
            bad(f"tensor {i} has batch {tuple(t.shape)[:1]}, expected {b}")
        if t.device != flat[0].device:
            bad("tensors live on different devices")
    if decoded_row_w is not None:
        if flat[0].dtype != torch.float32:
            raise ValueError(f"decoded tensor must be contiguous float32, got {flat[0].dtype}")
        if len(flat) != 1 or flat[0].dim() != 3 or flat[0].shape[2] != decoded_row_w:
            raise ValueError(f"decoded tensor must be (b, N, {decoded_row_w}), got {tuple(flat[0].shape)}")
        return _lib.INPUT_DECODED_ROWS
    kind = head_layout(family, flat)   # contiguous (NCHW) or, for the planes families, channels-last
    if family in ("yolov5", "yolov7"):
        if anchors is None:
            bad("anchors (L, A, 2) are required")
        L, A = int(anchors.shape[0]), int(anchors.shape[1])
        if len(flat) != L:
            bad(f"{len(flat)} levels but {L} anchor groups")
        for i, t in enumerate(flat):
            want = (b, A * (5 + C)) if family == "yolov5" else (b, A)
            if family == "yolov5" and (t.dim() != 4 or tuple(t.shape[:2]) != want):
                bad(f"level {i} must be (b, {A * (5 + C)}, H, W), got {tuple(t.shape)}")
            if family == "yolov7" and (t.dim() != 5 or tuple(t.shape[:2]) != want or t.shape[4] != 5 + C):
                bad(f"level {i} must be (b, {A}, H, W, {5 + C}), got {tuple(t.shape)}")
    elif family == "yolox":
        na = flat[0].shape[1] if flat[0].dim() == 5 else -1
        for i, t in enumerate(flat):
            if t.dim() != 5 or t.shape[1] != na or t.shape[2] != 5 + C:
                bad(f"level {i} must be (b, {na}, {5 + C}, H, W), got {tuple(t.shape)}")
    elif family == "yolov8":
        for i, t in enumerate(flat):
            if t.dim() != 4 or t.shape[1] != 4 * int(dfl_bins) + C:
                bad(f"level {i} must be (b, {4 * int(dfl_bins) + C}, H, W), got {tuple(t.shape)}")
    elif family in ("retinanet", "retinanet_exp"):
        w = 5 if family == "retinanet_exp" else 4
        if len(flat) != 2:
            bad("expected (reg, cls)")
        reg, cls = flat
        if reg.dim() != 3 or reg.shape[2] != w or cls.dim() != 3 or cls.shape[2] != C or reg.shape[1] != cls.shape[1]:
            bad(f"expected reg (b, N, {w}) and cls (b, N, {C}), got {tuple(reg.shape)} and {tuple(cls.shape)}")
    elif family == "fcos":
        if len(flat) % 3:
            bad("expected three lists (cls, reg, ctr) of equal length")
        n = len(flat) // 3
        for i in range(n):
            c, r, q = flat[i], flat[n + i], flat[2 * n + i]
            hw = tuple(c.shape[2:])
            if c.dim() != 4 or c.shape[1] != C or r.dim() != 4 or r.shape[1] != 4 or tuple(r.shape[2:]) != hw or \
                    q.dim() != 4 or q.shape[1] != 1 or tuple(q.shape[2:]) != hw:
                bad(f"level {i} must be cls (b, {C}, H, W), reg (b, 4, H, W), ctr (b, 1, H, W), got "
                    f"{tuple(c.shape)}, {tuple(r.shape)}, {tuple(q.shape)}")
    else:
        raise ValueError(f"unknown family {family!r}")
    return kind


class DetectionBuffers:
    """Per-call device outputs: rows (b, max_det, 6), candidate indices (b, max_det), counts (b)."""

    def __init__(self, batch, max_det, device):
        self.dets = torch.empty((batch, max_det, 6), dtype=torch.float32, device=device)
        self.det_idx = torch.empty((batch, max_det), dtype=torch.int32, device=device)
        self.det_cnt = torch.empty((batch,), dtype=torch.int32, device=device)
        self.matcher = None   # StepMatcher of PostProcessor.match, made on first use


class PostProcessor:
    """decode -> filter -> top-k -> class-aware NMS -> post-filter for one family / one head geometry.

    Buffers are allocated once per (batch, geometry) and reused; every call enqueues on torch's current stream.
    ``max_targets``: ground-truth boxes per image that ``match`` accepts.
    """

    def __init__(self, family, hyp, anchors=None, compute_metric=False, max_targets=1024):
        self.max_targets = check_max_targets(max_targets)
        self.family = family
        self.hyp = dict(hyp)
        self.anchors = anchors
        self.compute_metric = compute_metric
        self._lib = _lib.load()
        self._ops = _ops.load()
        self._cache = {}

    # ---- plumbing ------------------------------------------------------------------------------------------
    def _prepare(self, flat, batch, img_h, img_w, input_kind, tta=None):
        dev = flat[0].device
        if dev.type != "cuda":
            raise RuntimeError("yoloseries_b200 runs on CUDA devices only (no CPU fallback); got " + str(dev))
        raw = input_kind != _lib.INPUT_DECODED_ROWS
        if raw:
            # the layout picks the input kind: contiguous NCHW heads or channels-last ones
            input_kind = validate_heads(self.family, flat, self.hyp["num_class"], self.anchors, self.hyp.get("reg", 16))
            if input_kind == _lib.INPUT_RAW_HEADS_NHWC:
                k = nhwc_row_width(self.family, self.hyp["num_class"], self.hyp.get("reg", 16))
                if k > NHWC_MAX_ROW_WIDTH:
                    raise ValueError(f"{self.family} channels-last heads: rows of {k} values exceed the limit of "
                                     f"{NHWC_MAX_ROW_WIDTH} (NHWC_MAX_ROW_WIDTH); pass contiguous heads")
        else:
            for t in flat:
                if t.dtype != torch.float32 or not t.is_contiguous():
                    raise ValueError("head tensors must be contiguous float32")
        shapes = None
        if raw and self.family not in ("retinanet", "retinanet_exp"):
            shapes = _level_shapes(self.family, flat, self.hyp["num_class"])
        elif self.family not in ("retinanet", "retinanet_exp"):
            strides = _FIXED_STRIDES.get(self.family) or ((4, 8, 16, 32) if self.family == "yolov8" else (8, 16, 32))
            shapes = [(img_h // s, img_w // s) for s in strides]
        na = flat[0].shape[1] if (self.family == "yolox" and raw) else None
        rows = int(flat[0].shape[1]) if input_kind == _lib.INPUT_DECODED_ROWS else 0
        key = (batch, img_h, img_w, input_kind, tuple(shapes or ()), dev.index, na, rows, tta, flat[0].dtype)
        ent = self._cache.get(key)
        if ent is None:
            params = make_params(self.family, self.hyp, batch, img_h, img_w, shapes, self.anchors, input_kind,
                                 self.compute_metric, na, rows, tta, flat[0].dtype)
            n = ctypes.c_int64()
            rw = ctypes.c_int32()
            _lib.check(self._lib.ysb_num_candidates(ctypes.byref(params), ctypes.byref(n), ctypes.byref(rw)),
                       "ysb_num_candidates")
            ws = ctypes.c_size_t()
            _lib.check(self._lib.ysb_postprocess_workspace_bytes(ctypes.byref(params), ctypes.byref(ws)),
                       "ysb_postprocess_workspace_bytes")
            ent = dict(params=params, params_t=_ops.params_tensor(params), N=n.value, row_w=rw.value,
                       workspace=torch.empty(max(ws.value, 1), dtype=torch.uint8, device=dev),
                       out=DetectionBuffers(batch, params.max_det, dev))
            self._cache[key] = ent
        if raw and self.family in ("retinanet", "retinanet_exp") and flat[0].shape[1] != ent["N"]:
            raise ValueError(f"{self.family} heads: {flat[0].shape[1]} anchors per image, but a {img_h}x{img_w} input has {ent['N']}")
        if input_kind == _lib.INPUT_DECODED_ROWS:
            validate_heads(self.family, flat, self.hyp["num_class"], decoded_row_w=ent["row_w"])
        return ent

    @staticmethod
    def _stream(dev=None):
        """torch's current stream ON THE HEADS' DEVICE (not on whatever device happens to be current)."""
        return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    # ---- public ops ----------------------------------------------------------------------------------------
    def decode(self, heads, img_h, img_w):
        """do_inference: raw heads (float32, float16 or bfloat16) -> (b, N, C') float32 on the heads' device."""
        flat = flatten_heads(self.family, heads)
        batch = flat[0].shape[0]
        ent = self._prepare(flat, batch, img_h, img_w, _lib.INPUT_RAW_HEADS)
        return self._ops.decode(flat, ent["params_t"])

    def _letterbox(self, holder, params_list, info, batch, dev):
        """Stage the reference's per-image info dicts as the (b, 5) table the NMS kernel's row write reads (fused
        preds_postprocess, val_yolov5.py:166-172); ``info`` None switches the undo off."""
        ptr = None
        if info is not None:
            rows = torch.tensor(letterbox_rows(info, batch), dtype=torch.float32)
            if "lb" not in holder:
                holder["lb"] = torch.empty((batch, 5), dtype=torch.float32, device=dev)
            holder["lb"].copy_(rows, non_blocking=False)
            ptr = holder["lb"].data_ptr()
        for p in params_list:
            p.d_letterbox = ptr

    def _run_entry(self, heads, img_h, img_w, decoded):
        """(flat heads, cache entry) of one run; the entry is None for a batch of zero images."""
        flat = [heads] if decoded else flatten_heads(self.family, heads)
        if flat[0].shape[0] == 0:
            return flat, None
        kind = _lib.INPUT_DECODED_ROWS if decoded else _lib.INPUT_RAW_HEADS
        return flat, self._prepare(flat, flat[0].shape[0], img_h, img_w, kind)

    def _launch(self, flat, ent):
        """The whole path for an entry whose params (letterbox pointer included) are set."""
        out = ent["out"]
        # through the torch extension (csrc/torch_adapter.cpp): tensor checks, device guard, torch's current stream
        self._ops.postprocess(flat, ent["params_t"], ent["workspace"], out.dets, out.det_idx, out.det_cnt)
        return out

    def run(self, heads, img_h, img_w, decoded=False, info=None):
        """Whole path on the device.  Returns DetectionBuffers (views into reused storage).  ``info``: optional list of
        the reference's letterbox dicts (scale, pad_top, pad_left, org_shape): rows come out in original-picture pixels."""
        flat, ent = self._run_entry(heads, img_h, img_w, decoded)
        if ent is None:  # the reference loops over zero images and returns []
            return DetectionBuffers(0, int(self.hyp["max_predictions_per_img"]), flat[0].device)
        dev = flat[0].device
        with torch.cuda.device(dev):
            self._letterbox(ent, [ent["params"]], info, flat[0].shape[0], dev)
        return self._launch(flat, ent)

    # ---- test-time augmentation (trainer/eval_yolov5.py:152-179 and the same method of every evaluator) ------------
    def _tta_entries(self, passes, org_hw, batch=None):
        """passes: [(heads, img_h, img_w, scale, flip_axis), ...] -> [(flat heads, cache entry), ...].  ``batch``: the
        entries' image count when it is not the heads' (a sharded processor set up by a partial step)."""
        if not 1 <= len(passes) <= _lib.YSB_MAX_PASSES:
            raise ValueError(f"1..{_lib.YSB_MAX_PASSES} passes, got {len(passes)}")
        ents = []
        for heads, img_h, img_w, scale, flip in passes:
            flat = flatten_heads(self.family, heads)
            tta = (float(scale), int(flip or 0), int(org_hw[0]), int(org_hw[1]))
            b = flat[0].shape[0] if batch is None else batch
            ents.append((flat, self._prepare(flat, b, int(img_h), int(img_w), _lib.INPUT_RAW_HEADS, tta)))
        if len({e["params"].batch for _, e in ents}) != 1:
            raise ValueError("every pass must hold the same images")
        if len({e["params"].input_kind for _, e in ents}) != 1:
            raise ValueError("every pass must have heads of one layout (all contiguous or all channels-last)")
        return ents

    def decode_tta(self, passes, org_hw):
        """test_time_augmentation: every pass decoded, un-scaled and un-flipped straight into its slot of the merged
        (b, sum N_i, C') tensor.  Returns (merged, [per-pass views])."""
        ents = self._tta_entries(passes, org_hw)
        batch, total = ents[0][1]["params"].batch, sum(e["N"] for _, e in ents)
        out = torch.empty((batch, total, ents[0][1]["row_w"]), dtype=torch.float32, device=ents[0][0][0].device)
        off, views = 0, []
        dev = out.device
        for flat, ent in ents:
            self._ops.decode_into(flat, ent["params_t"], out, off)
            views.append(out[:, off:off + ent["N"]])
            off += ent["N"]
        return out, views

    def run_tta(self, passes, org_hw, info=None):
        """The whole path over several augmented passes without the merged tensor (ysb_postprocess_tta).  Candidate
        indices (det_idx) count through the passes in order, like rows of the reference's concatenated tensor."""
        ents = self._tta_entries(passes, org_hw)
        dev = ents[0][0][0].device
        batch = ents[0][1]["params"].batch
        if batch == 0:
            return DetectionBuffers(0, int(self.hyp["max_predictions_per_img"]), dev)
        n = len(ents)
        key = ("tta", dev.index) + tuple(id(e) for _, e in ents)
        bundle = self._cache.get(key)
        if bundle is None:
            arr = (YsbParams * n)(*[e["params"] for _, e in ents])
            ws = ctypes.c_size_t()
            _lib.check(self._lib.ysb_postprocess_tta_workspace_bytes(arr, n, ctypes.byref(ws)),
                       "ysb_postprocess_tta_workspace_bytes")
            bundle = dict(params=arr, workspace=torch.empty(max(ws.value, 1), dtype=torch.uint8, device=dev),
                          out=DetectionBuffers(batch, arr[0].max_det, dev), keep=[e for _, e in ents])
            self._cache[key] = bundle
        flat_all = [t for flat, _ in ents for t in flat]
        per_pass = (ctypes.c_int32 * n)(*[len(flat) for flat, _ in ents])
        out, ws = bundle["out"], bundle["workspace"]
        with torch.cuda.device(dev):
            self._letterbox(bundle, [bundle["params"][i] for i in range(n)], info, batch, dev)
            _lib.check(self._lib.ysb_postprocess_tta(bundle["params"], n, _lib.head_pointer_array(flat_all), per_pass,
                                                     ws.data_ptr(), ws.numel(), out.dets.data_ptr(), out.det_idx.data_ptr(),
                                                     out.det_cnt.data_ptr(), self._stream(dev)), "ysb_postprocess_tta")
        return out

    def capture(self, heads, img_h, img_w, decoded=False):
        """Capture {zero counters, filter kernel, NMS kernel} for THESE head tensors into a CUDA graph.

        Returns a callable: every call replays the graph on the current stream (one driver call instead of a Python
        -> ctypes -> three launches round trip; +47 % images/s at 8 images per batch) and returns the DetectionBuffers.
        The head tensors are baked in by address: refill them in place (as a CUDA-graphed model does).
        """
        self.run(heads, img_h, img_w, decoded=decoded)  # warm-up outside capture: function attributes, buffers
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=(heads if decoded else flatten_heads(self.family, heads)[0]).device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
            out = self.run(heads, img_h, img_w, decoded=decoded)
        keep_alive = heads

        def replay():
            graph.replay()
            return out

        replay.graph, replay.heads = graph, keep_alive
        return replay

    def filter_only(self, heads, img_h, img_w, decoded=False):
        """K1 alone: returns (keys (b, N) uint64 as int64 tensor, counts (b, 4) int32)."""
        flat = [heads] if decoded else flatten_heads(self.family, heads)
        batch = flat[0].shape[0]
        kind = _lib.INPUT_DECODED_ROWS if decoded else _lib.INPUT_RAW_HEADS
        ent = self._prepare(flat, batch, img_h, img_w, kind)
        dev = flat[0].device
        slots = ent["N"] * (int(self.hyp["num_class"]) if self.hyp["mutil_label"] else 1)
        keys = torch.empty((batch, slots), dtype=torch.int64, device=dev)
        counts = torch.empty((batch, 4), dtype=torch.int32, device=dev)
        self._ops.filter_candidates(flat, ent["params_t"], keys, counts)
        return keys, counts

    def undo_letterbox(self, out, info):
        """The box part of val_yolov5.py:140-179 (preds_postprocess) on the kept rows, in place, before the D2H copy.

        ``info``: per image the reference's dict (``scale``, ``pad_top``, ``pad_left``, ``org_shape`` = (h, w)).
        x = clamp((x - pad_left) / scale, 1, org_w - 1), y likewise with pad_top / org_h; float32, op by op.
        """
        if out.det_cnt.numel() == 0:
            return out
        if len(info) != out.det_cnt.numel():
            raise ValueError(f"need one info dict per image: {len(info)} != {out.det_cnt.numel()}")
        dev = out.dets.device
        table = torch.tensor(letterbox_table(info), dtype=torch.float32).to(dev, non_blocking=True)
        with torch.cuda.device(dev):
            _lib.check(self._lib.ysb_undo_letterbox(out.dets.data_ptr(), out.det_cnt.data_ptr(), out.dets.shape[0],
                                                    out.dets.shape[1], table.data_ptr(), self._stream(dev)),
                       "ysb_undo_letterbox")
        return out

    def match(self, out, targets, iou_thr=None):
        """mAP_v2.compute_tp for every image of a ``run`` / ``run_tta`` output, on the device rows, in one launch on the
        current stream: ``targets`` holds one (n_i, 5) array or tensor (x1, y1, x2, y2, cls; float32 or float64, one
        type per call, at most ``max_targets`` rows) per image.  Float32 ground truth matches in float32, float64 in
        float64 -- bit for bit what utils.mAP.compute_tp_batch returns for the images' rows.  Returns Matches (tp on
        the device, for MatchStats.add); its buffers are reused by the next match on the same output."""
        b, dev = out.dets.shape[0], out.dets.device
        with torch.cuda.device(dev):
            if out.matcher is None:
                out.matcher = StepMatcher(1, b, out.dets.shape[1], self.max_targets, dev)
            return out.matcher.run(out.dets.unsqueeze(0), out.det_cnt.unsqueeze(0), targets, range(b), iou_thr)

    @staticmethod
    def to_list(out, as_numpy=False, with_index=False):
        """DetectionBuffers -> the reference's output contract: list of CPU float32 (K, 6) tensors or None."""
        cnt = out.det_cnt.cpu()
        kmax = int(cnt.max().item()) if cnt.numel() else 0
        rows = out.dets[:, : max(kmax, 1)].cpu()
        idx = out.det_idx[:, : max(kmax, 1)].cpu() if with_index else None
        res, ids = [], []
        for i, c in enumerate(cnt.tolist()):
            if c < 0:
                res.append(None)
                ids.append(None)
                continue
            r = rows[i, :c].clone()
            res.append(r.numpy() if as_numpy else r)
            if with_index:
                ids.append(idx[i, :c].clone().numpy())
        if not with_index and not as_numpy:
            res = DetectionList(res)
            res.device_rows, res.device_cnt = out.dets[:, : max(kmax, 1)].clone(), out.det_cnt.clone()
        return (res, ids) if with_index else res


class PipelinedPostProcessor:
    """Several batches in flight: batch i runs filter -> NMS on CUDA stream ``i % lanes`` with its own buffers, so the
    NMS kernel of one batch overlaps the HBM-bound filter kernels of the next ones (the single-GPU form of
    dist.ShardedPostProcessor, which bench.py runs; 4 lanes hide the NMS kernel completely at 64 images per batch, batches
    below 64 images want 8).

        t = ppp.submit(heads, h, w)      # returns immediately
        dets = ppp.result(t)             # list[Tensor(K,6) | None], blocks on that batch only

    A ticket's buffers are reused ``lanes`` submissions later: fetch results before submitting that many new batches.
    With ``info`` (as for PostProcessor.run) a batch's rows come out in original-picture pixels; each lane uploads its
    own letterbox table on its stream (LetterboxStaging).

        m = ppp.match(t, targets)        # tp of the batch on the device, on its lane; MatchStats.add(m) accumulates
    """

    def __init__(self, family, hyp, anchors=None, compute_metric=False, lanes=4, max_targets=1024):
        self._pps = [PostProcessor(family, hyp, anchors, compute_metric, max_targets) for _ in range(lanes)]
        self._streams = None
        self._done = [None] * lanes   # per lane: the event recorded after its last batch
        self._next = 0
        self._layout = None   # contiguous or channels-last raw heads: fixed by the first submission

    def submit(self, heads, img_h, img_w, decoded=False, info=None):
        flat = [heads] if decoded else flatten_heads(self._pps[0].family, heads)
        if not decoded:
            kind = head_layout(self._pps[0].family, flat)
            if self._layout is None:
                self._layout = kind
            elif kind != self._layout:
                names = {_lib.INPUT_RAW_HEADS: "contiguous", _lib.INPUT_RAW_HEADS_NHWC: "channels-last"}
                raise ValueError(f"this processor was set up for {names[self._layout]} heads, got {names[kind]} ones")
        rows = None if info is None else letterbox_rows(info, flat[0].shape[0])
        dev = flat[0].device
        if self._streams is None:
            self._streams = [torch.cuda.Stream(device=dev) for _ in self._pps]
        i = self._next
        self._next = (i + 1) % len(self._pps)
        st = self._streams[i]
        st.wait_stream(torch.cuda.current_stream(dev))  # the heads were produced on the caller's stream
        with torch.cuda.stream(st):
            pp = self._pps[i]
            flat, ent = pp._run_entry(heads, img_h, img_w, decoded)
            if ent is None:   # zero images
                out = DetectionBuffers(0, int(pp.hyp["max_predictions_per_img"]), dev)
            else:
                ent["params"].d_letterbox = None
                if rows is not None:
                    if "staging" not in ent:   # allocated under the lane's stream, like the entry's other buffers
                        ent["staging"] = LetterboxStaging(flat[0].shape[0], dev)
                    # the lane's previous batch ended after any earlier copy out of this staging buffer
                    ent["params"].d_letterbox = ent["staging"].stage(rows, self._done[i])
                    ent["staging"].enqueue_copy()
                out = pp._launch(flat, ent)
            done = torch.cuda.Event()
            done.record(st)
            self._done[i] = done
        for t in flat:
            t.record_stream(st)
        return (i, done, out)

    def result(self, ticket, as_numpy=False, with_index=False):
        i, done, out = ticket
        done.synchronize()
        with torch.cuda.stream(self._streams[i]):
            return PostProcessor.to_list(out, as_numpy=as_numpy, with_index=with_index)

    def match(self, ticket, targets, iou_thr=None):
        """PostProcessor.match for a submitted batch, enqueued on its lane after its rows: ``targets`` holds one (n_i, 5)
        array per image, in ``result()`` order.  Returns Matches; no host wait."""
        i, _, out = ticket
        with torch.cuda.stream(self._streams[i]):
            return self._pps[i].match(out, targets, iou_thr)
