"""Drop-in mirrors of the per-image matching step of utils/mAP.py (the consumer of the kept rows, val_yolov5.py:388):

    iou(box1, box2)                     utils/mAP.py:18-42   (M,4), (N,4) ndarrays -> (M,N), the arrays' own precision
    compute_tp(gt, pred)                utils/mAP.py:70-100  (N,5), (M,6) ndarrays -> (M,10) bool
    compute_tp_batch(gts, preds)        the loop of utils/mAP.py:102-108 (compute_ap_per_class) as ONE launch
    MatchStats                          that loop's outputs accumulated on the device from the post-processors' match()

The AP integration / plotting half of mAP_v2 is bookkeeping on a few thousand numbers and stays with the caller;
dropin.install() rebinds ``mAP_v2.compute_tp`` so the reference's class keeps working unchanged.  Compute runs in
libysb_postproc.so (ysb_map_iou, ysb_compute_tp); no CPU path.
"""
import ctypes

import numpy as np
import torch

from .. import _lib, _ops
from ._common import cuda_device, stream_ptr

__all__ = ["iou", "compute_tp", "compute_tp_batch", "MatchStats", "IOU_THRESHOLDS"]

IOU_THRESHOLDS = np.linspace(0.5, 0.95, 10)   # mAP_v2.__init__, utils/mAP.py:64


def _common_dtype(*arrays):
    """numpy computes in the promoted dtype of the operands; anything that is not float32 all the way is float64."""
    dt = np.result_type(*[np.asarray(a).dtype for a in arrays])
    return np.float32 if dt == np.float32 else np.float64


def _to_dev(a, dt, dev):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)


def iou(box1, box2):
    """utils/mAP.py:18-42."""
    box1, box2 = np.asarray(box1), np.asarray(box2)
    assert box1.ndim == 2 and box2.ndim == 2 and box1.shape[1] >= 4 and box2.shape[1] >= 4
    dt = _common_dtype(box1, box2)
    dev = cuda_device()
    n, m = box1.shape[0], box2.shape[0]
    b1, b2 = _to_dev(box1[:, :4], dt, dev), _to_dev(box2[:, :4], dt, dev)
    out = torch.empty((n, m), dtype=torch.float32 if dt == np.float32 else torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().ysb_map_iou(b1.data_ptr(), n, 4, b2.data_ptr(), m, 4, int(dt == np.float64), out.data_ptr(),
                                           stream_ptr()), "ysb_map_iou")
    return out.cpu().numpy()


def compute_tp_batch(gts, preds, iou_thr=None):
    """[gt (N_i,5)], [pred (M_i,6)] -> [tp (M_i,10) bool]: every image of a validation run in one kernel launch."""
    if len(gts) != len(preds):
        raise ValueError(f"need one ground-truth array per prediction array: {len(gts)} != {len(preds)}")
    thr = np.ascontiguousarray(IOU_THRESHOLDS if iou_thr is None else iou_thr, dtype=np.float64)
    if thr.shape != (10,):
        raise ValueError("iou_thr must hold 10 thresholds (np.linspace(0.5, 0.95, 10) in the reference)")
    batch = len(gts)
    if batch == 0:
        return []
    gts = [np.asarray(g).reshape(-1, 5) for g in gts]
    preds = [np.asarray(p).reshape(-1, 6) for p in preds]
    dt = _common_dtype(*gts, *preds)
    dev = cuda_device()
    g_off = np.concatenate(([0], np.cumsum([g.shape[0] for g in gts]))).astype(np.int64)
    p_off = np.concatenate(([0], np.cumsum([p.shape[0] for p in preds]))).astype(np.int64)
    total_g, total_p = int(g_off[-1]), int(p_off[-1])
    d_gt = _to_dev(np.concatenate(gts, axis=0), dt, dev)
    d_pred = _to_dev(np.concatenate(preds, axis=0), dt, dev)
    d_goff, d_poff = torch.from_numpy(g_off).to(dev), torch.from_numpy(p_off).to(dev)
    lib = _lib.load()
    ws_bytes = ctypes.c_size_t()
    _lib.check(lib.ysb_compute_tp_workspace_bytes(total_g, ctypes.byref(ws_bytes)), "ysb_compute_tp_workspace_bytes")
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    tp = torch.empty((max(total_p, 1), 10), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ysb_compute_tp(d_gt.data_ptr(), d_goff.data_ptr(), total_g, d_pred.data_ptr(), d_poff.data_ptr(),
                                      total_p, batch, int(dt == np.float64), thr.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                      ws.data_ptr(), ws.numel(), tp.data_ptr(), stream_ptr()), "ysb_compute_tp")
    host = tp[:total_p].cpu().numpy().astype(bool)
    return [host[p_off[i]:p_off[i + 1]] for i in range(batch)]


def compute_tp(gt, pred, iou_thr=None):
    """mAP_v2.compute_tp(gt, pred), utils/mAP.py:70-100 -> (M, 10) bool."""
    return compute_tp_batch([gt], [pred], iou_thr)[0]


class MatchStats:
    """The per-image results of a validation run's matching, accumulated on the device: ``add`` appends a step's
    ``match`` result (PostProcessor, PipelinedPostProcessor or dist.ShardedPostProcessor) with one launch on the step's
    lane (ysb_match_compact), and ``arrays`` returns, at the end, what the AP integration of mAP_v2 consumes:

        tp (P, 10) bool, conf (P,) float32, pred_cls (P,) float32, target_cls (G,) float64

    equal to concatenating compute_tp(gt_i, pred_i), pred_i[:, 4], pred_i[:, 5] and gt_i[:, 4] over the images in the
    order ``result()`` lists them, step after step in ``add`` order (absent images of a partial step are skipped; an
    image whose rows are None adds its targets only).  AP sorts by confidence, so that order matters for equal scores.
    Storage grows with the rows the steps could hold (world * batch * max_det per step), without a host wait."""

    def __init__(self):
        self.device = None
        self._acc = None       # (2, 2) int64: {rows, targets} so far, ping-pong between the steps
        self._cur = 0
        self._rows_bound = self._targets = 0
        self._buf = None       # conf, pred_cls, tp (cap, 10), target_cls (cap_t)
        self._last = None      # event after the last compaction

    def _grow(self, rows, targets, dev, st):
        cap_r = self._buf[0].numel() if self._buf else 0
        cap_t = self._buf[3].numel() if self._buf else 0
        if self._buf is not None and rows <= cap_r and targets <= cap_t:
            return
        new_r, new_t = max(rows, 2 * cap_r, 4096), max(targets, 2 * cap_t, 4096)
        buf = (torch.empty(new_r, dtype=torch.float32, device=dev), torch.empty(new_r, dtype=torch.float32, device=dev),
               torch.empty((new_r, 10), dtype=torch.uint8, device=dev), torch.empty(new_t, dtype=torch.float64, device=dev))
        if self._buf is not None:
            for new, old in zip(buf, self._buf):
                new[:old.shape[0]].copy_(old)
                old.record_stream(st)
        self._buf = buf

    def add(self, matches):
        """Append one step (engine.Matches); enqueued on its lane after the previous add, no host wait."""
        st = matches.stream
        dev = matches.tp.device
        if self.device is None:
            self.device = dev
            with torch.cuda.device(dev), torch.cuda.stream(st):
                self._acc = torch.zeros((2, 2), dtype=torch.int64, device=dev)
        elif dev != self.device:
            raise ValueError(f"this MatchStats accumulates on {self.device}, got matches on {dev}")
        with torch.cuda.device(dev), torch.cuda.stream(st):
            if self._last is not None:
                st.wait_event(self._last)
            w, b, d = matches.tp.shape[:3]
            self._rows_bound += w * b * d
            self._targets += matches.n_targets
            self._grow(self._rows_bound, self._targets, dev, st)
            conf, cls, tp, tcls = self._buf
            _ops.load().match_compact(matches.rows, matches.cnt, matches.gt, matches.gt_cnt, matches.tp,
                                      self._acc[self._cur], self._acc[1 - self._cur], conf, cls, tp, tcls)
            self._cur = 1 - self._cur
            for t in (self._acc, *self._buf):   # used on several lanes: freed only after this one's work
                t.record_stream(st)
            self._last = torch.cuda.Event()
            self._last.record(st)

    def arrays(self):
        """(tp (P, 10) bool, conf (P,) float32, pred_cls (P,) float32, target_cls (G,) float64) on the host."""
        if self._last is None:
            return (np.zeros((0, 10), dtype=bool), np.zeros(0, dtype=np.float32), np.zeros(0, dtype=np.float32),
                    np.zeros(0, dtype=np.float64))
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(self._last)
            p, g = self._acc[self._cur].cpu().tolist()
            conf, cls, tp, tcls = self._buf
            return (tp[:p].cpu().numpy().astype(bool), conf[:p].cpu().numpy(), cls[:p].cpu().numpy(),
                    tcls[:g].cpu().numpy())


def _compute_tp_method(self, gt, pred):
    """Bound in place of mAP_v2.compute_tp by dropin.install(): same signature, the instance's own thresholds."""
    return compute_tp(gt, pred, getattr(self, "iou_thr", None))
