"""Image-sharded post-processing across the GPUs of one box + the one collective the path has.

Images are independent units (trainer/eval_yolov5.py:268 loops per image), so rank r simply owns images
[r*b/W, (r+1)*b/W) and no data-path collective is needed until the end, where the kept detections of every rank are
all-gathered for mAP evaluation.  The reference never gathers detections (its val sampler is not even rank-sliced,
dataset/data_sampler.py:185-192); the closest thing it has is the unused pickle-over-Gloo ``all_gather`` of
utils/dist.py:176-211.  Here the message is a fixed-stride buffer -- rows padded to max_det plus the per-image counts --
so there is no size pre-exchange, and on a B200 box it travels over NVLink/NVSwitch through NCCL.
Works with any torch.distributed backend (``gloo`` on CPU tensors is what the CPU tests use).
"""
import torch
import torch.distributed as dist


def shard_bounds(batch, rank, world):
    """[lo, hi) of the images rank ``rank`` owns; the first ``batch % world`` ranks take one extra image."""
    base, extra = divmod(batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def pack_detections(dets, cnt, per_rank):
    """(b_local, max_det, 6) f32 + (b_local,) i32 -> one flat f32 buffer sized for ``per_rank`` images."""
    b, max_det, _ = dets.shape
    buf = torch.zeros(per_rank * (max_det * 6 + 1), dtype=torch.float32, device=dets.device)
    buf[: b * max_det * 6] = dets.reshape(-1)
    cnt_f = torch.full((per_rank,), -2.0, dtype=torch.float32, device=dets.device)  # -2 marks padding images
    cnt_f[:b] = cnt.to(torch.float32)
    buf[per_rank * max_det * 6:] = cnt_f
    return buf


def gather_detections(dets, cnt, batch, group=None):
    """All-gather the kept detections of an image-sharded batch.

    ``dets`` (b_local, max_det, 6) and ``cnt`` (b_local,) are this rank's shard (in shard_bounds order); ``batch`` is the
    global image count.  Returns (dets_all (batch, max_det, 6), cnt_all (batch,)) on every rank; ``cnt == -1`` keeps
    meaning "the reference returns None for this image".
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return dets, cnt
    max_det = dets.shape[1]
    per_rank = (batch + world - 1) // world
    send = pack_detections(dets, cnt, per_rank)
    recv = torch.empty(world * send.numel(), dtype=torch.float32, device=dets.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    recv = recv.view(world, -1)
    rows = recv[:, : per_rank * max_det * 6].reshape(world, per_rank, max_det, 6)
    cnts = recv[:, per_rank * max_det * 6:].to(torch.int32)
    out_d, out_c = [], []
    for r in range(world):
        lo, hi = shard_bounds(batch, r, world)
        out_d.append(rows[r, : hi - lo])
        out_c.append(cnts[r, : hi - lo])
    return torch.cat(out_d, 0), torch.cat(out_c, 0)


# ----------------------------------------------------------------------------------------------------------------------
# The gather without a collective launch: symmetric receive buffers mapped over NVLink (CUDA IPC), written by the NMS
# kernel itself (include/ysb_postproc.h "multi-GPU", csrc/gather_kernels.cu).
# ----------------------------------------------------------------------------------------------------------------------
import ctypes
import os

from . import _lib

_LAYOUT_NAMES = {_lib.INPUT_RAW_HEADS: "contiguous", _lib.INPUT_RAW_HEADS_NHWC: "channels-last"}


def exchange_bytes(payload: bytes, group=None):
    """All-gather one small bytes object per rank (IPC handles) through torch.distributed; works on gloo and NCCL."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return [payload]
    out = [None] * world
    dist.all_gather_object(out, payload, group=group)
    return out


def bind_to_gpu_numa(local_rank):
    """Pin the calling process to the CPU cores next to GPU ``local_rank`` (NVML's ideal affinity) so that pinned host
    buffers allocated afterwards are first-touched on that GPU's NUMA node: with every rank's staging memory on node 0,
    H2D throughput stops scaling beyond two GPUs.  Best effort; returns the core count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(local_rank))
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cores = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        if cores:
            os.sched_setaffinity(0, cores)
            return len(cores)
    except Exception:
        return None
    return None


def default_lanes(batch, world):
    """Batches in flight per rank (one CUDA stream each) when the caller does not say.

    Large batches: 4 hide the NMS kernel behind the filter kernels of the next batches; with peers a lane also stays busy
    until every rank's rows have landed, which 6 lanes cover.  Batches below 64 images leave SMs idle per launch and want 8.
    Measured on B200 (YOLOv5s 640, images/s): b=64 4 / 6 lanes 738 k / 722 k on one GPU, 0.0944 / 0.0891 ms per step on
    two; b=32 603 k / 694 k (4 / 6); b=16 550 k / 618 k / 654 k (4 / 6 / 8); YOLOv5x-1280 b=16 174.5 k / 185.2 k / 187.7 k;
    b=8 476 k / 480 k / 485 k."""
    if int(batch) < 64:
        return 8
    return 4 if int(world) == 1 else 6


class _DevicePointer:
    """``__cuda_array_interface__`` holder: a zero-copy torch view of memory the C ABI allocated."""

    def __init__(self, ptr, shape, typestr, strides, owner):
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(shape), "typestr": typestr,
                                         "strides": tuple(strides), "version": 3}
        self._owner = owner


class DetectionGather:
    """Symmetric receive buffers of one rank + the mappings of every peer's buffer.

    ``mode``: 'p2p' (the NMS kernel stores rows into every peer's slot), 'local' (world == 1), decided at construction;
    a failed IPC mapping raises (callers that want the NCCL path ask for it explicitly, see ShardedPostProcessor)."""

    def __init__(self, batch, max_det, slots, device, group=None):
        self.lib = _lib.load()
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        if self.world > _lib.YSB_MAX_PEERS:
            raise ValueError(f"at most {_lib.YSB_MAX_PEERS} ranks")
        self.batch, self.max_det, self.slots, self.device = int(batch), int(max_det), int(slots), torch.device(device)
        nbytes = ctypes.c_size_t()
        _lib.check(self.lib.ysb_gather_buffer_bytes(self.world, self.slots, self.batch, self.max_det, ctypes.byref(nbytes)),
                   "ysb_gather_buffer_bytes")
        self.nbytes = nbytes.value
        own = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(_lib.YSB_IPC_HANDLE_BYTES)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ysb_gather_alloc(self.nbytes, ctypes.byref(own), handle), "ysb_gather_alloc")
        self._own = own.value
        self._opened = []
        g = _lib.YsbGather()
        g.world, g.rank, g.slots, g.batch, g.max_det = self.world, self.rank, self.slots, self.batch, self.max_det
        g.d_buf[self.rank] = self._own
        handles = exchange_bytes(handle.raw, group)
        with torch.cuda.device(self.device):
            for r, h in enumerate(handles):
                if r == self.rank:
                    continue
                p = ctypes.c_void_p()
                _lib.check(self.lib.ysb_gather_open(h, ctypes.byref(p)), f"ysb_gather_open(rank {r})")
                self._opened.append(p.value)
                g.d_buf[r] = p.value
        self.g = g
        rs, cs = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(self.lib.ysb_gather_strides(ctypes.byref(g), ctypes.byref(rs), ctypes.byref(cs)), "ysb_gather_strides")
        self._views = []
        for s in range(self.slots):
            rp, cp = ctypes.c_void_p(), ctypes.c_void_p()
            _lib.check(self.lib.ysb_gather_slot_views(ctypes.byref(g), s, ctypes.byref(rp), ctypes.byref(cp)),
                       "ysb_gather_slot_views")
            with torch.cuda.device(self.device):
                rows = torch.as_tensor(_DevicePointer(rp.value, (self.world, self.batch, self.max_det, 6), "<f4",
                                                      (rs.value, self.max_det * 24, 24, 4), self), device=self.device)
                cnt = torch.as_tensor(_DevicePointer(cp.value, (self.world, self.batch), "<i4", (cs.value, 4), self),
                                      device=self.device)
            self._views.append((rows, cnt))
        if self.world > 1:
            dist.barrier(group)   # every rank has mapped every buffer before anybody's kernels write into them

    def views(self, slot):
        """(rows (world, batch, max_det, 6) f32, counts (world, batch) i32) of this rank's receive slot."""
        return self._views[slot]

    def error(self):
        e = ctypes.c_uint32()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ysb_gather_error(ctypes.byref(self.g), ctypes.byref(e)), "ysb_gather_error")
        return e.value

    def close(self):
        """Collective: every rank stops using the buffers, then unmaps and frees."""
        if self._own is None:
            return
        with torch.cuda.device(self.device):
            torch.cuda.synchronize()
            if self.world > 1 and dist.is_initialized():
                dist.barrier(self.group)
            for p in self._opened:
                self.lib.ysb_gather_close(p)
            self._views = []
            self.lib.ysb_gather_free(self._own)
        self._own, self._opened = None, []


class ShardedPostProcessor:
    """The multi-GPU path as an API: every rank post-processes its own image shard, ``lanes`` batches in flight (default:
    4, 6 with peers, 8 for batches below 64 images), and the
    kept detections of ALL ranks end up on EVERY rank.

        spp = ShardedPostProcessor("yolov5", hyp, batch=8, img_h=640, img_w=640, anchors=anchors)
        t = spp.submit(heads)                  # filter -> NMS (+ stores into every peer's slot) -> arrival wait, async
        rows, cnt = spp.gathered(t)            # (world, batch, max_det, 6), (world, batch) device views, stream-ordered
        dets = spp.result(t)                   # list over world*batch images: CPU (K, 6) tensors / None

    Batch i runs on CUDA stream i % lanes with its own key/count buffers, so the latency-bound NMS kernel of one batch
    overlaps the HBM-bound filter kernels of the next ones.  gather = 'p2p': no collective launch at all (the NMS kernel
    writes over NVLink, flow control by two tiny kernels); 'nccl': one all_gather_into_tensor per batch on the lane's
    stream (fallback when CUDA IPC is unavailable); world == 1: plain local buffers.  With ``graph`` (default: batch <=
    16) the per-lane launch sequence is captured once per set of head tensors and replayed.
    A ticket's buffers are reused ``lanes`` submissions later.  The heads may be float32, float16 or bfloat16; the first
    submission fixes the type, and a later batch of another type raises ValueError.

    Test-time augmentation (hyp['use_tta'], trainer/eval_yolov5.py:152-179) goes through ``submit_tta`` with the passes
    of ``PostProcessor.run_tta``; ``img_h, img_w`` are then the un-augmented input size the boxes are mapped back to:

        passes = [(heads0, 640, 640, 1, None), (heads1, 640, 640, 0.83, 2), (heads2, 640, 640, 0.67, 3)]
        t = spp.submit_tta(passes)             # every pass's filter -> one merged NMS (+ peer stores) -> arrival wait
        rows, cnt = spp.gathered(t)            # as above; rows in un-augmented network-input pixels

    Contiguous (NCHW) and channels-last heads (YOLOv5, YOLOX, YOLOv8, FCOS; include/ysb_postproc.h) are both read as they
    are; like the dtype, the first submission fixes the layout and a later batch in the other one raises ValueError.

    Rows in original-picture pixels (the box half of preds_postprocess, val_yolov5.py:166-172): every rank passes the
    letterbox dicts of its own images, as for PostProcessor.run(info=...).  The NMS kernel maps the rows before it stores
    them into every rank's slot, so each rank receives mapped rows of all world*batch images without exchanging the dicts:

        t = spp.submit(heads, info=info)       # info: this rank's batch dicts (scale, pad_top, pad_left, org_shape)
        rows, cnt = spp.gathered(t)            # every rank's rows in its own original-picture pixels
        t = spp.submit_tta(passes, info=info)  # TTA undo first, then the letterbox undo, as in run_tta(info=...)

    ``info`` is decided per submission (None: network-input pixels); one dict per image, otherwise ValueError.

    Partial steps (the tail of a dataset that is not a multiple of world * batch): with ``partial=True`` a rank may
    submit any 0 <= n <= batch images, and ranks may differ within the step.  Every rank still submits once per step,
    with zero images if it has none (a rank that skips a step makes its peers time out).  The images a rank did not have
    read count -2 in ``gathered`` and are left out of ``result``.  Partial steps run as plain launches, never as graphs;
    their heads must have the per-image shapes, dtype and layout of the set-up.  The first submission must hold at least
    one image.  Without ``partial=True`` any count but ``batch`` raises ValueError: mid-run, a short batch is usually a
    sharding bug.

        lo, hi = shard_bounds(len(tail), rank, world)                  # the last, short step
        t = spp.submit([h[lo:hi] for h in heads], info=info[lo:hi], partial=True)   # hi - lo may be 0

    Lanes, graphs and the gather work as for ``submit``.

    Matching against ground truth for mAP (mAP_v2.compute_tp, val_yolov5.py:388) runs where the rows landed: ``match``
    enqueues it on the lane after the gather, and every rank matches all world*batch images of the step, so no ground
    truth or tp crosses ranks (each rank holds the dataset's labels, as YOLO datasets do):

        m = spp.match(t, targets)              # targets: one (n_i, 5) array per image, in result() order
        stats.add(m)                           # utils.mAP.MatchStats: the run's tp / conf / pred_cls / target_cls

    The first submission fixes the kind (plain or TTA): a processor
    takes only ``submit`` or only ``submit_tta`` calls.  For TTA it also fixes the number of passes, each pass's
    (img_h, img_w, scale, flip_axis) and the head shapes, and sizes the key buffers to the passes' summed key slots; a
    later submission that differs raises ValueError.
    """

    def __init__(self, family, hyp, batch, img_h, img_w, anchors=None, lanes=None, group=None, gather="auto", graph=None,
                 compute_metric=False, device=None, max_targets=1024):
        from .engine import PostProcessor, check_max_targets
        self.max_targets = check_max_targets(max_targets)
        self.family, self.batch, self.img_h, self.img_w = family, int(batch), int(img_h), int(img_w)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.lanes = max(1, int(lanes)) if lanes else default_lanes(self.batch, self.world)
        self.pp = PostProcessor(family, hyp, anchors=anchors, compute_metric=compute_metric)
        self.lib = _lib.load()
        self.max_det = int(hyp["max_predictions_per_img"])
        self.graph = (self.batch <= 16) if graph is None else bool(graph)
        want = os.environ.get("YSB_GATHER", gather)
        self.mode = "local" if self.world == 1 else ("p2p" if want in ("auto", "p2p") else "nccl")
        self.dg = None
        if self.mode == "p2p":
            ok = torch.ones(1, device=self.device)
            try:
                self.dg = DetectionGather(self.batch, self.max_det, self.lanes, self.device, group)
            except Exception as e:   # every rank must take the same path: agree on it below
                self._p2p_error = repr(e)
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if ok.item() == 0:
                if want == "p2p":
                    raise RuntimeError("P2P detection gather unavailable: " + getattr(self, "_p2p_error", "a peer failed"))
                if self.dg is not None:
                    self.dg.close()
                    self.dg = None
                self.mode = "nccl"
        self.streams = [torch.cuda.Stream(device=self.device) for _ in range(self.lanes)]
        self._ent = None
        self._kind = None      # "plain" (submit) or "tta" (submit_tta), fixed by the first submission
        self._tta = None       # TTA set-up: pass geometry, cache entries, ctypes params / heads-per-pass arrays
        self._slots = None
        self._graphs = {}
        self._warmed = False
        self._next = 0

    # ---- buffers ---------------------------------------------------------------------------------------------------
    def _prepare(self, flat):
        if self._ent is not None:
            return
        self._need_images(flat[0].shape[0])
        self._ent = self.pp._prepare(flat, self.batch, self.img_h, self.img_w, _lib.INPUT_RAW_HEADS)
        self._head_dtype = flat[0].dtype
        self._layout = self._ent["params"].input_kind
        self._set_shapes(flat)
        self._alloc_lanes(self._ent["N"] * self._slots_per_candidate())

    @staticmethod
    def _need_images(n):
        if n == 0:
            raise ValueError("the first submission must hold at least one image: it fixes the head shapes, dtype and "
                             "layout of the processor")

    def _slots_per_candidate(self):
        return int(self.pp.hyp["num_class"]) if self.pp.hyp["mutil_label"] else 1

    def _prepare_tta(self, ents, geom):
        """TTA set-up of the first submit_tta: params of every pass, key buffers sized to the summed key slots."""
        n = len(ents)
        params = (_lib.YsbParams * n)(*[e["params"] for _, e in ents])
        self._tta = dict(geom=geom, ents=[e for _, e in ents], params=params,
                         per_pass=(ctypes.c_int32 * n)(*[len(flat) for flat, _ in ents]))
        self._head_dtype = ents[0][0][0].dtype
        self._layout = ents[0][1]["params"].input_kind
        self._set_shapes([t for flat, _ in ents for t in flat])
        self._alloc_lanes(sum(e["N"] for _, e in ents) * self._slots_per_candidate())

    def _alloc_lanes(self, n):
        """Key / count / output buffers of every lane; ``n`` key slots per image."""
        from .engine import LetterboxStaging
        self._key_cap = n
        b, d, dev = self.batch, self.max_det, self.device
        self._slots = []
        cur = torch.cuda.current_stream(dev)
        for s in range(self.lanes):
            # A lane's buffers are allocated UNDER the lane's stream: the caching allocator hands out blocks whose last
            # use may still be pending on the stream they were freed on, which is only safe for work enqueued on that
            # same stream.  (Allocated on the caller's stream and written from the lane, a key buffer could share memory
            # with a temporary of a still-running producer kernel: corrupted keys -> wild candidate indices in the NMS
            # kernel.)  The lane also waits for everything the caller has enqueued so far.
            self.streams[s].wait_stream(cur)
            with torch.cuda.stream(self.streams[s]):
                sl = {"keys": torch.empty((b, n), dtype=torch.int64, device=dev),
                      "counts": torch.zeros((b, 4), dtype=torch.int32, device=dev),
                      "idx": torch.empty((b, d), dtype=torch.int32, device=dev),
                      "lb": LetterboxStaging(b, dev),
                      "done": torch.cuda.Event()}
                if self.mode == "p2p":
                    sl["rows"], sl["cnt"] = self.dg.views(s)
                elif self.mode == "nccl":
                    sl["send"] = torch.zeros(b * d * 6 + b, dtype=torch.float32, device=dev)
                    sl["send_cnt"] = sl["send"][b * d * 6:].view(torch.int32)
                    sl["recv"] = torch.empty((self.world, b * d * 6 + b), dtype=torch.float32, device=dev)
                    sl["rows"] = sl["recv"][:, : b * d * 6].view(self.world, b, d, 6)
                    sl["cnt"] = sl["recv"][:, b * d * 6:].view(torch.int32)
                else:
                    sl["rows"] = torch.zeros((1, b, d, 6), dtype=torch.float32, device=dev)
                    sl["cnt"] = torch.zeros((1, b), dtype=torch.int32, device=dev)
            self._slots.append(sl)

    def _enqueue(self, ptrs, nheads, lane, st, events=None, lb=None, n=None):
        """The launch sequence of one batch on stream ``st`` (plain C-ABI calls and a copy: capturable into a CUDA
        graph).  ``lb``: address of the lane's letterbox table, whose staged rows the sequence copies in first, or None
        for rows in network-input pixels.  ``n``: the image count of a partial step (fewer than ``batch``), else None."""
        lib, sl = self.lib, self._slots[lane]
        sp = ctypes.c_void_p(st.cuda_stream)
        # the plain and the TTA entry points take the same arguments after the heads; the params are shared by the lanes,
        # and every call copies them, so the lane's table pointer is set right before the calls.  A partial step gets its
        # own copy with batch = n: captured graphs and the other lanes read the shared ones.
        if self._kind == "tta":
            tta, sfx = self._tta, "_tta"
            params = tta["params"]
            if n is not None:
                params = (_lib.YsbParams * len(params))(*params)
                for p in params:
                    p.batch = n
            for p in params:
                p.d_letterbox = lb
            head = (params, len(params), ptrs, tta["per_pass"])
        else:
            sfx = ""
            params = self._ent["params"]
            if n is not None:
                params = _lib.YsbParams.from_buffer_copy(params)
                params.batch = n
            params.d_letterbox = lb
            head = (ctypes.byref(params), ptrs, nheads)
        filt, nms = getattr(lib, "ysb_filter_candidates" + sfx), getattr(lib, "ysb_select_nms" + sfx)
        nms_gather = getattr(lib, "ysb_select_nms" + sfx + ("_gather" if n is None else "_gather_partial"))
        if self.mode == "p2p":
            # first thing of the step: tell the peers this slot's previous contents have been consumed (they check it
            # right before storing into it, a filter + NMS pass from now)
            g = ctypes.byref(self.dg.g)
            _lib.check(lib.ysb_gather_begin(g, lane, None, 0, sp), "ysb_gather_begin")
        if lb is not None:
            with torch.cuda.stream(st):
                sl["lb"].enqueue_copy()
        if events:
            events[0].record(st)
        _lib.check(filt(*head, sl["keys"].data_ptr(), self._key_cap, sl["counts"].data_ptr(), sp),
                   "ysb_filter_candidates" + sfx)
        if events:
            events[1].record(st)
        if self.mode == "p2p":
            _lib.check(nms_gather(*head, sl["keys"].data_ptr(), self._key_cap, sl["counts"].data_ptr(), g, lane,
                                  sl["idx"].data_ptr(), sp), nms_gather.__name__)
            if events:
                events[2].record(st)
            _lib.check(lib.ysb_gather_wait(g, lane, sp), "ysb_gather_wait")
        else:
            if self.mode == "nccl":
                rows_ptr, cnt_ptr = sl["send"].data_ptr(), sl["send"].data_ptr() + self.batch * self.max_det * 24
            else:
                rows_ptr, cnt_ptr = sl["rows"].data_ptr(), sl["cnt"].data_ptr()
            _lib.check(nms(*head, sl["keys"].data_ptr(), self._key_cap, sl["counts"].data_ptr(), rows_ptr,
                           sl["idx"].data_ptr(), cnt_ptr, sp), "ysb_select_nms" + sfx)
            if n is not None:   # the images this rank did not have in a partial step
                with torch.cuda.stream(st):
                    (sl["send_cnt"] if self.mode == "nccl" else sl["cnt"][0])[n:].fill_(_lib.YSB_CNT_ABSENT)
            if events:
                events[2].record(st)

    # ---- public ----------------------------------------------------------------------------------------------------
    def submit(self, heads, events=None, sync_input=True, info=None, partial=False):
        """Enqueue one batch.  ``events``: optional 3 timing events (start, filter done, NMS done) recorded on the lane's
        stream.  ``sync_input=False`` skips the wait on the caller's current stream (heads known to be ready).  ``info``:
        this rank's letterbox dicts (scale, pad_top, pad_left, org_shape), one per image as for PostProcessor.run: its
        rows are then stored in original-picture pixels, into every rank's slot; None keeps network-input pixels.
        ``partial=True``: this rank may hold any 0 <= n <= batch images in this step (see the class docstring)."""
        from .engine import flatten_heads, head_layout, letterbox_rows
        if self._kind == "tta":
            raise ValueError("this processor was set up for test-time-augmented batches: use submit_tta")
        flat = flatten_heads(self.family, heads)
        n = flat[0].shape[0]
        if n != self.batch:
            self._check_count(n, partial)
        rows = None if info is None else letterbox_rows(info, n)
        self._prepare(flat)
        self._kind = "plain"
        if any(t.dtype != self._head_dtype for t in flat):
            raise ValueError(f"this processor was set up for {self._head_dtype} heads, got {sorted({str(t.dtype) for t in flat})}")
        if n:   # zero-image tensors count as contiguous whatever their strides: nothing of them is read
            self._check_layout(head_layout(self.family, flat))
        self._check_shapes(flat, n)
        return self._submit(flat, events, sync_input, rows, n)

    def _check_count(self, n, partial, where=""):
        if partial:
            if n > self.batch:
                raise ValueError(f"expected at most {self.batch} images per rank, got {n}{where}")
        elif n != self.batch:
            raise ValueError(f"expected {self.batch} images per rank, got {n}{where}")

    def _set_shapes(self, flat):
        """Cache the set-up's head shapes as torch.Size objects: per image, and of a full batch."""
        self._shapes = [t.shape[1:] for t in flat]
        self._full_shapes = [torch.Size((self.batch,) + tuple(s)) for s in self._shapes]

    def _check_shapes(self, flat, n):
        """Per-image head shapes against the set-up's.  submit is on the host's critical path at small batches, so a full
        batch compares one list of shapes with the cached one (the batch dimension matches by then)."""
        if n == self.batch:
            same = [t.shape for t in flat] == self._full_shapes
        else:
            same = [t.shape[1:] for t in flat] == self._shapes
        if not same:
            raise ValueError(f"the head shapes differ from those of the first submission: per image "
                             f"{[tuple(s) for s in self._shapes]}, got {[tuple(t.shape[1:]) for t in flat]}")

    def _check_layout(self, kind):
        if kind != self._layout:
            raise ValueError(f"this processor was set up for {_LAYOUT_NAMES[self._layout]} heads, got "
                             f"{_LAYOUT_NAMES[kind]} ones")

    def submit_tta(self, passes, events=None, sync_input=True, info=None, partial=False):
        """Enqueue one test-time-augmented batch: ``passes`` = [(heads, img_h, img_w, scale, flip_axis), ...] as for
        PostProcessor.run_tta, undone against the constructor's (img_h, img_w).  The passes' filter kernels append to one
        key list per image and one NMS kernel selects over all of them; rows are in un-augmented network-input pixels and
        the local det_idx counts through the passes in order.  With ``info`` (as for ``submit``) the letterbox undo
        follows the TTA undo, as in run_tta(info=...): rows in original-picture pixels.  ``events`` / ``sync_input`` /
        ``partial`` as for ``submit``; every pass holds the same images."""
        from .engine import flatten_heads, head_layout, letterbox_rows
        if self._kind == "plain":
            raise ValueError("this processor was set up for plain batches: use submit")
        passes = list(passes)
        if not 1 <= len(passes) <= _lib.YSB_MAX_PASSES:
            raise ValueError(f"1..{_lib.YSB_MAX_PASSES} passes, got {len(passes)}")
        flats = [flatten_heads(self.family, p[0]) for p in passes]
        n = flats[0][0].shape[0]
        for k, flat in enumerate(flats):
            self._check_count(flat[0].shape[0], partial, f" in pass {k}")
            if flat[0].shape[0] != n:
                raise ValueError(f"every pass must hold the same images: {n} in pass 0, {flat[0].shape[0]} in pass {k}")
        rows = None if info is None else letterbox_rows(info, n)
        geom = tuple((int(h), int(w), float(s), int(f or 0)) for _, h, w, s, f in passes)
        dtypes = {t.dtype for flat in flats for t in flat}
        if len(dtypes) != 1:
            raise ValueError(f"every pass must have heads of one dtype, got {sorted(map(str, dtypes))}")
        if self._tta is not None:
            if geom != self._tta["geom"]:
                raise ValueError(f"this processor was set up for the passes (img_h, img_w, scale, flip) "
                                 f"{list(self._tta['geom'])}, got {list(geom)}")
            if dtypes != {self._head_dtype}:
                raise ValueError(f"this processor was set up for {self._head_dtype} heads, got {sorted(map(str, dtypes))}")
        flat_all = [t for flat in flats for t in flat]
        if self._tta is not None and n != self.batch:
            # a partial step: no cache entries of its own (its params are a copy of the set-up's with batch = n)
            if n:
                self._check_layout(head_layout(self.family, flat_all))
            self._check_shapes(flat_all, n)
            return self._submit(flat_all, events, sync_input, rows, n)
        if self._tta is None:
            self._need_images(n)
        ents = self.pp._tta_entries(passes, (self.img_h, self.img_w), batch=self.batch)
        if self._tta is None:
            self._prepare_tta(ents, geom)
            self._kind = "tta"
        self._check_layout(ents[0][1]["params"].input_kind)
        if any(e is not k for (_, e), k in zip(ents, self._tta["ents"])):
            raise ValueError("the head shapes differ from those of the first submit_tta")
        return self._submit(flat_all, events, sync_input, rows, n)

    def _submit(self, flat, events, sync_input, lb_rows, n):
        """Lane choice, letterbox upload, plain launches / graph capture / replay and the NCCL all-gather of one batch
        whose heads (all passes' for TTA) are ``flat``; ``lb_rows``: letterbox_rows of its info, or None; ``n``: its
        image count (a partial step when below ``batch``: plain launches, never a graph)."""
        lane = self._next % self.lanes
        self._next += 1
        st = self.streams[lane]
        if sync_input:
            st.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.device(self.device):
            sl = self._slots[lane]
            # the lane's previous batch (its "done" event) ended after the previous copy out of the staging buffer; a
            # graph captures the table's address and the copy, so a replay copies in the rows staged here
            lb = None if not lb_rows else sl["lb"].stage(lb_rows, sl["done"])
            if n != self.batch:
                self._enqueue(_lib.head_pointer_array(flat), len(flat), lane, st, events, lb, n)
            elif self.graph and events is None and not self._warmed:
                # the very first batch runs as plain launches (lazy module load, function attributes) and counts as a
                # normal step; graphs are captured from the second submission on
                self._enqueue(_lib.head_pointer_array(flat), len(flat), lane, st, None, lb)
                torch.cuda.synchronize(self.device)
                self._warmed = True
            elif self.graph and events is None:
                key = (lane, lb is not None) + tuple(t.data_ptr() for t in flat)
                gr = self._graphs.get(key)
                if gr is None:
                    gr = self._capture(flat, lane, st, lb)
                    self._graphs[key] = gr
                with torch.cuda.stream(st):
                    gr.replay()
            else:
                self._enqueue(_lib.head_pointer_array(flat), len(flat), lane, st, events, lb)
            if self.mode == "nccl":
                with torch.cuda.stream(st):
                    dist.all_gather_into_tensor(sl["recv"].view(-1), sl["send"], group=self.group)
        sl["done"].record(st)
        if sync_input:
            for t in flat:
                t.record_stream(st)
        return lane

    def _capture(self, flat, lane, st, lb):
        ptrs = _lib.head_pointer_array(flat)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            self._enqueue(ptrs, len(flat), lane, st, None, lb)
        g._ysb_keep = (ptrs, flat, self._tta)   # pointer arrays, heads and (TTA) the params / heads-per-pass arrays
        return g

    def gathered(self, ticket):
        """Device views (rows (world, batch, max_det, 6), counts (world, batch)); the caller's current stream is made to
        wait for the batch (and, p2p, for every peer's rows).  Rank r's rows are in original-picture pixels when rank r
        submitted the batch with ``info``, otherwise in network-input pixels.  After a partial step the images a rank
        did not have read count YSB_CNT_ABSENT (-2), and their rows are unspecified."""
        sl = self._slots[ticket]
        torch.cuda.current_stream(self.device).wait_event(sl["done"])
        return sl["rows"], sl["cnt"]

    def result(self, ticket):
        """list over the images every rank had in this step, in rank order: CPU float32 (K, 6) tensors, or None (a4.3
        contract); pixels as for ``gathered``.  A full step gives world*batch entries; after a partial step the absent
        images are skipped, so with per-rank shard_bounds slices of a step's images the list is in their global order."""
        rows, cnt = self.gathered(ticket)
        cnt_h = cnt.cpu()
        kmax = max(int(cnt_h.max().item()), 1)
        rows_h = rows[:, :, :kmax].cpu()
        out = []
        for r in range(rows_h.shape[0]):
            for i in range(self.batch):
                c = int(cnt_h[r, i])
                if c != _lib.YSB_CNT_ABSENT:
                    out.append(None if c < 0 else rows_h[r, i, :c].clone())
        return out

    def match(self, ticket, targets, iou_thr=None):
        """mAP_v2.compute_tp for every image of the step, on the gathered rows, enqueued on the ticket's lane after the
        rows of every rank have landed (outside any captured graph).  ``targets``: one (n_i, 5) array or tensor per
        image (x1, y1, x2, y2, cls; float32 or float64, one type per step, at most ``max_targets`` rows), in ``result()``
        order, in the pixels of the rows.  Returns engine.Matches (tp (world, batch, max_det, 10) on the device) for
        utils.mAP.MatchStats.add; no host wait -- except after a partial step (fewer arrays than world * batch), where
        which images are absent is read back from the gathered counts once.  Raises ValueError for a wrong count of
        arrays, a wrong shape or dtype, mixed dtypes, or more than ``max_targets`` rows in an image."""
        from .engine import StepMatcher
        sl = self._slots[ticket]
        images = self.world * self.batch
        if len(targets) == images:
            positions = range(images)
        elif len(targets) > images:
            raise ValueError(f"need one target array per image of the step: {len(targets)} > {images}")
        else:
            sl["done"].synchronize()
            cnt = sl["cnt"].cpu().reshape(-1).tolist()
            positions = [k for k, c in enumerate(cnt) if c != _lib.YSB_CNT_ABSENT]
        with torch.cuda.device(self.device), torch.cuda.stream(self.streams[ticket]):
            if "matcher" not in sl:
                sl["matcher"] = StepMatcher(self.world, self.batch, self.max_det, self.max_targets, self.device)
            return sl["matcher"].run(sl["rows"], sl["cnt"], targets, positions, iou_thr)

    def drain(self):
        """The caller's current stream waits for everything submitted so far."""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def check(self):
        """Raises if a flow-control spin of the p2p gather timed out (host sync)."""
        if self.dg is not None:
            e = self.dg.error()
            if e:
                raise RuntimeError(f"detection gather timed out waiting for a peer (code {e})")

    def close(self):
        """Waits for the lanes, then releases the buffers (collective when the p2p gather is in use)."""
        with torch.cuda.device(self.device):
            torch.cuda.synchronize()
        self._graphs = {}
        if self.dg is not None:
            self.dg.close()
            self.dg = None
        self._slots, self._ent, self._tta = None, None, None
