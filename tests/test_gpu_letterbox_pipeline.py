"""Rows in original-picture pixels from the pipelined processors: ShardedPostProcessor.submit / submit_tta and
PipelinedPostProcessor.submit with ``info`` against PostProcessor.run / run_tta with the same ``info``, which
tests/test_gpu_api.py pins to the oracle's letterbox undo.  Both run the same kernels on the same inputs, so rows, counts
and candidate indices are compared bit for bit."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from conftest import golden_names, hyp_from_meta, load_golden, tta_pass_heads

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAMILIES = ["yolov5", "yolov7", "yolox", "yolov8", "retinanet", "fcos"]


def _anchors(family):
    from yoloseries_b200 import synth
    return torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


def _hyp(family, **over):
    hyp = oracle.default_hyp(num_class=80)
    if family == "fcos":
        hyp.update(cls_threshold=0.2, iou_threshold=0.35, max_predictions_per_img=100)
    if family == "yolox":   # the synthetic YOLOX boxes all fail the postprocess_bbox filter: no rows to compare
        hyp.update(postprocess_bbox=False)
    hyp.update(over)
    return hyp


def _pp(family, hyp):
    from yoloseries_b200.engine import PostProcessor
    return PostProcessor(family, hyp, anchors=_anchors(family))


def _sharded(family, hyp, batch, h, w, **kw):
    from yoloseries_b200.dist import ShardedPostProcessor
    return ShardedPostProcessor(family, hyp, batch, h, w, anchors=_anchors(family), **kw)


def _heads(family, batch, img, seed, dname="dense"):
    from yoloseries_b200 import synth
    return synth.make_heads(family, batch, img, img, 80, dname, seed, "cuda")


def _nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(_nest(v, fn) for v in x)


def _to_dev(x):
    if isinstance(x, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return type(x)(_to_dev(v) for v in x)


def make_info(batch, img, seed):
    """``batch`` letterbox dicts of pictures that were scaled into an ``img`` x ``img`` network input: scales above and
    below 1, pads on either side, and original sizes small enough that the clamp to the picture takes part."""
    rnd = random.Random(seed)
    out = []
    for _ in range(batch):
        scale = rnd.choice([0.25, 0.5, 0.731, 1.0, 1.6]) * rnd.uniform(0.9, 1.1)
        top, left = rnd.choice([(0, rnd.randint(0, 60)), (rnd.randint(0, 60), 0)])
        org_h = max(8, int((img - 2 * top) / scale) - rnd.randint(0, 40))
        org_w = max(8, int((img - 2 * left) / scale) - rnd.randint(0, 40))
        out.append(dict(scale=scale, pad_top=top, pad_left=left, org_shape=(org_h, org_w)))
    return out


def _reference(pp, heads, img, info):
    out = pp.run(heads, img, img, info=info)
    torch.cuda.synchronize()
    return out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone()


def _reference_tta(pp, passes, hw, info):
    out = pp.run_tta(passes, hw, info=info)
    torch.cuda.synchronize()
    return out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone()


def _snapshot(spp, ticket):
    rows, cnt = spp.gathered(ticket)
    idx = spp._slots[ticket]["idx"]
    torch.cuda.synchronize()
    return rows[0].clone(), cnt[0].clone(), idx.clone()


def _assert_same(got, want_rows, want_cnt, want_idx):
    rows, cnt, idx = got
    assert torch.equal(cnt, want_cnt), (cnt.tolist(), want_cnt.tolist())
    for i in range(cnt.numel()):
        c = max(int(cnt[i]), 0)
        assert torch.equal(rows[i, :c].view(torch.int32), want_rows[i, :c].view(torch.int32)), f"image {i}"
        assert torch.equal(idx[i, :c], want_idx[i, :c]), f"image {i} candidate indices"


def _mapped(want, unmapped):
    """The mapped reference differs from the unmapped rows: the comparison is not vacuous."""
    rows, cnt, _ = want
    assert int(cnt.max()) > 0
    c = int(cnt.max())
    assert not torch.equal(rows[:, :c], unmapped[0][:, :c])


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("family", FAMILIES)
def test_submit_with_info_equals_run_with_info(family, graph):
    """3 lanes, 7 steps, new info every step, two sets of head tensors (A A B A A B A): steps 4, 5 and 6 meet their lane's
    head tensors again, so with graphs they replay a captured step that must read the new table contents at the address
    it captured."""
    hyp = _hyp(family)
    pp = _pp(family, hyp)
    img, b = 256, 4
    sets = [_heads(family, b, img, 300), _heads(family, b, img, 301)]
    spp = _sharded(family, hyp, b, img, img, lanes=3, graph=graph)
    for step in range(7):
        heads = sets[1] if step % 3 == 2 else sets[0]
        info = make_info(b, img, 1000 * step + len(family))
        want = _reference(pp, heads, img, info)
        _mapped(want, _reference(pp, heads, img, None))
        _assert_same(_snapshot(spp, spp.submit(heads, info=info)), *want)
    if graph:   # step 0 runs as plain launches, steps 1-3 capture, steps 4-6 replay
        assert len(spp._graphs) == 3 and all(k[1] for k in spp._graphs)
    assert spp.mode == "local"
    spp.close()


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("name", golden_names("tta_"))
def test_submit_tta_with_info_equals_run_tta_with_info(name, graph):
    g = load_golden(name)
    meta = g["meta"]
    fam, h, w, b = meta["family"], meta["img_h"], meta["img_w"], meta["batch"]
    hyp = hyp_from_meta(meta)
    passes = [(_to_dev(tta_pass_heads(g, k)), h, w, s, f) for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    pp = _pp(fam, hyp)
    unmapped = _reference_tta(pp, passes, (h, w), None)
    spp = _sharded(fam, hyp, b, h, w, lanes=2, graph=graph)
    for step in range(4):   # more submissions than lanes: lanes are reused (and, with graphs, replayed)
        info = make_info(b, max(h, w), 77 + step)
        want = _reference_tta(pp, passes, (h, w), info)
        _mapped(want, unmapped)
        _assert_same(_snapshot(spp, spp.submit_tta(passes, info=info)), *want)
    spp.close()


@pytest.mark.parametrize("variant", ["float16", "bfloat16", "channels_last", "multi_label"])
def test_other_inputs(variant):
    family = "yolov8" if variant == "channels_last" else "yolov5"
    hyp = _hyp(family, mutil_label=variant == "multi_label")
    pp = _pp(family, hyp)
    img, b = 320, 4
    spp = _sharded(family, hyp, b, img, img, lanes=2)
    for step in range(3):
        heads = _heads(family, b, img, 40 + step)
        if variant in ("float16", "bfloat16"):
            heads = _nest(heads, lambda t: t.to(getattr(torch, variant)))
        elif variant == "channels_last":
            heads = _nest(heads, lambda t: t.contiguous(memory_format=torch.channels_last))
        info = make_info(b, img, 500 + step)
        want = _reference(pp, heads, img, info)
        _mapped(want, _reference(pp, heads, img, None))
        _assert_same(_snapshot(spp, spp.submit(heads, info=info)), *want)
    spp.close()


@pytest.mark.parametrize("graph", [False, True])
def test_mapped_and_unmapped_batches_mix(graph):
    hyp = _hyp("yolov5")
    pp = _pp("yolov5", hyp)
    img, b = 320, 4
    heads = _heads("yolov5", b, img, 9, "crowd")
    info = make_info(b, img, 9)
    mapped, unmapped = _reference(pp, heads, img, info), _reference(pp, heads, img, None)
    _mapped(mapped, unmapped)
    spp = _sharded("yolov5", hyp, b, img, img, lanes=1, graph=graph)
    for _ in range(2):
        for want in (mapped, unmapped, mapped):
            _assert_same(_snapshot(spp, spp.submit(heads, info=info if want is mapped else None)), *want)
    if graph:   # one graph per (lane, letterbox on/off, heads)
        assert len(spp._graphs) == 2
    spp.close()


def test_lanes_running_ahead():
    """b = 64 at 640x640: every lane gets a batch with its own info before any of them is read."""
    from yoloseries_b200.dist import default_lanes
    hyp = _hyp("yolov5")
    pp = _pp("yolov5", hyp)
    img, b = 640, 64
    lanes = default_lanes(b, 1)
    spp = _sharded("yolov5", hyp, b, img, img)
    assert spp.lanes == lanes and not spp.graph
    subs = []
    for k in range(lanes):
        heads = _heads("yolov5", b, img, 60 + k)
        info = make_info(b, img, 600 + k)
        subs.append((spp.submit(heads, info=info), heads, info))
    for ticket, heads, info in subs:
        _assert_same(_snapshot(spp, ticket), *_reference(pp, heads, img, info))
    spp.close()


def test_pipelined_submit_with_info():
    from yoloseries_b200.engine import PipelinedPostProcessor
    hyp = _hyp("yolov5")
    pp = _pp("yolov5", hyp)
    img, b = 320, 4
    ppp = PipelinedPostProcessor("yolov5", hyp, anchors=_anchors("yolov5"), lanes=3)
    subs = []
    for step in range(6):   # two rounds over the lanes, each lane's table reused; every other batch unmapped
        heads = _heads("yolov5", b, img, 80 + step, "crowd")
        info = make_info(b, img, 800 + step) if step % 2 == 0 else None
        subs.append((ppp.submit(heads, img, img, info=info), heads, info))
        if len(subs) == 3:
            for ticket, hh, ii in subs:
                rows, idx = ppp.result(ticket, as_numpy=True, with_index=True)
                want_rows, want_idx = pp.to_list(pp.run(hh, img, img, info=ii), as_numpy=True, with_index=True)
                for r, wr, x, wx in zip(rows, want_rows, idx, want_idx):
                    assert (r is None) == (wr is None)
                    if wr is not None:
                        np.testing.assert_array_equal(r.view(np.uint32), wr.view(np.uint32))
                        np.testing.assert_array_equal(x, wx)
            subs = []


def test_wrong_info_length_raises_and_the_processor_keeps_working():
    from yoloseries_b200.engine import PipelinedPostProcessor
    hyp = _hyp("yolov5")
    pp = _pp("yolov5", hyp)
    img, b = 320, 4
    heads = _heads("yolov5", b, img, 3)
    info = make_info(b, img, 3)
    want = _reference(pp, heads, img, info)
    spp = _sharded("yolov5", hyp, b, img, img, lanes=2)
    with pytest.raises(ValueError, match="one info dict per image"):
        spp.submit(heads, info=info[:3])
    assert spp._next == 0 and spp._kind is None   # refused before anything was set up or enqueued
    _assert_same(_snapshot(spp, spp.submit(heads, info=info)), *want)
    with pytest.raises(ValueError, match="one info dict per image"):
        spp.submit(heads, info=info + info[:1])
    _assert_same(_snapshot(spp, spp.submit(heads, info=info)), *want)
    spp.close()
    passes = [(_heads("yolov5", b, img, 5 + k), img, img, s, f) for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    want_t = _reference_tta(pp, passes, (img, img), info)
    tta = _sharded("yolov5", hyp, b, img, img, lanes=2)
    with pytest.raises(ValueError, match="one info dict per image"):
        tta.submit_tta(passes, info=info[:1])
    _assert_same(_snapshot(tta, tta.submit_tta(passes, info=info)), *want_t)
    tta.close()
    ppp = PipelinedPostProcessor("yolov5", hyp, anchors=_anchors("yolov5"), lanes=2)
    with pytest.raises(ValueError, match="one info dict per image"):
        ppp.submit(heads, img, img, info=info[:2])
    got = ppp.result(ppp.submit(heads, img, img, info=info), as_numpy=True)
    for i, r in enumerate(got):
        c = int(want[1][i])
        np.testing.assert_array_equal(r, want[0][i, :c].cpu().numpy())


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_every_rank_holds_every_ranks_mapped_rows(mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    port = 29650 + os.getpid() % 300 + (7 if mode == "nccl" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mgpu_letterbox_worker.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_LETTERBOX_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
