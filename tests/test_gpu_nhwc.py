"""Channels-last heads read natively (YSB_INPUT_RAW_HEADS_NHWC): every output is bit-identical to the run on the same values
in contiguous NCHW memory -- rows, det_idx, counts, decoded tensors and the filter kernel's survivor key sets."""
import os
import subprocess
import sys
from collections import OrderedDict

import numpy as np
import pytest
import torch

import oracle
from conftest import golden_heads, golden_names, hyp_from_meta, load_golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
FAMILIES = ["yolov5", "yolox", "yolov8", "fcos"]


def _map(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    if isinstance(x, np.ndarray):
        return fn(torch.from_numpy(np.ascontiguousarray(x)).cuda())
    if isinstance(x, (dict, OrderedDict)):
        return type(x)((k, _map(v, fn)) for k, v in x.items())
    return type(x)(_map(v, fn) for v in x)


def _nhwc_tensor(t, offset=0):
    """``t``'s values in channels-last memory: 4-D heads as torch.channels_last, YOLOX' 5-D (b, A, K, H, W) as the view of
    a channels-last (b, A*K, H, W) conv output.  ``offset`` elements in front of the data (misaligned tiles)."""
    five = t.dim() == 5
    x = t.reshape(t.shape[0], t.shape[1] * t.shape[2], t.shape[3], t.shape[4]) if five else t
    cl = x.contiguous(memory_format=torch.channels_last)
    if offset:
        buf = torch.empty(cl.numel() + offset, dtype=cl.dtype, device=cl.device)
        v = buf[offset:].as_strided(cl.shape, cl.stride())
        v.copy_(cl)
        cl = v
    out = cl.view(t.shape) if five else cl
    return out


def nhwc(heads, offset=0):
    return _map(heads, lambda t: _nhwc_tensor(t, offset))


def _to(heads, dtype):
    return _map(heads, lambda t: t.to(dtype).contiguous())


def _pp(family, hyp):
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None
    return PostProcessor(family, hyp, anchors=anchors)


def _hyp(family, C=80, **over):
    hyp = oracle.default_hyp(num_class=C)
    if family == "fcos":
        hyp.update(cls_threshold=0.2, iou_threshold=0.35, max_predictions_per_img=100)
    hyp.update(over)
    return hyp


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _same_lists(got, want):
    (rows_a, idx_a), (rows_b, idx_b) = got, want
    assert len(rows_a) == len(rows_b)
    for ra, rb, ia, ib in zip(rows_a, rows_b, idx_a, idx_b):
        assert (ra is None) == (rb is None)
        if ra is None:
            continue
        np.testing.assert_array_equal(_bits(ra), _bits(rb))
        np.testing.assert_array_equal(ia, ib)


def _run_lists(pp, out):
    return pp.to_list(out, as_numpy=True, with_index=True)


def _is_nhwc_run(pp, heads):
    from yoloseries_b200 import _lib, engine
    return engine.head_layout(pp.family, engine.flatten_heads(pp.family, heads)) == _lib.INPUT_RAW_HEADS_NHWC


def _check_run(pp, h, img_h, img_w, cl=None, **kw):
    cl = nhwc(h) if cl is None else cl
    assert _is_nhwc_run(pp, cl)
    got = _run_lists(pp, pp.run(cl, img_h, img_w, **kw))
    _same_lists(got, _run_lists(pp, pp.run(h, img_h, img_w, **kw)))
    return got


def _check_filter(pp, h, img_h, img_w, cl):
    keys_a, cnt_a = pp.filter_only(cl, img_h, img_w)
    keys_b, cnt_b = pp.filter_only(h, img_h, img_w)
    cnt_a, cnt_b = cnt_a.cpu().numpy(), cnt_b.cpu().numpy()
    np.testing.assert_array_equal(cnt_a, cnt_b)
    ka, kb = keys_a.cpu().numpy(), keys_b.cpu().numpy()
    for i in range(cnt_a.shape[0]):
        m = int(cnt_a[i, 0])
        np.testing.assert_array_equal(np.sort(ka[i, :m]), np.sort(kb[i, :m]))   # survivor key sets (arrival order is free)
    return cnt_a


def _check_decode(pp, h, img_h, img_w, cl):
    a = pp.decode(cl, img_h, img_w)
    np.testing.assert_array_equal(_bits(a.cpu().numpy()), _bits(pp.decode(h, img_h, img_w).cpu().numpy()))


def _check_all(family, hyp, h, img_h, img_w, offset=0):
    pp = _pp(family, hyp)
    cl = nhwc(h, offset)
    _check_decode(pp, h, img_h, img_w, cl)
    cnt = _check_filter(pp, h, img_h, img_w, cl)
    _check_run(pp, h, img_h, img_w, cl)
    return cnt


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("dist", ["dense", "sparse", "crowd"])
@pytest.mark.parametrize("family", FAMILIES)
def test_every_family_and_distribution(family, dist, dtype):
    from yoloseries_b200 import synth
    if dist == "crowd" and family != "yolov5":
        pytest.skip("crowd heads exist for the anchor-grid families")
    h = _to(synth.make_heads(family, 2, 256, 256, 80, dist, seed=41, device="cuda"), dtype)
    cnt = _check_all(family, _hyp(family), h, 256, 256)
    assert cnt[:, 0].sum() > 0


def _golden_nhwc_names():
    return [n for n in golden_names() if load_golden(n)["meta"]["family"] in FAMILIES]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", _golden_nhwc_names())
def test_golden_sizes(name, dtype):
    g = load_golden(name)
    meta = g["meta"]
    _check_all(meta["family"], hyp_from_meta(meta), _to(golden_heads(g), dtype), meta["img"], meta["img"])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family,img,batch,dist", [("yolov5", 640, 2, "dense"), ("yolox", 640, 2, "dense"),
                                                   ("yolov8", 640, 2, "dense"), ("fcos", 640, 2, "dense"),
                                                   ("yolov5", 1280, 1, "sparse")])
def test_full_baseline_sizes(family, img, batch, dist, dtype):
    """v5s 25 200, YOLOX 8 400, v8 8 400, FCOS 8 525 (with its 5x5 level) and v5x 100 800 candidates per image."""
    from yoloseries_b200 import synth
    h = _to(synth.make_heads(family, batch, img, img, 80, dist, seed=7, device="cuda"), dtype)
    _check_all(family, _hyp(family), h, img, img)


@pytest.mark.parametrize("family", FAMILIES)
def test_levels_off_the_tile_grid_and_misaligned_bases(family):
    """A*H*W not a multiple of the 128-row tile (200x200 input: 25x25, 13x13 ... levels; FCOS down to 2x2), and heads whose
    data start 1 element past an aligned address, so that no tile is 16-byte aligned (scalar staging)."""
    from yoloseries_b200 import synth
    for dtype in (torch.float32, torch.float16):
        h = _to(synth.make_heads(family, 2, 200, 200, 80, "dense", seed=43, device="cuda"), dtype)
        _check_all(family, _hyp(family), h, 200, 200)
        _check_all(family, _hyp(family), h, 200, 200, offset=1)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", FAMILIES)
def test_multi_label(family, dtype):
    from yoloseries_b200 import synth
    h = _to(synth.make_heads(family, 2, 128, 128, 20, "dense", seed=5, device="cuda"), dtype)
    _check_all(family, _hyp(family, C=20, mutil_label=True), h, 128, 128)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("family", FAMILIES)
def test_tta(family, dtype):
    from yoloseries_b200 import synth
    C = 6
    pp = _pp(family, _hyp(family, C=C))
    sizes = [(128, 160), (160, 192), (128, 128)]
    passes = [(_to(synth.make_heads(family, 2, ph, pw, C, "dense", seed=900 + k, device="cuda"), dtype), ph, pw, s, f)
              for k, ((ph, pw), s, f) in enumerate(zip(sizes, oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    cl = [(nhwc(h), ph, pw, s, f) for h, ph, pw, s, f in passes]
    org = (150, 170)
    a, _ = pp.decode_tta(cl, org)
    b, _ = pp.decode_tta(passes, org)
    np.testing.assert_array_equal(_bits(a.cpu().numpy()), _bits(b.cpu().numpy()))
    _same_lists(_run_lists(pp, pp.run_tta(cl, org)), _run_lists(pp, pp.run_tta(passes, org)))
    with pytest.raises(ValueError, match="one layout"):
        pp.run_tta([cl[0], passes[1]], org)


def test_decode_into_slots():
    from yoloseries_b200 import synth
    pp = _pp("yolov8", _hyp("yolov8"))
    h = synth.make_heads("yolov8", 2, 128, 128, 80, "dense", seed=44, device="cuda")
    cl = nhwc(h)
    from yoloseries_b200 import engine
    hf, cf = engine.flatten_heads("yolov8", h), engine.flatten_heads("yolov8", cl)
    ent_cl = pp._prepare(cf, 2, 128, 128, 0)
    ent = pp._prepare(hf, 2, 128, 128, 0)
    assert ent_cl is not ent and ent_cl["params"].input_kind == 2
    out_a = torch.full((2, 3 * ent["N"], ent["row_w"]), 7.0, device="cuda")
    out_b = out_a.clone()
    pp._ops.decode_into(cf, ent_cl["params_t"], out_a, ent["N"])
    pp._ops.decode_into(hf, ent["params_t"], out_b, ent["N"])
    np.testing.assert_array_equal(_bits(out_a.cpu().numpy()), _bits(out_b.cpu().numpy()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_fused_letterbox(dtype):
    from yoloseries_b200 import synth
    h = _to(synth.make_heads("yolov5", 2, 320, 320, 80, "crowd", seed=8, device="cuda"), dtype)
    info = [dict(scale=0.5, pad_top=20, pad_left=0, org_shape=(560, 640)),
            dict(scale=0.8, pad_top=0, pad_left=16, org_shape=(400, 360))]
    _check_run(_pp("yolov5", _hyp("yolov5")), h, 320, 320, info=info)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("family", ["yolov5", "yolov8"])
def test_both_nms_cta_flavours(family, dtype):
    from yoloseries_b200 import _lib, synth
    lib = _lib.load()
    h = _to(synth.make_heads(family, 4, 320, 320, 80, "crowd" if family == "yolov5" else "dense", seed=9,
                             device="cuda"), dtype)
    pp = _pp(family, _hyp(family))
    try:
        for threads in (512, 1024):
            assert lib.ysb_set_nms_cta_threads(threads) == 0
            _check_run(pp, h, 320, 320)
    finally:
        lib.ysb_set_nms_cta_threads(0)


def test_graph_capture():
    from yoloseries_b200 import synth
    pp = _pp("yolox", _hyp("yolox"))
    cl = nhwc(synth.make_heads("yolox", 2, 256, 256, 80, "dense", seed=10, device="cuda"))
    replay = pp.capture(cl, 256, 256)
    for seed in (11, 12):   # refill in place, replay, compare with a plain NCHW run
        fresh = synth.make_heads("yolox", 2, 256, 256, 80, "dense", seed=seed, device="cuda")
        for t, f in zip(cl, fresh):
            t.copy_(f)
        got = _run_lists(pp, replay())
        ref = _pp("yolox", _hyp("yolox"))
        _same_lists(got, _run_lists(ref, ref.run(fresh, 256, 256)))


def _same_det_lists(a_list, b_list):
    assert len(a_list) == len(b_list)
    for a, b in zip(a_list, b_list):
        assert (a is None) == (b is None)
        if a is not None:
            np.testing.assert_array_equal(_bits(a.numpy()), _bits(b.numpy()))


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_pipelined_and_sharded_processors(dtype, graph):
    from yoloseries_b200 import synth
    from yoloseries_b200.dist import ShardedPostProcessor
    from yoloseries_b200.engine import PipelinedPostProcessor
    hyp = _hyp("yolov5")
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    batches = [_to(synth.make_heads("yolov5", 4, 320, 320, 80, "crowd", seed=20 + k, device="cuda"), dtype)
               for k in range(3)]
    cls = [nhwc(h) for h in batches]
    ref = _pp("yolov5", hyp)
    want = [ref.to_list(ref.run(h, 320, 320)) for h in batches]
    ppp = PipelinedPostProcessor("yolov5", hyp, anchors=anchors, lanes=2)
    tickets = [ppp.submit(h, 320, 320) for h in cls[:2]]
    got = [ppp.result(t) for t in tickets]
    got.append(ppp.result(ppp.submit(cls[2], 320, 320)))
    with pytest.raises(ValueError, match="set up for channels-last"):
        ppp.submit(batches[0], 320, 320)
    spp = ShardedPostProcessor("yolov5", hyp, batch=4, img_h=320, img_w=320, anchors=anchors, lanes=2, graph=graph)
    try:
        # five steps over two lanes: graph capture on the second, replay when head tensors come back
        got_s = [spp.result(spp.submit(cls[k % 3])) for k in range(5)]
        with pytest.raises(ValueError, match="set up for channels-last"):
            spp.submit(batches[0])                     # the first submission fixed the layout
    finally:
        spp.close()
    for g, w in zip(got, want):
        _same_det_lists(g, w)
    for k, s in enumerate(got_s):
        _same_det_lists(s, want[k % 3])
    # and the other way round: an NCHW processor refuses channels-last heads
    spp = ShardedPostProcessor("yolov5", hyp, batch=4, img_h=320, img_w=320, anchors=anchors, lanes=2, graph=graph)
    try:
        spp.submit(batches[0])
        with pytest.raises(ValueError, match="set up for contiguous"):
            spp.submit(cls[0])
    finally:
        spp.close()


@pytest.mark.parametrize("graph", [False, True])
def test_sharded_submit_tta(graph):
    from yoloseries_b200 import synth
    from yoloseries_b200.dist import ShardedPostProcessor
    hyp = _hyp("yolov8", C=80)
    pp = _pp("yolov8", hyp)
    img = 256
    steps = []
    for step in range(4):
        passes = [(synth.make_heads("yolov8", 4, img, img, 80, "dense", seed=300 + 10 * step + k, device="cuda"), img, img,
                   s, f) for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
        steps.append(passes)
    want = [pp.to_list(pp.run_tta(p, (img, img))) for p in steps]
    spp = ShardedPostProcessor("yolov8", hyp, batch=4, img_h=img, img_w=img, lanes=2, graph=graph)
    try:
        cl_steps = [[(nhwc(h), ph, pw, s, f) for h, ph, pw, s, f in p] for p in steps]
        got = [spp.result(spp.submit_tta(p)) for p in cl_steps + cl_steps[:2]]
        with pytest.raises(ValueError, match="set up for channels-last"):
            spp.submit_tta(steps[0])
    finally:
        spp.close()
    for k, g in enumerate(got):
        _same_det_lists(g, want[k % 4])


def test_evaluator_with_a_channels_last_model():
    """A stub model that emits channels-last float16 heads: the evaluator hands them to the engine unchanged."""
    from yoloseries_b200 import synth, trainer
    base = _to(synth.make_heads("yolov5", 2, 256, 256, 80, "crowd", seed=30, device="cuda"), torch.float16)
    heads = nhwc(base)
    hyp = oracle.default_hyp(num_class=80)
    hyp.update(device="cuda", input_img_size=[256, 256], use_tta=False, wfb=False)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    seen = []
    ev = trainer.YOLOV5Evaluator(lambda x: heads, anchors, hyp)
    ev_c = trainer.YOLOV5Evaluator(lambda x: base, anchors, hyp)
    orig = ev._pp.run

    def spy(h, *a, **k):
        seen.append(h)
        return orig(h, *a, **k)
    ev._pp.run = spy
    x = torch.zeros(2, 3, 256, 256, device="cuda")
    got, want = ev(x), ev_c(x)
    assert seen and seen[0] is heads                      # no layout copy on the way in
    _same_det_lists(got, want)
    np.testing.assert_array_equal(_bits(ev.do_inference(x).cpu().numpy()), _bits(ev_c.do_inference(x).cpu().numpy()))
    # TTA through the evaluator: three channels-last forwards, one fused call
    hyp_t = dict(hyp, use_tta=True)
    _same_det_lists(trainer.YOLOV5Evaluator(lambda x: nhwc(base), anchors, hyp_t)(x),
                    trainer.YOLOV5Evaluator(lambda x: base, anchors, hyp_t)(x))


def test_rows_wider_than_the_tile():
    """YOLOX rows of 5 + 450 values: PostProcessor names the limit, the evaluator falls back to the contiguous copy."""
    from yoloseries_b200 import engine, synth, trainer
    C = 450
    h = synth.make_heads("yolox", 1, 64, 64, C, "dense", seed=31, device="cuda")
    cl = nhwc(h)
    pp = _pp("yolox", _hyp("yolox", C=C))
    with pytest.raises(ValueError, match="NHWC_MAX_ROW_WIDTH"):
        pp.run(cl, 64, 64)
    assert engine.native_heads(cl, "yolox", C)[0].is_contiguous()
    hyp = oracle.default_hyp(num_class=C)
    hyp.update(device="cuda", input_img_size=[64, 64], use_tta=False, wfb=False)
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    _same_det_lists(trainer.YOLOXEvaluator(lambda x: cl, hyp)(x), trainer.YOLOXEvaluator(lambda x: h, hyp)(x))


def test_layout_errors():
    from yoloseries_b200 import engine, synth
    pp = _pp("yolox", _hyp("yolox", C=4))
    h = engine.flatten_heads("yolox", synth.make_heads("yolox", 1, 64, 64, 4, "dense", seed=1, device="cuda"))
    cl = nhwc(h)
    # mixed levels: one channels-last, the others contiguous
    with pytest.raises(ValueError, match="contiguous float32"):
        pp.run([cl[0], h[1], h[2]], 64, 64)
    # the torch adapter checks the strides against params.input_kind, after the heads and the params blob
    ent_c = pp._prepare(h, 1, 64, 64, 0)
    ent_n = pp._prepare(cl, 1, 64, 64, 0)
    out = ent_c["out"]
    with pytest.raises(ValueError, match="heads: expected a contiguous"):
        pp._ops.postprocess(cl, ent_c["params_t"], ent_c["workspace"], out.dets, out.det_idx, out.det_cnt)
    with pytest.raises(ValueError, match="heads: expected channels-last"):
        pp._ops.postprocess([t.transpose(3, 4) for t in cl], ent_n["params_t"], ent_n["workspace"], out.dets,
                            out.det_idx, out.det_cnt)
    # the same processor still works afterwards
    _check_run(pp, h, 64, 64)


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_multi_gpu_gathers(mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    port = 29650 + os.getpid() % 300 + (7 if mode == "nccl" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mgpu_nhwc_worker.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_NHWC_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
