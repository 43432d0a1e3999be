"""float16 / bfloat16 heads read natively: every output is bit-identical to the same call on the widened heads, h.float()."""
from collections import OrderedDict

import numpy as np
import pytest
import torch

import oracle
from conftest import close_rel, golden_heads, golden_names, hyp_from_meta, load_golden

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
FAMILIES = ["yolov5", "yolov7", "yolox", "yolov8", "retinanet", "retinanet_exp", "fcos"]


def _map(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    if isinstance(x, np.ndarray):
        return fn(torch.from_numpy(np.ascontiguousarray(x)).cuda())
    if isinstance(x, (dict, OrderedDict)):
        return type(x)((k, _map(v, fn)) for k, v in x.items())
    return type(x)(_map(v, fn) for v in x)


def _to(heads, dtype):
    return _map(heads, lambda t: t.to(dtype).contiguous())


def _widen(heads):
    return _map(heads, lambda t: t.float())


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
    """float32 array -> its bit patterns (NaN-safe bit equality)."""
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _same_lists(got, want, merged_boxes=False):
    """merged_boxes (RetinaNet): the box of a kept row is a score-weighted sum over the survivors that overlap it, added in
    the order they reach the kernel, which varies from run to run for float32 heads as well -- those four columns agree to
    1e-5 (as in the float32 parity tests), everything else bit for bit."""
    (rows_a, idx_a), (rows_b, idx_b) = got, want
    assert len(rows_a) == len(rows_b)
    for ra, rb, ia, ib in zip(rows_a, rows_b, idx_a, idx_b):
        assert (ra is None) == (rb is None)
        if ra is None:
            continue
        if merged_boxes:
            assert ra.shape == rb.shape and close_rel(ra[:, :4], rb[:, :4], 1e-5).all()
            ra, rb = ra[:, 4:], rb[:, 4:]
        np.testing.assert_array_equal(_bits(ra), _bits(rb))
        np.testing.assert_array_equal(ia, ib)


def _run_lists(pp, out):
    return pp.to_list(out, as_numpy=True, with_index=True)


def _check_run(pp, h16, img_h, img_w, **kw):
    got = _run_lists(pp, pp.run(h16, img_h, img_w, **kw))
    want = _run_lists(pp, pp.run(_widen(h16), img_h, img_w, **kw))
    _same_lists(got, want, pp.family.startswith("retinanet"))
    return got


def _check_filter(pp, h16, img_h, img_w):
    keys_a, cnt_a = pp.filter_only(h16, img_h, img_w)
    keys_b, cnt_b = pp.filter_only(_widen(h16), img_h, img_w)
    cnt_a, cnt_b = cnt_a.cpu().numpy(), cnt_b.cpu().numpy()
    np.testing.assert_array_equal(cnt_a, cnt_b)
    ka, kb = keys_a.cpu().numpy(), keys_b.cpu().numpy()
    for i in range(cnt_a.shape[0]):
        m = int(cnt_a[i, 0])
        np.testing.assert_array_equal(np.sort(ka[i, :m]), np.sort(kb[i, :m]))   # survivor key sets (arrival order is free)
    return cnt_a


def _check_decode(pp, h16, img_h, img_w):
    a = pp.decode(h16, img_h, img_w)
    assert a.dtype == torch.float32
    np.testing.assert_array_equal(_bits(a.cpu().numpy()), _bits(pp.decode(_widen(h16), img_h, img_w).cpu().numpy()))


def _check_all(family, hyp, h16, img_h, img_w):
    pp = _pp(family, hyp)
    _check_decode(pp, h16, img_h, img_w)
    cnt = _check_filter(pp, h16, img_h, img_w)
    _check_run(pp, h16, img_h, img_w)
    return cnt


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("dist", ["dense", "sparse", "crowd"])
@pytest.mark.parametrize("family", FAMILIES)
def test_every_family_and_distribution(family, dist, dtype):
    from yoloseries_b200 import synth
    if dist == "crowd" and family not in ("yolov5", "yolov7"):
        pytest.skip("crowd heads exist for the anchor-grid families")
    h16 = _to(synth.make_heads(family, 2, 256, 256, 80, dist, seed=41, device="cuda"), dtype)
    cnt = _check_all(family, _hyp(family), h16, 256, 256)
    assert cnt[:, 0].sum() > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", golden_names())
def test_golden_sizes(name, dtype):
    g = load_golden(name)
    meta = g["meta"]
    h16 = _to(golden_heads(g), dtype)
    _check_all(meta["family"], hyp_from_meta(meta), h16, meta["img"], meta["img"])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family,img,batch,dist", [("yolov5", 640, 2, "dense"), ("yolox", 640, 2, "dense"),
                                                   ("retinanet", 640, 2, "sparse"), ("yolov5", 1280, 1, "sparse")])
def test_full_baseline_sizes(family, img, batch, dist, dtype):
    """v5s 25 200, YOLOX 8 400, RetinaNet 76 725 and v5x 100 800 candidates per image."""
    from yoloseries_b200 import synth
    h16 = _to(synth.make_heads(family, batch, img, img, 80, dist, seed=7, device="cuda"), dtype)
    _check_all(family, _hyp(family), h16, img, img)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", ["yolov5", "yolov7", "yolox", "yolov8", "fcos"])
def test_multi_label(family, dtype):
    from yoloseries_b200 import synth
    h16 = _to(synth.make_heads(family, 2, 128, 128, 20, "dense", seed=5, device="cuda"), dtype)
    _check_all(family, _hyp(family, C=20, mutil_label=True), h16, 128, 128)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", ["yolov5", "yolov8", "retinanet", "fcos"])
def test_tta(family, dtype):
    from yoloseries_b200 import synth
    C = 6
    pp = _pp(family, _hyp(family, C=C))
    sizes = [(128, 160), (160, 192), (128, 128)]
    passes = [(_to(synth.make_heads(family, 2, ph, pw, C, "dense", seed=900 + k, device="cuda"), dtype), ph, pw, s, f)
              for k, ((ph, pw), s, f) in enumerate(zip(sizes, oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    wide = [(_widen(h), ph, pw, s, f) for h, ph, pw, s, f in passes]
    org = (150, 170)
    a, _ = pp.decode_tta(passes, org)
    b, _ = pp.decode_tta(wide, org)
    np.testing.assert_array_equal(_bits(a.cpu().numpy()), _bits(b.cpu().numpy()))
    _same_lists(_run_lists(pp, pp.run_tta(passes, org)), _run_lists(pp, pp.run_tta(wide, org)), family == "retinanet")


@pytest.mark.parametrize("dtype", DTYPES)
def test_fused_letterbox(dtype):
    from yoloseries_b200 import synth
    h16 = _to(synth.make_heads("yolov5", 2, 320, 320, 80, "crowd", seed=8, device="cuda"), dtype)
    info = [dict(scale=0.5, pad_top=20, pad_left=0, org_shape=(560, 640)),
            dict(scale=0.8, pad_top=0, pad_left=16, org_shape=(400, 360))]
    _check_run(_pp("yolov5", _hyp("yolov5")), h16, 320, 320, info=info)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", ["yolov5", "yolov8"])
def test_both_nms_cta_flavours(family, dtype):
    from yoloseries_b200 import _lib, synth
    lib = _lib.load()
    h16 = _to(synth.make_heads(family, 4, 320, 320, 80, "crowd" if family == "yolov5" else "dense", seed=9,
                               device="cuda"), dtype)
    pp = _pp(family, _hyp(family))
    try:
        for threads in (512, 1024):
            assert lib.ysb_set_nms_cta_threads(threads) == 0
            _check_run(pp, h16, 320, 320)
    finally:
        lib.ysb_set_nms_cta_threads(0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_graph_capture(dtype):
    from yoloseries_b200 import synth
    pp = _pp("yolov5", _hyp("yolov5"))
    h16 = _to(synth.make_heads("yolov5", 2, 256, 256, 80, "crowd", seed=10, device="cuda"), dtype)
    replay = pp.capture(h16, 256, 256)
    for seed in (11, 12):   # refill in place, replay, compare with a plain float32 run
        fresh = _to(synth.make_heads("yolov5", 2, 256, 256, 80, "crowd", seed=seed, device="cuda"), dtype)
        for t, f in zip(h16, fresh):
            t.copy_(f)
        got = _run_lists(pp, replay())
        ref = _pp("yolov5", _hyp("yolov5"))
        _same_lists(got, _run_lists(ref, ref.run(_widen(h16), 256, 256)))


@pytest.mark.parametrize("dtype", DTYPES)
def test_pipelined_and_sharded_processors(dtype):
    from yoloseries_b200 import synth
    from yoloseries_b200.dist import ShardedPostProcessor
    from yoloseries_b200.engine import PipelinedPostProcessor
    hyp = _hyp("yolov5")
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    batches = [_to(synth.make_heads("yolov5", 4, 320, 320, 80, "crowd", seed=20 + k, device="cuda"), dtype)
               for k in range(3)]
    ref = _pp("yolov5", hyp)
    want = [ref.to_list(ref.run(_widen(h), 320, 320)) for h in batches]
    ppp = PipelinedPostProcessor("yolov5", hyp, anchors=anchors, lanes=2)
    tickets = [ppp.submit(h, 320, 320) for h in batches[:2]]
    got = [ppp.result(t) for t in tickets]
    got.append(ppp.result(ppp.submit(batches[2], 320, 320)))
    spp = ShardedPostProcessor("yolov5", hyp, batch=4, img_h=320, img_w=320, anchors=anchors, lanes=2)
    try:
        got_s = [spp.result(spp.submit(h)) for h in batches]
        with pytest.raises(ValueError, match="set up for"):
            spp.submit(_widen(batches[0]))            # the first submission fixed the dtype
    finally:
        spp.close()
    for g, s, w in zip(got, got_s, want):
        assert len(g) == len(s) == len(w)
        for a, b, c in zip(g, s, w):
            assert (a is None) == (b is None) == (c is None)
            if c is not None:
                np.testing.assert_array_equal(_bits(a.numpy()), _bits(c.numpy()))
                np.testing.assert_array_equal(_bits(b.numpy()), _bits(c.numpy()))


def test_evaluator_mirror_with_a_half_precision_model():
    """A stub model that emits float16 heads: the evaluator hands them to the engine unchanged."""
    from yoloseries_b200 import synth, trainer
    heads = _to(synth.make_heads("yolov5", 2, 256, 256, 80, "crowd", seed=30, device="cuda"), torch.float16)
    hyp = oracle.default_hyp(num_class=80)
    hyp.update(device="cuda", input_img_size=[256, 256], use_tta=False, wfb=False)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    seen = []
    ev = trainer.YOLOV5Evaluator(lambda x: heads, anchors, hyp)
    ev_wide = trainer.YOLOV5Evaluator(lambda x: _widen(heads), anchors, hyp)
    orig = ev._pp.run

    def spy(h, *a, **k):
        seen.append(h)
        return orig(h, *a, **k)
    ev._pp.run = spy
    x = torch.zeros(2, 3, 256, 256, device="cuda")
    got, want = ev(x), ev_wide(x)
    assert seen and seen[0] is heads                      # no conversion pass on the way in
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert (a is None) == (b is None)
        if a is not None:
            np.testing.assert_array_equal(_bits(a.numpy()), _bits(b.numpy()))
    dec = ev.do_inference(x)
    np.testing.assert_array_equal(_bits(dec.cpu().numpy()), _bits(ev_wide.do_inference(x).cpu().numpy()))


def _specials(dtype):
    fi = torch.finfo(dtype)
    sub = fi.smallest_normal / 4                                 # a subnormal of the format
    return [0.0, -0.0, sub, -sub, fi.smallest_normal, fi.max, -fi.max, float("inf"), float("-inf")]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", ["yolov5", "yolox", "yolov7", "retinanet", "fcos"])
def test_subnormal_largest_and_infinite_values(family, dtype):
    """Each format's subnormals, largest finite values and +-inf, scattered over every channel (class and objectness
    logits, box channels: exp() of the largest values overflows to inf boxes in YOLOX / RetinaNet)."""
    from yoloseries_b200 import synth
    heads = synth.make_heads(family, 2, 128, 128, 20, "dense", seed=50, device="cuda")
    vals = torch.tensor(_specials(dtype), device="cuda")
    g = torch.Generator(device="cuda")
    g.manual_seed(51)

    def poke(t):
        flat = t.view(-1)
        pos = torch.randint(0, flat.numel(), (max(flat.numel() // 50, 1),), generator=g, device="cuda")
        flat[pos] = vals[torch.randint(0, vals.numel(), pos.shape, generator=g, device="cuda")]
        return t
    h16 = _to(_map(heads, poke), dtype)
    _check_all(family, _hyp(family, C=20), h16, 128, 128)


def test_bf16_dense_exact_score_ties():
    """bfloat16 keeps 8 significant bits: class logits drawn from a handful of values make the top two classes of most
    candidates exactly equal, so the near-tie re-evaluation runs for nearly every candidate."""
    from yoloseries_b200 import synth
    for family in ("yolov5", "yolov7", "retinanet"):
        heads = synth.make_heads(family, 2, 128, 128, 80, "dense", seed=60, device="cuda")
        levels = torch.tensor([-1.0, 0.5, 1.0, 1.0078125, 2.0], device="cuda")
        g = torch.Generator(device="cuda")
        g.manual_seed(61)

        def quantise(t):
            return levels[torch.randint(0, levels.numel(), t.shape, generator=g, device="cuda")]
        h = _to(_map(heads, quantise), torch.bfloat16)
        _check_all(family, _hyp(family), h, 128, 128)


def test_errors_are_refused_on_the_host_or_by_status():
    from yoloseries_b200 import synth
    pp = _pp("yolox", _hyp("yolox", C=4))
    h32 = synth.make_heads("yolox", 1, 64, 64, 4, "dense", seed=1, device="cuda")
    h16 = _to(h32, torch.float16)
    # the torch adapter: float16 heads against float32 params
    ent = pp._prepare(h32, 1, 64, 64, 0)
    out = ent["out"]
    with pytest.raises(ValueError, match="heads: expected"):
        pp._ops.postprocess(h16, ent["params_t"], ent["workspace"], out.dets, out.det_idx, out.det_cnt)
    # one call, two element types
    with pytest.raises(ValueError, match="one dtype"):
        pp.run([h16[0], h32[1], h16[2]], 64, 64)
    # TTA passes of different types: the C ABI returns YSB_ERR_BAD_ARG
    with pytest.raises(ValueError, match="bad argument"):
        pp.run_tta([(h16, 64, 64, 1, None), (_to(h32, torch.bfloat16), 64, 64, 0.83, 2)], (64, 64))
    # a 16-bit decoded tensor
    dec = pp.decode(h16, 64, 64)
    with pytest.raises(ValueError, match="float32"):
        pp.run(dec.half(), 64, 64, decoded=True)
    # the same processor still works afterwards
    _check_run(pp, h16, 64, 64)
