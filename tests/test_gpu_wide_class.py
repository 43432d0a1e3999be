"""1025..2048 classes (the wide sort key) and rows wider than the filter kernel's shared tile (k_filter_rows_wide) on the
GPU: oracle parity of every family, the padding invariant (C = 80 heads padded with -inf classes give the C = 80 results
bit for bit), 16-bit heads, class-aware NMS at the top class ids, multi-label, TTA, letterbox, graphs, the sharded
processor and an evaluator's seams."""
import numpy as np
import pytest
import torch

import oracle
from conftest import close_rel, v8_box_scale

pytestmark = pytest.mark.gpu

FAMILIES = ["yolov5", "yolov7", "yolox", "yolov8", "retinanet", "retinanet_exp", "fcos"]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]


def _anchors(family):
    from yoloseries_b200 import synth
    return torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


def _pp(family, hyp):
    from yoloseries_b200.engine import PostProcessor
    return PostProcessor(family, hyp, anchors=_anchors(family))


def _hyp(family, C, **over):
    hyp = oracle.default_hyp(num_class=C)
    if family == "fcos":
        hyp.update(cls_threshold=0.2, iou_threshold=0.35, max_predictions_per_img=100)
    hyp.update(over)
    return hyp


def _nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(_nest(v, fn) for v in x)


def _numpy(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else type(x)(_numpy(v) for v in x)


def _oracle_decode(family, heads, img, C):
    h = _numpy(heads)
    if family == "yolov5":
        return oracle.decode_yolov5(h, num_class=C)
    if family == "yolov7":
        return oracle.decode_yolov7(h, num_class=C)
    if family == "yolox":
        return oracle.decode_yolox(h, img, num_class=C)
    if family == "yolov8":
        return oracle.decode_yolov8(h, img, num_class=C)
    if family in ("retinanet", "retinanet_exp"):
        return oracle.decode_retinanet(h[0], h[1], img, img)
    return oracle.decode_fcos(h[0], h[1], h[2], img)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _check_oracle(family, hyp, heads, img, check_decode=True):
    """Fused raw-heads run == oracle NMS on ysb_decode's output (rows, candidate indices, None); ysb_decode == the oracle
    decode to 1e-5."""
    pp = _pp(family, hyp)
    decoded = pp.decode(heads, img, img).cpu().numpy()
    if check_decode:
        ref = _oracle_decode(family, _nest(heads, lambda t: t.float()), img, hyp["num_class"])
        assert decoded.shape == ref.shape
        if family == "yolov8":   # box sides are differences of values of magnitude s * (grid + reg): relative to those
            assert close_rel(decoded[..., 4:], ref[..., 4:], 1e-5).all()
            mag = v8_box_scale({"img": img}, hyp.get("reg", 16))[None, :, None]
            assert (np.abs(decoded[..., :4].astype(np.float64) - ref[..., :4]) <= 1e-5 * mag).all()
        else:
            assert close_rel(decoded, ref, 1e-5).all()
    want = oracle.evaluator_nms(family, decoded, hyp)
    rows, idx = pp.to_list(pp.run(heads, img, img), as_numpy=True, with_index=True)
    assert len(rows) == len(want)
    kept = 0
    for i, w in enumerate(want):
        assert (rows[i] is None) == (w.rows is None), f"image {i}"
        if w.rows is None:
            continue
        assert rows[i].shape == w.rows.shape, f"image {i}"
        if family.startswith("retinanet"):   # merged boxes: score-weighted float32 sums
            np.testing.assert_array_equal(rows[i][:, 4:], w.rows[:, 4:])
            assert close_rel(rows[i][:, :4], w.rows[:, :4], 1e-5).all()
        else:
            np.testing.assert_array_equal(_bits(rows[i]), _bits(w.rows))
        np.testing.assert_array_equal(idx[i], w.cand_index)
        kept += len(w.rows)
    return kept, decoded


def _heads(family, C, dist, img=128, batch=2, seed=7):
    from yoloseries_b200 import synth
    return synth.make_heads(family, batch, img, img, C, dist, seed=seed, device="cuda")


# ---- oracle parity --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dist", ["dense", "sparse", "crowd"])
@pytest.mark.parametrize("C", [450, 601, 1024, 1025, 1203, 2048])
@pytest.mark.parametrize("family", FAMILIES)
def test_oracle_parity(family, C, dist):
    if dist == "crowd" and family not in ("yolov5", "yolov7"):
        pytest.skip("crowd heads exist for the anchor-grid families")
    _check_oracle(family, _hyp(family, C), _heads(family, C, dist, seed=C), 128)


@pytest.mark.parametrize("family", FAMILIES)
def test_oracle_parity_640(family):
    dist = {"yolov5": "crowd", "yolov7": "crowd", "yolox": "dense", "yolov8": "dense"}.get(family, "sparse")
    hyp = _hyp(family, 1203, postprocess_bbox=dist != "dense")
    kept, _ = _check_oracle(family, hyp, _heads(family, 1203, dist, img=640, batch=1, seed=3), 640,
                            check_decode=family not in ("retinanet", "retinanet_exp"))
    assert kept > 0


def test_decoded_rows_seam():
    """PostProcessor.run(decoded=True) on wide decoded rows (the evaluators' numba_nms / do_nms input) == the oracle."""
    for family, C in (("yolov5", 601), ("yolov8", 1203), ("retinanet", 2048)):
        hyp = _hyp(family, C)
        pp = _pp(family, hyp)
        dec = pp.decode(_heads(family, C, "dense", seed=C + 1), 128, 128)
        want = oracle.evaluator_nms(family, dec.cpu().numpy(), hyp)
        rows, idx = pp.to_list(pp.run(dec, 128, 128, decoded=True), as_numpy=True, with_index=True)
        for i, w in enumerate(want):
            assert (rows[i] is None) == (w.rows is None)
            if w.rows is not None:
                np.testing.assert_array_equal(rows[i][:, 4:], w.rows[:, 4:])
                assert close_rel(rows[i][:, :4], w.rows[:, :4], 1e-5).all()
                np.testing.assert_array_equal(idx[i], w.cand_index)


# ---- padding invariant: C = 80 heads widened with classes at -inf --------------------------------------------------
def pad_classes(family, heads, C0, C):
    """The same heads with classes C0..C-1 appended at logit -inf."""
    def cat(t, dim):
        shape = list(t.shape)
        shape[dim] = C - C0
        return torch.cat([t, torch.full(shape, float("-inf"), dtype=t.dtype, device=t.device)], dim).contiguous()
    if family == "yolov5":
        return [cat(t.view(t.shape[0], 3, 5 + C0, t.shape[2], t.shape[3]), 2).view(t.shape[0], 3 * (5 + C), t.shape[2], t.shape[3])
                for t in heads]
    if family == "yolov7":
        return [cat(t, 4) for t in heads]
    if family == "yolox":
        return [cat(t, 2) for t in heads]
    if family == "yolov8":
        return [cat(t, 1) for t in heads]
    if family in ("retinanet", "retinanet_exp"):
        return heads[0], cat(heads[1], 2)
    return [cat(t, 1) for t in heads[0]], heads[1], heads[2]


def _lists(pp, out):
    return pp.to_list(out, as_numpy=True, with_index=True)


def _same(got, want):
    (ra, ia), (rb, ib) = got, want
    assert len(ra) == len(rb)
    for a, b, x, y in zip(ra, rb, ia, ib):
        assert (a is None) == (b is None)
        if a is None:
            continue
        np.testing.assert_array_equal(_bits(a), _bits(b))
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("family", FAMILIES)
def test_padding_invariant(family, dtype):
    from yoloseries_b200 import _lib
    lib = _lib.load()
    dist = "crowd" if family in ("yolov5", "yolov7") else "dense"
    base = _nest(_heads(family, 80, dist, img=256, batch=2, seed=21), lambda t: t.to(dtype))
    ref_pp = _pp(family, _hyp(family, 80, postprocess_bbox=False))
    try:
        for threads in (512, 1024):
            assert lib.ysb_set_nms_cta_threads(threads) == 0
            want = _lists(ref_pp, ref_pp.run(base, 256, 256))
            assert any(r is not None and len(r) for r in want[0])
            for C in (1203, 2048):
                pp = _pp(family, _hyp(family, C, postprocess_bbox=False))
                _same(_lists(pp, pp.run(pad_classes(family, base, 80, C), 256, 256)), want)
    finally:
        lib.ysb_set_nms_cta_threads(0)


# ---- 16-bit heads ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("family", FAMILIES)
def test_16_bit_heads_equal_float32_on_the_widened_heads(family, dtype):
    hyp = _hyp(family, 1203)
    h = _nest(_heads(family, 1203, "dense", seed=31), lambda t: t.to(dtype))
    pp = _pp(family, hyp)
    wide = _nest(h, lambda t: t.float())
    _same(_lists(pp, pp.run(h, 128, 128)), _lists(pp, pp.run(wide, 128, 128)))
    np.testing.assert_array_equal(_bits(pp.decode(h, 128, 128).cpu().numpy()), _bits(pp.decode(wide, 128, 128).cpu().numpy()))


@pytest.mark.parametrize("family", ["yolov7", "retinanet", "yolov5"])
def test_bfloat16_exact_ties_on_wide_rows(family):
    """Logits rounded to a coarse bfloat16 grid: the top class logit is tied in most rows."""
    hyp = _hyp(family, 1203)
    h = _nest(_heads(family, 1203, "dense", seed=33), lambda t: (t * 2).round().div(2).to(torch.bfloat16))
    pp = _pp(family, hyp)
    _same(_lists(pp, pp.run(h, 128, 128)), _lists(pp, pp.run(_nest(h, lambda t: t.float()), 128, 128)))
    _check_oracle(family, hyp, h, 128, check_decode=False)


# ---- class-aware NMS at the top class ids --------------------------------------------------------------------------
@pytest.mark.parametrize("span", [4095.0, 4096.0])
def test_class_aware_nms_near_class_2047(span):
    """Decoded YOLOv5 rows whose winning classes are 2040..2047 and whose boxes span `span` px in x: the class offsets
    pass 2^23, and at 4095 px the class-bucket walk is taken, at 4096 px every pair is tested."""
    C = 2048
    hyp = _hyp("yolov5", C, max_predictions_per_img=300, agnostic=True)
    rng = np.random.default_rng(5)
    n = 600
    rows = np.zeros((1, n, 5 + C), np.float32)
    w = rng.uniform(1, 60, n).astype(np.float32)
    w[0] = w[1] = 1.0
    cx = rng.uniform(w / 2, span - w / 2).astype(np.float32)   # boxes [cx - w/2, cx + w/2] inside [0, span]
    cx[0], cx[1] = 0.5, span - 0.5
    rows[0, :, 0] = cx
    rows[0, :, 1] = rng.uniform(0, 64, n)
    rows[0, :, 2] = w
    rows[0, :, 3] = rng.uniform(1, 60, n)
    rows[0, :, 4] = rng.uniform(0.05, 1, n)
    cls = rng.integers(C - 8, C, n)
    rows[0, np.arange(n), 5 + cls] = rng.uniform(0.05, 1, n)
    dec = torch.from_numpy(rows).cuda()
    pp = _pp("yolov5", hyp)
    want = oracle.evaluator_nms("yolov5", rows, hyp)
    got, idx = pp.to_list(pp.run(dec, 640, 640, decoded=True), as_numpy=True, with_index=True)
    np.testing.assert_array_equal(_bits(got[0]), _bits(want[0].rows))
    np.testing.assert_array_equal(idx[0], want[0].cand_index)
    assert set(got[0][:, 5].astype(int)) <= set(range(C - 8, C)) and len(got[0]) > 0


# ---- multi-label ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["yolov5", "yolov7", "yolox", "yolov8", "fcos"])
def test_multi_label(family):
    hyp = _hyp(family, 1203, mutil_label=True, postprocess_bbox=False)
    if family != "fcos":
        hyp.update(cls_threshold=0.8, conf_threshold=0.3)
    kept, _ = _check_oracle(family, hyp, _heads(family, 1203, "dense", seed=41), 128, check_decode=False)
    assert kept > 0


# ---- TTA, letterbox, graphs, sharded processor, evaluator ------------------------------------------------------------
def _passes(family, C, batch, img, seed, dist="dense"):
    from yoloseries_b200 import synth
    return [(synth.make_heads(family, batch, img, img, C, dist, seed + k, "cuda"), img, img, s, f)
            for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]


@pytest.mark.parametrize("family", ["yolov5", "yolov7", "retinanet"])
def test_tta_run_and_sharded_submit(family):
    from yoloseries_b200.dist import ShardedPostProcessor
    C = 1203
    hyp = _hyp(family, C)
    pp = _pp(family, hyp)
    passes = _passes(family, C, 2, 128, 50)
    out = pp.run_tta(passes, (128, 128))
    torch.cuda.synchronize()
    want_rows, want_cnt, want_idx = out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone()
    assert int(want_cnt.max()) > 0
    spp = ShardedPostProcessor(family, hyp, 2, 128, 128, anchors=_anchors(family), lanes=2)
    for _ in range(3):
        t = spp.submit_tta(passes)
        rows, cnt = spp.gathered(t)
        idx = spp._slots[t]["idx"]
        torch.cuda.synchronize()
        assert torch.equal(cnt[0], want_cnt)
        for i in range(cnt[0].numel()):
            c = max(int(cnt[0][i]), 0)
            assert torch.equal(rows[0][i, :c].view(torch.int32), want_rows[i, :c].view(torch.int32))
            assert torch.equal(idx[i, :c], want_idx[i, :c])
    spp.close()


def test_sharded_submit_graphs_and_letterbox():
    from yoloseries_b200.dist import ShardedPostProcessor
    C = 1203
    for family in ("yolov7", "yolov8"):
        hyp = _hyp(family, C)
        pp = _pp(family, hyp)
        spp = ShardedPostProcessor(family, hyp, 2, 128, 128, anchors=_anchors(family), lanes=2, graph=True)
        heads = _heads(family, C, "dense", seed=61)
        want = _lists(pp, pp.run(heads, 128, 128))
        for _ in range(3):
            t = spp.submit(heads)
            res = spp.result(t)
            assert len(res) == 2
            for r, w in zip(res, want[0]):
                assert (r is None) == (w is None)
                if w is not None:
                    np.testing.assert_array_equal(_bits(np.asarray(r.cpu() if isinstance(r, torch.Tensor) else r)), _bits(w))
        spp.close()
        # fused letterbox and graph capture of PostProcessor
        info = [dict(scale=0.5, pad_top=20, pad_left=0, org_shape=(216, 256)),
                dict(scale=0.8, pad_top=0, pad_left=16, org_shape=(160, 120))]
        fused = _lists(pp, pp.run(heads, 128, 128, info=info))
        plain = pp.run(heads, 128, 128)
        pp.undo_letterbox(plain, info)   # in place, the same arithmetic as the fused row write
        _same(fused, _lists(pp, plain))
        replay = pp.capture(heads, 128, 128)
        _same(_lists(pp, replay()), want)


def test_evaluator_end_to_end():
    from yoloseries_b200.trainer.evaluators import YOLOV7Evaluator
    C = 1203
    hyp = _hyp("yolov7", C)
    hyp.update(device="cuda", use_tta=False, input_img_size=[128, 128])
    heads = _heads("yolov7", C, "dense", seed=71)
    ev = YOLOV7Evaluator(lambda x: heads, _anchors("yolov7"), hyp)
    x = torch.zeros(2, 3, 128, 128, device="cuda")
    got = ev(x)
    dec = ev.do_inference(x)
    seam = ev.numba_nms(dec)
    want = oracle.evaluator_nms("yolov7", dec.cpu().numpy(), hyp)
    for g, s, w in zip(got, seam, want):
        assert (g is None) == (w.rows is None) == (s is None)
        if w.rows is not None:
            g = g.cpu().numpy() if isinstance(g, torch.Tensor) else np.asarray(g)
            np.testing.assert_array_equal(_bits(g), _bits(w.rows))
            np.testing.assert_array_equal(_bits(np.asarray(s)), _bits(w.rows))
