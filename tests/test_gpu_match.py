"""Matching kept rows against ground truth on the device (ysb_match_tp / ysb_match_compact through match() and
MatchStats): the reference's goldens bit for bit in the padded layout, equality with utils.mAP.compute_tp_batch (the
existing ysb_compute_tp launch) on PostProcessor outputs, random images against the oracle, the pipelined and sharded
processors (lane reuse, graphs, TTA with letterbox info, channels-last float16 heads, partial steps), and, with two or
more GPUs, a torchrun worker over the P2P and NCCL gathers with uneven partial steps."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from conftest import golden_heads, load_golden
from oracle import evalside

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, IMG = 8, 320


def _hyp(meta, **over):
    from oracle import default_hyp
    hyp = default_hyp(num_class=meta["num_class"], conf_threshold=meta["compute_metric_conf_threshold"],
                      cls_threshold=meta["compute_metric_cls_threshold"], iou_threshold=meta["compute_metric_iou_threshold"],
                      max_predictions_per_img=meta["max_predictions_per_img"], mutil_label=meta["mutil_label"],
                      agnostic=meta["agnostic"], postprocess_bbox=meta["postprocess_bbox"])
    hyp.update(over)
    return hyp


def _anchors():
    from yoloseries_b200 import synth
    return torch.tensor(synth.V5_ANCHORS_PX)


def make_targets(rows, seed, dtype=np.float32, cap=12, full=None):
    """Ground truth for a list of (K, 6) rows (or None): per image 0..cap boxes, most of them jittered copies of kept
    rows (same class, so they match at various IoUs), some random; image ``full`` gets exactly ``cap`` boxes."""
    r = np.random.default_rng(seed)
    out = []
    for i, p in enumerate(rows):
        p = np.zeros((0, 6), np.float32) if p is None else np.asarray(p, dtype=np.float32)
        n = cap if i == full else int(r.integers(0, cap + 1))
        g = np.zeros((n, 5), dtype=np.float64)
        for k in range(n):
            if len(p) and r.random() < 0.8:
                src = p[int(r.integers(0, len(p)))]
                wh = np.maximum(src[2:4] - src[0:2], 1.0)
                g[k, :4] = src[:4] + r.normal(0, 0.08, 4) * np.concatenate([wh, wh])
                g[k, 4] = src[5]
            else:
                xy = r.uniform(0, IMG, 2)
                g[k, :4] = np.concatenate([xy, xy + r.uniform(2, 120, 2)])
                g[k, 4] = float(r.integers(0, 80))
        out.append(g.astype(dtype))
    return out


def _rows_np(rows):
    return [np.zeros((0, 6), np.float32) if p is None else np.asarray(p, dtype=np.float32) for p in rows]


def _expected(targets, rows):
    """compute_tp_batch (ysb_compute_tp, one launch) over the images' rows, and the arrays MatchStats must return."""
    from yoloseries_b200.utils.mAP import compute_tp_batch
    rows = _rows_np(rows)
    tps = compute_tp_batch(targets, rows)
    return tps, (np.concatenate(tps + [np.zeros((0, 10), bool)]),
                 np.concatenate([p[:, 4] for p in rows] + [np.zeros(0, np.float32)]),
                 np.concatenate([p[:, 5] for p in rows] + [np.zeros(0, np.float32)]),
                 np.concatenate([np.asarray(t, np.float64)[:, 4] for t in targets] + [np.zeros(0)]))


def _same_arrays(got, want):
    names = ("tp", "conf", "pred_cls", "target_cls")
    for name, a, b in zip(names, got, want):
        assert a.dtype == b.dtype and a.shape == b.shape, (name, a.dtype, b.dtype, a.shape, b.shape)
        assert np.array_equal(a.view(np.uint8) if a.dtype == bool else a, b.view(np.uint8) if b.dtype == bool else b), name


# ---- the goldens -----------------------------------------------------------------------------------------------------
def test_goldens_in_the_padded_layout():
    """utils_extra.npz tp_* (outputs of the reference's compute_tp): images of one dtype per call, two ranks whose rows
    and counts lie 256 bytes apart (a gather slot's padding); float32 rows (the goldens hold with rows rounded to float32,
    also for the float64 images)."""
    g = load_golden("utils_extra")
    thr = [float(v) for v in g["tp_thr"]]
    ops = torch.ops.ysb
    from yoloseries_b200 import _ops
    _ops.load()
    for ids in ([0, 1, 2, 4], [3, 5]):
        world, batch = 2, len(ids) // 2
        preds = [g[f"tp_pred_{i}"].astype(np.float32) for i in ids]
        gts = [g[f"tp_gt_{i}"] for i in ids]
        D = max(p.shape[0] for p in preds)
        M = max(1, max(t.shape[0] for t in gts))
        pad = 64   # floats: 256 bytes between the ranks
        rank_f = batch * D * 6 + pad
        rows_buf = torch.full((world * rank_f,), float("nan"), dtype=torch.float32)
        cnt_buf = torch.full((world * 64,), 7, dtype=torch.int32)
        gt = np.zeros((world, batch, M, 5), dtype=gts[0].dtype)
        gt_cnt = np.zeros((world, batch), np.int32)
        for k, (p, t) in enumerate(zip(preds, gts)):
            r, i = divmod(k, batch)
            o = r * rank_f + i * D * 6
            rows_buf[o:o + p.size] = torch.from_numpy(p.reshape(-1))
            cnt_buf[r * 64 + i] = p.shape[0]
            gt[r, i, :t.shape[0]] = t
            gt_cnt[r, i] = t.shape[0]
        rows = rows_buf.cuda().as_strided((world, batch, D, 6), (rank_f, D * 6, 6, 1))
        cnt = cnt_buf.cuda().as_strided((world, batch), (64, 1))
        tp = torch.full((world, batch, D, 10), 9, dtype=torch.uint8, device="cuda")
        ops.match_tp(rows, cnt, torch.from_numpy(gt).cuda(), torch.from_numpy(gt_cnt).cuda(), thr, tp)
        tp = tp.cpu().numpy()
        for k, i in enumerate(ids):
            r, j = divmod(k, batch)
            got = tp[r, j, :preds[k].shape[0]]
            assert set(np.unique(got)) <= {0, 1}
            np.testing.assert_array_equal(got.astype(bool), g[f"tp_out_{i}"], err_msg=f"image {i}")
            assert (tp[r, j, preds[k].shape[0]:] == 9).all()   # rows past the count are not written


# ---- PostProcessor outputs against compute_tp_batch ------------------------------------------------------------------
def _pp_case(name, **over):
    from yoloseries_b200.engine import PostProcessor
    g = load_golden(name)
    meta = g["meta"]
    heads = [torch.from_numpy(np.ascontiguousarray(h)).cuda() for h in golden_heads(g)]
    kw = {k: over.pop(k) for k in ("max_targets",) if k in over}
    pp = PostProcessor("yolov5", _hyp(meta, **over), anchors=_anchors(), **kw)   # the hyp holds the metric profile
    return pp, heads, meta["img"]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("name", ["yolov5_dense", "yolov5_crowd", "yolov5_sparse"])
def test_postprocessor_match_equals_compute_tp_batch(name, dtype):
    from yoloseries_b200.utils.mAP import MatchStats
    pp, heads, img = _pp_case(name)
    out = pp.run(heads, img, img)
    if name == "yolov5_sparse":   # an image the reference returns None for (no candidate left)
        out.det_cnt[-1] = -1
    rows = pp.to_list(out, as_numpy=True)
    stats = MatchStats()
    want_all = [[], [], [], []]
    for seed in range(3):   # the same buffers again: staging and tp reused
        targets = make_targets(rows, seed, dtype)
        if seed == 1:
            targets[0] = np.zeros((0, 5), dtype)   # empty ground truth
        m = pp.match(out, targets)
        tps, want = _expected(targets, rows)
        got = m.to_list()
        assert len(got) == len(rows)
        for a, b in zip(got, tps):
            np.testing.assert_array_equal(a, b)
        stats.add(m)
        for acc, w in zip(want_all, want):
            acc.append(w)
    _same_arrays(stats.arrays(), [np.concatenate(w) for w in want_all])
    if name != "yolov5_sparse":   # the sparse heads keep no rows at this profile
        assert stats.arrays()[0].any()   # some rows matched: the comparison is not vacuous


def test_max_det_1024_and_targets_at_the_capacity():
    from yoloseries_b200.utils.mAP import MatchStats
    cap = 300
    pp, heads, img = _pp_case("yolov5_crowd", max_predictions_per_img=1024, max_targets=cap)
    out = pp.run(heads, img, img)
    assert out.dets.shape[1] == 1024
    rows = pp.to_list(out, as_numpy=True)
    assert max(len(r) for r in rows if r is not None) > 0
    for dtype in (np.float32, np.float64):
        targets = make_targets(rows, 5, dtype, cap=cap, full=0)
        assert targets[0].shape[0] == cap
        m = pp.match(out, targets)
        tps, want = _expected(targets, rows)
        for a, b in zip(m.to_list(), tps):
            np.testing.assert_array_equal(a, b)
        stats = MatchStats()
        stats.add(m)
        _same_arrays(stats.arrays(), want)
        with pytest.raises(ValueError, match="max_targets"):
            pp.match(out, make_targets(rows, 5, dtype, cap=cap + 1, full=0))
    with pytest.raises(ValueError, match="one target array per image"):
        pp.match(out, targets[:-1])
    with pytest.raises(ValueError, match="one dtype"):
        pp.match(out, [t.astype(np.float64) if i == 1 else t.astype(np.float32) for i, t in enumerate(targets)])


def test_images_without_rows_and_an_empty_batch():
    """An image whose count is 0 and one the reference returns None for: no tp rows, their targets still count."""
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    from yoloseries_b200.utils.mAP import MatchStats
    pp = PostProcessor("yolov5", synth.map_profile_hyp(num_class=80), anchors=_anchors())
    heads = synth.make_heads("yolov5", 4, IMG, IMG, 80, "sparse", 3, "cuda")
    out = pp.run(heads, IMG, IMG)
    out.det_cnt[1] = 0
    out.det_cnt[2] = -1
    rows = pp.to_list(out, as_numpy=True)
    targets = make_targets(rows, 9)
    targets[1], targets[2] = make_targets([rows[0]], 1, cap=4, full=0)[0], make_targets([None], 2, cap=3, full=0)[0]
    stats = MatchStats()
    m = pp.match(out, targets)
    tps, want = _expected(targets, rows)
    assert [len(t) for t in m.to_list()][1:3] == [0, 0]
    stats.add(m)
    empty = pp.run([h[:0] for h in heads], IMG, IMG)
    stats.add(pp.match(empty, []))
    _same_arrays(stats.arrays(), want)


def test_random_images_against_the_oracle():
    """200 random images (rows and ground truth drawn around each other) through the padded layout vs
    oracle.evalside.compute_tp, in both ground-truth types (float32 rows widened for float64)."""
    from yoloseries_b200.engine import PostProcessor, DetectionBuffers
    r = np.random.default_rng(11)
    n_img, D = 200, 64
    pp = PostProcessor("yolov5", oracle.default_hyp(max_predictions_per_img=D), anchors=_anchors())
    out = DetectionBuffers(n_img, D, torch.device("cuda"))
    rows = []
    for i in range(n_img):
        k = int(r.integers(0, D + 1))
        xy = r.uniform(0, 200, (k, 2))
        box = np.concatenate([xy, xy + r.uniform(1, 60, (k, 2))], 1)
        rows.append(np.concatenate([box, r.random((k, 1)), r.integers(0, 4, (k, 1))], 1).astype(np.float32))
    host = np.zeros((n_img, D, 6), np.float32)
    for i, p in enumerate(rows):
        host[i, :len(p)] = p
    out.dets.copy_(torch.from_numpy(host))
    out.det_cnt.copy_(torch.tensor([len(p) for p in rows], dtype=torch.int32))
    for dtype in (np.float32, np.float64):
        targets = make_targets(rows, 17, dtype, cap=20)
        got = pp.match(out, targets).to_list()
        for i, (t, p) in enumerate(zip(targets, rows)):
            want = evalside.compute_tp(t, p.astype(dtype), np.linspace(0.5, 0.95, 10))
            np.testing.assert_array_equal(got[i], want, err_msg=f"image {i} {dtype.__name__}")


# ---- pipelines -------------------------------------------------------------------------------------------------------
def _heads(seed, n=B, dtype=None, channels_last=False):
    from yoloseries_b200 import synth
    h = synth.make_heads("yolov5", B, IMG, IMG, 80, "dense", seed, "cuda")
    h = [t[:n] for t in h]
    if dtype is not None:
        h = [t.to(dtype) for t in h]
    if channels_last:
        h = [t.contiguous(memory_format=torch.channels_last) for t in h]
    return h


def _info(n, seed):
    from test_gpu_partial_batches import make_info
    return make_info(n, seed)


def test_pipelined_processor():
    """More submissions than lanes; every batch's tp and the run's MatchStats equal compute_tp over result()."""
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PipelinedPostProcessor
    from yoloseries_b200.utils.mAP import MatchStats
    ppp = PipelinedPostProcessor("yolov5", synth.map_profile_hyp(num_class=80), anchors=_anchors(), lanes=2)
    stats, want_all = MatchStats(), [[], [], [], []]
    tickets = []
    for step in range(5):
        info = _info(B, step) if step % 2 else None
        t = ppp.submit(_heads(100 + step), IMG, IMG, info=info)
        rows = [None if r is None else r.numpy() for r in ppp.result(t)]
        targets = make_targets(rows, step, np.float64 if step == 3 else np.float32)
        m = ppp.match(t, targets)
        stats.add(m)
        tps, want = _expected(targets, rows)
        for a, b in zip(m.to_list(), tps):
            np.testing.assert_array_equal(a, b)
        for acc, w in zip(want_all, want):
            acc.append(w)
        tickets.append(t)
    _same_arrays(stats.arrays(), [np.concatenate(w) for w in want_all])


def _sharded_run(graph, tta=False, with_info=False, seq=(8, 8, 8, 8, 5), **heads_kw):
    """A one-rank ShardedPostProcessor over ``seq`` steps (3 lanes: more steps than lanes, a partial last step); every
    step's match and the run's MatchStats equal compute_tp over result() in order."""
    from yoloseries_b200 import synth
    from yoloseries_b200.dist import ShardedPostProcessor
    from yoloseries_b200.utils.mAP import MatchStats
    spp = ShardedPostProcessor("yolov5", synth.map_profile_hyp(num_class=80), B, IMG, IMG, anchors=_anchors(), lanes=3,
                               graph=graph)
    keep = {}   # graphs replay by head address: reuse the tensors of lane 1
    stats, want_all = MatchStats(), [[], [], [], []]
    for step, n in enumerate(seq):
        info = _info(n, step) if with_info else None
        if tta:
            x = [(_heads(10 * step + k, n, **heads_kw), IMG, IMG, s, f)
                 for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
            t = spp.submit_tta(x, info=info, partial=n < B)
        else:
            x = _heads(10 * step, n, **heads_kw)
            if n == B and step % 3 == 1:
                if "h" not in keep:
                    keep["h"] = x
                else:
                    for d, s in zip(keep["h"], x):
                        d.copy_(s)
                x = keep["h"]
            t = spp.submit(x, info=info, partial=n < B)
        rows = [None if r is None else r.numpy() for r in spp.result(t)]
        assert len(rows) == n
        targets = make_targets(rows, 50 + step, np.float64 if step == 2 else np.float32)
        m = spp.match(t, targets)
        stats.add(m)
        tps, want = _expected(targets, rows)
        got = m.to_list()
        assert len(got) == n
        for a, b in zip(got, tps):
            np.testing.assert_array_equal(a, b)
        for acc, w in zip(want_all, want):
            acc.append(w)
    _same_arrays(stats.arrays(), [np.concatenate(w) for w in want_all])
    assert stats.arrays()[0].any()
    if graph:
        assert spp._graphs
    with pytest.raises(ValueError, match="one target array per image"):
        spp.match(t, targets + targets + [targets[0]] * 20)
    spp.close()


@pytest.mark.parametrize("graph", [False, True])
def test_sharded_one_rank(graph):
    _sharded_run(graph)


def test_sharded_tta_with_info():
    _sharded_run(True, tta=True, with_info=True)


def test_sharded_channels_last_float16():
    _sharded_run(True, with_info=True, dtype=torch.float16, channels_last=True)


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_two_gpus(mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    port = 29350 + os.getpid() % 300 + (7 if mode == "nccl" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mgpu_match_worker.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_MATCH_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
