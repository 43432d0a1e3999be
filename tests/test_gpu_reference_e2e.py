"""End-to-end parity (iv): raw heads -> fused CUDA path  vs  the UNMODIFIED reference's own rows on the same heads.

The reference runs in a child process (baseline/ref_worker.py) from /root/reference or, on the GPU box, from the staged
byte-for-byte copy baseline/_ref/:
  mode B  hyp['device'] = 'cuda': ATen CUDA decode + host numba NMS -- the reference's deployment path and, per SURVEY.md
          8c, the end-to-end bit-exact oracle for kept indices;
  mode A  hyp['device'] = 'cpu': the path the goldens were generated with (CPU ATen sigmoid/exp differ from CUDA's by an
          ulp, so score bits may differ; every disagreement is counted and attributed to its stage, oracle/parity.py).
Without the upstream sources these tests skip.  test_fused_path_vs_oracle_* then make the same comparisons against the
oracle (oracle/, pinned to upstream by the fixtures under tests/golden), less the two checks that would compare the
oracle or the engine with itself there (_oracle_runs).
Sizes: BASELINE C1 (YOLOv5s 640^2, 25 200 candidates, dense/sparse/crowd), YOLOX-s 8 400, YOLOv7, YOLOv8, RetinaNet,
FCOS at sizes the reference's O(K*M) loop finishes in seconds, and the 1280^2 crowd case.
"""
import ast
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import close_rel

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FCOS = {"compute_metric_cls_threshold": 0.2, "compute_metric_iou_threshold": 0.35, "max_predictions_per_img": 100}

CASES = [
    dict(name="v5_c1_dense", family="yolov5", img=640, dist="dense", batch=1, seed=501),
    dict(name="v5_c1_sparse", family="yolov5", img=640, dist="sparse", batch=2, seed=502),
    dict(name="v5_c1_sparse_nopp", family="yolov5", img=640, dist="sparse", batch=2, seed=505, hyp={"postprocess_bbox": False}),
    dict(name="v5_c1_crowd", family="yolov5", img=640, dist="crowd", batch=1, seed=503),
    dict(name="v5_1280_crowd", family="yolov5", img=1280, dist="crowd", batch=1, seed=504),
    dict(name="v7_sparse", family="yolov7", img=640, dist="sparse", batch=2, seed=511),
    dict(name="v7_sparse_nopp", family="yolov7", img=640, dist="sparse", batch=1, seed=513, hyp={"postprocess_bbox": False}),
    dict(name="v7_crowd", family="yolov7", img=640, dist="crowd", batch=1, seed=512),
    dict(name="yolox_c3_dense", family="yolox", img=640, dist="dense", batch=1, seed=521),
    dict(name="yolox_sparse", family="yolox", img=640, dist="sparse", batch=2, seed=522),
    dict(name="yolox_sparse_nopp", family="yolox", img=640, dist="sparse", batch=1, seed=523, hyp={"postprocess_bbox": False}),
    dict(name="v8_dense_320", family="yolov8", img=320, dist="dense", batch=1, seed=531),
    dict(name="v8_640_thr02", family="yolov8", img=640, dist="sparse", batch=1, seed=532,
         hyp={"compute_metric_cls_threshold": 0.02}),
    dict(name="retina_dense_256", family="retinanet", img=256, dist="dense", batch=1, seed=541),
    dict(name="retina_c4_thr05", family="retinanet", img=640, dist="sparse", batch=1, seed=542,
         hyp={"compute_metric_cls_threshold": 0.05}),
    dict(name="retina_exp_dense_256", family="retinanet_exp", img=256, dist="dense", batch=1, seed=543),
    dict(name="fcos_dense", family="fcos", img=640, dist="dense", batch=2, seed=551, hyp=FCOS),
    dict(name="fcos_sparse", family="fcos", img=640, dist="sparse", batch=1, seed=552,
         hyp=dict(FCOS, compute_metric_cls_threshold=0.05)),
]


def _numpy(x):
    return x.numpy() if isinstance(x, torch.Tensor) else type(x)(_numpy(v) for v in x)


def _oracle_decode(fam, heads, img):
    import oracle
    h = _numpy(heads)
    if fam == "yolov5":
        return oracle.decode_yolov5(h)
    if fam == "yolov7":
        return oracle.decode_yolov7(h)
    if fam == "yolox":
        return oracle.decode_yolox(h, img)
    if fam == "yolov8":
        return oracle.decode_yolov8(h, img)
    if fam in ("retinanet", "retinanet_exp"):
        return oracle.decode_retinanet(h[0], h[1], img, img)
    return oracle.decode_fcos(h[0], h[1], h[2], img)


def _oracle_runs(tmp):
    """The reference side of CASES from the oracle (oracle/), pinned to upstream outputs stored
    in tests/golden -- on upstream's decoded tensors its NMS reproduces upstream's rows bit for bit, and its decode is
    within 1e-5 of upstream's CPU decode.  One npz per case and mode, in the format of baseline/ref_worker.py:
      mode A  the oracle's numpy decode (upstream's CPU path restated) -> oracle NMS;
      mode B  the engine's CUDA decode -> oracle NMS: kept rows and candidate indices are held bit-exact given the same
              CUDA decode, as upstream's CUDA-decode mode held them; the decode itself is held to 1e-5 by mode A."""
    import oracle
    from oracle import refharness
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    out = {mode: os.path.join(tmp, mode) for mode in ("A", "B")}
    for d in out.values():
        os.makedirs(d)
    for case in CASES:
        fam, img = case["family"], case["img"]
        meta = {k: v for k, v in refharness.reference_hyp((img, img), **case.get("hyp", {})).items()
                if isinstance(v, (int, float, bool, str))}
        hyp = _hyp(meta)
        heads = synth.make_heads(fam, case["batch"], img, img, 80, case["dist"], case["seed"], "cpu")
        anchors = torch.tensor(synth.V5_ANCHORS_PX) if fam in ("yolov5", "yolov7") else None
        decoded = {"A": _oracle_decode(fam, heads, img),
                   "B": PostProcessor(fam, hyp, anchors=anchors).decode(_engine_outputs(case), img, img).cpu().numpy()}
        for mode, dec in decoded.items():
            res = oracle.evaluator_nms(fam, dec, hyp)
            rows = np.zeros((len(res), max([1] + [r.rows.shape[0] for r in res if r.rows is not None]), 6), np.float32)
            counts = np.full(len(res), -1, np.int32)
            for i, r in enumerate(res):
                if r.rows is not None:
                    counts[i] = r.rows.shape[0]
                    rows[i, :counts[i]] = r.rows
            np.savez(os.path.join(out[mode], case["name"] + ".npz"), decoded=dec, rows=rows, counts=counts,
                     meta=np.array(repr(meta)))
    return out


@pytest.fixture(scope="module")
def oracle_runs(tmp_path_factory):
    return _oracle_runs(str(tmp_path_factory.mktemp("oracle")))


@pytest.fixture(scope="module")
def reference_runs(tmp_path_factory):
    """Runs the unmodified reference over CASES once per mode (two child processes side by side)."""
    sys.path.insert(0, ROOT)
    from oracle import refharness
    if not (refharness.available() or os.path.isdir(os.path.join(refharness.STAGED_ROOT, "trainer"))):
        pytest.skip("the upstream YOLOSeries sources are not present (test_fused_path_vs_oracle_* run without them)")
    tmp = str(tmp_path_factory.mktemp("reference"))
    spec = os.path.join(tmp, "spec.json")
    with open(spec, "w") as f:
        json.dump(CASES, f)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    procs = {}
    for mode, dev in (("B", "cuda"), ("A", "cpu")):
        out = os.path.join(tmp, mode)
        # mode A: hide the GPUs from the child -- the reference's GPUAnchor picks 'cuda' whenever one is visible
        # (utils/anchor.py:138), whatever hyp['device'] says
        e = dict(env, CUDA_VISIBLE_DEVICES="") if mode == "A" else env
        procs[mode] = (out, subprocess.Popen(
            [sys.executable, os.path.join(ROOT, "baseline", "ref_worker.py"), "cases", "--spec", spec, "--device", dev,
             "--out", out], cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    res = {}
    for mode, (out, p) in procs.items():
        log, _ = p.communicate(timeout=1500)
        assert p.returncode == 0, f"reference run (mode {mode}) failed:\n{log[-3000:]}"
        res[mode] = out
    return res


def _engine_outputs(case):
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    fam, img, C = case["family"], case["img"], case.get("num_class", 80)

    def to_dev(x):
        return x.cuda() if isinstance(x, torch.Tensor) else type(x)(to_dev(v) for v in x)
    heads = to_dev(synth.make_heads(fam, case["batch"], img, img, C, case["dist"], case["seed"], "cpu"))
    return heads


def _hyp(meta):
    from conftest import hyp_from_meta
    return hyp_from_meta(meta)


def _report(case, ref_dir):
    from oracle import parity
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    g = dict(np.load(os.path.join(ref_dir, case["name"] + ".npz"), allow_pickle=False))
    meta = ast.literal_eval(str(g["meta"]))
    meta.setdefault("family", case["family"])
    hyp = _hyp(meta)
    fam, img = case["family"], case["img"]
    heads = _engine_outputs(case)
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if fam in ("yolov5", "yolov7") else None
    pp = PostProcessor(fam, hyp, anchors=anchors)
    decoded = pp.decode(heads, img, img).cpu().numpy()
    keys, counts = pp.filter_only(heads, img, img)
    keys = keys.cpu().numpy().view(np.uint64)
    counts = counts.cpu().numpy()
    out = pp.run(heads, img, img)
    rows, idx = pp.to_list(out, as_numpy=True, with_index=True)
    reps = []
    for i in range(case["batch"]):
        rc = int(g["counts"][i])
        gc = -1 if rows[i] is None else rows[i].shape[0]
        reps.append(parity.image_report(
            fam, hyp, g["decoded"][i], g["rows"][i, :max(rc, 0)], rc, keys[i], int(counts[i, 0]),
            rows[i] if rows[i] is not None else np.zeros((0, 6), np.float32),
            idx[i] if idx[i] is not None else np.zeros((0,), np.int32), gc))
    return decoded, g["decoded"], reps, parity.summarize(reps)


def _decode_ok(fam, got, ref, img):
    ok = close_rel(got, ref, 1e-5)
    if fam.startswith("retinanet"):
        bad = ~ok   # round_() turns a 1-ulp exp() difference into 1 px when the value sits on x.5
        return bad.sum() <= max(2, got.shape[1] // 5000) and bool(np.all(np.abs(got[bad] - ref[bad]) <= 1.0))
    if fam == "yolov8":
        from conftest import v8_box_scale
        scale = v8_box_scale({"img": img})
        return bool(ok[..., 4:].all() and (np.abs(got[..., :4] - ref[..., :4]) <= 1e-5 * scale[None, :, None]).all())
    return bool(ok.all())


def _dump(tag, case, summary, reps):
    d = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, "parity_e2e.jsonl"), "a") as f:
            f.write(json.dumps({"mode": tag, "case": case["name"], "summary": summary,
                                "images": [r for r in reps if r["stage"] != "ok"]}) + "\n")


def _check_cuda_decode(case, ref_dir, tag, upstream):
    """Kept rows and kept candidate indices bit-exact (RetinaNet's merged boxes: 1e-5, the reference's own sgemm order is
    unspecified).  ``upstream``: the rows and the decoded tensor come from an upstream run, so the oracle's reproduction
    of those rows and the decode are checked too; otherwise the rows are the oracle's own, on the engine's decode."""
    dec, ref_dec, reps, summary = _report(case, ref_dir)
    _dump(tag, case, summary, reps)
    if upstream:
        assert summary["oracle_reproduces_reference"], summary
        assert _decode_ok(case["family"], dec, ref_dec, case["img"]), "decoded tensor beyond 1e-5 of the reference's"
    fam = case["family"]
    for r in reps:
        if fam.startswith("retinanet") or fam == "yolov8":
            # RetinaNet: merged boxes come from an sgemm whose summation order is unspecified; YOLOv8: ATen's CUDA softmax
            # reduces the 16 DFL bins in another order than the sequential sum of the CPU path this engine mirrors
            assert r.get("kept_indices_equal", r.get("rows_bit_exact")) and r.get("rows_max_rel_err", 0.0) <= 1e-5, (r, summary)
            assert r.get("score_bits_differ", 0) == 0 and r["stage"] in ("ok", "rows"), (r, summary)
        else:
            assert r["stage"] == "ok" and r["rows_bit_exact"], (r, summary)


def _check_cpu_decode(case, ref_dir, tag, upstream):
    """Decoded tensors within 1e-5; kept rows compared and every disagreement attributed.  A disagreement is accepted only
    when it is explained by differing score bits (CPU vs CUDA sigmoid/exp ulps) or by an IoU within 1e-6 of the
    threshold -- never by the NMS stage on identical inputs.  ``upstream``: see _check_cuda_decode."""
    dec, ref_dec, reps, summary = _report(case, ref_dir)
    _dump(tag, case, summary, reps)
    if upstream:
        assert summary["oracle_reproduces_reference"], summary
    assert _decode_ok(case["family"], dec, ref_dec, case["img"]), "decoded tensor beyond 1e-5 of the reference's"
    for r in reps:
        if r["stage"] == "nms":
            assert r.get("iou_within_eps_of_threshold", 0) > 0 or r.get("score_bits_differ", 0) > 0, (r, summary)
        if r["stage"] in ("ok", "rows"):
            assert r.get("rows_max_rel_err", 0.0) <= 1e-5, (r, summary)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_fused_path_vs_reference_cuda_mode_b(case, reference_runs):
    """Mode B: against the reference run with hyp['device']='cuda'."""
    _check_cuda_decode(case, reference_runs["B"], "B", upstream=True)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_fused_path_vs_reference_cpu_mode_a(case, reference_runs):
    """Mode A: against the reference run with hyp['device']='cpu' (CPU ATen decode)."""
    _check_cpu_decode(case, reference_runs["A"], "A", upstream=True)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_fused_path_vs_oracle_cuda_decode(case, oracle_runs):
    """The oracle's NMS on the engine's own CUDA decode: the select, sort, NMS and post-filter kernels at full size."""
    _check_cuda_decode(case, oracle_runs["B"], "oracle-B", upstream=False)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_fused_path_vs_oracle_cpu_decode(case, oracle_runs):
    """The oracle's numpy decode (upstream's CPU path restated) and its NMS: the engine's decode within 1e-5 of it and
    every disagreement in the kept rows attributed."""
    _check_cpu_decode(case, oracle_runs["A"], "oracle-A", upstream=False)
