import ast
import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """The in-tree libysb_postproc.so normally travels with the snapshot; a fresh checkout (the .so is git-ignored)
    gets it built once per session.  Building is not a fallback: without nvcc this raises and every test fails loudly."""
    from yoloseries_b200 import _lib, _ops, build
    if not os.path.exists(_lib.LIB_PATH) and not os.environ.get("YSB_LIBRARY"):
        build.build()
    if not os.path.exists(_ops.ADAPTER_PATH):
        build.build_torch_adapter()
    yield


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def golden_names(prefix=""):
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    # tta_* fixtures hold three head sets and the merged tensor, c1_* fixtures are seed-only full-size cases (heads are
    # regenerated, see full_size_golden): both are asked for explicitly, golden_names("tta_") / golden_names("c1_")
    return [n for n in names if n.startswith(prefix) and not n.startswith("utils_")
            and (prefix or not n.startswith(("tta_", "c1_", "wfb_")))]


def full_size_golden(name):
    """c1_* fixture -> (data, heads regenerated on the CPU generator and checked against the stored checksum, the
    reference's decoded tensor rebuilt from its stored pre-mask survivors or None)."""
    import hashlib

    from yoloseries_b200 import synth
    g = load_golden(name)
    meta = g["meta"]
    heads = synth.make_heads(meta["family"], 1, meta["img"], meta["img"], meta["num_class"], meta["dist"], meta["seed"], "cpu")
    sha = hashlib.sha1()
    for h in heads:
        sha.update(np.ascontiguousarray(h.numpy()).tobytes())
    if sha.hexdigest() != str(g["heads_sha1"]):
        # torch's CPU generator / vector math did not reproduce the generation-time bits on this machine: the stored
        # outputs no longer belong to these heads.  The decoded-tensor part of the fixture stays usable.
        heads = None
    decoded = None
    if "decoded_rows" in g:
        # stored: box + objectness of every survivor and its largest class probability; the single-label path reads
        # nothing else of the class columns, so the others stay zero
        decoded = np.zeros(tuple(int(x) for x in g["decoded_shape"]), dtype=np.float32)
        idx = g["decoded_index"]
        decoded[0, idx, :5] = g["decoded_rows"]
        decoded[0, idx, 5 + g["decoded_cls_id"]] = g["decoded_cls_max"]
    return g, heads, decoded


def load_golden(name):
    data = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    if "meta" in data:
        data["meta"] = ast.literal_eval(str(data["meta"]))
    return data


def golden_heads(data):
    """Rebuild the nested head structure saved by oracle/gen_golden.py::_flat_np."""
    fam = data["meta"]["family"]
    keys = sorted(k for k in data if k.startswith("head_"))
    if fam in ("retinanet", "retinanet_exp"):
        return data["head_0"], data["head_1"]
    if fam == "fcos":
        groups = []
        for gi in range(3):
            ks = sorted((k for k in keys if k.startswith(f"head_{gi}_")), key=lambda s: int(s.split("_")[-1]))
            groups.append([data[k] for k in ks])
        return tuple(groups)
    ks = sorted(keys, key=lambda s: int(s.split("_")[-1]))
    return [data[k] for k in ks]


def tta_pass_heads(data, k):
    """Head structure of pass k of a tta_* fixture (keys p{k}_head_...)."""
    sub = {key[len(f"p{k}_"):]: v for key, v in data.items() if key.startswith(f"p{k}_head")}
    sub["meta"] = data["meta"]
    return golden_heads(sub)


def hyp_from_meta(meta):
    """Oracle-style hyp (thresholds already resolved to the compute_metric_* profile used at generation)."""
    from oracle import default_hyp
    return default_hyp(
        num_class=meta["num_class"], conf_threshold=meta["compute_metric_conf_threshold"],
        cls_threshold=meta["compute_metric_cls_threshold"], iou_threshold=meta["compute_metric_iou_threshold"],
        max_predictions_per_img=meta["max_predictions_per_img"], min_prediction_box_wh=meta["min_prediction_box_wh"],
        mutil_label=meta["mutil_label"], agnostic=meta["agnostic"], postprocess_bbox=meta["postprocess_bbox"],
        pre_nms_topk=meta["pre_nms_topk"], pre_nms_thresh=meta["pre_nms_thresh"], thresh_with_ctr=meta["thresh_with_ctr"],
    )


def close_rel(a, b, tol=1e-5):
    """north-star tolerance: |a-b| <= tol * max(|b|, 1)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) <= tol * np.maximum(np.abs(b), 1.0)


def v8_box_scale(meta, reg=16):
    """Per-candidate magnitude s * (max(gx, gy) + reg) of the operands of the v8 box subtraction."""
    img = meta["img"]
    out = []
    for s in (4, 8, 16, 32):
        h = img // s
        n = np.arange(h * h)
        g = np.maximum(n % h, n // h) + 0.5
        out.append(s * (g + reg))
    return np.concatenate(out)
