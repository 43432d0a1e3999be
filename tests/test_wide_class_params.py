"""Host side of 1025..2048-class calls: the header constants, the C ABI's limits (classes, the wide key's candidate limit,
TTA bases), rows inputs wider than the filter tile, the multi-label workspace, the wide key unpacking and the Python
refusal above 2048 classes -- no GPU."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import oracle
from oracle import parity
from yoloseries_b200 import _lib, engine, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAMILIES = ["yolov5", "yolov7", "yolox", "yolov8", "retinanet", "retinanet_exp", "fcos"]
HEADS = (ctypes.c_void_p * 15)(*[0x100000 * (k + 1) for k in range(15)])


@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


def test_limits_match_the_header():
    src = ('#include <stdio.h>\n#include "ysb_postproc.h"\nint main(){printf("%d %d %d %d", YSB_MAX_CLASSES, '
           'YSB_MAX_CANDIDATES, YSB_MAX_CANDIDATES_WIDE, YSB_ABI_VERSION);return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        classes, cand, cand_wide, abi = map(int, subprocess.check_output([exe]).split())
    assert (classes, cand, cand_wide) == (_lib.YSB_MAX_CLASSES, _lib.YSB_MAX_CANDIDATES, _lib.YSB_MAX_CANDIDATES_WIDE)
    assert (classes, cand, cand_wide) == (2048, (1 << 22) - 1, (1 << 21) - 1)
    assert abi == _lib.ABI_VERSION == 6


def params(family, C, img=128, kind=_lib.INPUT_RAW_HEADS, batch=2, tta=None, **over):
    hyp = oracle.default_hyp(num_class=C)
    hyp.update(over)
    shapes = None if family.startswith("retinanet") else synth.level_shapes(family, img, img)
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None
    return engine.make_params(family, hyp, batch, img, img, shapes, anchors, input_kind=kind, tta=tta)


def num_candidates(lib, p):
    n, rw = ctypes.c_int64(), ctypes.c_int32()
    st = lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw))
    return st, n.value, rw.value


def workspace(lib, p):
    ws = ctypes.c_size_t()
    return lib.ysb_postprocess_workspace_bytes(ctypes.byref(p), ctypes.byref(ws)), ws.value


def _align256(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("C", [1025, 1203, 2048])
def test_wide_class_counts_are_accepted(lib, family, C):
    st, n, rw = num_candidates(lib, params(family, C))
    assert st == 0 and n > 0
    assert rw == {"yolov8": 4 + C, "retinanet": C + 4, "retinanet_exp": C + 5}.get(family, 5 + C)
    st, ws = workspace(lib, params(family, C))
    assert st == 0 and ws == _align256(8 * n * 2) + _align256(16 * 2) + 256
    dec = params(family, C, kind=_lib.INPUT_DECODED_ROWS)
    assert num_candidates(lib, dec) == (0, n, rw)
    assert workspace(lib, dec) == (0, ws)


@pytest.mark.parametrize("family", FAMILIES)
def test_more_than_2048_classes_is_a_limit(lib, family):
    for kind in (_lib.INPUT_RAW_HEADS, _lib.INPUT_DECODED_ROWS):
        p = params(family, 2049, kind=kind)
        assert num_candidates(lib, p)[0] == _lib.YSB_ERR_LIMIT
        assert workspace(lib, p)[0] == _lib.YSB_ERR_LIMIT
        assert lib.ysb_filter_candidates(ctypes.byref(p), HEADS, 15, 0x1000, 1 << 40, 0x2000, None) == _lib.YSB_ERR_LIMIT
        assert lib.ysb_postprocess(ctypes.byref(p), HEADS, 15, 0x1000, 1 << 40, 0x2000, 0x3000, 0x4000, None) == \
            _lib.YSB_ERR_LIMIT
    with pytest.raises(ValueError, match="beyond the engine limits"):
        _lib.check(_lib.YSB_ERR_LIMIT, "ysb_num_candidates")


def test_wide_key_candidate_limit(lib):
    # YOLOv5 at 6144^2: 3 * (768^2 + 384^2 + 192^2) = 2 322 432 candidates, between the two limits
    p = params("yolov5", 1024, img=6144)
    st, n, _ = num_candidates(lib, p)
    assert st == 0 and n == 2322432 and _lib.YSB_MAX_CANDIDATES_WIDE < n <= _lib.YSB_MAX_CANDIDATES
    assert workspace(lib, p)[0] == 0
    wide = params("yolov5", 1025, img=6144)
    assert num_candidates(lib, wide)[0] == _lib.YSB_ERR_LIMIT
    assert workspace(lib, wide)[0] == _lib.YSB_ERR_LIMIT
    assert lib.ysb_decode(ctypes.byref(wide), HEADS, 3, 0x1000, None) == _lib.YSB_ERR_LIMIT
    assert lib.ysb_filter_candidates(ctypes.byref(wide), HEADS, 3, 0x1000, 1 << 40, 0x2000, None) == _lib.YSB_ERR_LIMIT
    # decoded rows: the row count given in the params counts against the same limit
    dec = params("yolov5", 1203, kind=_lib.INPUT_DECODED_ROWS)
    dec.decoded_rows = _lib.YSB_MAX_CANDIDATES_WIDE
    assert num_candidates(lib, dec)[:2] == (0, _lib.YSB_MAX_CANDIDATES_WIDE)
    dec.decoded_rows = _lib.YSB_MAX_CANDIDATES_WIDE + 1
    assert num_candidates(lib, dec)[0] == _lib.YSB_ERR_LIMIT
    dec.num_classes = 1024
    assert num_candidates(lib, dec)[0] == 0


def test_wide_key_limit_on_summed_tta_bases(lib):
    # YOLOv5 at 4096^2: 1 032 192 candidates per pass; three passes (3 096 576) fit 22 candidate bits, not 21
    def passes(C, n):
        return (_lib.YsbParams * n)(*[params("yolov5", C, img=4096, batch=1, tta=(1.0, None, 4096, 4096))
                                      for _ in range(n)])
    ws = ctypes.c_size_t()
    assert num_candidates(lib, params("yolov5", 1203, img=4096))[1] == 1032192
    assert lib.ysb_postprocess_tta_workspace_bytes(passes(1024, 3), 3, ctypes.byref(ws)) == 0
    assert lib.ysb_postprocess_tta_workspace_bytes(passes(1203, 2), 2, ctypes.byref(ws)) == 0
    assert ws.value == _align256(8 * 2 * 1032192) + _align256(16) + 256
    for C in (1025, 2048):
        assert lib.ysb_postprocess_tta_workspace_bytes(passes(C, 3), 3, ctypes.byref(ws)) == _lib.YSB_ERR_LIMIT
        per = (ctypes.c_int32 * 3)(3, 3, 3)
        assert lib.ysb_filter_candidates_tta(passes(C, 3), 3, HEADS, per, 0x1000, 1 << 40, 0x2000, None) == \
            _lib.YSB_ERR_LIMIT
    # RetinaNet at 1280^2 (306 900 candidates): four passes fit the wide key
    r = (_lib.YsbParams * 4)(*[params("retinanet", 1203, img=1280, batch=1, tta=(1.0, None, 1280, 1280))
                               for _ in range(4)])
    assert num_candidates(lib, r[0])[1] == 306900
    assert lib.ysb_postprocess_tta_workspace_bytes(r, 4, ctypes.byref(ws)) == 0


@pytest.mark.parametrize("family,kind", [("yolov7", _lib.INPUT_RAW_HEADS), ("retinanet", _lib.INPUT_RAW_HEADS),
                                         ("retinanet_exp", _lib.INPUT_RAW_HEADS), ("yolov5", _lib.INPUT_DECODED_ROWS),
                                         ("yolov8", _lib.INPUT_DECODED_ROWS), ("retinanet", _lib.INPUT_DECODED_ROWS)])
def test_rows_wider_than_the_filter_tile_are_accepted(lib, family, kind):
    # row width of the filter kernel's input: YOLOv7 5 + C, RetinaNet class rows C, decoded rows the family's C'
    in_w = {"yolov7": 5, "retinanet": 0, "retinanet_exp": 0}[family] if kind == _lib.INPUT_RAW_HEADS else None
    for C in range(440, 470):
        p = params(family, C, kind=kind)
        st, n, rw = num_candidates(lib, p)
        width = C + in_w if in_w is not None else rw
        assert st == 0, (C, width)
        assert workspace(lib, p)[0] == 0
    for C in (601, 1024, 1025, 1203, 2047, 2048):
        assert num_candidates(lib, params(family, C, kind=kind))[0] == 0


def test_channels_last_rows_wider_than_the_tile_stay_refused(lib):
    for C in (engine.NHWC_MAX_ROW_WIDTH - 4, 601, 1203, 2048):
        p = params("yolov5", C, kind=_lib.INPUT_RAW_HEADS_NHWC)
        assert num_candidates(lib, p)[0] == _lib.YSB_ERR_LIMIT
        assert lib.ysb_decode(ctypes.byref(p), HEADS, 3, 0x1000, None) == _lib.YSB_ERR_LIMIT
        assert num_candidates(lib, params("yolov5", C))[0] == 0


@pytest.mark.parametrize("family", ["yolov5", "yolov7", "yolox", "yolov8", "fcos"])
def test_multilabel_workspace_at_2048_classes(lib, family):
    p = params(family, 2048, img=640, batch=64, mutil_label=True)
    st, n, _ = num_candidates(lib, p)
    assert st == 0
    st, ws = workspace(lib, p)
    assert st == 0 and ws == _align256(8 * n * 2048 * 64) + _align256(16 * 64) + 256
    assert ws > 1 << 32   # N * 2048 key slots * 64 images * 8 bytes: past 32 bits, computed in 64
    for fam in ("retinanet", "retinanet_exp"):
        assert num_candidates(lib, params(fam, 2048, mutil_label=True))[0] == _lib.YSB_ERR_UNSUPPORTED


def _pack(score, cand, cls, cls_bits):
    cand_mask = (1 << (32 - cls_bits)) - 1
    cls_mask = (1 << cls_bits) - 1
    hi = np.asarray(score, dtype=np.float32).view(np.uint32).astype(np.uint64) << np.uint64(32)
    lo = ((cand_mask - np.asarray(cand, dtype=np.uint64)) << np.uint64(cls_bits)) | (cls_mask - np.asarray(cls, dtype=np.uint64))
    return hi | lo


@pytest.mark.parametrize("C,cls_bits,max_cand,max_cls", [(1024, 10, _lib.YSB_MAX_CANDIDATES, 1023),
                                                         (2048, 11, _lib.YSB_MAX_CANDIDATES_WIDE, 2047)])
def test_unpack_keys_round_trips_both_layouts(C, cls_bits, max_cand, max_cls):
    rng = np.random.default_rng(3)
    n = 4096
    score = rng.random(n, dtype=np.float32)
    cand = np.concatenate([[0, max_cand], rng.integers(0, max_cand + 1, n - 2)])
    cls = np.concatenate([[max_cls, 0], rng.integers(0, max_cls + 1, n - 2)])
    keys = _pack(score, cand, cls, cls_bits)
    s, c, k = _lib.unpack_keys(keys, C)
    if cls_bits == 10:   # the narrow layout is the one the parity report reads
        assert all(np.array_equal(a, b) for a, b in zip((s, c, k), parity.unpack_keys(keys)))
    assert np.array_equal(s.view(np.uint32), score.view(np.uint32))
    assert np.array_equal(c, cand) and np.array_equal(k, cls)
    # descending key order = (score desc, candidate asc, class asc)
    order = np.argsort(keys)[::-1]
    want = np.lexsort((cls, cand, -score.astype(np.float64)))
    assert np.array_equal(order, want)


@pytest.mark.parametrize("family", FAMILIES)
def test_validate_heads_refuses_more_than_2048_classes(family):
    for C in (2049, 0):
        with pytest.raises(ValueError, match="YSB_MAX_CLASSES"):
            engine.validate_heads(family, [torch.zeros(1, 8, 2, 2)], C, torch.tensor(synth.V5_ANCHORS_PX))
