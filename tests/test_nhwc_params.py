"""Host side of channels-last heads (YSB_INPUT_RAW_HEADS_NHWC): the header value, the C ABI's refusals, the layout helper,
validate_heads, make_params and native_heads -- no GPU."""
import ctypes
import os
import subprocess
import tempfile

import pytest
import torch

import oracle
from yoloseries_b200 import _lib, engine, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NHWC = _lib.INPUT_RAW_HEADS_NHWC


def test_nhwc_input_kind_matches_the_header():
    src = ('#include <stdio.h>\n#include "ysb_postproc.h"\nint main(){printf("%d %d %d %zu %d", YSB_INPUT_RAW_HEADS, '
           'YSB_INPUT_DECODED_ROWS, YSB_INPUT_RAW_HEADS_NHWC, sizeof(ysb_params), YSB_ABI_VERSION);return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        raw, dec, nhwc, size, abi = map(int, subprocess.check_output([exe]).split())
    assert (raw, dec, nhwc) == (_lib.INPUT_RAW_HEADS, _lib.INPUT_DECODED_ROWS, _lib.INPUT_RAW_HEADS_NHWC) == (0, 1, 2)
    assert size == ctypes.sizeof(_lib.YsbParams) and abi == _lib.ABI_VERSION == 6


# ---- heads ----------------------------------------------------------------------------------------------------------
def _flat(family, b=2, img=64, C=5, dtype=torch.float32):
    flat = engine.flatten_heads(family, synth.make_heads(family, b, img, img, C, "dense", 3, "cpu"))
    return [t.to(dtype) for t in flat]


def to_nhwc(family, t):
    """The same values in channels-last memory: 4-D heads via torch.channels_last, YOLOX' 5-D (b, A, K, H, W) as the view
    of a channels-last (b, A*K, H, W) conv output."""
    if t.dim() == 4:
        return t.contiguous(memory_format=torch.channels_last)
    b, A, K, H, W = t.shape
    return t.reshape(b, A * K, H, W).contiguous(memory_format=torch.channels_last).view(b, A, K, H, W)


def _anchors(family):
    return torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


@pytest.mark.parametrize("family", ["yolov5", "yolox", "yolov8", "fcos"])
def test_layout_helper_recognises_channels_last_heads(family):
    flat = _flat(family)
    assert engine.head_layout(family, flat) == _lib.INPUT_RAW_HEADS
    cl = [to_nhwc(family, t) for t in flat]
    assert not all(t.is_contiguous() for t in cl)
    assert engine.head_layout(family, cl) == NHWC
    assert all(torch.equal(a, b) for a, b in zip(flat, cl))
    assert engine.validate_heads(family, cl, 5, _anchors(family), 16) == NHWC
    assert engine.validate_heads(family, flat, 5, _anchors(family), 16) == _lib.INPUT_RAW_HEADS


def test_yolox_view_of_a_channels_last_conv_output():
    conv = torch.zeros(2, 3 * 85, 8, 8).contiguous(memory_format=torch.channels_last)
    view = conv.view(2, 3, 85, 8, 8)
    assert engine.is_channels_last_head("yolox", view)
    assert not engine.is_channels_last_head("yolov5", view)   # 5-D is not a YOLOv5 layout
    assert engine.head_layout("yolox", [view]) == NHWC


def test_size_one_dims_and_both_patterns():
    # a 1-channel ctr and 1x1 levels satisfy both patterns: NCHW wins when every tensor is contiguous
    ctr = torch.zeros(2, 1, 8, 8)
    assert engine.is_channels_last_head("fcos", ctr) and ctr.is_contiguous()
    one = torch.zeros(2, 85, 1, 1)
    assert engine.is_channels_last_head("yolov5", one) and one.is_contiguous()
    assert engine.head_layout("yolov5", [one]) == _lib.INPUT_RAW_HEADS
    # ... and count as channels-last next to channels-last levels
    cls = torch.zeros(2, 5, 8, 8).contiguous(memory_format=torch.channels_last)
    reg = torch.zeros(2, 4, 8, 8).contiguous(memory_format=torch.channels_last)
    assert engine.head_layout("fcos", [cls, reg, ctr]) == NHWC
    big = torch.zeros(2, 85, 4, 4).contiguous(memory_format=torch.channels_last)
    assert engine.head_layout("yolov5", [big, torch.zeros(2, 85, 1, 1)]) == NHWC


def test_mixed_and_transposed_layouts_are_refused():
    flat = _flat("yolov5")
    mixed = [to_nhwc("yolov5", flat[0])] + flat[1:]
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.head_layout("yolov5", mixed)
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.validate_heads("yolov5", mixed, 5, _anchors("yolov5"))
    tr = [t.transpose(2, 3) for t in flat]               # H and W swapped: neither pattern
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.head_layout("yolov5", tr)
    cl_tr = [to_nhwc("yolov5", t).transpose(2, 3) for t in flat]
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.head_layout("yolov5", cl_tr)
    # the rows families have no channels-last variant
    v7 = _flat("yolov7")
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.head_layout("yolov7", [t.permute(0, 1, 3, 2, 4) for t in v7])
    # the permuted (b, A, H, W, 85) view is no channels-last pattern of any family
    view = torch.zeros(2, 85, 3, 8, 8).permute(0, 2, 3, 4, 1)
    for fam in engine.NHWC_FAMILIES:
        assert not engine.is_channels_last_head(fam, view)


def test_make_params_carries_the_nhwc_kind(lib):
    hyp = oracle.default_hyp()
    shapes = [(8, 8), (4, 4), (2, 2)]
    p = engine.make_params("yolox", hyp, 1, 64, 64, shapes, input_kind=NHWC, head_dtype=torch.float16)
    assert p.input_kind == NHWC and p.head_dtype == _lib.DTYPE_F16
    n, rw = ctypes.c_int64(), ctypes.c_int32()
    assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == 0
    q = engine.make_params("yolox", hyp, 1, 64, 64, shapes)
    n2, rw2 = ctypes.c_int64(), ctypes.c_int32()
    assert lib.ysb_num_candidates(ctypes.byref(q), ctypes.byref(n2), ctypes.byref(rw2)) == 0
    assert (n.value, rw.value) == (n2.value, rw2.value)
    ws, ws2 = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.ysb_postprocess_workspace_bytes(ctypes.byref(p), ctypes.byref(ws)) == 0
    assert lib.ysb_postprocess_workspace_bytes(ctypes.byref(q), ctypes.byref(ws2)) == 0
    assert ws.value == ws2.value


# ---- native_heads ---------------------------------------------------------------------------------------------------
def test_native_heads_without_a_family_is_unchanged():
    cl = [to_nhwc("yolov5", t) for t in _flat("yolov5", dtype=torch.float16)]
    out = engine.native_heads(cl)                      # one argument: today's behaviour, a contiguous float32 copy
    assert all(t.dtype == torch.float32 and t.is_contiguous() for t in out)
    flat = _flat("yolov5")
    assert engine.native_heads(flat) is flat


@pytest.mark.parametrize("family", ["yolov5", "yolox", "yolov8", "fcos"])
def test_native_heads_passes_channels_last_outputs_through(family):
    heads = synth.make_heads(family, 2, 64, 64, 5, "dense", 3, "cpu")
    if family == "fcos":
        cl = tuple([to_nhwc(family, t) for t in lst] for lst in heads)
    elif isinstance(heads, dict):
        cl = type(heads)((k, to_nhwc(family, v)) for k, v in heads.items())
    else:
        cl = type(heads)(to_nhwc(family, t) for t in heads)
    assert engine.native_heads(cl, family, 5, 16) is cl
    with pytest.raises(ValueError, match="num_class"):
        engine.native_heads(cl, family)
    # another family's pattern, or a layout mix, still goes through normalise_heads
    other = "yolox" if family != "yolox" else "yolov5"
    out = engine.native_heads(cl, other, 5, 16)
    assert out is not cl and all(t.is_contiguous() for t in engine._leaves(out))


def test_native_heads_copies_rows_wider_than_the_tile():
    C = engine.NHWC_MAX_ROW_WIDTH + 1 - 4 * 16          # YOLOv8 rows of 4*16 + C = 454 values: one too wide
    t = torch.zeros(1, 4 * 16 + C, 2, 2).contiguous(memory_format=torch.channels_last)
    assert not t.is_contiguous()
    out = engine.native_heads([t], "yolov8", C, 16)
    assert out[0].is_contiguous()
    assert engine.native_heads([t], "yolov8", C - 1, 16)[0] is t
    ok = torch.zeros(1, engine.NHWC_MAX_ROW_WIDTH, 2, 2).contiguous(memory_format=torch.channels_last)
    heads = [ok]
    assert engine.native_heads(heads, "fcos", engine.NHWC_MAX_ROW_WIDTH) is heads
    assert engine.nhwc_row_width("fcos", 7) == 7 and engine.nhwc_row_width("yolov8", 80, 16) == 144


# ---- C ABI refusals before any CUDA call ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


HEADS = (ctypes.c_void_p * 15)(*[0x100000 * (k + 1) for k in range(15)])


def test_abi_refuses_nhwc_for_the_rows_families_and_unknown_kinds(lib):
    hyp = oracle.default_hyp()
    n, rw = ctypes.c_int64(), ctypes.c_int32()
    for fam in ("yolov7", "retinanet", "retinanet_exp"):
        shapes = synth.level_shapes(fam, 64, 64) if fam == "yolov7" else None
        anchors = torch.tensor(synth.V5_ANCHORS_PX) if fam == "yolov7" else None
        p = engine.make_params(fam, hyp, 1, 64, 64, shapes, anchors)
        assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == 0
        p.input_kind = NHWC
        assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == _lib.YSB_ERR_BAD_ARG
        assert lib.ysb_postprocess(ctypes.byref(p), HEADS, 3, 0x1000, 1 << 30, 0x2000, 0x3000, 0x4000, None) == \
            _lib.YSB_ERR_BAD_ARG
    for fam in engine.NHWC_FAMILIES:
        p = engine.make_params(fam, hyp, 1, 256, 256, synth.level_shapes(fam, 256, 256),
                               torch.tensor(synth.V5_ANCHORS_PX) if fam == "yolov5" else None, input_kind=NHWC)
        assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == 0
        for kind in (3, -1):
            p.input_kind = kind
            assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == _lib.YSB_ERR_BAD_ARG
            ws = ctypes.c_size_t()
            assert lib.ysb_postprocess_workspace_bytes(ctypes.byref(p), ctypes.byref(ws)) == _lib.YSB_ERR_BAD_ARG
            assert lib.ysb_decode(ctypes.byref(p), HEADS, 3, 0x1000, None) == _lib.YSB_ERR_BAD_ARG


def _v5(kind, tta=None, C=None, **over):
    hyp = oracle.default_hyp()
    hyp.update(over)
    if C is not None:
        hyp["num_class"] = C
    return engine.make_params("yolov5", hyp, 2, 64, 64, synth.level_shapes("yolov5", 64, 64),
                              torch.tensor(synth.V5_ANCHORS_PX), input_kind=kind, tta=tta)


def test_abi_refuses_tta_passes_of_mixed_kinds(lib):
    a = _v5(_lib.INPUT_RAW_HEADS, (1, None, 64, 64))
    b = _v5(NHWC, (0.83, 2, 64, 64))
    c = _v5(NHWC, (1, None, 64, 64))
    ws = ctypes.c_size_t()
    assert lib.ysb_postprocess_tta_workspace_bytes((_lib.YsbParams * 2)(c, b), 2, ctypes.byref(ws)) == 0
    arr = (_lib.YsbParams * 2)(a, b)
    assert lib.ysb_postprocess_tta_workspace_bytes(arr, 2, ctypes.byref(ws)) == _lib.YSB_ERR_BAD_ARG
    per = (ctypes.c_int32 * 2)(3, 3)
    assert lib.ysb_filter_candidates_tta(arr, 2, HEADS, per, 0x1000, 1 << 20, 0x2000, None) == _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_select_nms_tta(arr, 2, HEADS, per, 0x1000, 1 << 20, 0x2000, 0x3000, 0x4000, 0x5000, None) == \
        _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_postprocess_tta(arr, 2, HEADS, per, 0x1000, 1 << 30, 0x3000, 0x4000, 0x5000, None) == \
        _lib.YSB_ERR_BAD_ARG


def test_abi_refuses_rows_wider_than_the_tile(lib):
    n, rw = ctypes.c_int64(), ctypes.c_int32()
    C = engine.NHWC_MAX_ROW_WIDTH - 5                    # 5 + C = 453: the widest row that fits
    assert lib.ysb_num_candidates(ctypes.byref(_v5(NHWC, C=C)), ctypes.byref(n), ctypes.byref(rw)) == 0
    wide = _v5(NHWC, C=C + 1)
    assert lib.ysb_num_candidates(ctypes.byref(wide), ctypes.byref(n), ctypes.byref(rw)) == _lib.YSB_ERR_LIMIT
    assert lib.ysb_decode(ctypes.byref(wide), HEADS, 3, 0x1000, None) == _lib.YSB_ERR_LIMIT
    assert lib.ysb_filter_candidates(ctypes.byref(wide), HEADS, 3, 0x1000, 1 << 30, 0x2000, None) == _lib.YSB_ERR_LIMIT
    # the same classes in NCHW memory are fine
    assert lib.ysb_num_candidates(ctypes.byref(_v5(_lib.INPUT_RAW_HEADS, C=C + 1)), ctypes.byref(n), ctypes.byref(rw)) == 0
