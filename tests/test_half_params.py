"""Host side of float16 / bfloat16 heads: the head_dtype field of ysb_params, validate_heads and make_params -- no GPU."""
import ctypes
import os
import subprocess
import tempfile

import pytest
import torch

import oracle
from yoloseries_b200 import _lib, engine, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_head_dtype_field_matches_the_header():
    src = ('#include <stdio.h>\n#include "ysb_postproc.h"\nint main(){printf("%zu %zu %zu %d %d %d %d", sizeof(ysb_params), '
           '__builtin_offsetof(ysb_params, head_dtype), sizeof(((ysb_params *)0)->head_dtype), YSB_F32, YSB_F16, YSB_BF16, '
           'YSB_ABI_VERSION);return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        size, off, fsize, f32, f16, bf16, abi = map(int, subprocess.check_output([exe]).split())
    assert ctypes.sizeof(_lib.YsbParams) == size
    assert _lib.YsbParams.head_dtype.offset == off and fsize == 4
    assert (f32, f16, bf16) == (_lib.DTYPE_F32, _lib.DTYPE_F16, _lib.DTYPE_BF16)
    assert abi == _lib.ABI_VERSION == 6
    # the last member: a zero-filled struct of an older caller reads as float32
    assert off == max(f.offset for f in (getattr(_lib.YsbParams, n) for n, _ in _lib.YsbParams._fields_))
    assert _lib.YsbParams().head_dtype == _lib.DTYPE_F32


def _heads(family, dtype, b=2, img=64, C=5):
    flat = engine.flatten_heads(family, synth.make_heads(family, b, img, img, C, "dense", 3, "cpu"))
    return [t.to(dtype) for t in flat]


def _anchors(family):
    return torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("family", ["yolov5", "yolov7", "yolox", "yolov8", "retinanet", "retinanet_exp", "fcos"])
def test_validate_heads_accepts_the_three_dtypes(family, dtype):
    engine.validate_heads(family, _heads(family, dtype), 5, _anchors(family), 16)


@pytest.mark.parametrize("family", ["yolov5", "retinanet", "retinanet_exp", "fcos"])
def test_validate_heads_rejects_mixed_dtypes(family):
    flat = _heads(family, torch.float16)
    for i in range(len(flat)):   # any one tensor of another type: RetinaNet reg vs cls, FCOS cls / reg / ctr, v5 levels
        mixed = list(flat)
        mixed[i] = mixed[i].to(torch.bfloat16 if i % 2 else torch.float32)
        with pytest.raises(ValueError, match="one dtype"):
            engine.validate_heads(family, mixed, 5, _anchors(family), 16)


def test_validate_heads_rejects_double_and_16_bit_decoded_rows():
    good = _heads("yolov5", torch.float16)
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.validate_heads("yolov5", [good[0].double(), good[1].double(), good[2].double()], 5, _anchors("yolov5"))
    with pytest.raises(ValueError, match="contiguous float32"):
        engine.validate_heads("yolov5", [good[0].transpose(2, 3), good[1], good[2]], 5, _anchors("yolov5"))
    for dtype in (torch.float16, torch.bfloat16):
        with pytest.raises(ValueError, match="decoded tensor must be contiguous float32"):
            engine.validate_heads("yolov5", [torch.zeros(2, 7, 10, dtype=dtype)], 5, decoded_row_w=10)
    engine.validate_heads("yolov5", [torch.zeros(2, 7, 10)], 5, decoded_row_w=10)


def test_make_params_carries_the_dtype():
    hyp = oracle.default_hyp()
    shapes = [(8, 8), (4, 4), (2, 2)]
    want = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}
    for dtype, code in want.items():
        assert engine.make_params("yolox", hyp, 1, 64, 64, shapes, head_dtype=dtype).head_dtype == code
        assert engine.make_params("retinanet", hyp, 1, 64, 64, head_dtype=dtype).head_dtype == code
    assert engine.make_params("yolox", hyp, 1, 64, 64, shapes).head_dtype == _lib.DTYPE_F32
    with pytest.raises(ValueError, match="head_dtype"):
        engine.make_params("yolox", hyp, 1, 64, 64, shapes, head_dtype=torch.float64)


def test_native_heads_passes_16_bit_outputs_unchanged():
    from collections import OrderedDict
    half = [torch.zeros(2, 255, 8, 8, dtype=torch.float16), torch.zeros(2, 255, 4, 4, dtype=torch.float16)]
    assert engine.native_heads(half) is half
    f32 = (torch.zeros(2, 4, 5), torch.zeros(2, 4, 80))
    assert engine.native_heads(f32) is f32
    fcos = ([torch.zeros(2, 4, 8, 8, dtype=torch.bfloat16)], [torch.zeros(2, 4, 8, 8, dtype=torch.bfloat16)],
            [torch.zeros(2, 1, 8, 8, dtype=torch.bfloat16)])
    assert engine.native_heads(fcos) is fcos
    # mixed types, a view or double: the conversion of normalise_heads (float32, contiguous)
    mixed = OrderedDict(p0=torch.zeros(2, 3, 8, 8, 85, dtype=torch.float16), p1=torch.zeros(2, 3, 4, 4, 85))
    out = engine.native_heads(mixed)
    assert isinstance(out, OrderedDict) and all(t.dtype == torch.float32 for t in out.values())
    view = [torch.zeros(2, 85, 3, 8, 8, dtype=torch.float16).permute(0, 2, 3, 4, 1)]
    out = engine.native_heads(view)
    assert out[0].dtype == torch.float32 and out[0].is_contiguous()
    assert engine.native_heads([torch.zeros(2, 5, dtype=torch.float64)])[0].dtype == torch.float32


@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


def test_abi_refuses_bad_dtypes_without_a_device(lib):
    """Argument checks run before any CUDA call: unknown dtype, 16-bit decoded rows, TTA passes of different types."""
    hyp = oracle.default_hyp()
    shapes = [(8, 8), (4, 4), (2, 2)]
    p = engine.make_params("yolox", hyp, 1, 64, 64, shapes)
    n, rw = ctypes.c_int64(), ctypes.c_int32()
    for code, status in ((0, 0), (1, 0), (2, 0), (3, _lib.YSB_ERR_BAD_ARG), (-1, _lib.YSB_ERR_BAD_ARG)):
        p.head_dtype = code
        assert lib.ysb_num_candidates(ctypes.byref(p), ctypes.byref(n), ctypes.byref(rw)) == status
    d = engine.make_params("yolox", hyp, 1, 64, 64, shapes, input_kind=_lib.INPUT_DECODED_ROWS)
    assert lib.ysb_num_candidates(ctypes.byref(d), ctypes.byref(n), ctypes.byref(rw)) == 0
    d.head_dtype = _lib.DTYPE_F16
    assert lib.ysb_num_candidates(ctypes.byref(d), ctypes.byref(n), ctypes.byref(rw)) == _lib.YSB_ERR_BAD_ARG
    a = engine.make_params("yolox", hyp, 1, 64, 64, shapes, head_dtype=torch.float16)
    b = engine.make_params("yolox", hyp, 1, 64, 64, shapes, head_dtype=torch.bfloat16)
    ws = ctypes.c_size_t()
    assert lib.ysb_postprocess_tta_workspace_bytes((_lib.YsbParams * 2)(a, a), 2, ctypes.byref(ws)) == 0
    assert lib.ysb_postprocess_tta_workspace_bytes((_lib.YsbParams * 2)(a, b), 2, ctypes.byref(ws)) == _lib.YSB_ERR_BAD_ARG
