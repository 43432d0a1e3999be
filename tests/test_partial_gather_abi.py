"""Host side of partial steps in the detection gather (ysb_select_nms_gather_partial, ysb_select_nms_tta_gather_partial):
the absent mark, the signature table, and the argument checks that return before any CUDA call, so no GPU is needed."""
import ctypes
import os
import re

import pytest
import torch

import oracle
from yoloseries_b200 import _lib, engine, synth

B, IMG, N = 4, 640, 25200
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


def _params(batch=B, scale=1, flip=None):
    return engine.make_params("yolov5", oracle.default_hyp(), batch, IMG, IMG, synth.level_shapes("yolov5", IMG, IMG),
                              anchors=torch.tensor(synth.V5_ANCHORS_PX), tta=(scale, flip, IMG, IMG))


# fake, never dereferenced device addresses: every refused call below must return before touching them
HEADS = (ctypes.c_void_p * 9)(*[0x100000 * (k + 1) for k in range(9)])
PER_PASS = (ctypes.c_int32 * 3)(3, 3, 3)
KEYS, COUNTS, IDX = 0x2000000, 0x3000000, 0x5000000


def _gather(batch=B, max_det=None):
    g = _lib.YsbGather()
    g.world, g.rank, g.slots, g.batch = 1, 0, 2, batch
    g.max_det = _params().max_det if max_det is None else max_det
    g.d_buf[0] = 0x7000000
    return g


def _call(lib, which, batch, g=None, slot=0, keys=KEYS, counts=COUNTS, heads=HEADS, strict=False):
    """One call of the plain or TTA gather entry (the partial one unless ``strict``) for a plan of ``batch`` images."""
    gp = None if g is False else ctypes.byref(g if g is not None else _gather())
    if which == "plain":
        p = _params(batch)
        fn = lib.ysb_select_nms_gather if strict else lib.ysb_select_nms_gather_partial
        return fn(ctypes.byref(p), heads, 3, keys, N, counts, gp, slot, IDX, None)
    arr = (_lib.YsbParams * 3)(*[_params(batch, s, f) for s, f in zip(oracle.TTA_SCALES, oracle.TTA_FLIPS)])
    fn = lib.ysb_select_nms_tta_gather if strict else lib.ysb_select_nms_tta_gather_partial
    return fn(arr, 3, heads, PER_PASS, keys, 3 * N, counts, gp, slot, IDX, None)


WHICH = ["plain", "tta"]


def test_absent_mark_matches_the_header():
    with open(os.path.join(ROOT, "include", "ysb_postproc.h")) as f:
        m = re.search(r"#define\s+YSB_CNT_ABSENT\s+\((-?\d+)\)", f.read())
    assert m and int(m.group(1)) == _lib.YSB_CNT_ABSENT == -2
    assert _lib.ABI_VERSION == 6


def test_partial_entry_points_are_in_the_signature_table(lib):
    for name in ("ysb_select_nms_gather_partial", "ysb_select_nms_tta_gather_partial"):
        assert name in _lib.EXPORTED_SYMBOLS
        assert getattr(lib, name).restype is ctypes.c_int


@pytest.mark.parametrize("which", WHICH)
def test_more_images_than_the_gather_holds(lib, which):
    assert _call(lib, which, B + 1) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", WHICH)
def test_negative_batch(lib, which):
    assert _call(lib, which, -1) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", WHICH)
def test_max_det_must_still_match(lib, which):
    assert _call(lib, which, B - 1, g=_gather(max_det=_params().max_det - 2)) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, 0, g=_gather(max_det=_params().max_det + 2)) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", WHICH)
def test_bad_slot_and_null_pointers(lib, which):
    assert _call(lib, which, B - 1, slot=2) == _lib.YSB_ERR_BAD_ARG       # two slots
    assert _call(lib, which, B - 1, slot=-1) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, B - 1, g=False) == _lib.YSB_ERR_BAD_ARG      # no gather
    unmapped = _gather()
    unmapped.world = 2                                                    # peer buffer missing
    assert _call(lib, which, B - 1, g=unmapped) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, B - 1, keys=None) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, B - 1, counts=None) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, B - 1, heads=None) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", WHICH)
def test_short_plans_pass_validation(lib, which):
    """batch 0 and batch < g->batch get past every argument check of the partial entry (the strict one refuses them);
    the first thing after the checks is a kernel launch, which fails without a device.  On a machine with a GPU the
    launches would be real, into the fake addresses above, so the check runs where there is none
    (tests/test_gpu_partial_batches.py runs the entries on the device)."""
    if torch.cuda.is_available():
        pytest.skip("would launch kernels into fake addresses")
    for n in (0, 1, B - 1):
        assert _call(lib, which, n, strict=True) == _lib.YSB_ERR_BAD_ARG
        assert _call(lib, which, n) == _lib.YSB_ERR_CUDA


@pytest.mark.parametrize("family", ["yolov5", "yolox", "yolov8", "fcos"])
@pytest.mark.parametrize("channels_last", [False, True])
def test_zero_image_heads_flatten_and_pass_the_layout_check(family, channels_last):
    """A rank without images in a partial step slices zero images out of the model's outputs: those heads flatten and
    pass head_layout in both memory layouts (zero-element tensors read as contiguous: nothing of them is read)."""
    heads = synth.make_heads(family, 2, 64, 64, 3, "sparse", 1, "cpu")
    if channels_last:
        heads = _to_channels_last(family, heads)
    empty = _nest(heads, lambda t: t[:0])
    flat = engine.flatten_heads(family, empty)
    assert flat and all(t.shape[0] == 0 for t in flat)
    assert engine.head_layout(family, flat) == _lib.INPUT_RAW_HEADS
    if channels_last:   # the full batch keeps its layout
        assert engine.head_layout(family, engine.flatten_heads(family, heads)) == _lib.INPUT_RAW_HEADS_NHWC


def _nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(_nest(v, fn) for v in x)


def _to_channels_last(family, heads):
    def cl(t):
        if t.dim() == 5:   # YOLOX (b, A, K, H, W): the view of a channels-last (b, A*K, H, W) conv output
            b, a, k, h, w = t.shape
            return t.reshape(b, a * k, h, w).contiguous(memory_format=torch.channels_last).view(b, a, k, h, w)
        return t.contiguous(memory_format=torch.channels_last)
    return _nest(heads, cl)
