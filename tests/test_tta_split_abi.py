"""Host-side refusals of the split test-time-augmentation entry points (ysb_filter_candidates_tta, ysb_select_nms_tta,
ysb_select_nms_tta_gather): every bad argument returns its status before any CUDA call, so no GPU is needed."""
import ctypes

import pytest
import torch

import oracle
from yoloseries_b200 import _lib, engine, synth

B, IMG, N = 4, 640, 25200


@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


def _params(scale=1, flip=None, **over):
    hyp = oracle.default_hyp()
    hyp.update(over)
    p = engine.make_params("yolov5", hyp, B, IMG, IMG, synth.level_shapes("yolov5", IMG, IMG),
                           anchors=torch.tensor(synth.V5_ANCHORS_PX), tta=(scale, flip, IMG, IMG))
    return p


def _passes(*ps):
    return (_lib.YsbParams * len(ps))(*ps)


def _three(**over):
    return _passes(*[_params(s, f, **over) for s, f in zip(oracle.TTA_SCALES, oracle.TTA_FLIPS)])


# fake, never dereferenced device addresses: every call below must be refused on the host
HEADS = (ctypes.c_void_p * 9)(*[0x100000 * (k + 1) for k in range(9)])
PER_PASS = (ctypes.c_int32 * 3)(3, 3, 3)
KEYS, COUNTS, DETS, IDX, CNT = 0x2000000, 0x3000000, 0x4000000, 0x5000000, 0x6000000


def _gather(batch=B, max_det=None):
    g = _lib.YsbGather()
    g.world, g.rank, g.slots, g.batch = 1, 0, 2, batch
    g.max_det = _params().max_det if max_det is None else max_det
    g.d_buf[0] = 0x7000000
    return g


def _call(lib, which, arr, n, heads=HEADS, per_pass=PER_PASS, keys=KEYS, cap=3 * N, counts=COUNTS, g=None):
    if which == "filter":
        return lib.ysb_filter_candidates_tta(arr, n, heads, per_pass, keys, cap, counts, None)
    if which == "select":
        return lib.ysb_select_nms_tta(arr, n, heads, per_pass, keys, cap, counts, DETS, IDX, CNT, None)
    return lib.ysb_select_nms_tta_gather(arr, n, heads, per_pass, keys, cap, counts,
                                         ctypes.byref(g if g is not None else _gather()), 0, IDX, None)


ENTRY_POINTS = ["filter", "select", "gather"]


def _summed_slots(lib, arr, n, multi):
    """Key slots per image implied by ysb_postprocess_tta_workspace_bytes (keys region minus the counts and padding)."""
    ws = ctypes.c_size_t()
    assert lib.ysb_postprocess_tta_workspace_bytes(arr, n, ctypes.byref(ws)) == _lib.YSB_OK
    al = lambda x: (x + 255) & ~255   # noqa: E731
    slots = sum(N * (80 if multi else 1) for _ in range(n))
    assert ws.value == al(8 * slots * B) + al(16 * B) + 256
    return slots


@pytest.mark.parametrize("which", ENTRY_POINTS)
def test_null_keys_counts_and_heads(lib, which):
    arr = _three()
    assert _call(lib, which, arr, 3, keys=None) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, arr, 3, counts=None) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, arr, 3, heads=None) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, arr, 3, per_pass=None) == _lib.YSB_ERR_BAD_ARG
    holes = (ctypes.c_void_p * 9)(*HEADS)
    holes[4] = None                                            # one head tensor of pass 1 missing
    assert _call(lib, which, arr, 3, heads=holes) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, None, 3) == _lib.YSB_ERR_BAD_ARG


def test_select_needs_rows_and_counts(lib):
    arr = _three()
    assert lib.ysb_select_nms_tta(arr, 3, HEADS, PER_PASS, KEYS, 3 * N, COUNTS, None, IDX, CNT, None) == _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_select_nms_tta(arr, 3, HEADS, PER_PASS, KEYS, 3 * N, COUNTS, DETS, IDX, None, None) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", ENTRY_POINTS)
def test_pass_count(lib, which):
    five = _passes(*[_params() for _ in range(5)])
    per5 = (ctypes.c_int32 * 5)(3, 3, 3, 3, 3)
    heads15 = (ctypes.c_void_p * 15)(*[0x100000 * (k + 1) for k in range(15)])
    assert _call(lib, which, five, 0, heads=heads15, per_pass=per5, cap=5 * N) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, five, 5, heads=heads15, per_pass=per5, cap=5 * N) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("which", ENTRY_POINTS)
def test_passes_whose_thresholds_differ(lib, which):
    arr = _three()
    arr[2].iou_thr = 0.5                                       # one evaluator, one hyp
    assert _call(lib, which, arr, 3) == _lib.YSB_ERR_BAD_ARG
    arr = _three()
    arr[1].cls_thr = arr[0].cls_thr + 0.01
    assert _call(lib, which, arr, 3) == _lib.YSB_ERR_BAD_ARG
    arr = _three()
    arr[1].head_dtype = _lib.DTYPE_F16
    assert _call(lib, which, arr, 3) == _lib.YSB_ERR_BAD_ARG
    arr = _three()
    arr[2].tta_flip = 1                                        # the reference flips along dims 2 or 3 only
    assert _call(lib, which, arr, 3) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, which, _three(), 3, per_pass=(ctypes.c_int32 * 3)(3, 2, 3)) == _lib.YSB_ERR_BAD_ARG


@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("which", ENTRY_POINTS)
def test_key_capacity_one_below_the_summed_slots(lib, which, multi):
    arr = _three(mutil_label=multi)
    slots = _summed_slots(lib, arr, 3, multi)
    assert slots == 3 * N * (80 if multi else 1)
    assert _call(lib, which, arr, 3, cap=slots - 1) == _lib.YSB_ERR_WORKSPACE
    assert _call(lib, which, arr, 3, cap=0) == _lib.YSB_ERR_WORKSPACE
    # two passes: the sum of those two
    two = _passes(arr[0], arr[1])
    slots2 = _summed_slots(lib, two, 2, multi)
    assert _call(lib, which, two, 2, per_pass=(ctypes.c_int32 * 2)(3, 3), cap=slots2 - 1) == _lib.YSB_ERR_WORKSPACE


def test_gather_that_does_not_match_the_passes(lib):
    arr = _three()
    cap = _summed_slots(lib, arr, 3, False)
    assert _call(lib, "gather", arr, 3, cap=cap, g=_gather(batch=B + 1)) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, "gather", arr, 3, cap=cap, g=_gather(batch=B - 1)) == _lib.YSB_ERR_BAD_ARG
    assert _call(lib, "gather", arr, 3, cap=cap, g=_gather(max_det=arr[0].max_det - 2)) == _lib.YSB_ERR_BAD_ARG
    bad_slot = _gather()
    assert lib.ysb_select_nms_tta_gather(arr, 3, HEADS, PER_PASS, KEYS, cap, COUNTS, ctypes.byref(bad_slot), 2, IDX,
                                         None) == _lib.YSB_ERR_BAD_ARG          # slot out of range
    unmapped = _gather()
    unmapped.world = 2                                         # peer buffer missing
    assert _call(lib, "gather", arr, 3, cap=cap, g=unmapped) == _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_select_nms_tta_gather(arr, 3, HEADS, PER_PASS, KEYS, cap, COUNTS, None, 0, IDX,
                                         None) == _lib.YSB_ERR_BAD_ARG


def test_new_entry_points_are_in_the_signature_table():
    for name in ("ysb_filter_candidates_tta", "ysb_select_nms_tta", "ysb_select_nms_tta_gather"):
        assert name in _lib.EXPORTED_SYMBOLS
    assert _lib.ABI_VERSION == 6
