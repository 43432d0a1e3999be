"""Host side of matching kept rows against ground truth on the device (ysb_match_tp, ysb_match_compact, match(),
MatchStats): the struct layout, every argument refusal of the C ABI (they return before any CUDA call, so no GPU is
needed), the Python argument checks, and where a step's target arrays land in the padded block for full and partial
steps."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from yoloseries_b200 import _lib, engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, B, D, G = 2, 4, 300, 16

# fake, never dereferenced device addresses: every refused call below must return before touching them
ROWS, CNT, GT, GT_CNT, TP, WS = 0x1000000, 0x2000000, 0x3000000, 0x4000000, 0x5000000, 0x6000000
ACC_IN, ACC_OUT, CONF, CLS, TP_OUT, TCLS = 0x7000000, 0x7000100, 0x8000000, 0x9000000, 0xa000000, 0xb000000
THR = (ctypes.c_double * 10)(*np.linspace(0.5, 0.95, 10))


@pytest.fixture(scope="module")
def lib():
    from yoloseries_b200 import build
    build.build()
    return _lib.load()


def _step(**kw):
    s = _lib.YsbMatchStep()
    s.world, s.batch, s.max_det, s.max_gt = W, B, D, G
    s.d_rows, s.rows_rank_bytes = ROWS, B * D * 24 + 256
    s.d_cnt, s.cnt_rank_bytes = CNT, 256
    s.d_gt, s.d_gt_cnt, s.gt_dtype = GT, GT_CNT, _lib.DTYPE_F32
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def _tp(lib, s, thr=THR, ws=WS, ws_bytes=1 << 20, tp=TP):
    return lib.ysb_match_tp(None if s is None else ctypes.byref(s), thr, ws, ws_bytes, tp, None)


def _compact(lib, s, tp=TP, acc_in=ACC_IN, acc_out=ACC_OUT, conf=CONF, cls=CLS, tp_out=TP_OUT, row_cap=100, tcls=TCLS,
             tgt_cap=100):
    return lib.ysb_match_compact(None if s is None else ctypes.byref(s), tp, acc_in, acc_out, conf, cls, tp_out, row_cap,
                                 tcls, tgt_cap, None)


def test_struct_layout_matches_the_compiler(tmp_path):
    src = tmp_path / "m.c"
    src.write_text('#include <stdio.h>\n#include "ysb_postproc.h"\nint main(){printf("%zu %zu %zu", sizeof(ysb_match_step), '
                   '__builtin_offsetof(ysb_match_step, rows_rank_bytes), __builtin_offsetof(ysb_match_step, gt_dtype));'
                   'return 0;}\n')
    exe = tmp_path / "m"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(_lib.YsbMatchStep), _lib.YsbMatchStep.rows_rank_bytes.offset,
                   _lib.YsbMatchStep.gt_dtype.offset]


def test_entry_points_are_in_the_signature_table(lib):
    for name in ("ysb_match_tp_workspace_bytes", "ysb_match_tp", "ysb_match_compact"):
        assert name in _lib.EXPORTED_SYMBOLS
        assert getattr(lib, name).restype is ctypes.c_int
    assert _lib.ABI_VERSION == lib.ysb_abi_version() == 6


def test_workspace_query(lib):
    n = ctypes.c_size_t()
    assert lib.ysb_match_tp_workspace_bytes(ctypes.byref(_step()), ctypes.byref(n)) == _lib.YSB_OK
    assert n.value == 4 * W * B * G
    assert lib.ysb_match_tp_workspace_bytes(ctypes.byref(_step()), None) == _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_match_tp_workspace_bytes(None, ctypes.byref(n)) == _lib.YSB_ERR_BAD_ARG
    assert lib.ysb_match_tp_workspace_bytes(ctypes.byref(_step(world=0)), ctypes.byref(n)) == _lib.YSB_ERR_BAD_ARG


REFUSED_STEPS = {
    "world 0": (dict(world=0), _lib.YSB_ERR_BAD_ARG),
    "too many ranks": (dict(world=_lib.YSB_MAX_PEERS + 1), _lib.YSB_ERR_BAD_ARG),
    "negative batch": (dict(batch=-1), _lib.YSB_ERR_BAD_ARG),
    "negative max_det": (dict(max_det=-1), _lib.YSB_ERR_BAD_ARG),
    "negative max_gt": (dict(max_gt=-1), _lib.YSB_ERR_BAD_ARG),
    "max_det beyond the limit": (dict(max_det=_lib.YSB_MAX_DET_LIMIT + 1, rows_rank_bytes=1 << 30), _lib.YSB_ERR_LIMIT),
    "unknown dtype": (dict(gt_dtype=_lib.DTYPE_F16), _lib.YSB_ERR_BAD_ARG),
    "dtype out of range": (dict(gt_dtype=7), _lib.YSB_ERR_BAD_ARG),
    "rows stride below a rank's rows": (dict(rows_rank_bytes=B * D * 24 - 4), _lib.YSB_ERR_BAD_ARG),
    "counts stride below a rank's counts": (dict(cnt_rank_bytes=B * 4 - 4), _lib.YSB_ERR_BAD_ARG),
    "null rows": (dict(d_rows=None), _lib.YSB_ERR_BAD_ARG),
    "null counts": (dict(d_cnt=None), _lib.YSB_ERR_BAD_ARG),
    "null gt": (dict(d_gt=None), _lib.YSB_ERR_BAD_ARG),
    "null gt counts": (dict(d_gt_cnt=None), _lib.YSB_ERR_BAD_ARG),
    "first_pred index beyond int32": (dict(max_gt=1 << 29), _lib.YSB_ERR_LIMIT),
}


@pytest.mark.parametrize("case", sorted(REFUSED_STEPS))
def test_step_refusals(lib, case):
    kw, status = REFUSED_STEPS[case]
    assert _tp(lib, _step(**kw)) == status
    assert _compact(lib, _step(**kw)) == status


def test_call_refusals(lib):
    s = _step()
    assert _tp(lib, None) == _lib.YSB_ERR_BAD_ARG
    assert _tp(lib, s, thr=None) == _lib.YSB_ERR_BAD_ARG
    nan = (ctypes.c_double * 10)(*([float("nan")] + [0.5] * 9))
    assert _tp(lib, s, thr=nan) == _lib.YSB_ERR_BAD_ARG
    assert _tp(lib, s, tp=None) == _lib.YSB_ERR_BAD_ARG
    assert _tp(lib, s, ws=None) == _lib.YSB_ERR_WORKSPACE
    assert _tp(lib, s, ws_bytes=4 * W * B * G - 1) == _lib.YSB_ERR_WORKSPACE
    assert _compact(lib, None) == _lib.YSB_ERR_BAD_ARG
    for k in ("tp", "acc_in", "acc_out", "conf", "cls", "tp_out", "tcls"):
        assert _compact(lib, s, **{k: None}) == _lib.YSB_ERR_BAD_ARG, k
    assert _compact(lib, s, acc_out=ACC_IN) == _lib.YSB_ERR_BAD_ARG       # the counters must not alias
    assert _compact(lib, s, row_cap=-1) == _lib.YSB_ERR_BAD_ARG
    assert _compact(lib, s, tgt_cap=-1) == _lib.YSB_ERR_BAD_ARG


def test_empty_steps_need_no_device_buffers(lib):
    """batch 0: nothing to match (no launch, no pointers needed); one rank's strides are not used."""
    s = _step(batch=0, d_rows=None, d_cnt=None, d_gt=None, d_gt_cnt=None, rows_rank_bytes=0, cnt_rank_bytes=0)
    assert _tp(lib, s, ws=None, ws_bytes=0, tp=None) == _lib.YSB_OK


def test_valid_calls_pass_validation(lib):
    """Past every check the first thing is a launch, which fails without a device (on a machine with a GPU it would
    launch into the fake addresses above, so the check runs where there is none; tests/test_gpu_match.py runs them)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("would launch kernels into fake addresses")
    for kw in (dict(), dict(gt_dtype=_lib.DTYPE_F64), dict(world=1, rows_rank_bytes=B * D * 24, cnt_rank_bytes=B * 4),
               dict(max_det=_lib.YSB_MAX_DET_LIMIT, rows_rank_bytes=B * _lib.YSB_MAX_DET_LIMIT * 24)):
        assert _tp(lib, _step(**kw)) == _lib.YSB_ERR_CUDA
        assert _compact(lib, _step(**kw)) == _lib.YSB_ERR_CUDA


# ---- Python side ------------------------------------------------------------------------------------------------------
def _boxes(n, dtype=np.float32, seed=0):
    r = np.random.default_rng(seed)
    xy = r.uniform(0, 500, (n, 2))
    return np.concatenate([xy, xy + r.uniform(5, 100, (n, 2)), r.integers(0, 80, (n, 1))], 1).astype(dtype)


def test_pack_targets_full_step():
    arrs = [_boxes(n, seed=n) for n in (3, 0, 7, 1)]
    out, dtype, max_n = engine.pack_targets(arrs, range(4), 4, 1024)
    assert dtype == np.float32 and max_n == 7
    for a, b in zip(arrs, out):
        assert np.array_equal(a, b)


def test_pack_targets_partial_step_positions():
    """A partial step lists only the images every rank had, in result() order: rank-major, then image, absent skipped.
    The present positions come from the gathered counts."""
    cnt = np.array([[3, -1, -2, -2], [0, 5, 2, -2]])          # world 2, batch 4; -2 = absent
    positions = [k for k, c in enumerate(cnt.reshape(-1)) if c != _lib.YSB_CNT_ABSENT]
    assert positions == [0, 1, 4, 5, 6]
    arrs = [_boxes(k + 1, np.float64, k) for k in range(5)]
    out, dtype, max_n = engine.pack_targets(arrs, positions, 8, 8)
    assert dtype == np.float64 and max_n == 5 and len(out) == 5


def test_pack_targets_refusals():
    with pytest.raises(ValueError, match="one target array per image"):
        engine.pack_targets([_boxes(2)] * 3, range(4), 4, 1024)
    with pytest.raises(ValueError, match=r"\(n, 5\)"):
        engine.pack_targets([_boxes(2)[:, :4]], range(1), 1, 1024)
    with pytest.raises(ValueError, match="float32 or float64"):
        engine.pack_targets([_boxes(2).astype(np.int64)], range(1), 1, 1024)
    with pytest.raises(ValueError, match="one dtype"):
        engine.pack_targets([_boxes(2), _boxes(2, np.float64)], range(2), 2, 1024)
    with pytest.raises(ValueError, match="max_targets"):
        engine.pack_targets([_boxes(9)], range(1), 1, 8)
    out, dtype, _ = engine.pack_targets([_boxes(8), np.zeros((0, 5))], range(2), 2, 8)   # at the capacity; empty: any dtype
    assert dtype == np.float32
    with pytest.raises(ValueError, match="max_targets must be at least 1"):
        engine.check_max_targets(0)


def test_torch_targets_are_accepted():
    import torch
    t = torch.from_numpy(_boxes(4, np.float64))
    out, dtype, max_n = engine.pack_targets([t, []], range(2), 2, 16)
    assert dtype == np.float64 and max_n == 4 and np.array_equal(out[0], t.numpy()) and out[1].shape == (0, 5)


def test_match_stats_is_empty_before_any_step():
    from yoloseries_b200.utils.mAP import MatchStats
    tp, conf, cls, tcls = MatchStats().arrays()
    assert tp.shape == (0, 10) and tp.dtype == bool and conf.dtype == cls.dtype == np.float32
    assert tcls.dtype == np.float64 and tcls.shape == (0,)
