"""Test-time-augmented batches through ShardedPostProcessor.submit_tta (lanes, CUDA graphs, the detection gather) against
PostProcessor.run_tta, which tests/test_gpu_tta.py pins to the reference goldens and the oracle.  Both run the same kernels
on the same inputs, so rows, counts and candidate indices are compared bit for bit, RetinaNet included."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from conftest import golden_names, hyp_from_meta, load_golden, tta_pass_heads

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _to_dev(x):
    if isinstance(x, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return type(x)(_to_dev(v) for v in x)


def _nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(_nest(v, fn) for v in x)


def _anchors(family):
    from yoloseries_b200.synth import V5_ANCHORS_PX
    return torch.tensor(V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


def _sharded(family, hyp, batch, h, w, **kw):
    from yoloseries_b200.dist import ShardedPostProcessor
    return ShardedPostProcessor(family, hyp, batch, h, w, anchors=_anchors(family), **kw)


def _v5_passes(batch, img, dname, seed, dtype=None):
    from yoloseries_b200 import synth
    out = []
    for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS)):
        heads = synth.make_heads("yolov5", batch, img, img, 80, dname, seed + k, "cuda")
        if dtype is not None:
            heads = _nest(heads, lambda t: t.to(dtype))
        out.append((heads, img, img, s, f))
    return out


def _snapshot(spp, ticket):
    rows, cnt = spp.gathered(ticket)
    idx = spp._slots[ticket]["idx"]
    torch.cuda.synchronize()
    return rows[0].clone(), cnt[0].clone(), idx.clone()


def _assert_same(got, want_rows, want_cnt, want_idx=None):
    rows, cnt, idx = got
    assert torch.equal(cnt, want_cnt), (cnt.tolist(), want_cnt.tolist())
    for i in range(cnt.numel()):
        c = max(int(cnt[i]), 0)
        assert torch.equal(rows[i, :c].view(torch.int32), want_rows[i, :c].view(torch.int32)), f"image {i}"
        if want_idx is not None:
            assert torch.equal(idx[i, :c], want_idx[i, :c]), f"image {i} candidate indices"


def _reference(pp, passes, h, w):
    out = pp.run_tta(passes, (h, w))
    torch.cuda.synchronize()
    return out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone()


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("name", golden_names("tta_"))
def test_tta_goldens_through_submit_tta(name, graph):
    from yoloseries_b200.engine import PostProcessor
    g = load_golden(name)
    meta = g["meta"]
    fam, h, w = meta["family"], meta["img_h"], meta["img_w"]
    hyp = hyp_from_meta(meta)
    passes = [(_to_dev(tta_pass_heads(g, k)), h, w, s, f) for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    pp = PostProcessor(fam, hyp, anchors=_anchors(fam))
    want = _reference(pp, passes, h, w)
    assert int(want[1].max()) > 0
    spp = _sharded(fam, hyp, meta["batch"], h, w, lanes=2, graph=graph)
    for _ in range(4):   # more submissions than lanes: lanes are reused (and, with graphs, replayed)
        _assert_same(_snapshot(spp, spp.submit_tta(passes)), *want)
    assert spp.mode == "local" and spp._key_cap == sum(e["N"] for e in spp._tta["ents"])
    spp.close()


@pytest.mark.parametrize("dname", ["dense", "crowd", "sparse"])
def test_full_size_yolov5_lanes_and_graphs(dname):
    """YOLOv5 640x640, 8 images, 3 lanes, 7 steps: some steps reuse the previous head tensors (graph replay), the others
    allocate new ones (capture)."""
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    hyp = synth.map_profile_hyp(num_class=80)
    pp = PostProcessor("yolov5", hyp, anchors=_anchors("yolov5"))
    spp = _sharded("yolov5", hyp, 8, 640, 640, lanes=3)
    assert spp.graph
    for step in range(7):
        if step % 3 != 1:
            passes = _v5_passes(8, 640, dname, 100 * step)
        want = _reference(pp, passes, 640, 640)
        _assert_same(_snapshot(spp, spp.submit_tta(passes)), *want)
        if dname == "dense":   # rows from the augmented passes take part
            assert max(int(want[2][i, :c].max()) for i, c in enumerate(want[1].tolist()) if c > 0) >= 25200
    assert len(spp._graphs) >= 3
    res = spp.result(spp.submit_tta(passes))
    assert len(res) == 8
    spp.close()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_16_bit_heads_equal_the_float32_run_on_the_widened_heads(dtype):
    from yoloseries_b200 import synth
    hyp = synth.map_profile_hyp(num_class=80)
    half = _sharded("yolov5", hyp, 8, 640, 640, lanes=2)
    f32 = _sharded("yolov5", hyp, 8, 640, 640, lanes=2)
    for step in range(3):
        passes = _v5_passes(8, 640, "dense", 40 + 10 * step, dtype)
        wide = [(_nest(p[0], lambda t: t.float()), *p[1:]) for p in passes]
        want = _snapshot(f32, f32.submit_tta(wide))
        _assert_same(_snapshot(half, half.submit_tta(passes)), *want)
    with pytest.raises(ValueError, match="heads"):
        half.submit_tta(wide)
    half.close()
    f32.close()


def test_multi_label_key_capacity():
    """mutil_label: N*C key slots per pass; the lane's key buffer holds all three passes' slots."""
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    hyp = oracle.default_hyp(num_class=80, mutil_label=True)
    pp = PostProcessor("yolov5", hyp, anchors=_anchors("yolov5"))
    spp = _sharded("yolov5", hyp, 4, 320, 320, lanes=2)
    for step in range(3):
        passes = _v5_passes(4, 320, "dense", 500 + step)
        want = _reference(pp, passes, 320, 320)
        _assert_same(_snapshot(spp, spp.submit_tta(passes)), *want)
    assert spp._key_cap == 3 * synth.num_candidates("yolov5", 320, 320) * 80
    assert spp._slots[0]["keys"].shape == (4, spp._key_cap)
    spp.close()


def test_events_give_the_same_rows():
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    hyp = synth.map_profile_hyp(num_class=80)
    pp = PostProcessor("yolov5", hyp, anchors=_anchors("yolov5"))
    spp = _sharded("yolov5", hyp, 8, 640, 640, lanes=2)
    for step in range(3):
        passes = _v5_passes(8, 640, "crowd", 900 + step)
        want = _reference(pp, passes, 640, 640)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        _assert_same(_snapshot(spp, spp.submit_tta(passes, events=ev)), *want)
        assert ev[0].elapsed_time(ev[1]) > 0 and ev[1].elapsed_time(ev[2]) > 0
    assert not spp._graphs   # timed submissions run as plain launches
    spp.close()


def test_set_up_mismatches_raise():
    from yoloseries_b200 import synth
    hyp = synth.map_profile_hyp(num_class=80)
    passes = _v5_passes(4, 320, "dense", 7)
    spp = _sharded("yolov5", hyp, 4, 320, 320, lanes=2)
    spp.submit_tta(passes)
    with pytest.raises(ValueError, match="submit_tta"):
        spp.submit(passes[0][0])
    with pytest.raises(ValueError, match="passes"):
        spp.submit_tta(passes[:2])
    with pytest.raises(ValueError, match="passes"):
        spp.submit_tta([passes[0], passes[1], (passes[2][0], 320, 320, 0.5, 3)])
    with pytest.raises(ValueError, match="passes"):
        spp.submit_tta([passes[0], passes[1], (passes[2][0], 320, 320, 0.67, 2)])
    with pytest.raises(ValueError, match="heads"):
        spp.submit_tta([(_nest(p[0], lambda t: t.half()), *p[1:]) for p in passes])
    with pytest.raises(ValueError, match="one dtype"):
        spp.submit_tta([passes[0], passes[1], (_nest(passes[2][0], lambda t: t.half()), *passes[2][1:])])
    with pytest.raises(ValueError, match="images per rank"):
        spp.submit_tta(_v5_passes(3, 320, "dense", 7))
    with pytest.raises(ValueError, match="head shapes"):
        spp.submit_tta([(h, 320, 320, s, f) for h, _, _, s, f in _v5_passes(4, 256, "dense", 7)])
    with pytest.raises(ValueError):
        spp.submit_tta([])
    spp.submit_tta(passes)   # the processor still works after the refusals
    spp.close()
    plain = _sharded("yolov5", hyp, 4, 320, 320, lanes=2)
    plain.submit(passes[0][0])
    with pytest.raises(ValueError, match="submit"):
        plain.submit_tta(passes)
    plain.close()


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_every_rank_holds_every_ranks_tta_rows(mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    port = 29950 + os.getpid() % 300 + (7 if mode == "nccl" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mgpu_tta_worker.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_TTA_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
