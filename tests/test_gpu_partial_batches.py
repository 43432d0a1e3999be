"""Partial steps through ShardedPostProcessor (submit / submit_tta with partial=True): the images a rank holds give the
rows, counts and candidate indices PostProcessor.run / run_tta gives on the same images, bit for bit; the others read
count -2; full steps before and after a partial one (graph replays included) are unchanged.  With two or more GPUs a
torchrun worker checks the P2P and NCCL gathers with ranks of different image counts."""
import os
import random
import subprocess
import sys

import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, IMG = 8, 320
SEQ = (8, 8, 5, 0, 8, 8)   # images per step; 3 lanes, so partial steps land on lanes that full steps reuse


def _anchors():
    from yoloseries_b200 import synth
    return torch.tensor(synth.V5_ANCHORS_PX)


def _nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(_nest(v, fn) for v in x)


def _channels_last(t):
    return t.contiguous(memory_format=torch.channels_last)


def _heads(seed, dtype=None, channels_last=False):
    from yoloseries_b200 import synth
    h = synth.make_heads("yolov5", B, IMG, IMG, 80, "dense", seed, "cuda")
    if dtype is not None:
        h = _nest(h, lambda t: t.to(dtype))
    if channels_last:
        h = _nest(h, _channels_last)
    return h


def _passes(seed, **kw):
    return [(_heads(seed + k, **kw), IMG, IMG, s, f) for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]


def _first(x, n):
    """The first ``n`` images of heads or TTA passes."""
    if isinstance(x, list) and x and isinstance(x[0], tuple):
        return [(_first(p[0], n), *p[1:]) for p in x]
    return _nest(x, lambda t: t[:n])


def _refill(dst, src):
    """Copy new values into the tensors of ``dst`` in place (a graph replays reads them by address)."""
    if isinstance(dst, torch.Tensor):
        dst.copy_(src)
        return
    for d, s in zip(dst, src):
        _refill(d[0] if isinstance(d, tuple) else d, s[0] if isinstance(s, tuple) else s)


def make_info(n, seed):
    rnd = random.Random(seed)
    out = []
    for _ in range(n):
        scale = rnd.choice([0.25, 0.5, 0.731, 1.0, 1.6]) * rnd.uniform(0.9, 1.1)
        top, left = rnd.choice([(0, rnd.randint(0, 30)), (rnd.randint(0, 30), 0)])
        out.append(dict(scale=scale, pad_top=top, pad_left=left,
                        org_shape=(max(8, int((IMG - 2 * top) / scale) - rnd.randint(0, 20)),
                                   max(8, int((IMG - 2 * left) / scale) - rnd.randint(0, 20)))))
    return out


def _check_step(spp, ticket, want, n):
    """Rows, counts and det_idx of images [0, n) equal the reference's; images [n, B) read -2; result() has n entries."""
    rows, cnt = spp.gathered(ticket)
    idx = spp._slots[ticket]["idx"]
    torch.cuda.synchronize()
    rows, cnt, idx = rows[0].clone(), cnt[0].clone(), idx.clone()
    w_rows, w_cnt, w_idx = want
    assert torch.equal(cnt[:n], w_cnt), (cnt.tolist(), w_cnt.tolist())
    assert (cnt[n:] == -2).all(), cnt.tolist()
    for i in range(n):
        c = max(int(w_cnt[i]), 0)
        assert torch.equal(rows[i, :c].view(torch.int32), w_rows[i, :c].view(torch.int32)), f"image {i}"
        assert torch.equal(idx[i, :c], w_idx[i, :c]), f"image {i} candidate indices"
    res = spp.result(ticket)
    assert len(res) == n
    for i, r in enumerate(res):
        c = int(w_cnt[i])
        assert (r is None) if c < 0 else torch.equal(r, w_rows[i, :c].cpu())


def _run_sequence(tta, graph, with_info, **heads_kw):
    from yoloseries_b200.dist import ShardedPostProcessor
    from yoloseries_b200.engine import PostProcessor
    from yoloseries_b200 import synth
    hyp = synth.map_profile_hyp(num_class=80)
    pp = PostProcessor("yolov5", hyp, anchors=_anchors())
    spp = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=_anchors(), lanes=3, graph=graph)
    make = (lambda s: _passes(s, **heads_kw)) if tta else (lambda s: _heads(s, **heads_kw))
    again = make(10)   # the head tensors of steps 1 and 4 (lane 1 both times): a graph replay after the partial steps
    seen = 0
    for step, n in enumerate(SEQ):
        if step == 1:
            x = again
        elif step == 4:
            _refill(again, make(40))
            x = again
        else:
            x = make(100 * step + 7)
        x = _first(x, n) if n < B else x
        info = make_info(n, step) if with_info else None
        if tta:
            out = pp.run_tta(x, (IMG, IMG), info=info)
            want = (out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone())
            t = spp.submit_tta(x, info=info, partial=n < B)
        else:
            out = pp.run(x, IMG, IMG, info=info)
            want = (out.dets.clone(), out.det_cnt.clone(), out.det_idx.clone())
            t = spp.submit(x, info=info, partial=n < B)
        _check_step(spp, t, want, n)
        seen += int((want[1] > 0).sum())
    assert seen > 0   # some image kept rows: the comparison is not vacuous
    assert spp.mode == "local"
    if graph:   # step 0 warms up, steps 1 and 5 capture, step 4 replays; partial steps never capture
        assert len(spp._graphs) == 2
    else:
        assert not spp._graphs
    spp.close()


@pytest.mark.parametrize("with_info", [False, True])
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("tta", [False, True])
def test_partial_steps_equal_the_single_gpu_run(tta, graph, with_info):
    _run_sequence(tta, graph, with_info)


def test_float16_heads():
    _run_sequence(False, True, False, dtype=torch.float16)


def test_channels_last_heads():
    _run_sequence(False, True, True, channels_last=True)


def test_refusals_leave_the_processor_working():
    from yoloseries_b200 import synth
    from yoloseries_b200.dist import ShardedPostProcessor
    hyp = synth.map_profile_hyp(num_class=80)
    spp = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=_anchors(), lanes=2)
    heads = _heads(3)
    with pytest.raises(ValueError, match="at least one image"):
        spp.submit(_first(heads, 0), partial=True)
    spp.submit(heads)
    nine = [torch.cat([t, t[:1]]) for t in heads]
    with pytest.raises(ValueError, match="at most 8 images per rank"):
        spp.submit(nine, partial=True)
    with pytest.raises(ValueError, match="expected 8 images per rank, got 5"):
        spp.submit(_first(heads, 5))
    with pytest.raises(ValueError, match="info"):
        spp.submit(_first(heads, 5), info=make_info(B, 1), partial=True)
    with pytest.raises(ValueError, match="info"):
        spp.submit(_first(heads, 0), info=make_info(1, 1), partial=True)
    other = synth.make_heads("yolov5", B, 256, 256, 80, "dense", 3, "cuda")   # 256x256 levels on a 320x320 set-up
    with pytest.raises(ValueError, match="head shapes"):
        spp.submit(other)
    with pytest.raises(ValueError, match="head shapes"):
        spp.submit(_first(other, 3), partial=True)
    with pytest.raises(ValueError, match="head shapes"):
        spp.submit(_first(other, 0), partial=True)
    with pytest.raises(ValueError, match="heads"):
        spp.submit(_first(_nest(heads, lambda t: t.half()), 4), partial=True)
    with pytest.raises(ValueError, match="channels-last"):
        spp.submit(_first(_nest(heads, _channels_last), 4), partial=True)
    # still working: a partial and a full step
    for n in (4, B):
        t = spp.submit(_first(heads, n), partial=True)
        assert len(spp.result(t)) == n
    spp.close()
    tta = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=_anchors(), lanes=2)
    passes = _passes(5)
    tta.submit_tta(passes)
    with pytest.raises(ValueError, match="images per rank"):
        tta.submit_tta(_first(passes, 5))
    with pytest.raises(ValueError, match="same images"):
        tta.submit_tta([_first(passes, 5)[0]] + passes[1:], partial=True)
    small = [(synth.make_heads("yolov5", 2, 256, 256, 80, "dense", 3 + k, "cuda"), IMG, IMG, s, f)
             for k, (s, f) in enumerate(zip(oracle.TTA_SCALES, oracle.TTA_FLIPS))]
    with pytest.raises(ValueError, match="head shapes"):
        tta.submit_tta(small, partial=True)
    t = tta.submit_tta(_first(passes, 2), partial=True)
    assert len(tta.result(t)) == 2
    tta.close()


@pytest.mark.parametrize("mode", ["p2p", "nccl"])
def test_ranks_with_different_image_counts(mode):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    port = 29650 + os.getpid() % 300 + (7 if mode == "nccl" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mgpu_partial_worker.py"), mode]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_PARTIAL_OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
