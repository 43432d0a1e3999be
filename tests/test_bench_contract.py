"""bench.py contract on the CPU: the reference arm runs here (it is the CPU baseline) and prints the agreed JSON line;
the product arm refuses to run without a CUDA device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None, timeout=300):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=e, timeout=timeout,
                          capture_output=True, text=True)


def test_reference_arm_prints_the_contract_line():
    from oracle import refharness
    if not refharness.available():
        pytest.skip("the reference arm runs the upstream YOLOSeries sources, which are not part of this repository")
    # a small YOLOX picture keeps the unmodified reference's O(K*M) numba loop at a fraction of a second per image
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--family", "yolox", "--img", "320")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_steps_detections(tmp_path):
    """--dump-outputs writes the rows and counts of the last timed step; the heads are seeded, so the same rows come out
    of a PostProcessor run on heads generated here."""
    import numpy as np
    import torch

    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    r = _run("--batch", "8", "--steps", "3", "--warmup", "1", "--no-extras", "--no-cpu-baseline",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 3
    assert sorted(p.name for p in tmp_path.iterdir()) == ["counts.npy", "rows.npy"]
    rows, counts = np.load(tmp_path / "rows.npy"), np.load(tmp_path / "counts.npy")
    assert rows.dtype == counts.dtype == np.float32 and rows.shape == (1, 8, 300, 6) and counts.shape == (1, 8)
    heads = synth.make_heads("yolov5", 8, 640, 640, 80, "dense", 1234, "cuda:0")
    pp = PostProcessor("yolov5", synth.map_profile_hyp(num_class=80), anchors=torch.tensor(synth.V5_ANCHORS_PX))
    want = pp.to_list(pp.run(heads, 640, 640), as_numpy=True)
    for i, w in enumerate(want):
        assert counts[0, i] == (-1 if w is None else w.shape[0])
        k = 0 if w is None else w.shape[0]
        np.testing.assert_array_equal(rows[0, i, :k], w if k else rows[0, i, :0])
        assert not rows[0, i, k:].any()


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = _run("--steps", "1", "--warmup", "0", timeout=120)
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
