"""Cost of the mAP matching step (mAP_v2.compute_tp, val_yolov5.py:388) over a COCO-sized validation run, three ways:

  per_image   the drop-in's mAP_v2.compute_tp once per image (utils.mAP.compute_tp: upload, launch, sync, download)
  batch       ShardedPostProcessor.result() per step, then utils.mAP.compute_tp_batch over the step's images
  device      ShardedPostProcessor.match() + utils.mAP.MatchStats.add() per step, MatchStats.arrays() at the end

Workload: 5000 images, YOLOv5s 640x640, 80 classes, dense synthetic heads, 64 images per step (78 full steps + one
partial step of 8), one GPU (world 1; more GPUs are not run by this script).  Ground truth: a geometric count per
image with mean ~7, at most 100, mostly jittered copies of kept rows.  Each arm's time runs from the first submission
to its final host arrays and ends in a device synchronise (host clock).  The run without any matching ("none": submit
every step, synchronise) gives the step time without match; "device" minus "none" is what match adds.  The arms
alternate for --rounds rounds; medians are reported.  Before timing, the arms' arrays are compared (tp, conf, pred_cls,
target_cls equal); a difference aborts.

Usage: python profiles/tools/match_bench.py --out profiles/r6_match_bench.json [--rounds 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import PostProcessor  # noqa: E402
from yoloseries_b200.utils import mAP  # noqa: E402

IMG, C, B, IMAGES, SETS = 640, 80, 64, 5000, 4


def targets_for(rows, rng):
    out = []
    for p in rows:
        n = min(100, int(rng.geometric(1 / 7.0)) - 1 + int(rng.random() < 0.01) * 60)
        g = np.zeros((n, 5), np.float32)
        for k in range(n):
            if p is not None and len(p) and rng.random() < 0.8:
                src = p[int(rng.integers(0, len(p)))]
                wh = np.maximum(src[2:4] - src[0:2], 1.0)
                g[k, :4] = src[:4] + rng.normal(0, 0.08, 4) * np.concatenate([wh, wh])
                g[k, 4] = src[5]
            else:
                xy = rng.uniform(0, IMG, 2)
                g[k, :4] = np.concatenate([xy, xy + rng.uniform(4, 200, 2)])
                g[k, 4] = float(rng.integers(0, C))
        out.append(g)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    hyp = synth.map_profile_hyp(num_class=C)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    heads = [synth.make_heads("yolov5", B, IMG, IMG, C, "dense", 100 + k, dev) for k in range(SETS)]
    pp = PostProcessor("yolov5", hyp, anchors=anchors)
    rows_of = [PostProcessor.to_list(pp.run(h, IMG, IMG), as_numpy=True) for h in heads]
    steps = [B] * (IMAGES // B) + ([IMAGES % B] if IMAGES % B else [])
    rng = np.random.default_rng(7)
    # per step: its head set and its ground truth (rows of a head set are the same every time it is used)
    plan = [(s % SETS, n, targets_for(rows_of[s % SETS][:n], rng)) for s, n in enumerate(steps)]
    spp = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=anchors)

    def submit(k, n):
        h = heads[k]
        return spp.submit(h if n == B else [t[:n] for t in h], partial=n < B)

    def arm_none():
        for k, n, _ in plan:
            submit(k, n)
        torch.cuda.synchronize()
        return None

    def arm_per_image():
        tp, conf, cls, tcls = [], [], [], []
        for k, n, tg in plan:
            for g, p in zip(tg, spp.result(submit(k, n))):
                p = np.zeros((0, 6), np.float32) if p is None else p.numpy()
                tp.append(mAP.compute_tp(g, p))
                conf.append(p[:, 4]), cls.append(p[:, 5]), tcls.append(g[:, 4].astype(np.float64))
        torch.cuda.synchronize()
        return [np.concatenate(x) for x in (tp, conf, cls, tcls)]

    def arm_batch():
        tp, conf, cls, tcls = [], [], [], []
        for k, n, tg in plan:
            rows = [np.zeros((0, 6), np.float32) if p is None else p.numpy() for p in spp.result(submit(k, n))]
            tp += mAP.compute_tp_batch(tg, rows)
            conf += [p[:, 4] for p in rows]
            cls += [p[:, 5] for p in rows]
            tcls += [g[:, 4].astype(np.float64) for g in tg]
        torch.cuda.synchronize()
        return [np.concatenate(x) for x in (tp, conf, cls, tcls)]

    def arm_device():
        stats = mAP.MatchStats()
        for k, n, tg in plan:
            stats.add(spp.match(submit(k, n), tg))
        out = stats.arrays()
        torch.cuda.synchronize()
        return list(out)

    arms = {"none": arm_none, "per_image": arm_per_image, "batch": arm_batch, "device": arm_device}
    ref = None
    for name in ("per_image", "batch", "device"):   # warm-up + agreement
        got = arms[name]()
        if ref is None:
            ref = got
        for a, b in zip(got, ref):
            if a.shape != b.shape or not np.array_equal(a, b):
                raise SystemExit(f"arm {name} disagrees with per_image")
    arm_none()
    times = {k: [] for k in arms}
    order = list(arms)
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            arms[name]()
            times[name].append(time.perf_counter() - t0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    med = {k: statistics.median(v) for k, v in times.items()}
    res = dict(
        gpu=smi[0] if smi else torch.cuda.get_device_name(0), world=1, images=IMAGES, batch=B, steps=len(steps),
        lanes=spp.lanes, targets=int(ref[3].shape[0]), kept_rows=int(ref[1].shape[0]), rounds=args.rounds,
        seconds_median=med, seconds_all=times,
        ms_per_step={k: 1e3 * v / len(steps) for k, v in med.items()},
        match_ms_per_step_added=1e3 * (med["device"] - med["none"]) / len(steps),
        speedup_vs_per_image={k: med["per_image"] / med[k] for k in ("batch", "device")},
        timing="host clock from the first submission to the final host arrays, ending in torch.cuda.synchronize()",
    )
    spp.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
