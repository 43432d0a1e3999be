"""Cost of rows in original-picture pixels on the sharded path: ShardedPostProcessor.submit with ``info=None`` vs with
``info`` (a distinct list of letterbox dicts every step: per-lane table upload + the fused undo in the NMS row write).

Workload: YOLOv5s (C2), 80 classes, dense synthetic heads, 640x640.  Configs, per head dtype (float32, float16):
  b64_default  64 images per rank, default lanes (4 at world 1), no CUDA graphs (the default at 64 images)
  b8_graphs    8 images per rank, 8 lanes, CUDA graphs
Arms: none (info=None) and info.  Every arm cycles over head sets that together exceed the 126 MB L2.  Before timing, the
rows, counts and candidate indices of both arms are checked bit for bit against PostProcessor.run(heads, info=...) (and
info=None) on every head set; a difference aborts.  The arms alternate for --rounds rounds, each going first in every
other round; the median round is reported.
With two or more GPUs visible, world N (one rank per GPU, torch.distributed.run) is measured the same way.

Usage: python profiles/tools/letterbox_shard_bench.py --out profiles/r6_letterbox_shard_bench.json [--steps 200]
"""
import argparse
import json
import math
import os
import random
import statistics
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import PostProcessor  # noqa: E402

IMG, C = 640, 80
L2_BYTES = 126 << 20
DTYPES = {"float32": torch.float32, "float16": torch.float16}
CONFIGS = {"b64_default": dict(batch=64, lanes=None, graph=None), "b8_graphs": dict(batch=8, lanes=8, graph=True)}


def head_sets(batch, dtype, dev, seed):
    """Enough head sets to exceed twice the L2 together (at least 2, a power of two so that (lane, set) pairs repeat)."""
    one = [t.to(dtype) for t in synth.make_heads("yolov5", batch, IMG, IMG, C, "dense", seed, dev)]
    nbytes = sum(t.numel() * t.element_size() for t in one)
    n = 1 << max(1, math.ceil(math.log2(2 * L2_BYTES / nbytes)))
    return [one] + [[t.to(dtype) for t in synth.make_heads("yolov5", batch, IMG, IMG, C, "dense", seed + s, dev)]
                    for s in range(1, n)], nbytes


def make_info(batch, seed):
    rnd = random.Random(seed)
    out = []
    for _ in range(batch):
        scale = rnd.uniform(0.2, 1.6)
        top, left = rnd.choice([(0, rnd.randint(0, 100)), (rnd.randint(0, 100), 0)])
        out.append(dict(scale=scale, pad_top=top, pad_left=left,
                        org_shape=(int((IMG - 2 * top) / scale), int((IMG - 2 * left) / scale))))
    return out


class Arm:
    def __init__(self, hyp, batch, sets, infos, lanes, graph, group=None):
        self.sets, self.infos = sets, infos   # infos None: the info=None arm
        self.spp = ShardedPostProcessor("yolov5", hyp, batch, IMG, IMG, anchors=torch.tensor(synth.V5_ANCHORS_PX),
                                        lanes=lanes, graph=graph, group=group)

    def step(self, k):
        info = None if self.infos is None else self.infos[k % len(self.infos)]
        return self.spp.submit(self.sets[k % len(self.sets)], sync_input=False, info=info)

    def measure(self, steps, warmup):
        # every (lane, head set) pair before the clock: graphs are captured there, not in the timed window
        for k in range(max(warmup, 2 * self.spp.lanes * len(self.sets) + 2)):
            self.step(k)
        self.spp.drain()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        cur = torch.cuda.current_stream()
        e0.record(cur)
        for st in self.spp.streams:
            st.wait_stream(cur)
        for k in range(steps):
            self.step(k)
        self.spp.drain()
        e1.record(cur)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps


def check(arm, pp, sets, infos):
    """Both arms' own rows == PostProcessor.run(heads, info=...) bit for bit, on every head set."""
    for k in range(len(sets)):
        info = None if infos is None else infos[k % len(infos)]
        arm.spp.drain()
        t = arm.step(k)
        rows, cnt = arm.spp.gathered(t)
        idx = arm.spp._slots[t]["idx"]
        out = pp.run(sets[k % len(sets)], IMG, IMG, info=info)
        torch.cuda.synchronize()
        r = arm.spp.rank
        valid = torch.arange(rows.shape[2], device=rows.device)[None, :] < out.det_cnt[:, None]
        if not (torch.equal(cnt[r], out.det_cnt) and torch.equal(rows[r].view(torch.int32)[valid], out.dets.view(torch.int32)[valid])
                and torch.equal(idx[valid], out.det_idx[valid])):
            raise SystemExit(f"rows of the {'info' if infos else 'none'} arm differ from PostProcessor.run (head set {k})")


def run_config(name, cfg, dname, dev, args, rank=0, group=None):
    hyp = synth.map_profile_hyp(num_class=C)
    batch = cfg["batch"]
    sets, set_bytes = head_sets(batch, DTYPES[dname], dev, 4321 + 1000 * rank)
    # a distinct dict list for every step of the longest run (warm-up + timed window)
    infos = [make_info(batch, 7919 * rank + s) for s in range(max(args.steps, 2 * 8 * len(sets) + 2) + 1)]
    arms = {"none": Arm(hyp, batch, sets, None, cfg["lanes"], cfg["graph"], group),
            "info": Arm(hyp, batch, sets, infos, cfg["lanes"], cfg["graph"], group)}
    pp = PostProcessor("yolov5", hyp, anchors=torch.tensor(synth.V5_ANCHORS_PX))
    check(arms["none"], pp, sets, None)
    check(arms["info"], pp, sets, infos)
    ms = {a: [] for a in arms}
    for r in range(args.rounds):
        for a in (("none", "info") if r % 2 == 0 else ("info", "none")):   # each arm goes first in every other round
            if group is not None:
                torch.distributed.barrier(group)
            ms[a].append(arms[a].measure(args.steps, args.warmup))
    spp = arms["none"].spp
    out = {"batch": batch, "dtype": dname, "lanes": spp.lanes, "cuda_graphs": spp.graph, "gather": spp.mode,
           "world": spp.world, "head_sets": len(sets), "head_set_bytes": set_bytes,
           "bit_identical_to_PostProcessor_run": True, "arms": {}}
    for a, v in ms.items():
        step = statistics.median(v)
        out["arms"][a] = {"ms_per_step_rounds": v, "ms_per_step": step, "images_per_s": spp.world * batch / (step * 1e-3)}
    out["info_over_none_step_time"] = out["arms"]["info"]["ms_per_step"] / out["arms"]["none"]["ms_per_step"]
    # the same arm's spread across rounds, for comparison with the difference between the arms
    out["none_round_spread"] = (max(ms["none"]) - min(ms["none"])) / statistics.median(ms["none"])
    for arm in arms.values():
        arm.spp.close()
    del arms, sets, pp
    torch.cuda.empty_cache()
    return out


def multi_gpu_worker(args):
    """One rank at world N; the slowest rank's median step sets the pace.  Rank 0 writes the configs to args.part."""
    import torch.distributed as dist
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    res = {}
    for name, cfg in CONFIGS.items():
        for dname in args.dtypes:
            out = run_config(name, cfg, dname, dev, args, rank, dist.group.WORLD)
            for a in out["arms"].values():
                t = torch.tensor([a["ms_per_step"]], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                a["ms_per_step"] = float(t.item())
                a["images_per_s"] = out["world"] * out["batch"] / (a["ms_per_step"] * 1e-3)
            out["info_over_none_step_time"] = out["arms"]["info"]["ms_per_step"] / out["arms"]["none"]["ms_per_step"]
            res[f"{name}_{dname}_w{out['world']}"] = out
    if rank == 0:
        with open(args.part, "w") as f:
            json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--dtypes", default="float32,float16", type=lambda s: s.split(","))
    ap.add_argument("--part", help=argparse.SUPPRESS)   # set for the torchrun workers of world N
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("letterbox_shard_bench.py needs a CUDA device")
    if args.part:
        return multi_gpu_worker(args)
    if not args.out:
        ap.error("--out is required")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    rec = {"gpu": smi[0] if smi else None, "gpus_visible": torch.cuda.device_count(),
           "workload": "YOLOv5s 640x640, 80 classes, dense; ShardedPostProcessor.submit, info=None vs a new info list per step",
           "steps": args.steps, "rounds": args.rounds, "configs": {}}
    for name, cfg in CONFIGS.items():
        for dname in args.dtypes:
            out = run_config(name, cfg, dname, dev, args)
            rec["configs"][f"{name}_{dname}_w1"] = out
            print(name, dname, json.dumps({a: round(v["images_per_s"]) for a, v in out["arms"].items()}),
                  round(out["info_over_none_step_time"], 4), flush=True)
    n = torch.cuda.device_count()
    if n >= 2:
        with tempfile.TemporaryDirectory() as d:
            part = os.path.join(d, "part.json")
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                   "127.0.0.1", "--master-port", str(29800 + os.getpid() % 150), os.path.abspath(__file__), "--part", part,
                   "--steps", str(args.steps), "--warmup", str(args.warmup), "--rounds", str(args.rounds),
                   "--dtypes", ",".join(args.dtypes)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise SystemExit(f"world {n} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
            with open(part) as f:
                rec["configs"].update(json.load(f))
    else:
        rec["multi_gpu"] = f"not measured: {n} GPU visible"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"]}))


if __name__ == "__main__":
    main()
