"""Test-time-augmented batches: PostProcessor.run_tta one after the other vs ShardedPostProcessor.submit_tta.

Workload: YOLOv5s 640x640, 80 classes, dense synthetic heads, the evaluator's three passes (scale 1 / 0.83 / 0.67, flip
none / along h / along w; scale_img pads every pass back to 640x640, so each has 25 200 candidates).
Arms, per (batch per rank, head dtype):
  run_tta      (a) PostProcessor.run_tta back to back on one stream -- the one TTA path before submit_tta
  submit_tta   (b) ShardedPostProcessor.submit_tta, world 1, default lanes, CUDA graphs as default (batch <= 16)
  sharded_wN   (c) (b) at world N under torch.distributed.run, one rank per GPU (only when >= 2 GPUs are visible)
Every arm cycles over two head sets (three passes each) that together exceed the 126 MB L2.  Before timing, rows and
counts of (a) and (b) are checked bit for bit on both head sets at the timed size; a difference aborts.  (a) and (b)
alternate for --rounds rounds; the median round is reported.

Usage: python profiles/tools/tta_shard_bench.py --out r3_tta_shard_bench.json [--steps 100] [--rounds 3]
"""
import argparse
import json
import os
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
SCALES, FLIPS = (1, 0.83, 0.67), (None, 2, 3)   # trainer/eval_yolov5.py:158-168
DTYPES = {"float32": torch.float32, "float16": torch.float16}


def copy_peak_gbs(dev):
    """Device-to-device copy of 4 GiB (read + write bytes over event time): the attainable HBM rate of this card."""
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 10 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def head_sets(batch, dtype, dev, seed):
    """Two sets of three passes [(heads, h, w, scale, flip), ...]."""
    out = []
    for s in range(2):
        passes = []
        for k, (sc, fl) in enumerate(zip(SCALES, FLIPS)):
            heads = [t.to(dtype) for t in synth.make_heads("yolov5", batch, IMG, IMG, C, "dense", seed + 10 * s + k, dev)]
            passes.append((heads, IMG, IMG, sc, fl))
        out.append(passes)
    return out


def set_bytes(passes):
    return sum(t.numel() * t.element_size() for p in passes for t in p[0])


def timed(stream, fn, steps, drain=None, lanes=()):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for st in lanes:
        st.wait_stream(stream)
    for k in range(steps):
        fn(k)
    if drain:
        drain()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


class RunTTA:
    def __init__(self, hyp, sets):
        self.pp, self.sets = PostProcessor("yolov5", hyp, anchors=torch.tensor(synth.V5_ANCHORS_PX)), sets

    def step(self, k):
        return self.pp.run_tta(self.sets[k % 2], (IMG, IMG))

    def rows(self, k):
        out = self.step(k)
        torch.cuda.synchronize()
        return out.dets.clone(), out.det_cnt.clone()

    def measure(self, steps, warmup):
        for k in range(warmup):
            self.step(k)
        return timed(torch.cuda.current_stream(), self.step, steps)


class SubmitTTA:
    def __init__(self, hyp, batch, sets, group=None):
        self.sets = sets
        self.spp = ShardedPostProcessor("yolov5", hyp, batch, IMG, IMG, anchors=torch.tensor(synth.V5_ANCHORS_PX), group=group)

    def step(self, k):
        return self.spp.submit_tta(self.sets[k % 2], sync_input=False)

    def rows(self, k):
        self.spp.drain()
        rows, cnt = self.spp.gathered(self.step(k))
        torch.cuda.synchronize()
        return rows[self.spp.rank].clone(), cnt[self.spp.rank].clone()

    def measure(self, steps, warmup):
        # every (lane, head set) pair once before the clock: graphs are captured there, not in the timed window
        for k in range(max(warmup, 2 * self.spp.lanes + 2)):
            self.step(k)
        self.spp.drain()
        return timed(torch.cuda.current_stream(), self.step, steps, self.spp.drain, self.spp.streams)


def same(a, b):
    (ra, ca), (rb, cb) = a, b
    valid = torch.arange(ra.shape[1], device=ra.device)[None, :] < ca[:, None]   # slots past a count are stale
    return torch.equal(ca, cb) and torch.equal(ra.view(torch.int32)[valid], rb.view(torch.int32)[valid])


def single_gpu(args, dev, peak):
    hyp = synth.map_profile_hyp(num_class=C)
    configs = {}
    for batch in args.batches:
        for dname in args.dtypes:
            dtype = DTYPES[dname]
            sets = head_sets(batch, dtype, dev, 4321)
            a, b = RunTTA(hyp, sets), SubmitTTA(hyp, batch, sets)
            for k in range(2):
                if not same(a.rows(k), b.rows(k)):
                    raise SystemExit(f"b={batch} {dname}: submit_tta rows differ from run_tta (head set {k})")
            ms = {"run_tta": [], "submit_tta": []}
            for _ in range(args.rounds):
                ms["run_tta"].append(a.measure(args.steps, args.warmup))
                ms["submit_tta"].append(b.measure(args.steps, args.warmup))
            logits = batch * 3 * 25200 * C * dtype.itemsize   # class logits the filter kernels read per step
            out = {"batch": batch, "dtype": dname, "passes": 3, "candidates_per_image": 3 * 25200,
                   "head_set_bytes": set_bytes(sets[0]), "head_sets": 2, "class_logit_bytes_per_step": logits,
                   "bit_identical_rows_and_counts": True, "lanes": b.spp.lanes, "cuda_graphs": b.spp.graph, "arms": {}}
            for arm, v in ms.items():
                step = statistics.median(v)
                out["arms"][arm] = {"ms_per_step_rounds": v, "ms_per_step": step, "images_per_s": batch / (step * 1e-3),
                                    "class_logit_read_frac_of_copy_peak": logits / (step * 1e-3) / 1e9 / peak}
            out["speedup_submit_tta_over_run_tta"] = out["arms"]["run_tta"]["ms_per_step"] / out["arms"]["submit_tta"]["ms_per_step"]
            b.spp.close()
            del a, b, sets
            torch.cuda.empty_cache()
            name = f"yolov5s_640_b{batch}_{dname}"
            configs[name] = out
            print(name, json.dumps({k: round(v["images_per_s"]) for k, v in out["arms"].items()}), flush=True)
    return configs


def multi_gpu_worker(args):
    """One rank of arm (c): submit_tta at world N; rank 0 writes the per-config step times to args.part."""
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=C)
    res = {}
    for batch in args.batches:
        for dname in args.dtypes:
            sets = head_sets(batch, DTYPES[dname], dev, 4321 + 1000 * rank)
            arm = SubmitTTA(hyp, batch, sets)
            v = []
            for _ in range(args.rounds):
                dist.barrier()
                v.append(arm.measure(args.steps, args.warmup))
            t = torch.tensor([statistics.median(v)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)   # the slowest rank sets the pace
            res[f"yolov5s_640_b{batch}_{dname}"] = {"world": world, "gather": arm.spp.mode, "lanes": arm.spp.lanes,
                                                     "ms_per_step": float(t.item()),
                                                     "images_per_s": world * batch / (float(t.item()) * 1e-3)}
            arm.spp.close()
            del arm, sets
            torch.cuda.empty_cache()
    if rank == 0:
        with open(args.part, "w") as f:
            json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batches", default="64,8", type=lambda s: [int(x) for x in s.split(",")])
    ap.add_argument("--dtypes", default="float32,float16", type=lambda s: s.split(","))
    ap.add_argument("--part", help=argparse.SUPPRESS)   # set for the torchrun workers of arm (c)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tta_shard_bench.py needs a CUDA device")
    if args.part:
        return multi_gpu_worker(args)
    if not args.out:
        ap.error("--out is required")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    peak = copy_peak_gbs(dev)
    rec = {"gpu": smi[0] if smi else None, "gpus_visible": torch.cuda.device_count(), "copy_peak_gbs": peak,
           "copy_peak_note": "torch device-to-device copy of 4 GiB, read + write bytes over event time, this run",
           "workload": "YOLOv5s 640x640, 80 classes, dense, 3 TTA passes (scale 1/0.83/0.67, flip none/2/3)",
           "steps": args.steps, "rounds": args.rounds, "configs": single_gpu(args, dev, peak)}
    n = torch.cuda.device_count()
    if n >= 2:
        with tempfile.TemporaryDirectory() as d:
            part = os.path.join(d, "part.json")
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                   "127.0.0.1", "--master-port", str(29700 + os.getpid() % 200), os.path.abspath(__file__),
                   "--part", part, "--steps", str(args.steps), "--warmup", str(args.warmup), "--rounds", str(args.rounds),
                   "--batches", ",".join(map(str, args.batches)), "--dtypes", ",".join(args.dtypes)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise SystemExit(f"arm (c) failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
            with open(part) as f:
                for name, v in json.load(f).items():
                    rec["configs"][name]["arms"][f"sharded_w{n}"] = v
    else:
        rec["sharded_multi_gpu"] = f"not measured: {n} GPU visible"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "copy_peak_gbs": round(peak)}))


if __name__ == "__main__":
    main()
