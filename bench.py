#!/usr/bin/env python
"""bench.py -- post-processing throughput (images/s) of the B200 engine on BASELINE.json's configs.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  (the UNMODIFIED reference on the host cores)
  python bench.py --config c3|c4|c5 ...                    (the other BASELINE configs; c2 is the default / headline)

A "step" is one pass of the hot path (decode-score + filter + compaction kernel, select + sort + class-aware NMS +
post-filter kernel) over one batch of synthetic head tensors, through yoloseries_b200.dist.ShardedPostProcessor -- the
package's own multi-GPU API: every rank owns `batch` images per step (weak scaling), several batches in flight on
separate CUDA streams, and at N > 1 the NMS kernel stores the kept rows straight into every peer's receive slot over
NVLink (no collective launch).  Headline (c2): YOLOv5s 640x640, 3 levels, 25 200 candidates/image, 80 classes,
conf = cls = 0.001, iou = 0.65, max_det = 300, class-aware, 64 images per GPU per step.

Output: ONE JSON line on rank 0.  Besides the contract keys it carries `distributions` (the same shape on sparse and
crowd inputs), `c2_strong` (BASELINE's "batch 64 sharded over N GPUs" = 64/N images per rank, CUDA-graph path),
`roofline`, `cpu_baseline` (the unmodified reference on one host core), `parity` (fused path vs the reference's rows).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "post-proc images/s (YOLOv5s 640^2, conf=0.001)"
UNIT = "images/s"

CONFIGS = {
    # BASELINE.json configs[1..4]; batch = images per GPU per step
    "c2": dict(family="yolov5", img=640, batch=64, what="configs[1]: YOLOv5s decode+NMS, 64 images/GPU at 640^2"),
    "c3": dict(family="yolox", img=640, batch=256, what="configs[2]: YOLOX-s anchor-free decode (8 400 points), batch 256"),
    "c4": dict(family="retinanet", img=640, batch=64, what="configs[3]: RetinaNet 640^2 (76 725 anchors/image), batch 64"),
    "c5": dict(family="yolov5", img=1280, batch=16, what="configs[4]: YOLOv5x 1280^2 (100 800 candidates/image)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="images per rank per step (default: the config's)")
    ap.add_argument("--family", default="")
    ap.add_argument("--img", type=int, default=0)
    ap.add_argument("--dist", default="dense", choices=["dense", "sparse", "crowd"])
    ap.add_argument("--lanes", type=int, default=0, help="batches in flight per rank, one CUDA stream each (0: the package default -- 4 on one GPU, 6 with peers, 8 for batches below 64 images)")
    ap.add_argument("--graph", type=int, default=-1, help="replay captured CUDA graphs (-1: when batch <= 16)")
    ap.add_argument("--gather", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sparse/crowd/strong-scaling sub-measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's outputs, float32: DIR/rows.npy (world, batch, max_det, 6), slots past "
                         "an image's count zeroed, and DIR/counts.npy (world, batch), -1 = no candidate.  Above 64 MB a "
                         "fixed, seeded sample of k images: rows (k, max_det, 6), counts (k,), their flat image indices "
                         "in DIR/images.npy.  Inputs are seeded: two builds run with the same arguments can be compared "
                         "output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = CONFIGS[args.config]
    args.family = args.family or cfg["family"]
    args.img = args.img or cfg["img"]
    args.batch = args.batch or cfg["batch"]
    return args


def workload_config(args, world, batch=None, dist_name=None):
    batch = batch or args.batch
    return {
        "workload": f"{args.family} {args.img}x{args.img} decode+filter+top-k+class-aware NMS, "
                    f"{batch} images/GPU/step, 80 classes, conf=cls=0.001, iou=0.65, max_det=300, "
                    f"postprocess_bbox=true, distribution={dist_name or args.dist}",
        "baseline_config": CONFIGS[args.config]["what"],
        "images_per_gpu_per_step": batch,
        "global_batch": batch * world,
        "distribution": dist_name or args.dist,
        "parallelism": f"image-sharded x{world}" + (", kept detections all-gathered (rows stored into every peer's slot by the NMS kernel)" if world > 1 else ""),
        "l2": "inputs per step exceed the 126 MB L2 (548 MB at 64 v5s images) and are streamed once per step",
    }


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, rows, counts):
    """Writes what a caller of ShardedPostProcessor.gathered() receives for one step: rows.npy (world, batch, max_det, 6)
    with the slots past each image's count zeroed, and counts.npy (world, batch; -1: no candidate passed the filter), both
    float32.  Beyond DUMP_CAP_BYTES a fixed, seeded sample of the images is written instead, their flat indices in
    images.npy."""
    import numpy as np
    rows, counts = rows.cpu().numpy(), counts.cpu().numpy()
    rows = np.where((np.arange(rows.shape[2]) < counts[..., None])[..., None], rows, np.float32(0))
    os.makedirs(out_dir, exist_ok=True)
    per_image = rows[0, 0].nbytes + 4
    n = counts.size
    if n * per_image > DUMP_CAP_BYTES:
        images = np.sort(np.random.default_rng(0).choice(n, DUMP_CAP_BYTES // per_image, replace=False))
        rows, counts = rows.reshape(n, *rows.shape[2:])[images], counts.reshape(n)[images]
        np.save(os.path.join(out_dir, "images.npy"), images.astype(np.float64))
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float32))
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float32))


def bench_hyp(family="yolov5"):
    from yoloseries_b200 import synth
    hyp = synth.map_profile_hyp(num_class=80)
    if family == "fcos":  # config/train_fcos.yaml:110-116
        hyp.update(cls_threshold=0.2, iou_threshold=0.35, max_predictions_per_img=100)
    return hyp


# ----------------------------------------------------------------------------------------------------------------
# clocks: sampled with NVML while the timed workload is running
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._armed = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            if self._armed.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    r = get_reasons(self.h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(0.01)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def arm(self, on):
        (self._armed.set if on else self._armed.clear)()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


# ----------------------------------------------------------------------------------------------------------------
# CPU legs.  The reference itself (baseline/ref_worker.py: /root/reference or the staged copy baseline/_ref) always
# runs in child processes; the oracle port (oracle/) is the second, labelled figure.
# ----------------------------------------------------------------------------------------------------------------
def port_images_per_second(args, n_images, threads):
    """The C/numpy port (oracle/) of the same algorithm, full greedy loop like the reference: labelled 'port'."""
    from concurrent.futures import ThreadPoolExecutor

    import oracle
    from yoloseries_b200 import synth
    if args.family != "yolov5":
        return None
    oracle.load_library()
    hyp = bench_hyp()
    heads_np = [h.numpy() for h in synth.make_heads("yolov5", n_images, args.img, args.img, 80, args.dist, 4321, "cpu")]

    def one(i):
        dec = oracle.decode_yolov5([h[i:i + 1] for h in heads_np])
        return oracle.evaluator_nms("yolov5", dec, hyp, full_nms=True)

    t0 = time.perf_counter()
    if threads <= 1:
        for i in range(n_images):
            one(i)
    else:
        with ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(one, range(n_images)))
    dt = time.perf_counter() - t0
    return {"value": n_images / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_images} images, C/numpy port of the reference algorithm (oracle/), full greedy NMS loop, {dt:.1f} s"}


def reference_available():
    from oracle import refharness
    return os.path.isdir(os.path.join(refharness.REFERENCE_ROOT, "trainer"))


def run_reference(args):
    """The reference arm: the UNMODIFIED reference's XEvaluator.__call__ (do_inference + numba_nms) on the host cores,
    one single-threaded process per core (the reference is single-threaded), one image per process and step."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if not reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "neither /root/reference nor baseline/_ref (staged copy) is present"}))
        return
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import ref_worker
    procs = os.cpu_count() or 1
    # RetinaNet 640^2 and v5x 1280^2 cost minutes per image on one core: one step is then the whole bounded sample
    res = ref_worker.throughput(args.family, args.img, args.dist, procs, max(args.steps, 1), min(args.warmup, 1), 150.0)
    value = res["images_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": res["steps"],
        "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * res["seconds"] / res["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (+f64 IoU)", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "reference",
                         "sample": f"{procs} images per step (one per single-threaded process, the reference is "
                                   f"single-threaded), {res['steps']} step(s), {res['seconds']:.1f} s; unmodified "
                                   "trainer/eval_*.py XEvaluator.__call__ = do_inference + numba_nms (utils/nms.py:10-27, "
                                   "full greedy loop, truncation to max_det afterwards); numba JIT and imports "
                                   f"({res['setup_s']:.0f} s) outside the timing",
                         "s_per_image_1core": res["s_per_image_1core"], "kept_rows": res["kept_rows"][:4]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:
        port = port_images_per_second(args, procs, procs)
        if port:
            line["cpu_port"] = port
    except Exception as e:  # the port is a courtesy figure
        line["cpu_port"] = {"unavailable": repr(e)}
    print(json.dumps(line))


def reference_children(args, seed=4321):
    """Starts the two 1-image reference runs of the N=1 bench (child processes): mode A (CPU, timed = cpu_baseline) and
    mode B (hyp['device']='cuda', the parity oracle).  Returns a function that waits and returns their npz paths."""
    import tempfile
    tmp = tempfile.mkdtemp(prefix="ysb_bench_ref_")
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    procs = {}
    for mode, dev in (("A", "cpu"), ("B", "cuda")):
        out = os.path.join(tmp, f"{mode}.npz")
        cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_worker.py"), "case", "--family", args.family,
               "--img", str(args.img), "--dist", args.dist, "--batch", "1", "--seed", str(seed), "--device", dev,
               "--out", out]
        # mode A: no GPU visible to the child (the reference's GPUAnchor picks 'cuda' whenever one is, utils/anchor.py:138)
        e = dict(env, CUDA_VISIBLE_DEVICES="") if mode == "A" else env
        procs[mode] = (out, subprocess.Popen(cmd, cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))

    def wait():
        res = {}
        for mode, (out, p) in procs.items():
            try:
                so, se = p.communicate(timeout=900)
            except subprocess.TimeoutExpired:
                p.kill()
                res[mode] = {"error": "timeout"}
                continue
            if p.returncode != 0:
                res[mode] = {"error": se[-400:]}
            else:
                res[mode] = {"npz": out, "timing": json.loads(so.strip().splitlines()[-1])}
        return res
    return wait


def parity_vs_reference(args, npz_path, seed=4321):
    """Fused CUDA path on the same single image the reference child processed; stage-attributed counters."""
    import ast

    import numpy as np
    import torch

    from oracle import parity
    from yoloseries_b200 import synth
    from yoloseries_b200.engine import PostProcessor
    g = dict(np.load(npz_path, allow_pickle=False))
    hyp = bench_hyp(args.family)
    heads = synth.make_heads(args.family, 1, args.img, args.img, 80, args.dist, seed, "cpu")
    heads = [h.cuda() for h in heads] if isinstance(heads, list) else tuple(h.cuda() for h in heads)
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if args.family in ("yolov5", "yolov7") else None
    pp = PostProcessor(args.family, hyp, anchors=anchors)
    dec = pp.decode(heads, args.img, args.img).cpu().numpy()
    rel = np.abs(dec - g["decoded"]) / np.maximum(np.abs(g["decoded"]), 1.0)
    keys, counts = pp.filter_only(heads, args.img, args.img)
    rows, idx = pp.to_list(pp.run(heads, args.img, args.img), as_numpy=True, with_index=True)
    rc = int(g["counts"][0])
    rep = parity.image_report(args.family, hyp, g["decoded"][0], g["rows"][0, :max(rc, 0)], rc,
                              keys.cpu().numpy().view(np.uint64)[0], int(counts[0, 0].item()),
                              rows[0] if rows[0] is not None else np.zeros((0, 6), np.float32),
                              idx[0] if idx[0] is not None else np.zeros((0,), np.int32),
                              -1 if rows[0] is None else rows[0].shape[0])
    out = parity.summarize([rep])
    out["decoded_max_rel_err"] = float(rel.max())
    out["decoded_within_1e-5"] = bool(rel.max() <= 1e-5)
    return out


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes

    import torch
    import torch.distributed as dist

    from yoloseries_b200 import _lib, synth
    from yoloseries_b200.dist import ShardedPostProcessor, bind_to_gpu_numa
    from yoloseries_b200.engine import flatten_heads
    if not os.path.exists(_lib.LIB_PATH):  # fresh checkout: the built library is git-ignored
        if int(os.environ.get("LOCAL_RANK", "0")) == 0:
            from yoloseries_b200 import build as ysb_build
            print("bench.py: libysb_postproc.so missing, building it with nvcc ...", file=sys.stderr)
            ysb_build.build_all()
        else:  # the other ranks wait for rank 0's build (the link is renamed into place atomically)
            deadline = time.time() + 900
            while not os.path.exists(_lib.LIB_PATH) and time.time() < deadline:
                time.sleep(1.0)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the engine has no CPU fallback")
    numa_cores = bind_to_gpu_numa(local)   # before any pinned allocation: staging buffers land on the GPU's NUMA node
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    lib = _lib.load()
    stream = torch.cuda.current_stream()
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if args.family in ("yolov5", "yolov7") else None
    hyp = bench_hyp(args.family)
    graph = None if args.graph < 0 else bool(args.graph)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    class Workload:
        """Heads of one (batch, distribution) resident in HBM + the package's sharded post-processor for them."""

        def __init__(self, batch, dist_name, seed):
            self.batch, self.dist_name = batch, dist_name
            self.heads = synth.make_heads(args.family, batch, args.img, args.img, 80, dist_name, seed, dev)
            self.flat = flatten_heads(args.family, self.heads)
            self.spp = ShardedPostProcessor(args.family, hyp, batch, args.img, args.img, anchors=anchors, lanes=args.lanes or None,
                                            gather=args.gather, graph=graph)

        def fork(self):
            for st in self.spp.streams:
                st.wait_stream(stream)

        def measure(self, steps, warmup, events=False):
            """Exactly `steps` timed steps bracketed by barrier + synchronize; device time, max over ranks."""
            spp = self.spp
            # (with CUDA graphs every lane captures its launch sequence on its second use: all of that stays untimed)
            for _ in range(max(warmup, 3, spp.lanes + 2 if spp.graph else 0)):
                spp.submit(self.heads, sync_input=False)
            spp.drain()
            sync_all()
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)] if events else None
            e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e_beg.record(stream)
            self.fork()
            for k in range(steps):
                self.last_lane = spp.submit(self.heads, events=evs[k] if evs else None, sync_input=False)
            spp.drain()
            e_end.record(stream)
            sync_all()
            spp.check()
            total_ms = max_over_ranks(e_beg.elapsed_time(e_end))
            out = {"total_ms": total_ms, "ms_per_step": total_ms / steps,
                   "images_per_s": world * self.batch * steps / (total_ms * 1e-3)}
            if evs:
                out["filter_ms"] = [e[0].elapsed_time(e[1]) for e in evs]
                out["nms_ms"] = [e[1].elapsed_time(e[2]) for e in evs]
            return out

        def filter_alone_ms(self, reps=50):
            """The dominant kernel by itself (no concurrent NMS kernel), CUDA events around each launch."""
            spp = self.spp
            sl, params = spp._slots[0], spp._ent["params"]
            ptrs = _lib.head_pointer_array(self.flat)
            iso = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(reps)]
            for a, b_ in iso:
                a.record(stream)
                _lib.check(lib.ysb_filter_candidates(ctypes.byref(params), ptrs, len(self.flat), sl["keys"].data_ptr(),
                                                     spp._key_cap, sl["counts"].data_ptr(),
                                                     ctypes.c_void_p(stream.cuda_stream)), "ysb_filter_candidates")
                b_.record(stream)
            torch.cuda.synchronize()
            return statistics.mean(a.elapsed_time(b_) for a, b_ in iso)

        def survivors(self):
            return float(self.spp._slots[0]["counts"][:, 0].float().mean().item())

        def kept(self):
            rows, cnt = self.spp.gathered(0)
            return float(cnt[self.spp.rank].clamp(min=0).float().mean().item())

        def close(self):
            self.spp.close()
            del self.heads, self.flat

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()

    main = Workload(args.batch, args.dist, 1234 + rank)
    main.measure(3, max(args.warmup, 3))   # untimed shake-out: lazy module load, graph capture, peer mappings
    if sampler:
        sampler.arm(True)   # sampled through the timed region and the identical-load hold phase that follows it
    graphed = main.spp.graph
    timed = main.measure(args.steps, args.warmup, events=not graphed)
    total_ms = timed["total_ms"]
    last_out = None
    if args.dump_outputs and rank == 0:
        # copied on the device before the hold steps reuse the lane's buffers; written to disk once the sampler is off
        last_out = [t.clone() for t in main.spp.gathered(main.last_lane)]
        stream.synchronize()
    # Keep the identical load running ~1.5 s so NVML (10 ms period) sees the clocks this workload runs at; the step count
    # is derived from the all-reduced step time, so every rank issues the same sequence.
    hold_steps = int(min(200000, max(100, 1500.0 / max(total_ms / args.steps, 1e-3))))
    hold_steps -= hold_steps % 64
    for i in range(hold_steps):
        main.spp.submit(main.heads, sync_input=False)
        if i % 64 == 63:
            main.spp.drain()
            torch.cuda.synchronize()
    main.spp.drain()
    torch.cuda.synchronize()
    if sampler:
        sampler.arm(False)
    if last_out is not None:
        dump_outputs(args.dump_outputs, *last_out)
        del last_out
    sync_all()
    main.spp.check()
    iso_ms = main.filter_alone_ms()
    m_mean = main.survivors()
    kept_mean = main.kept()
    iso_per_rank = [iso_ms]
    if world > 1:
        tt = torch.tensor([iso_ms], dtype=torch.float64, device=dev)
        allv = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allv, tt)
        iso_per_rank = [float(x) for x in allv.tolist()]

    # ---- end to end through the public API: pinned host heads -> H2D -> kernels (-> peers) -> D2H of rows + counts ----
    spp = main.spp
    n_buf = min(2, spp.lanes)
    host_heads = [torch.empty(t_.shape, dtype=t_.dtype, pin_memory=True).copy_(t_) for t_ in main.flat]
    dev_bufs = [[torch.empty_like(t_) for t_ in main.flat] for _ in range(n_buf)]
    b_loc, max_det = args.batch, spp.max_det
    host_rows = [torch.empty((b_loc, max_det, 6), dtype=torch.float32, pin_memory=True) for _ in range(n_buf)]
    host_cnt = [torch.empty((b_loc,), dtype=torch.int32, pin_memory=True) for _ in range(n_buf)]
    copy_streams = [torch.cuda.Stream(device=dev) for _ in range(n_buf)]
    read_done = [torch.cuda.Event() for _ in range(n_buf)]

    def rebuild(bufs):
        """the family's head container around flat device tensors"""
        if args.family in ("retinanet", "retinanet_exp"):
            return (bufs[0], bufs[1])
        if args.family == "fcos":
            n = len(bufs) // 3
            return (bufs[:n], bufs[n:2 * n], bufs[2 * n:])
        return list(bufs)

    def e2e_run(steps):
        """Step k: H2D of its heads on copy stream k % 2 (overlaps the kernels and the D2H of step k-1), kernels on the
        package's lane, D2H of this rank's rows + counts; the host waits for step k-1's result while step k is in flight."""
        pending = None
        for k in range(steps):
            j = k % n_buf
            cs = copy_streams[j]
            cs.wait_event(read_done[j])            # the kernels that read this staging buffer two steps ago are done
            with torch.cuda.stream(cs):
                for d, h in zip(dev_bufs[j], host_heads):
                    d.copy_(h, non_blocking=True)
                lane = spp.submit(rebuild(dev_bufs[j]), sync_input=True)
                rows, cnt = spp.gathered(lane)
                host_rows[j].copy_(rows[spp.rank], non_blocking=True)
                host_cnt[j].copy_(cnt[spp.rank], non_blocking=True)
                read_done[j].record(cs)
            if pending is not None:
                read_done[pending].synchronize()   # the caller reads step k-1's rows on the host
            pending = j
        read_done[pending].synchronize()

    e2e_steps = max(4, min(args.steps, 12))
    was_graph = spp.graph
    spp.graph = False      # the staging buffers alternate: plain launches
    e2e_run(2)
    sync_all()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    torch.cuda.synchronize()
    e2e_local_ms = (time.perf_counter() - t0) * 1e3
    sync_all()
    e2e_ms = max_over_ranks(e2e_local_ms)
    spp.graph = was_graph
    spp.check()
    h2d = sum(t_.numel() * 4 for t_ in main.flat)
    d2h = host_rows[0].numel() * 4 + host_cnt[0].numel() * 4
    del dev_bufs, host_heads

    clocks = sampler.stop() if sampler else None

    # ---- the same shape on the other input distributions, and BASELINE's "batch 64 sharded over N GPUs" -----------------
    extras = {}
    if not args.no_extras:
        ex_steps = max(10, min(args.steps, 200))
        if args.family in ("yolov5", "yolov7") and args.dist == "dense":
            dists = {}
            for dname in ("sparse", "crowd"):
                w = Workload(args.batch, dname, 2234 + rank)
                r = w.measure(ex_steps, 3)
                dists[dname] = {"value": r["images_per_s"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": ex_steps,
                                "survivors_per_image": w.survivors(), "kept_per_image": w.kept(),
                                "filter_alone_ms": w.filter_alone_ms(20)}
                w.close()
            extras["distributions"] = dists
        if args.config == "c2" and args.batch == 64:
            per_rank = 64 // world if world > 1 else 8
            if per_rank >= 1 and (world == 1 or 64 % world == 0):
                w = Workload(per_rank, args.dist, 3234 + rank)
                r = w.measure(max(ex_steps, 40), 5)
                extras["c2_strong"] = {
                    "what": ("BASELINE configs[1] as written: global batch 64 sharded over %d GPUs = %d images per rank" % (world, per_rank))
                            if world > 1 else "the 8-images-per-rank shard of configs[1] at 8 GPUs, on one GPU",
                    "images_per_rank": per_rank, "global_batch": per_rank * world, "value": r["images_per_s"], "unit": UNIT,
                    "ms_per_step": r["ms_per_step"], "cuda_graph": bool(w.spp.graph), "lanes": w.spp.lanes}
                w.close()

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        C, N = 80, main.spp._ent["N"]
        # channels the filter kernel must read per candidate: class logits (+ objectness / centerness / conf when the
        # family has one); box channels are not read by it
        n_read_ch = C + (0 if args.family in ("yolov8", "retinanet") else 1)
        algo_bytes = args.batch * (N * n_read_ch * 4 + m_mean * 8)
        # Several batches are in flight, so launches of the dominant kernel overlap each other and the NMS kernels: its
        # average duration over the timed region is the region divided by the launches it contains.
        region_launch_ms = total_ms / args.steps
        achieved = algo_bytes / (region_launch_ms * 1e-3) / 1e9
        kernel = ("k_filter_rows" if args.family in ("yolov7", "retinanet", "retinanet_exp") else
                  "k_filter_planes_v4" if args.family in ("yolov5", "yolox", "yolov8") else "k_filter_planes")
        launches_per_step = 4 if spp.mode == "p2p" else 2
        line = {
            "metric": METRIC, "value": timed["images_per_s"], "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (+f64 IoU test)",
            "data": "synthetic", "config": workload_config(args, world),
            "clocks": clocks,
            "e2e": {"value": world * args.batch * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": "ShardedPostProcessor.submit(heads staged from pinned host memory) -> gathered() -> pinned host rows/counts; "
                           "H2D of step k+1 overlaps the kernels and D2H of step k (two staging buffers)",
                    "numa_bound_cores": numa_cores},
            "gpu_launches": launches_per_step * args.steps,
            "gather": spp.mode, "lanes": spp.lanes, "cuda_graph": bool(graphed),
            "filter_alone_ms_per_rank": [round(x, 5) for x in iso_per_rank],
            "roofline": {"kernel": kernel + " (decode-sigmoid + filter + class pick + compaction)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src, "traffic": None,
                         "traffic_note": "not measurable inside the run; the ncu --set full capture of this kernel is "
                                         "profiles/r2_filter_ncu_raw.txt (dram__bytes_read.sum + dram__bytes_write.sum)",
                         "launch_ms_alone": iso_ms, "achieved_alone": algo_bytes / (iso_ms * 1e-3) / 1e9,
                         "frac_alone": algo_bytes / (iso_ms * 1e-3) / 1e9 / peak,
                         "note": "achieved/frac: algorithmic bytes of the K filter launches / duration of the timed region "
                                 "(launches of consecutive batches overlap each other and the NMS kernels); *_alone: the "
                                 "same kernel timed by itself with CUDA events",
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "bytes_per_image": f"N*{n_read_ch}*4 read + M*8 written = {N * n_read_ch * 4} + {m_mean * 8:.0f}",
                         "launch_ms": region_launch_ms},
            "survivors_per_image": m_mean, "kept_per_image": kept_mean,
        }
        if "filter_ms" in timed:
            line["stages_ms"] = {"filter_compact": statistics.mean(timed["filter_ms"]),
                                 "select_sort_nms": statistics.mean(timed["nms_ms"]),
                                 "filter_p50": statistics.median(timed["filter_ms"]),
                                 "nms_p50": statistics.median(timed["nms_ms"])}
        line.update(extras)
        if not args.no_cpu_baseline and world == 1:
            slow = (args.family, args.img) in (("retinanet", 640), ("retinanet_exp", 640)) or args.img > 640
            if reference_available() and not slow:
                res = reference_children(args)()
                a, b_ = res.get("A", {}), res.get("B", {})
                if "timing" in a:
                    s_img = a["timing"]["decode_s"] + a["timing"]["nms_s"]
                    line["cpu_baseline"] = {
                        "value": 1.0 / s_img, "unit": UNIT, "cores": 1, "kind": "reference",
                        "sample": f"1 image of the same workload, unmodified reference (do_inference {a['timing']['decode_s']:.3f} s + "
                                  f"numba_nms {a['timing']['nms_s']:.1f} s) in a single-threaded child process, numba JIT excluded"}
                else:
                    line["cpu_baseline"] = {"unavailable": a.get("error", "?")}
                par = {}
                for mode, r_ in (("vs_reference_cuda_decode", b_), ("vs_reference_cpu_decode", a)):
                    if "npz" in r_:
                        try:
                            par[mode] = parity_vs_reference(args, r_["npz"])
                        except Exception as e:
                            par[mode] = {"error": repr(e)}
                    else:
                        par[mode] = {"unavailable": r_.get("error", "?")}
                line["parity"] = par
            port = None
            try:
                port = port_images_per_second(args, 2, 1)
            except Exception as e:
                port = {"unavailable": repr(e)}
            if port:
                line["cpu_port"] = port
                if "cpu_baseline" not in line:
                    line["cpu_baseline"] = port
        print(json.dumps(line))
    main.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
