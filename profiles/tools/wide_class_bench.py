"""Large class counts on the fused path (ShardedPostProcessor, world 1, default lanes, no CUDA graphs).

Arms (seeded dense heads, synth.make_heads / map_profile_hyp; every input is larger than the 126 MB L2, and every arm
cycles over two head sets):
  yolov5s_640_b16_c1203_{float32,float16}   planes kernels with the wide (11-bit class) sort key
  yolov7_640_b16_c601                        k_filter_rows_wide, narrow key (rows of 606 values)
  yolov7_640_b16_c1203                       k_filter_rows_wide, wide key (rows of 1208 values)
  retinanet_640_b4_c1203                     k_filter_rows_wide on the class rows
  decoded_yolov5_640_b16_c1203               k_filter_rows_wide on the decoded (b, N, 5 + C) tensor (numba_nms seam;
                                             PostProcessor.run(decoded=True), as ShardedPostProcessor takes raw heads)
Before timing, image 0 of every arm is checked against the oracle (oracle.evaluator_nms on ysb_decode's output): rows and
candidate indices bit for bit (RetinaNet boxes to 1e-5); a difference aborts.

Per arm: ms/step and images/s; the filter kernel timed alone (CUDA events around single launches) and its rate over the
head bytes (computed from shapes: every head tensor once, e.g. 25 200 * 1208 * 4 B = 121.8 MB per YOLOv5s image at
C = 1203), as a fraction of the device-to-device copy rate measured in the same run (read + write bytes).  The card's name
and power limit are read in the same run.

Usage: python profiles/tools/wide_class_bench.py --out profiles/r5_wide_class_bench.json [--steps 40] [--rounds 3]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from yoloseries_b200 import _lib, synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import PostProcessor, flatten_heads, make_params  # noqa: E402

ARMS = {   # name: (family, img, batch, C, dtype, decoded)
    "yolov5s_640_b16_c1203_float32": ("yolov5", 640, 16, 1203, torch.float32, False),
    "yolov5s_640_b16_c1203_float16": ("yolov5", 640, 16, 1203, torch.float16, False),
    "yolov7_640_b16_c601": ("yolov7", 640, 16, 601, torch.float32, False),
    "yolov7_640_b16_c1203": ("yolov7", 640, 16, 1203, torch.float32, False),
    "retinanet_640_b4_c1203": ("retinanet", 640, 4, 1203, torch.float32, False),
    "decoded_yolov5_640_b16_c1203": ("yolov5", 640, 16, 1203, torch.float32, True),
}


def nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(nest(v, fn) for v in x)


def copy_rate_gbs(dev):
    """Device-to-device copy of 4 GiB, read + write bytes over event time."""
    a = torch.ones(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
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


def anchors(family):
    return torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None


def check_image0(family, hyp, img, inp, decoded, spp_rows, spp_cnt, spp_idx):
    """Image 0 of the arm's sharded run against the oracle on ysb_decode's output."""
    pp = PostProcessor(family, hyp, anchors=anchors(family))
    one = nest(inp, lambda t: t[:1].contiguous())
    dec = one if decoded else pp.decode(one, img, img)
    want = oracle.evaluator_nms(family, dec.float().cpu().numpy(), hyp)[0]
    c = int(spp_cnt[0])
    if want.rows is None:
        return c == -1
    got = spp_rows[0, :c].cpu().numpy()
    if got.shape != want.rows.shape or not np.array_equal(spp_idx[0, :c].cpu().numpy(), want.cand_index):
        return False
    if family.startswith("retinanet"):
        return np.array_equal(got[:, 4:], want.rows[:, 4:]) and np.allclose(got[:, :4], want.rows[:, :4], rtol=1e-5, atol=1e-5)
    return np.array_equal(got.view(np.uint32), want.rows.view(np.uint32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--arms", default=",".join(ARMS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_class_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    copy = copy_rate_gbs(dev)
    rec = {"gpu": smi[0] if smi else None, "copy_rate_gbs": copy, "steps": args.steps, "rounds": args.rounds,
           "cuda_graphs": False, "arms": {}}
    lib = _lib.load()
    for name in args.arms.split(","):
        family, img, batch, C, dtype, decoded = ARMS[name]
        hyp = synth.map_profile_hyp(num_class=C)
        pp = PostProcessor(family, hyp, anchors=anchors(family))
        sets = []
        for s in range(2):
            h = nest(synth.make_heads(family, batch, img, img, C, "dense", seed=1234 + s, device=dev), lambda t: t.to(dtype).contiguous())
            sets.append(pp.decode(h, img, img) if decoded else h)
            del h
        head_bytes = sum(t.numel() * t.element_size() for t in flatten_heads(family, sets[0])) if not decoded else \
            sets[0].numel() * 4
        stream = torch.cuda.current_stream()
        if decoded:
            spp = None
            submit = (lambda k: pp.run(sets[k % 2], img, img, decoded=True))
            res = submit(0)
            rows, cnt, idx = res.dets[None], res.det_cnt[None], res.det_idx
        else:
            spp = ShardedPostProcessor(family, hyp, batch, img, img, anchors=anchors(family), graph=False)
            submit = (lambda k: spp.submit(sets[k % 2], sync_input=False))
            t = submit(0)
            rows, cnt = spp.gathered(t)
            idx = spp._slots[t]["idx"]
        # ---- image 0 against the oracle -------------------------------------------------------------------------------
        torch.cuda.synchronize()
        if not check_image0(family, hyp, img, sets[0], decoded, rows[0], cnt[0], idx):
            raise SystemExit(f"{name}: image 0 differs from the oracle")
        drain = spp.drain if spp is not None else torch.cuda.synchronize
        drain()
        # ---- end to end ------------------------------------------------------------------------------------------------
        ms = []
        for _ in range(args.rounds):
            for k in range(args.warmup):
                submit(k)
            drain()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for st in (spp.streams if spp is not None else []):
                st.wait_stream(stream)
            for k in range(args.steps):
                submit(k)
            drain()
            e1.record(stream)
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1) / args.steps)
        # ---- the filter kernel alone -----------------------------------------------------------------------------------
        shapes = None if family.startswith("retinanet") else synth.level_shapes(family, img, img)
        params = make_params(family, hyp, batch, img, img, shapes, anchors(family),
                             input_kind=_lib.INPUT_DECODED_ROWS if decoded else _lib.INPUT_RAW_HEADS, head_dtype=dtype)
        n_c = synth.num_candidates(family, img, img)
        keys = torch.empty((batch, n_c), dtype=torch.int64, device=dev)
        counts = torch.empty((batch, 4), dtype=torch.int32, device=dev)
        sp = ctypes.c_void_p(stream.cuda_stream)
        flats = [[s] if decoded else flatten_heads(family, s) for s in sets]
        ptrs = [_lib.head_pointer_array(f) for f in flats]
        tf = []
        for k in range(24):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record(stream)
            _lib.check(lib.ysb_filter_candidates(ctypes.byref(params), ptrs[k % 2], len(flats[k % 2]), keys.data_ptr(),
                                                 n_c, counts.data_ptr(), sp), "ysb_filter_candidates")
            e[1].record(stream)
            torch.cuda.synchronize()
            if k >= 4:
                tf.append(e[0].elapsed_time(e[1]))
        f_ms = statistics.median(tf)
        step = statistics.median(ms)
        rate = head_bytes / (f_ms * 1e-3) / 1e9
        out = {"family": family, "img": img, "batch": batch, "num_class": C, "dtype": str(dtype).replace("torch.", ""),
               "input": "decoded rows" if decoded else "raw heads", "candidates_per_image": n_c,
               "head_bytes_per_image": head_bytes / batch, "ms_per_step_rounds": ms, "ms_per_step": step,
               "images_per_s": batch / (step * 1e-3), "filter_alone_ms": f_ms, "filter_gbs": rate,
               "filter_fraction_of_copy_rate": rate / copy,
               "path": "PostProcessor.run(decoded=True)" if decoded else f"ShardedPostProcessor, {spp.lanes} lanes"}
        if spp is not None:
            spp.close()
        del sets, flats, ptrs, spp, pp, keys, counts
        torch.cuda.empty_cache()
        rec["arms"][name] = out
        print(name, json.dumps({k: round(out[k], 3) for k in ("images_per_s", "filter_alone_ms", "filter_fraction_of_copy_rate")}),
              flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "copy_rate_gbs": round(copy, 1)}))


if __name__ == "__main__":
    main()
