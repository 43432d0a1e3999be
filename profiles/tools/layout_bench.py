"""Channels-last (NHWC) heads read natively vs contiguous NCHW heads vs today's copy path, on the fused path
(ShardedPostProcessor, world 1, default lanes).

Arms, on the same seeded heads (synth.make_heads, then the arm's dtype):
  nchw    contiguous heads, read natively
  nhwc    the same values in channels-last memory (torch.channels_last; YOLOX: the 5-D view of a channels-last conv
          output), read natively through the filter kernel's rows path
  copy    the channels-last heads through engine.native_heads without a family -> normalise_heads (a float32, contiguous
          copy), then the float32 NCHW run: what a channels-last model cost before the engine read that layout
Before timing, rows and counts of every arm are checked bit for bit against nchw at the timed size; any difference aborts.
Arms alternate in one process for --rounds rounds; every arm cycles over two head sets so that consecutive steps never find
their heads in L2.  Plain launches (no CUDA graphs): the copy arm allocates new tensors every step.

Per config and arm: ms/step, images/s, and for nchw / nhwc the filter kernel alone and the selection/NMS kernel alone
(CUDA events around single launches).  The card's name and power limit are read in the same run.

Usage: python profiles/tools/layout_bench.py --out r4_layout_bench.json [--steps 200] [--rounds 3]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from yoloseries_b200 import _lib, synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import flatten_heads, head_layout, native_heads  # noqa: E402

CONFIGS = {   # name: (family, img, batch)
    "c2_yolov5s_640_b64": ("yolov5", 640, 64),
    "c3_yolox_640_b256": ("yolox", 640, 256),
    "c5_yolov5x_1280_b16": ("yolov5", 1280, 16),
    "yolov8_640_b64": ("yolov8", 640, 64),
    "fcos_640_b256": ("fcos", 640, 256),
}
DTYPES = {"float32": torch.float32, "float16": torch.float16}
ARMS = ("nchw", "nhwc", "copy")
C = 80


def nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(nest(v, fn) for v in x)


def to_nhwc(t):
    if t.dim() == 4:
        return t.contiguous(memory_format=torch.channels_last)
    b, A, K, H, W = t.shape   # YOLOX (b, A, 5+C, H, W): the view of a channels-last (b, A*(5+C), H, W) conv output
    return t.reshape(b, A * K, H, W).contiguous(memory_format=torch.channels_last).view(b, A, K, H, W)


class Arm:
    def __init__(self, family, img, batch, hyp, sets, convert):
        self.sets, self.convert, self.batch, self.family = sets, convert, batch, family
        anchors = torch.tensor(synth.V5_ANCHORS_PX) if family == "yolov5" else None
        self.spp = ShardedPostProcessor(family, hyp, batch, img, img, anchors=anchors, graph=False)
        self.stream = torch.cuda.current_stream()

    def step(self, k, events=None):
        h = self.sets[k % len(self.sets)]
        if self.convert:   # today's channels-last user: native_heads(h) copies to contiguous float32
            return self.spp.submit(native_heads(h), events=events)
        return self.spp.submit(h, events=events, sync_input=False)

    def rows(self, k):
        self.spp.drain()
        lane = self.step(k)
        rows, cnt = self.spp.gathered(lane)
        torch.cuda.synchronize()
        return rows.clone(), cnt.clone()

    def measure(self, steps, warmup):
        for k in range(max(warmup, self.spp.lanes + 2)):
            self.step(k)
        self.spp.drain()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for st in self.spp.streams:
            st.wait_stream(self.stream)
        for k in range(steps):
            self.step(k)
        self.spp.drain()
        e1.record(self.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def alone_ms(self, reps=40):
        """Filter kernel alone and selection/NMS kernel alone: one launch at a time on an otherwise idle device."""
        lib, spp = _lib.load(), self.spp
        sl, params = spp._slots[0], spp._ent["params"]
        sp = ctypes.c_void_p(self.stream.cuda_stream)
        flats = [flatten_heads(self.family, h) for h in self.sets]
        ptrs = [_lib.head_pointer_array(f) for f in flats]
        tf, tn = [], []
        for k in range(reps):
            f, pa = flats[k % 2], ptrs[k % 2]
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(self.stream)
            _lib.check(lib.ysb_filter_candidates(ctypes.byref(params), pa, len(f), sl["keys"].data_ptr(), spp._key_cap,
                                                 sl["counts"].data_ptr(), sp), "ysb_filter_candidates")
            e[1].record(self.stream)
            _lib.check(lib.ysb_select_nms(ctypes.byref(params), pa, len(f), sl["keys"].data_ptr(), spp._key_cap,
                                          sl["counts"].data_ptr(), sl["rows"].data_ptr(), sl["idx"].data_ptr(),
                                          sl["cnt"].data_ptr(), sp), "ysb_select_nms")
            e[2].record(self.stream)
            torch.cuda.synchronize()
            if k >= 4:
                tf.append(e[0].elapsed_time(e[1]))
                tn.append(e[1].elapsed_time(e[2]))
        return statistics.mean(tf), statistics.mean(tn), float(sl["counts"][:, 0].float().mean())

    def close(self):
        self.spp.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--dtypes", default=",".join(DTYPES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("layout_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    rec = {"gpu": smi[0] if smi else None, "steps": args.steps, "rounds": args.rounds, "cuda_graphs": False, "configs": {}}
    for name in args.configs.split(","):
        family, img, batch = CONFIGS[name]
        hyp = synth.map_profile_hyp(num_class=C)
        for dname in args.dtypes.split(","):
            dtype = DTYPES[dname]
            nchw = [nest(synth.make_heads(family, batch, img, img, C, "dense", seed=1234 + s, device=dev),
                         lambda t: t.to(dtype).contiguous()) for s in range(2)]
            nhwc = [nest(h, to_nhwc) for h in nchw]
            assert head_layout(family, flatten_heads(family, nhwc[0])) == _lib.INPUT_RAW_HEADS_NHWC
            sets = {"nchw": nchw, "nhwc": nhwc, "copy": nhwc}
            arms = {a: Arm(family, img, batch, hyp, sets[a], a == "copy") for a in ARMS}
            # ---- outputs: bit-identical at the timed size, or no timing ----------------------------------------------
            for k in range(2):
                wr, wc = arms["nchw"].rows(k)
                valid = torch.arange(wr.shape[2], device=dev)[None, None, :] < wc[..., None]   # slots past a count are stale
                for a in ("nhwc", "copy"):
                    gr, gc = arms[a].rows(k)
                    if not (torch.equal(gc, wc) and torch.equal(gr.view(torch.int32)[valid], wr.view(torch.int32)[valid])):
                        raise SystemExit(f"{name} {dname}: arm {a} differs from the NCHW run (set {k})")
            # ---- timing: arms alternate, several rounds ------------------------------------------------------------
            ms = {a: [] for a in ARMS}
            for _ in range(args.rounds):
                for a in ARMS:
                    ms[a].append(arms[a].measure(args.steps, args.warmup))
            out = {"family": family, "img": img, "batch": batch, "dtype": dname, "dist": "dense",
                   "candidates_per_image": arms["nchw"].spp._ent["N"], "arms": {}}
            for a in ARMS:
                step = statistics.median(ms[a])
                out["arms"][a] = {"ms_per_step_rounds": ms[a], "ms_per_step": step, "images_per_s": batch / (step * 1e-3),
                                  "lanes": arms[a].spp.lanes}
                if a != "copy":
                    f_alone, n_alone, m = arms[a].alone_ms()
                    out["arms"][a].update(filter_alone_ms=f_alone, nms_alone_ms=n_alone, survivors_per_image=m)
            for a in ARMS:
                arms[a].close()
            del arms, sets, nchw, nhwc
            torch.cuda.empty_cache()
            rec["configs"][f"{name}_{dname}"] = out
            print(name, dname, json.dumps({a: round(out["arms"][a]["images_per_s"]) for a in ARMS}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"]}))


if __name__ == "__main__":
    main()
