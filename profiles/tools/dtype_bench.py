"""Native float16 / bfloat16 heads vs float32 on the fused path (ShardedPostProcessor, world 1, default lanes).

Arms, on the same seeded heads (synth.make_heads in float32, rounded to 16 bits; the float32 arms get the widened 16-bit
tensors, so every arm computes the same rows):
  f16     float16 heads read natively           bf16    bfloat16 heads read natively
  f32     the widened float16 heads              today   float16 heads -> engine.normalise_heads -> the float32 run
Before timing, rows and counts of every arm are checked bit for bit at the timed size (f16 / today vs f32, bf16 vs a float32
run on the widened bfloat16 heads); any difference aborts.  Arms alternate in one process for --rounds rounds; every arm
cycles over two head sets so that consecutive steps never find their heads in L2.  Plain launches (no CUDA graphs): the
conversion arm allocates new tensors every step.

Per config and arm: ms/step, images/s, the filter kernel alone and the selection/NMS kernel alone (CUDA events around
single launches), the filter's algorithmic bytes and their fraction of the device-to-device copy rate measured in the
same run.  Also: C2 host -> host with pinned heads, and how often the filter kernel's near-tie re-evaluation runs.

Usage: python profiles/tools/dtype_bench.py --out r3_dtype_bench.json [--steps 200] [--rounds 3]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from yoloseries_b200 import _lib, synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import flatten_heads, normalise_heads  # noqa: E402

CONFIGS = {   # name: (family, img, batch)
    "c2_yolov5s_640_b64": ("yolov5", 640, 64),
    "c3_yolox_640_b256": ("yolox", 640, 256),
    "c4_retinanet_640_b64": ("retinanet", 640, 64),
    "c5_yolov5x_1280_b16": ("yolov5", 1280, 16),
    "yolov7_640_b64": ("yolov7", 640, 64),
    "yolov8_640_b64": ("yolov8", 640, 64),
}
ARMS = ("f16", "bf16", "f32", "today")
C = 80


def hyp_for(family):
    return synth.map_profile_hyp(num_class=C)


def nest(x, fn):
    if isinstance(x, torch.Tensor):
        return fn(x)
    return type(x)(nest(v, fn) for v in x)


def copy_peak_gbs(dev):
    """Device-to-device copy of 4 GiB (read + write bytes over event time): the attainable HBM rate of this card."""
    n = 1 << 30
    a = torch.empty(n, dtype=torch.float32, device=dev)
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


def guard_rate(family, flat, hyp):
    """Fraction of the candidates that reach the filter kernel's class decision and take its literal re-evaluation of
    near-tied classes: runner-up logit m2 not below guard_lo = m1 - 8e-6 * (1 + e^m1) (filter_kernels.cu, decide_candidate),
    computed with torch float32 ops on the same values.  The device's expf may differ from torch's by an ulp at the
    band's edge: a count, not a bit-exact replay."""
    reach = hit = total = 0
    for t in (flat[1:] if family.startswith("retinanet") else flat):
        t = t.float()
        if family in ("yolov5", "yolox"):
            v = t.view(t.shape[0], -1, 5 + C, t.shape[-2], t.shape[-1])
            cls, obj = v[:, :, 5:].movedim(2, -1), v[:, :, 4]
        elif family == "yolov7":
            cls, obj = t[..., 5:], t[..., 4]
        elif family == "yolov8":
            cls, obj = t[:, 64:].movedim(1, -1), None
        else:
            cls, obj = t, None
        top = torch.topk(cls, 2, dim=-1).values
        m1, m2 = top[..., 0], top[..., 1]
        e = torch.exp(-m1)
        smax = 1.0 / (1.0 + e)
        p = smax * torch.sigmoid(obj) if obj is not None else smax
        glo = m1 - 8.0e-6 * (1.0 + 1.0 / e)
        glo = torch.where((m1 < -80.0) | ~(p > 1e-30) | torch.isnan(glo), torch.full_like(glo, -float("inf")), glo)
        r = torch.ones_like(m1, dtype=torch.bool)
        if family == "yolov5":   # PRE_OBJ: candidates below conf_threshold leave before the class decision
            r = torch.sigmoid(obj) >= hyp["conf_threshold"]
        reach += int(r.sum())
        hit += int((r & ~(m2 < glo)).sum())
        total += m1.numel()
    return {"reach_decision": reach, "candidates": total, "reevaluated": hit,
            "rate_of_decisions": hit / max(reach, 1), "rate_of_candidates": hit / max(total, 1)}


class Arm:
    def __init__(self, family, img, batch, hyp, sets, convert):
        self.sets, self.convert, self.batch = sets, convert, batch
        anchors = torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None
        self.spp = ShardedPostProcessor(family, hyp, batch, img, img, anchors=anchors, graph=False)
        self.family = family
        self.stream = torch.cuda.current_stream()

    def step(self, k, events=None):
        h = self.sets[k % len(self.sets)]
        if self.convert:   # today's 16-bit user: a torch conversion pass to float32, then the float32 path
            return self.spp.submit(normalise_heads(h), events=events)
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

    def stage_ms(self, steps=60):
        """In-pipeline stage durations (events on the lane: start, filter done, NMS done)."""
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        for k in range(steps):
            self.step(k, events=evs[k])
        self.spp.drain()
        torch.cuda.synchronize()
        return (statistics.mean(e[0].elapsed_time(e[1]) for e in evs[4:]),
                statistics.mean(e[1].elapsed_time(e[2]) for e in evs[4:]))

    def alone_ms(self, reps=40):
        """Filter kernel alone and selection/NMS kernel alone: one launch at a time on an otherwise idle device."""
        lib, spp = _lib.load(), self.spp
        sl, params = spp._slots[0], spp._ent["params"]
        sp = ctypes.c_void_p(self.stream.cuda_stream)
        flats = [flatten_heads(self.family, normalise_heads(h) if self.convert else h) for h in self.sets]
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
        m = float(sl["counts"][:, 0].float().mean())
        return statistics.mean(tf), statistics.mean(tn), m

    def close(self):
        self.spp.close()


def host_to_host(family, img, batch, hyp, h, steps=12):
    """(grid families) Pinned host heads -> H2D (two staging buffers on two copy streams) -> kernels -> D2H of rows + counts."""
    anchors = torch.tensor(synth.V5_ANCHORS_PX) if family in ("yolov5", "yolov7") else None
    spp = ShardedPostProcessor(family, hyp, batch, img, img, anchors=anchors, graph=False)
    flat = flatten_heads(family, h)
    host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in flat]
    bufs = [[torch.empty_like(t) for t in flat] for _ in range(2)]
    hr = [torch.empty((batch, spp.max_det, 6), pin_memory=True) for _ in range(2)]
    hc = [torch.empty((batch,), dtype=torch.int32, pin_memory=True) for _ in range(2)]
    cs = [torch.cuda.Stream() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def run(n):
        pending = None
        for k in range(n):
            j = k % 2
            cs[j].wait_event(done[j])
            with torch.cuda.stream(cs[j]):
                for d, s in zip(bufs[j], host):
                    d.copy_(s, non_blocking=True)
                lane = spp.submit(list(bufs[j]))
                rows, cnt = spp.gathered(lane)
                hr[j].copy_(rows[0], non_blocking=True)
                hc[j].copy_(cnt[0], non_blocking=True)
                done[j].record(cs[j])
            if pending is not None:
                done[pending].synchronize()
            pending = j
        done[pending].synchronize()
    run(3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run(steps)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    spp.close()
    return {"ms_per_step": ms, "images_per_s": batch / (ms * 1e-3), "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in flat)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dtype_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    peak = copy_peak_gbs(dev)
    rec = {"gpu": smi[0] if smi else None, "copy_peak_gbs": peak,
           "copy_peak_note": "torch device-to-device copy of 4 GiB, read + write bytes over event time, this run",
           "steps": args.steps, "rounds": args.rounds, "cuda_graphs": False, "configs": {}}
    for name in args.configs.split(","):
        family, img, batch = CONFIGS[name]
        hyp = hyp_for(family)
        base = [synth.make_heads(family, batch, img, img, C, "dense", seed=1234 + s, device=dev) for s in range(2)]
        guard = {"f32_unrounded": guard_rate(family, flatten_heads(family, base[0]), hyp)}
        sets = {"f16": [nest(h, lambda t: t.half()) for h in base], "bf16": [nest(h, lambda t: t.bfloat16()) for h in base]}
        guard["f16"] = guard_rate(family, flatten_heads(family, sets["f16"][0]), hyp)
        guard["bf16"] = guard_rate(family, flatten_heads(family, sets["bf16"][0]), hyp)
        del base
        sets["f32"] = [nest(h, lambda t: t.float()) for h in sets["f16"]]
        sets["today"] = sets["f16"]
        arms = {a: Arm(family, img, batch, hyp, sets[a], a == "today") for a in ARMS}
        # ---- outputs: bit-identical at the timed size, or no timing --------------------------------------------------
        bf_ref = Arm(family, img, batch, hyp, [nest(h, lambda t: t.float()) for h in sets["bf16"]], False)
        for k in range(2):
            f32 = arms["f32"].rows(k)
            want = {"f16": f32, "today": f32, "bf16": bf_ref.rows(k)}
            for a, (wr, wc) in want.items():
                gr, gc = arms[a].rows(k)
                valid = torch.arange(wr.shape[2], device=dev)[None, None, :] < wc[..., None]   # slots past a count are stale
                if not (torch.equal(gc, wc) and torch.equal(gr.view(torch.int32)[valid], wr.view(torch.int32)[valid])):
                    raise SystemExit(f"{name}: arm {a} differs from the float32 run on its widened heads (set {k})")
        bf_ref.close()
        del bf_ref
        # ---- timing: arms alternate, several rounds ----------------------------------------------------------------
        ms = {a: [] for a in ARMS}
        for _ in range(args.rounds):
            for a in ARMS:
                ms[a].append(arms[a].measure(args.steps, args.warmup))
        N = arms["f32"].spp._ent["N"]
        n_read_ch = C + (0 if family in ("yolov8", "retinanet") else 1)
        out = {"family": family, "img": img, "batch": batch, "candidates_per_image": N, "dist": "dense",
               "guard_band_reevaluation": guard, "arms": {}}
        for a in ARMS:
            f_alone, n_alone, m = arms[a].alone_ms()
            f_stage, n_stage = arms[a].stage_ms()
            esize = 4 if a in ("f32", "today") else 2
            algo = batch * (N * n_read_ch * esize + m * 8)
            step = statistics.median(ms[a])
            out["arms"][a] = {
                "ms_per_step_rounds": ms[a], "ms_per_step": step, "images_per_s": batch / (step * 1e-3),
                "filter_alone_ms": f_alone, "nms_alone_ms": n_alone,
                "filter_stage_ms_in_pipeline": f_stage, "nms_stage_ms_in_pipeline": n_stage,
                "survivors_per_image": m, "filter_algorithmic_bytes": algo,
                "filter_alone_frac_of_copy_peak": algo / (f_alone * 1e-3) / 1e9 / peak,
                "filter_bytes_per_step_frac_of_copy_peak": algo / (step * 1e-3) / 1e9 / peak,
                "lanes": arms[a].spp.lanes,
            }
            if a == "today":
                out["arms"][a]["note"] = ("filter_*: the float32 kernels on the converted heads; the step also reads the "
                                          "16-bit heads and writes their float32 copy in the conversion pass")
        for a in ARMS:
            arms[a].close()
        del arms
        if name.startswith("c2_"):
            out["host_to_host"] = {a: host_to_host(family, img, batch, hyp, sets[a][0]) for a in ("f16", "f32")}
        del sets
        torch.cuda.empty_cache()
        rec["configs"][name] = out
        print(name, json.dumps({a: round(out["arms"][a]["images_per_s"]) for a in ARMS}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "copy_peak_gbs": round(peak)}))


if __name__ == "__main__":
    main()
