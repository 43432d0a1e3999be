"""torchrun worker: match() + MatchStats through ShardedPostProcessor (P2P detection gather or its NCCL fallback) with
uneven partial steps.  Every rank matches all images of every step against the same ground truth (generated from a
seed, as every rank of a YOLO validation run holds all labels); its arrays must equal compute_tp over the step's
result() images computed by a single process, the same on every rank.  Exit code 0 = all of that holds on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor, shard_bounds  # noqa: E402
from yoloseries_b200.utils.mAP import MatchStats, compute_tp_batch  # noqa: E402
from test_gpu_match import make_targets  # noqa: E402

B, IMG = 8, 320


def counts(step, rank, world):
    """Full steps, a step whose counts differ per rank, the tail of a dataset split with shard_bounds (5 images)."""
    plan = [B, (3 + 5 * rank) % (B + 1), B, B, shard_bounds(5, rank, world)]
    n = plan[step]
    return n[1] - n[0] if isinstance(n, tuple) else n


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    mode = sys.argv[1] if len(sys.argv) > 1 else "p2p"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=80)
    ok = True
    for graph in (True, False):
        spp = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=torch.tensor(synth.V5_ANCHORS_PX), lanes=2,
                                   gather=mode, graph=graph)
        assert spp.mode == mode, (spp.mode, getattr(spp, "_p2p_error", None))
        stats = MatchStats()
        want = [[], [], [], []]
        for step in range(5):
            n = counts(step, rank, world)
            x = [h[:n] for h in synth.make_heads("yolov5", B, IMG, IMG, 80, "crowd", 1000 * step + 10 * rank, dev)]
            t = spp.submit(x, partial=n < B)
            rows = [np.zeros((0, 6), np.float32) if r is None else r.numpy() for r in spp.result(t)]
            assert len(rows) == sum(counts(step, r, world) for r in range(world))
            targets = make_targets(rows, 77 + step, np.float64 if step == 3 else np.float32)
            stats.add(spp.match(t, targets))
            tps = compute_tp_batch(targets, rows)
            want[0] += tps
            want[1] += [p[:, 4] for p in rows]
            want[2] += [p[:, 5] for p in rows]
            want[3] += [np.asarray(g, np.float64)[:, 4] for g in targets]
        got = stats.arrays()
        for name, a, w in zip(("tp", "conf", "pred_cls", "target_cls"), got, want):
            w = np.concatenate(w)
            if a.shape != w.shape or not np.array_equal(a, w):
                ok = False
                print(f"[rank {rank}] MISMATCH graph={graph} {name}: {a.shape} vs {w.shape}", flush=True)
        # every rank holds the same arrays
        digest = torch.tensor([float(got[0].sum()), float(got[1].astype(np.float64).sum()), float(got[3].sum()),
                               float(len(got[1]))], dtype=torch.float64, device=dev)
        lo, hi = digest.clone(), digest.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        if not torch.equal(lo, hi):
            ok = False
            print(f"[rank {rank}] ranks disagree: {digest.tolist()}", flush=True)
        try:
            spp.check()
        except RuntimeError as e:
            ok = False
            print(f"[rank {rank}] {e}", flush=True)
        spp.close()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_MATCH_OK" if flag.item() else "MGPU_MATCH_FAILED", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
