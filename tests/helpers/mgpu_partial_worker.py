"""torchrun worker: partial steps through ShardedPostProcessor (P2P detection gather or its NCCL fallback).  Ranks hold
different image counts within a step, one step has ranks without images, and there are more steps than lanes.  Every
rank's gathered rows of every rank's present images must equal each rank's own PostProcessor.run (run_tta) rows
exchanged with a plain NCCL all-gather, absent images must read -2, and result() must list exactly the present images.
Exit code 0 = all of that holds on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor, shard_bounds  # noqa: E402
from yoloseries_b200.engine import PostProcessor  # noqa: E402

SCALES, FLIPS = (1, 0.83, 0.67), (None, 2, 3)   # test_time_augmentation, trainer/eval_yolov5.py:158-168
B, IMG = 8, 320


def counts(step, rank, world):
    """Images of ``rank`` in ``step``: full steps, a step whose counts differ per rank (some full, some not), the tail of
    a dataset split with shard_bounds (5 images), a step where only rank 0 has images."""
    plan = [B, (3 + 5 * rank) % (B + 1), B, shard_bounds(5, rank, world), B if rank == 0 else 0, B, B]
    n = plan[step]
    return n[1] - n[0] if isinstance(n, tuple) else n


STEPS = 7


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    mode = sys.argv[1] if len(sys.argv) > 1 else "p2p"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=80)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    assert any(counts(s, r, world) == 0 for s in range(STEPS) for r in range(world))
    ok = True
    for tta, graph in ((False, True), (False, False), (True, True)):
        spp = ShardedPostProcessor("yolov5", hyp, B, IMG, IMG, anchors=anchors, lanes=3, gather=mode, graph=graph)
        assert spp.mode == mode, (spp.mode, getattr(spp, "_p2p_error", None))
        pp = PostProcessor("yolov5", hyp, anchors=anchors)
        for step in range(STEPS):
            n = counts(step, rank, world)
            seed = 1000 * step + 10 * rank
            if tta:
                x = [([t[:n] for t in synth.make_heads("yolov5", B, IMG, IMG, 80, "dense", seed + k, dev)], IMG, IMG, s, f)
                     for k, (s, f) in enumerate(zip(SCALES, FLIPS))]
                t = spp.submit_tta(x, partial=n < B)
                loc = pp.run_tta(x, (IMG, IMG))
            else:
                x = [h[:n] for h in synth.make_heads("yolov5", B, IMG, IMG, 80, "crowd", seed, dev)]
                t = spp.submit(x, partial=n < B)
                loc = pp.run(x, IMG, IMG)
            rows, cnt = spp.gathered(t)
            rows, cnt = rows.clone(), cnt.clone()
            # this rank's rows padded to B images, absent ones marked -2, then exchanged by a plain all-gather
            mine_rows = torch.zeros((B, spp.max_det, 6), dtype=torch.float32, device=dev)
            mine_cnt = torch.full((B,), -2, dtype=torch.int32, device=dev)
            mine_rows[:n] = loc.dets
            mine_cnt[:n] = loc.det_cnt
            want_rows = [torch.empty_like(mine_rows) for _ in range(world)]
            want_cnt = [torch.empty_like(mine_cnt) for _ in range(world)]
            dist.all_gather(want_rows, mine_rows)
            dist.all_gather(want_cnt, mine_cnt)
            for r in range(world):
                c = want_cnt[r]
                same_c = torch.equal(cnt[r], c)
                same_r = all(torch.equal(rows[r, i, :max(int(c[i]), 0)], want_rows[r][i, :max(int(c[i]), 0)])
                             for i in range(B))
                if not (same_c and same_r):
                    ok = False
                    print(f"[rank {rank}] MISMATCH tta={tta} graph={graph} step={step} from rank {r}: counts {same_c} "
                          f"rows {same_r} {cnt[r].tolist()} vs {c.tolist()}", flush=True)
            total = sum(counts(step, r, world) for r in range(world))
            if len(spp.result(t)) != total:
                ok = False
                print(f"[rank {rank}] result() of step {step} has {len(spp.result(t))} entries, expected {total}", flush=True)
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
        print("MGPU_PARTIAL_OK" if flag.item() else "MGPU_PARTIAL_FAILED", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
