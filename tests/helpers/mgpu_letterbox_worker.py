"""torchrun worker: ShardedPostProcessor.submit / submit_tta with each rank's own letterbox ``info`` (P2P detection gather or
its NCCL fallback) vs each rank's PostProcessor.run / run_tta with the same ``info``, exchanged with a plain NCCL
all-gather.  Exit code 0 = every rank holds every rank's rows in that rank's original-picture pixels, bit for bit.

Odd ranks read every batch right after submitting it.  Even ranks submit all batches back to back and read only the last
``lanes`` of them, so their lanes queue up behind the gather's flow control while their host keeps uploading tables: a
letterbox staging buffer overwritten before its previous copy ran would show up as wrongly mapped rows on the odd ranks.
Every rank submits the same sequence of batches."""
import os
import random
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import PostProcessor  # noqa: E402

SCALES, FLIPS = (1, 0.83, 0.67), (None, 2, 3)   # test_time_augmentation, trainer/eval_yolov5.py:158-168
LANES = 3
STEPS = 4 * LANES


def make_info(batch, img, seed):
    rnd = random.Random(seed)
    out = []
    for _ in range(batch):
        scale = rnd.choice([0.25, 0.5, 0.731, 1.0, 1.6]) * rnd.uniform(0.9, 1.1)
        top, left = rnd.choice([(0, rnd.randint(0, 60)), (rnd.randint(0, 60), 0)])
        org_h = max(8, int((img - 2 * top) / scale) - rnd.randint(0, 40))
        org_w = max(8, int((img - 2 * left) / scale) - rnd.randint(0, 40))
        out.append(dict(scale=scale, pad_top=top, pad_left=left, org_shape=(org_h, org_w)))
    return out


def gathered_reference(loc, world):
    rows = [torch.empty_like(loc.dets) for _ in range(world)]
    cnt = [torch.empty_like(loc.det_cnt) for _ in range(world)]
    dist.all_gather(rows, loc.dets.contiguous())
    dist.all_gather(cnt, loc.det_cnt.contiguous())
    return rows, cnt


def same(rows, cnt, want, world, batch):
    """Per source rank: (counts equal, rows equal)."""
    want_rows, want_cnt = want
    out = []
    for r in range(world):
        c = want_cnt[r]
        out.append((torch.equal(cnt[r], c),
                    all(torch.equal(rows[r, i, :max(int(c[i]), 0)].view(torch.int32),
                                    want_rows[r][i, :max(int(c[i]), 0)].view(torch.int32)) for i in range(batch))))
    return out


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    mode = sys.argv[1] if len(sys.argv) > 1 else "p2p"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=80)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    ok = True
    reads_ahead = rank % 2 == 0
    for tta, batch, graph, img in ((False, 8, True, 320), (False, 5, False, 320), (True, 8, True, 320)):
        spp = ShardedPostProcessor("yolov5", hyp, batch, img, img, anchors=anchors, lanes=LANES, gather=mode, graph=graph)
        assert spp.mode == mode, (spp.mode, getattr(spp, "_p2p_error", None))
        pp = PostProcessor("yolov5", hyp, anchors=anchors)
        # two head sets per rank: a lane meets the same heads every 2 * LANES steps (graph replay with a new table)
        sets = [[synth.make_heads("yolov5", batch, img, img, 80, "crowd", 100 * s + 10 * k + rank, dev) for k in range(3)]
                for s in range(2)]
        steps = []
        for step in range(STEPS):
            heads = sets[step % 2]
            # each rank decides per batch; now and then one sends its rows unmapped
            info = None if (step + rank) % 5 == 4 else make_info(batch, img, 1000 * rank + step)
            if tta:
                passes = [(h, img, img, s, f) for h, s, f in zip(heads, SCALES, FLIPS)]
                loc = pp.run_tta(passes, (img, img), info=info)
            else:
                passes = heads[0]
                loc = pp.run(passes, img, img, info=info)
            steps.append((passes, info, gathered_reference(loc, world)))   # every rank's collectives in the same order
        tickets = []
        for step, (passes, info, want) in enumerate(steps):
            t = spp.submit_tta(passes, info=info) if tta else spp.submit(passes, info=info)
            tickets.append(t)
            if not reads_ahead:
                rows, cnt = spp.gathered(t)
                for r, (sc, sr) in enumerate(same(rows, cnt, want, world, batch)):
                    if not (sc and sr):
                        ok = False
                        print(f"[rank {rank}] MISMATCH tta={tta} batch={batch} step={step} from rank {r}: counts {sc} "
                              f"rows {sr}", flush=True)
        if reads_ahead:
            for step in range(STEPS - LANES, STEPS):
                rows, cnt = spp.gathered(tickets[step])
                for r, (sc, sr) in enumerate(same(rows, cnt, steps[step][2], world, batch)):
                    if not (sc and sr):
                        ok = False
                        print(f"[rank {rank}] MISMATCH tta={tta} batch={batch} step={step} from rank {r}: counts {sc} "
                              f"rows {sr}", flush=True)
        assert len(spp.result(tickets[-1])) == world * batch
        spp.check()
        spp.close()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_LETTERBOX_OK" if flag.item() else "MGPU_LETTERBOX_FAILED", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
