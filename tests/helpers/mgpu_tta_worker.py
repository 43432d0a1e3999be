"""torchrun worker: test-time-augmented batches through ShardedPostProcessor.submit_tta (P2P detection gather or its NCCL
fallback) vs each rank's own PostProcessor.run_tta rows exchanged with a plain NCCL all-gather.  Exit code 0 = every rank
holds every rank's rows, bit for bit."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from yoloseries_b200 import synth  # noqa: E402
from yoloseries_b200.dist import ShardedPostProcessor  # noqa: E402
from yoloseries_b200.engine import PostProcessor  # noqa: E402

SCALES, FLIPS = (1, 0.83, 0.67), (None, 2, 3)   # test_time_augmentation, trainer/eval_yolov5.py:158-168


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    mode = sys.argv[1] if len(sys.argv) > 1 else "p2p"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=80)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    ok = True
    for batch, dname, graph, img in ((8, "crowd", True, 320), (5, "dense", False, 320), (8, "dense", True, 640)):
        spp = ShardedPostProcessor("yolov5", hyp, batch, img, img, anchors=anchors, lanes=3, gather=mode, graph=graph)
        assert spp.mode == mode, (spp.mode, getattr(spp, "_p2p_error", None))
        pp = PostProcessor("yolov5", hyp, anchors=anchors)
        for step in range(7):   # more steps than lanes: slots are reused, flow control is exercised
            # every third step reuses the previous head tensors (graph replay), the others allocate new ones (capture)
            if step % 3 != 1:
                passes = [(synth.make_heads("yolov5", batch, img, img, 80, dname, 100 * step + 10 * k + rank, dev), img, img,
                           s, f) for k, (s, f) in enumerate(zip(SCALES, FLIPS))]
            t = spp.submit_tta(passes)
            rows, cnt = spp.gathered(t)
            rows, cnt = rows.clone(), cnt.clone()
            loc = pp.run_tta(passes, (img, img))
            want_rows = [torch.empty_like(loc.dets) for _ in range(world)]
            want_cnt = [torch.empty_like(loc.det_cnt) for _ in range(world)]
            dist.all_gather(want_rows, loc.dets.contiguous())
            dist.all_gather(want_cnt, loc.det_cnt.contiguous())
            for r in range(world):
                c = want_cnt[r]
                same_c = torch.equal(cnt[r], c)
                same_r = all(torch.equal(rows[r, i, :max(int(c[i]), 0)], want_rows[r][i, :max(int(c[i]), 0)]) for i in range(batch))
                if not (same_c and same_r):
                    ok = False
                    print(f"[rank {rank}] MISMATCH batch={batch} dist={dname} step={step} from rank {r}: counts {same_c} rows {same_r}", flush=True)
        lst = spp.result(t)
        assert len(lst) == world * batch
        spp.check()
        spp.close()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_TTA_OK" if flag.item() else "MGPU_TTA_FAILED", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
