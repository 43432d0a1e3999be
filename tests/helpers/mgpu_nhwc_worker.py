"""torchrun worker: channels-last heads through ShardedPostProcessor.submit / submit_tta (P2P detection gather or its NCCL
fallback) vs each rank's own PostProcessor run on the same values in contiguous memory, exchanged with a plain NCCL
all-gather.  Exit code 0 = every rank holds every rank's rows, bit for bit."""
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


def nhwc(heads):
    return type(heads)(t.contiguous(memory_format=torch.channels_last) for t in heads)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    mode = sys.argv[1] if len(sys.argv) > 1 else "p2p"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    hyp = synth.map_profile_hyp(num_class=80)
    anchors = torch.tensor(synth.V5_ANCHORS_PX)
    ok = True
    for tta, batch, graph, img in ((False, 8, True, 320), (False, 5, False, 320), (True, 8, True, 320)):
        spp = ShardedPostProcessor("yolov5", hyp, batch, img, img, anchors=anchors, lanes=3, gather=mode, graph=graph)
        assert spp.mode == mode, (spp.mode, getattr(spp, "_p2p_error", None))
        pp = PostProcessor("yolov5", hyp, anchors=anchors)
        for step in range(7):   # more steps than lanes: slots are reused, flow control is exercised
            if step % 3 != 1:   # every third step reuses the previous head tensors (graph replay)
                heads = [synth.make_heads("yolov5", batch, img, img, 80, "crowd", 100 * step + 10 * k + rank, dev)
                         for k in range(3 if tta else 1)]
                cl = [nhwc(h) for h in heads]
            if tta:
                t = spp.submit_tta([(c, img, img, s, f) for c, s, f in zip(cl, SCALES, FLIPS)])
                loc = pp.run_tta([(h, img, img, s, f) for h, s, f in zip(heads, SCALES, FLIPS)], (img, img))
            else:
                t = spp.submit(cl[0])
                loc = pp.run(heads[0], img, img)
            rows, cnt = spp.gathered(t)
            rows, cnt = rows.clone(), cnt.clone()
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
                    print(f"[rank {rank}] MISMATCH tta={tta} batch={batch} step={step} from rank {r}: counts {same_c} rows {same_r}", flush=True)
        assert len(spp.result(t)) == world * batch
        spp.check()
        spp.close()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_NHWC_OK" if flag.item() else "MGPU_NHWC_FAILED", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
