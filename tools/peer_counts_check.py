"""Run under torchrun with >= 2 ranks (one GPU each): the fused count gather of the matcher's last kernel
(PeerCounts: multimem.st through the NVSwitch multicast address, or peer stores) against ncclAllGather."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from linetr_b200 import _native as N, _ops, synthetic as syn
from linetr_b200.engine import PeerCounts, gather_counts

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
P, n0, n1 = 6, 200, 180
ok = True
for multicast in (True, False):
    pc = PeerCounts(P, multicast=multicast)
    for step in range(19):    # > 2 * GATHER_SLOTS: slots and epochs wrap
        thr = 0.3 + 0.1 * ((step + rank) % 5)     # different counts per rank and step
        pairs = [syn.make_descriptor_pair(1000 * rank + 10 * step + i, n0, n1)[:2] for i in range(P)]
        d0 = torch.from_numpy(np.concatenate([a.T for a, _ in pairs], 0).copy()).to(dev)
        d1 = torch.from_numpy(np.concatenate([b.T for _, b in pairs], 0).copy()).to(dev)
        out = _ops.match_descriptors(d0, d1, N.LAYOUT_ROWS, P, thr, True, n0=n0, n1=n1, want_dist=False, gather=pc.publish())
        want = gather_counts(out["counts"], P * world)
        got = pc.collect() if step % 2 == 0 else pc.collect_async().result().to(dev)   # device-side / host-side consumer
        torch.cuda.synchronize()
        if not torch.equal(got, want):
            ok = False
            print(f"rank {rank} multicast={multicast} step {step}: mismatch\n got {got.tolist()}\n want {want.tolist()}", flush=True)
    if rank == 0:
        print(f"multicast requested={multicast} used={pc.multicast}: {'ok' if ok else 'FAILED'}", flush=True)
t = torch.tensor([int(ok)], device=dev)
dist.all_reduce(t, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(t[0]) == 1 else 1)
