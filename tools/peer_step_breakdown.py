#!/usr/bin/env python
"""Run under torchrun (R ranks): where the time of one row-sharded step goes in peer-exchange mode.
Captures the step (ShardedSupConLoss + autograd, exactly bench.py's) as a CUDA graph under several settings and
times 20 replays each (CUDA events, L2 flushed, max over ranks):
  full           the real step
  noz            rows are NOT pushed / waited for (stale z: timing only)  -> full - noz  = exposed z exchange
  nostats        statistics are NOT pushed / waited for                   -> full - this = exposed stats exchange
  noz,nostats    neither                                                  -> kernels + launch structure only
"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist
from wav2vec_contr_loss_b200 import _cabi, distributed as D

# The variants leave an exchange out by skipping its push and its wait (the flag ids of the exchanges they drop)
SKIPS = {"noz": _cabi.PEER_FLAG_Z, "nostats": _cabi.PEER_FLAG_STATS}
skipped = set()
_peer_push, _peer_wait = D.Fn.peer_push, D.Fn.peer_wait


def peer_push(desc, src0, dst_off0, src1, dst_off1, flag_id, **kw):
    if flag_id not in skipped:
        _peer_push(desc, src0, dst_off0, src1, dst_off1, flag_id, **kw)


def peer_wait(desc, flag_id, device):
    if flag_id not in skipped:
        _peer_wait(desc, flag_id, device)


D.Fn.peer_push, D.Fn.peer_wait = peer_push, peer_wait

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dev = torch.device("cuda", lr)
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
nl = n // world
g = torch.Generator().manual_seed(1337)
z = torch.nn.functional.normalize(torch.randn(n, 256, generator=g), dim=1).to(torch.bfloat16)
y = torch.zeros(n, dtype=torch.int32); y[torch.randperm(n, generator=g)[: n // 2]] = 1
zl, yl = z[rank * nl:(rank + 1) * nl].to(dev), y[rank * nl:(rank + 1) * nl].to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
out = {"world": world, "N": n}
keep = []      # modules, graphs and outputs stay alive: freeing symmetric memory during a later capture is an error
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 2     # the whole list is measured `rounds` times: order effects show
for rnd, exchange in [(r_, e_) for r_ in range(rounds) for e_ in ("peer", "nccl")]:
    for variant in (("", "noz", "nostats", "noz,nostats") if exchange == "peer" else ("",)):
        skipped = {SKIPS[v] for v in variant.split(",") if v}
        mod = D.ShardedSupConLoss(0.07, "cosine", exchange=exchange)
        mod.assume_unit_rows = True
        keep.append(mod)

        def step(mod=mod):
            zz = zl.detach().requires_grad_(True)
            loss = mod(zz, yl, topk_neg=15, alpha=0.0)
            (dz,) = torch.autograd.grad(loss, zz)
            return loss, dz
        for _ in range(3):
            step()
        torch.cuda.synchronize(); dist.barrier()
        gr = torch.cuda.CUDAGraph(); side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(); torch.cuda.synchronize(); dist.barrier()
            with torch.cuda.graph(gr, stream=side, capture_error_mode="thread_local"):
                res = step()
        torch.cuda.synchronize(); dist.barrier()
        for _ in range(3):
            gr.replay()
        tot = 0.0
        for _ in range(12):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier(); torch.cuda.synchronize()
            e0.record(); gr.replay(); e1.record(); torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        t = torch.tensor([tot / 12], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out.setdefault(f"{exchange}/{variant or 'full'}_ms", []).append(round(float(t), 4))
        keep.extend([gr, res, step])
if rank == 0:
    print(json.dumps(out), flush=True)
torch.cuda.synchronize(); dist.barrier()
sys.stdout.flush()
os._exit(0)
