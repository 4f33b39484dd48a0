"""The layer-mean store sharded over the GPUs of a node (feature_store.ShardedLayerMeanStore), one process per GPU:

    torchrun --nproc-per-node R tools/sharded_store_bench.py [--out profiles/r07_sharded_store_bench_rR.json]

Measured in one run, each rank reading its own card's name, power limit and max SM clock in the same run:

* pool: head_sharded_store_pool_fwd_kernel at B = 64, F = 1024, T = 199 on a --store-clips store (13.4 GB at 16 k,
  split R ways) for rows of this rank's shard only (local), of the other ranks' only (remote, R > 1), and uniform
  random rows, in eval and with dropout 0.1; beside head_store_pool_fwd_kernel on a single-GPU store of the same
  clips in the same process.  Rates are over the 64 rows read (52 MB).
* graphed_step: one GraphedHeadStep(store=sharded, grad_sync=GradSync) replay per rank: FusedCompressionHead(1024,
  256, 0.1), ShardedSupConLoss (global batch R x 64), AdamW, alpha 0.5, fresh random rows every replay.
* build: --clips synthetic 4 s clips through a random-init XLS-R-300M (tools/store_step_bench.py's encoder), frozen,
  batch 64: build_layer_mean_store on rank 0 alone, then build_sharded_layer_mean_store on all R ranks; then
  --epochs epochs of train_one_epoch_from_store from the sharded store (BalancedBatchSampler(rank=, world_size=),
  ShardedSupConLoss, GradSync).

Kernel and step times are CUDA events, median over --iters launches after warm-up; build and epoch times are host
clocks around work that ends in a device synchronise and a barrier.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from graphed_step_bench import median_ms  # noqa: E402

B, F, T = 64, 1024, 199


def card(dev):
    out = {"name": torch.cuda.get_device_name(dev), "index": dev.index}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def pool(dev, rank, world, n, iters):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore, ShardedLayerMeanStore
    sharded = ShardedLayerMeanStore(n, F, T, dev)
    sharded.rows.normal_()
    sharded.labels.copy_(torch.arange(n, device=dev) % 2)
    sharded.filled = n
    single = LayerMeanStore(n, F, T, dev)
    single.rows.normal_()
    single.filled = n
    torch.cuda.synchronize(dev)
    dist.barrier()
    g = torch.Generator().manual_seed(3 + rank)
    slots = torch.arange(n)
    sets = {"local": slots[slots % world == rank], "random": slots}
    if world > 1:
        sets["remote"] = slots[slots % world != rank]
    rng = torch.tensor([7, 0], dtype=torch.int64, device=dev)
    out = {"store_clips": n, "shard_GB": sharded.rows.numel() * 4 / 1e9, "rows_read_MB": B * F * T * 4 / 1e6}
    for name, pick in sets.items():
        idx = [pick[torch.randint(0, len(pick), (B,), generator=g)].to(dev) for _ in range(64)]
        for p in (0.0, 0.1):
            for which, store in (("sharded", sharded), ("single_gpu", single)):
                if which == "single_gpu" and name == "remote":
                    continue
                it = iter(idx * (iters // 16 + 2))
                ms = median_ms(lambda: store.pool(next(it), p, 0.01, rng if p else None), iters)  # noqa: B023
                out[f"{name}/p{p}/{which}"] = {"us": ms * 1e3, "GB_per_s": B * F * T * 4 / ms / 1e6}
    del single
    torch.cuda.empty_cache()
    return sharded, out


def graphed_step(dev, store, iters):
    from wav2vec_contr_loss_b200 import FusedCompressionHead
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss
    torch.manual_seed(0)
    head = FusedCompressionHead(F, 256, 0.1).to(dev).train()
    opt = torch.optim.AdamW(head.parameters(), lr=1e-4, weight_decay=3e-3, capturable=True)
    g = torch.Generator().manual_seed(5)
    idx = [torch.randperm(store.n, generator=g)[:B].to(dev) for _ in range(8)]
    step = S.GraphedHeadStep(head, ShardedSupConLoss(0.1, "cosine"), opt, idx[0], topk_neg=15, store=store,
                             grad_sync=S.GradSync(head.parameters()))
    it = iter(idx * (iters + 8))
    return {"ms": median_ms(lambda: step(next(it), alpha=0.5), iters)}


def build_and_epochs(dev, rank, world, n_clips, n_epochs):
    from types import SimpleNamespace
    from torch.utils.data import DataLoader, Subset
    from store_step_bench import Clips, XlsrStandIn
    from wav2vec_contr_loss_b200 import FusedCompressionHead
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss
    from wav2vec_contr_loss_b200.feature_store import (build_layer_mean_store, build_sharded_layer_mean_store,
                                                       shard_slots)
    torch.manual_seed(1337)
    enc = XlsrStandIn().to(dev).eval()
    ds = Clips(n_clips)
    res = {"clips": n_clips, "encoder": "random-init XLS-R-300M, frozen, fp32, batch 64"}
    with torch.no_grad():                                     # warm-up: cuDNN / cuBLAS choices for the shapes used
        w = ds.wave[:B].to(dev)
        enc(w, attention_mask=(w != 0).long())

    def timed(fn):
        torch.cuda.synchronize(dev)
        dist.barrier()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize(dev)
        dist.barrier()
        return out, time.perf_counter() - t0

    def one_gpu():
        if rank == 0:
            store = build_layer_mean_store(enc, DataLoader(ds, batch_size=B), dev)
            del store
    _, res["build_one_gpu_s"] = timed(one_gpu)
    torch.cuda.empty_cache()
    mine = DataLoader(Subset(ds, list(shard_slots(n_clips, rank, world))), batch_size=B)
    store, res["build_sharded_s"] = timed(lambda: build_sharded_layer_mean_store(enc, mine, dev, n=n_clips))
    res["build_speedup"] = res["build_one_gpu_s"] / res["build_sharded_s"]
    del enc
    torch.cuda.empty_cache()
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=15, warmup_epochs=0,
                          alpha_ramp_epochs=1, alpha_end=0.5)
    head = FusedCompressionHead(F, 256, 0.1).to(dev)
    opt = torch.optim.AdamW(head.parameters(), lr=1e-4, weight_decay=3e-3)
    loss_fn = ShardedSupConLoss(0.1, "cosine")
    sampler = S.BalancedBatchSampler(ds, B, seed=0, rank=rank, world_size=world)
    per_epoch = []
    for epoch in range(1, n_epochs + 1):
        sampler.set_epoch(epoch)
        batches = list(sampler)
        (loss, _), s = timed(lambda: S.train_one_epoch_from_store(  # noqa: B023
            head, loss_fn, store, batches, opt, dev, epoch, cfg, grad_sync=S.GradSync(head.parameters())))
        per_epoch.append(s)
    res["steps_per_epoch"] = len(sampler)
    res["epoch_s"] = per_epoch
    res["steady_epoch_s"] = statistics.median(per_epoch[1:]) if len(per_epoch) > 1 else per_epoch[0]
    store.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="rank 0 writes the JSON of every rank here (default: print only)")
    ap.add_argument("--store-clips", type=int, default=16384)
    ap.add_argument("--clips", type=int, default=16384, help="clips of the build and epoch measurement")
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--skip-build", action="store_true", help="kernels and graphed steps only")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    from wav2vec_contr_loss_b200 import build
    from wav2vec_contr_loss_b200 import stage1 as S
    build.build()
    is_dist, rank, world, local = S.setup_distributed("nccl")
    if not is_dist:                                           # one process: a group of one rank
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        torch.cuda.set_device(0)
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    dev = torch.device("cuda", torch.cuda.current_device())
    try:
        res = {"world": world, "card": card(dev)}
        store, res["pool"] = pool(dev, rank, world, args.store_clips, args.iters)
        res["graphed_step"] = graphed_step(dev, store, args.iters)
        store.close()
        del store
        torch.cuda.empty_cache()
        if not args.skip_build:
            res["build"] = build_and_epochs(dev, rank, world, args.clips, args.epochs)
        every = [None] * world
        dist.all_gather_object(every, res)
        if rank == 0:
            text = json.dumps({"ranks": every}, indent=1)
            print(text)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "w") as fh:
                    fh.write(text + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
