"""The layer-mean store in fp16 against fp32, on the same content, in one process:

    python tools/store_fp16_bench.py [--clips 4096] [--dir /tmp] [--out profiles/r09_store_fp16_bench.json]

1. pool: the gather-pool kernel (LayerMeanStore.pool, batch 64) on a 16 k-clip store of (1024, 199) rows: fp32
   (13.4 GB) against fp16 (6.7 GB).  The fp32 store holds the fp16 store's values widened, so the two pool the same
   bits (checked).  Eval and dropout 0.1; CUDA events around each launch, the two dtypes alternated launch by launch,
   median of --iters; random indices, so the rows read (52 / 26 MB a launch) come mostly from HBM, not L2.
2. graphed step: GraphedHeadStep(store=) (FusedCompressionHead 1024 -> 256, SupConBinaryLoss, AdamW) from each of
   those stores, median of --iters replays.
3. clips: --clips synthetic 4 s clips through a random-init XLS-R-300M (tools/store_step_bench.py's encoder),
   frozen, fp32, batch 64: build_layer_mean_store per dtype; save and load per dtype (time, file size, the share of
   rows.npy in the page cache before the load: caches are not dropped); three epochs from each store with the same
   head, sampler and dropout stream (per-epoch loss relative difference and max |delta head weight|); the largest
   |layer mean| of the fp32 build.
4. capacity: an fp16 store of more clips than the free memory would hold in fp32; its last rows written and pooled,
   checked against head.layer_time_pool of the widened rows.

The card's name, power limit and max SM clock are read in the same run.
"""
import argparse
import copy
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from graphed_step_bench import median_ms  # noqa: E402
from sharded_store_bench import card  # noqa: E402
from store_io_bench import resident_share  # noqa: E402

B, F, T = 64, 1024, 199
F16 = torch.float16


def pool_leg(dev, n, iters):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    s16 = LayerMeanStore(n, F, T, dev, dtype=F16)
    s16.rows.normal_()
    s32 = LayerMeanStore(n, F, T, dev)
    s32.rows.copy_(s16.rows)
    s16.filled = s32.filled = n
    g = torch.Generator().manual_seed(3)
    idx = [torch.randint(0, n, (B,), generator=g).to(dev) for _ in range(iters + 3)]
    rng = torch.tensor([7, 0], dtype=torch.int64, device=dev)
    out = {"store_clips": n, "fp32_store_GB": s32.rows.nbytes / 1e9, "fp16_store_GB": s16.rows.nbytes / 1e9}
    for p in (0.0, 0.1):
        r = rng if p else None
        same = all(torch.equal(s16.pool(i, p, 0.01, r), s32.pool(i, p, 0.01, r)) for i in idx[:3])
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
              for k in ("fp32", "fp16")}
        torch.cuda.synchronize(dev)
        for it in range(iters):
            for name, store in (("fp32", s32), ("fp16", s16)):
                s, e = ev[name][it]
                s.record()
                store.pool(idx[it], p, 0.01, r)
                e.record()
        torch.cuda.synchronize(dev)
        us = {k: statistics.median(s.elapsed_time(e) for s, e in v) * 1e3 for k, v in ev.items()}
        out[f"p{p}"] = {"fp32_us": us["fp32"], "fp16_us": us["fp16"], "fp16_over_fp32": us["fp16"] / us["fp32"],
                        "fp32_bytes_read": B * F * T * 4, "fp16_bytes_read": B * F * T * 2,
                        "fp16_equals_widened_fp32_bit_for_bit": same}
    return s32, s16, out


def graphed_leg(dev, stores, iters):
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    out = {}
    for name, store in stores.items():
        store.labels[: store.filled] = torch.arange(store.filled, device=dev) % 2
        torch.manual_seed(0)
        head = FusedCompressionHead(F, 256, 0.1).to(dev).train()
        opt = torch.optim.AdamW(head.parameters(), lr=1e-4, weight_decay=3e-3, capturable=True)
        g = torch.Generator().manual_seed(5)
        idx = [torch.randperm(store.filled, generator=g)[:B].to(dev) for _ in range(8)]
        step = S.GraphedHeadStep(head, SupConBinaryLoss(0.1, "cosine"), opt, idx[0], topk_neg=15, store=store)
        it = iter(idx * (iters + 8))
        out[name] = {"ms": median_ms(lambda: step(next(it), alpha=0.5), iters)}
    return out


def timed(dev, fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(dev)
    return out, time.perf_counter() - t0


def clips_leg(dev, n_clips, root):
    from types import SimpleNamespace
    from torch.utils.data import DataLoader
    from store_step_bench import Clips, XlsrStandIn
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss
    from wav2vec_contr_loss_b200 import feature_store as FS
    from wav2vec_contr_loss_b200 import stage1 as S
    torch.manual_seed(1337)
    enc = XlsrStandIn().to(dev).eval()
    ds = Clips(n_clips)
    res = {"clips": n_clips, "encoder": "random-init XLS-R-300M, frozen, fp32, batch 64 (trained XLS-R layer-mean "
                                        "magnitudes are not measured here)"}
    with torch.no_grad():                                      # warm-up: cuDNN / cuBLAS choices for the shapes used
        w = ds.wave[:B].to(dev)
        enc(w, attention_mask=(w != 0).long())
    stores = {}
    for name, dtype in (("fp32", torch.float32), ("fp16", F16)):
        stores[name], s = timed(dev, lambda: FS.build_layer_mean_store(enc, DataLoader(ds, batch_size=B), dev,
                                                                       dtype=dtype))
        res[f"{name}_build_s"] = s
    del enc
    torch.cuda.empty_cache()
    s32, s16 = stores["fp32"], stores["fp16"]
    res["fp16_rows_equal_fp32_rows_half"] = bool(torch.equal(s16.rows.view(torch.int16),
                                                             s32.rows.half().view(torch.int16)))
    res["max_abs_layer_mean"] = float(s32.rows.abs().max())
    res["io"] = {}
    for name, store in stores.items():
        path = os.path.join(root, name)
        _, save_s = timed(dev, lambda: store.save(path))
        rows_file = os.path.join(path, FS.ROWS_FILE)
        cached = resident_share(rows_file)
        loaded, load_s = timed(dev, lambda: FS.load_layer_mean_store(path, dev, dtype=store.dtype))
        same = bool(torch.equal(loaded.rows.view(torch.int8), store.rows.view(torch.int8)))
        res["io"][name] = {"rows_file_bytes": os.path.getsize(rows_file), "save_s": save_s, "load_s": load_s,
                           "load_GB_per_s": os.path.getsize(rows_file) / load_s / 1e9,
                           "rows_file_share_in_page_cache_before_load": cached, "loaded_equals_saved": same}
        del loaded
        torch.cuda.empty_cache()
    res["io_note"] = "caches were not dropped: each load read rows.npy from the page cache (share above)"
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=15, warmup_epochs=0,
                          alpha_ramp_epochs=1, alpha_end=0.5)
    torch.manual_seed(0)
    heads = {"fp32": FusedCompressionHead(F, 256, 0.1).to(dev)}
    heads["fp16"] = copy.deepcopy(heads["fp32"])
    opts = {k: torch.optim.AdamW(h.parameters(), lr=1e-4, weight_decay=3e-3) for k, h in heads.items()}
    losses = {k: SupConBinaryLoss(0.1, "cosine") for k in heads}
    samplers = {k: S.BalancedBatchSampler(ds, B, seed=0) for k in heads}
    res["epochs"] = []
    for epoch in (1, 2, 3):
        got = {}
        for k in heads:
            samplers[k].set_epoch(epoch)
            (loss, _), s = timed(dev, lambda: S.train_one_epoch_from_store(heads[k], losses[k], stores[k],
                                                                           list(samplers[k]), opts[k], dev, epoch,
                                                                           cfg))
            got[k] = (loss, s)
        wa, wb = (torch.cat([p.detach().reshape(-1) for p in heads[k].parameters()]) for k in ("fp32", "fp16"))
        res["epochs"].append({"epoch": epoch, "fp32_loss": got["fp32"][0], "fp16_loss": got["fp16"][0],
                              "loss_rel_diff": abs(got["fp16"][0] - got["fp32"][0]) / abs(got["fp32"][0]),
                              "max_abs_head_weight_diff": float((wa - wb).abs().max()),
                              "fp32_epoch_s": got["fp32"][1], "fp16_epoch_s": got["fp16"][1]})
    return res


def capacity_leg(dev):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    from wav2vec_contr_loss_b200.head import layer_time_pool
    torch.cuda.empty_cache()
    free, total = torch.cuda.mem_get_info(dev)
    row32 = F * T * 4 + 8
    fp32_fit = free // row32
    n = int(fp32_fit * 1.1)
    store = LayerMeanStore(n, F, T, dev, dtype=F16)
    last = torch.arange(n - B, n, device=dev)
    torch.manual_seed(11)
    store.rows[n - B:].normal_()
    store.filled = n
    rng = torch.tensor([3, 1], dtype=torch.int64, device=dev)
    hs = store.rows[last].float().unsqueeze(1)
    ok = bool(torch.equal(store.pool(last, 0.1, 0.01, rng), layer_time_pool(hs, 0.1, 0.01, rng)))
    out = {"free_GB_before": free / 1e9, "fp32_clips_that_fit": int(fp32_fit), "fp16_store_clips": n,
           "fp16_store_GB": store.rows.nbytes / 1e9, "fp32_would_need_GB": n * row32 / 1e9,
           "last_rows_pool_equals_layer_time_pool": ok}
    del store, hs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--clips", type=int, default=4096)
    ap.add_argument("--store-clips", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--dir", default=tempfile.gettempdir(), help="where the stores are saved (and removed)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    from wav2vec_contr_loss_b200 import build
    build.build()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card(dev), "batch": B, "row_shape": [F, T]}
    s32, s16, res["pool"] = pool_leg(dev, args.store_clips, args.iters)
    res["graphed_step"] = graphed_leg(dev, {"fp32": s32, "fp16": s16}, args.iters)
    del s32, s16
    torch.cuda.empty_cache()
    root = tempfile.mkdtemp(dir=args.dir, prefix="store_fp16_bench_")
    try:
        res["clips_through_xlsr"] = clips_leg(dev, args.clips, root)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    torch.cuda.empty_cache()
    res["capacity"] = capacity_leg(dev)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
