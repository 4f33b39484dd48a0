"""Stage-1 head training from a device-resident store of layer means (wav2vec_contr_loss_b200.feature_store).

    python tools/store_step_bench.py [--out profiles/r06_store_step_bench.json] [--clips 2048] [--store-clips 16384]

Measured in one run, with the card's name, power limit and max SM clock read in the same run:

* layer_mean: head_layer_mean_kernel alone on hs = (64, 25, 1024, 199), fp32 and bf16 (the store build's kernel);
  rate over algorithmic bytes = hs read once + the (64, 1024, 199) fp32 rows written once.
* store_pool: head_store_pool_fwd_kernel alone at B = 64, F = 1024, T = 199, eval and dropout 0.1, gathering random
  rows of a store of --store-clips clips (13.4 GB at 16 k, a hundred times the 126 MB L2, so rows come from HBM);
  rate over the 64 rows read.
* graphed_step: one GraphedHeadStep replay (FusedCompressionHead(1024, 256, 0.1), SupConBinaryLoss, AdamW, alpha 0.5)
  on the (64, 25, 1024, 199) fp32 hs - produced in the step's static buffer, and copied into it before each replay -
  against the same step captured with store= on the store, fed new random rows every replay.
* epoch: --clips synthetic 4 s clips through a random-init XLS-R-300M (the architecture of bench.py --workload
  stage1, built with transformers; hs = its 25 hidden states as (B, 25, 1024, 199)), frozen, batch 64 from
  BalancedBatchSampler: one train_one_epoch, against build_layer_mean_store + train_one_epoch_from_store on the same
  batches, seeds and dropout stream, then further epochs from the store (the steady per-epoch time).  The two runs'
  epoch losses and head weights are reported side by side: the encoder's GEMMs may round differently at the build's
  batch composition than at the training batches', so they agree to rounding, not bit for bit.

Kernel and step times are CUDA events, median over the timed launches after warm-up; epoch times are host clocks
around work that ends in a device synchronise.
"""
import argparse
import copy
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from graphed_step_bench import card, median_ms  # noqa: E402

B, K, F, T = 64, 25, 1024, 199


def layer_mean(dev, iters):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    out = {}
    for dtype in (torch.float32, torch.bfloat16):
        hs = torch.randn(B, K, F, T, device=dev).to(dtype)
        store = LayerMeanStore(B, F, T, dev)
        y = torch.zeros(B, dtype=torch.int64, device=dev)

        def write():
            store.filled = 0
            store.append(hs, y)
        ms = median_ms(write, iters)
        nbytes = hs.numel() * hs.element_size() + B * F * T * 4
        out[str(dtype).replace("torch.", "")] = {"ms": ms, "GB_per_s": nbytes / ms / 1e6, "bytes": nbytes}
        del hs, store
    return out


def store_pool(dev, n_store, iters):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    store = LayerMeanStore(n_store, F, T, dev)
    store.rows.normal_()
    store.filled = n_store
    g = torch.Generator().manual_seed(3)
    idx = [torch.randint(0, n_store, (B,), generator=g).to(dev) for _ in range(iters + 3)]
    rng = torch.tensor([7, 0], dtype=torch.int64, device=dev)
    out = {"store_clips": n_store, "store_GB": store.rows.numel() * 4 / 1e9}
    for p in (0.0, 0.1):
        it = iter(idx * 2)

        def pool():
            store.pool(next(it), p, 0.01, rng if p else None)
        ms = median_ms(pool, iters)
        nbytes = B * F * T * 4
        out[f"p{p}"] = {"ms": ms, "GB_per_s": nbytes / ms / 1e6, "bytes_read": nbytes}
    return store, out


def graphed_steps(dev, store, iters):
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    y = (torch.arange(B) % 2).to(dev)
    store.labels[: store.filled] = torch.arange(store.filled, device=dev) % 2
    hs = torch.randn(B, K, F, T, device=dev)
    g = torch.Generator().manual_seed(5)
    idx = [torch.randperm(store.filled, generator=g)[:B].to(dev) for _ in range(8)]
    out = {}
    for name in ("hs_in_place", "hs_copied", "store"):
        torch.manual_seed(0)
        head = FusedCompressionHead(F, 256, 0.1).to(dev).train()
        opt = torch.optim.AdamW(head.parameters(), lr=1e-4, weight_decay=3e-3, capturable=True)
        loss_fn = SupConBinaryLoss(0.1, "cosine")
        if name == "hs_in_place":                   # the encoder writes its output into step.hs: no copy
            step = S.GraphedHeadStep(head, loss_fn, opt, hs, y, topk_neg=15)
            fn = lambda: step(step.hs, step.labels, 0.5)   # noqa: E731
        elif name == "hs_copied":                   # hs copied into step.hs before each replay (1.3 GB)
            step = S.GraphedHeadStep(head, loss_fn, opt, hs, y, topk_neg=15)
            fn = lambda: step(hs, y, 0.5)          # noqa: E731
        else:
            step = S.GraphedHeadStep(head, loss_fn, opt, idx[0], topk_neg=15, store=store)
            it = iter(idx * (iters + 8))
            fn = lambda: step(next(it), alpha=0.5)  # noqa: E731
        out[name] = {"ms": median_ms(fn, iters)}
    out["speedup_vs_hs_in_place"] = out["hs_in_place"]["ms"] / out["store"]["ms"]
    return out


class XlsrStandIn(torch.nn.Module):
    """random-init XLS-R-300M (bench.py --workload stage1's config); forward -> (B, 25, 1024, frames)"""

    def __init__(self):
        super().__init__()
        from transformers import Wav2Vec2Config, Wav2Vec2Model
        cfg = Wav2Vec2Config(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                             feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True, conv_dim=(512,) * 7,
                             conv_stride=(5, 2, 2, 2, 2, 2, 2), conv_kernel=(10, 3, 3, 3, 3, 2, 2),
                             num_conv_pos_embeddings=128, num_conv_pos_embedding_groups=16, layerdrop=0.0)
        self.model = Wav2Vec2Model(cfg)

    def forward(self, waveforms, attention_mask=None):
        out = self.model(waveforms, attention_mask=attention_mask, output_hidden_states=True)
        return torch.stack(out.hidden_states, dim=1).transpose(2, 3).contiguous()


class Clips(torch.utils.data.Dataset):
    def __init__(self, n, seed=1337):
        g = torch.Generator().manual_seed(seed)
        self.wave = torch.randn(n, 64000, generator=g)
        self.y = torch.arange(n) % 2
        self.data = [(f"utt{i}", int(self.y[i])) for i in range(n)]

    def __len__(self):
        return len(self.data)

    def __getitem__(self, i):
        return self.wave[i], self.y[i]


def epochs(dev, n_clips, store_epochs):
    from types import SimpleNamespace
    from torch.utils.data import DataLoader
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    torch.manual_seed(1337)
    enc = XlsrStandIn().to(dev).eval()
    n_params = sum(p.numel() for p in enc.parameters())
    ds = Clips(n_clips)
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=15, warmup_epochs=0,
                          alpha_ramp_epochs=1, alpha_end=0.5)
    head_a = FusedCompressionHead(F, 256, 0.1).to(dev)
    head_b = copy.deepcopy(head_a)
    opt_a = torch.optim.AdamW(head_a.parameters(), lr=1e-4, weight_decay=3e-3)
    opt_b = torch.optim.AdamW(head_b.parameters(), lr=1e-4, weight_decay=3e-3)
    sampler_a, sampler_b = S.BalancedBatchSampler(ds, B, seed=0), S.BalancedBatchSampler(ds, B, seed=0)
    res = {"clips": n_clips, "steps_per_epoch": len(sampler_a),
           "encoder": f"random-init XLS-R-300M ({n_params / 1e6:.1f} M params), frozen, fp32"}

    with torch.no_grad():                                     # warm-up: cuDNN / cuBLAS choices for the shapes used
        w = ds.wave[:B].to(dev)
        enc(w, attention_mask=(w != 0).long())
    torch.cuda.synchronize()
    sampler_a.set_epoch(1)
    t0 = time.perf_counter()
    loss_a, _ = S.train_one_epoch(enc, head_a, SupConBinaryLoss(0.1, "cosine"), DataLoader(ds, batch_sampler=sampler_a),
                                  opt_a, dev, 1, cfg)
    torch.cuda.synchronize()
    res["train_one_epoch_s"] = time.perf_counter() - t0

    t0 = time.perf_counter()
    store = build_layer_mean_store(enc, DataLoader(ds, batch_size=B), dev)
    torch.cuda.synchronize()
    res["store_build_s"] = time.perf_counter() - t0
    res["store_GB"] = store.rows.numel() * 4 / 1e9
    loss_fn_b = SupConBinaryLoss(0.1, "cosine")
    per_epoch = []
    for epoch in range(1, store_epochs + 1):
        sampler_b.set_epoch(epoch)
        batches = list(sampler_b)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss_b, _ = S.train_one_epoch_from_store(head_b, loss_fn_b, store, batches, opt_b, dev, epoch, cfg)
        torch.cuda.synchronize()
        per_epoch.append(time.perf_counter() - t0)
        if epoch == 1:
            res["epoch1_loss"] = {"train_one_epoch": loss_a, "from_store": loss_b,
                                  "rel_diff": abs(loss_a - loss_b) / abs(loss_a)}
            wa = torch.cat([p.detach().reshape(-1) for p in head_a.parameters()])
            wb = torch.cat([p.detach().reshape(-1) for p in head_b.parameters()])
            res["epoch1_head_weights"] = {"max_abs_diff": float((wa - wb).abs().max()),
                                          "rel_l2_diff": float((wa - wb).norm() / wa.norm()),
                                          "bit_identical": bool(torch.equal(wa, wb))}
    res["from_store_epoch_s"] = per_epoch
    res["from_store_steady_epoch_s"] = statistics.median(per_epoch[1:]) if len(per_epoch) > 1 else per_epoch[0]
    res["build_plus_first_store_epoch_s"] = res["store_build_s"] + per_epoch[0]
    res["steady_speedup_vs_train_one_epoch"] = res["train_one_epoch_s"] / res["from_store_steady_epoch_s"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON here (default: print only)")
    ap.add_argument("--clips", type=int, default=2048, help="clips of the epoch comparison")
    ap.add_argument("--store-clips", type=int, default=16384, help="clips of the store the gather-pool reads")
    ap.add_argument("--store-epochs", type=int, default=4)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--skip-epochs", action="store_true", help="kernels and graphed steps only")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    from wav2vec_contr_loss_b200 import build
    build.build()
    dev = torch.device("cuda:0")
    res = {"card": card(), "shape": {"B": B, "K": K, "F": F, "T": T}}
    res["layer_mean"] = layer_mean(dev, args.iters)
    store, res["store_pool"] = store_pool(dev, args.store_clips, args.iters)
    res["graphed_step"] = graphed_steps(dev, store, args.iters)
    del store
    torch.cuda.empty_cache()
    if not args.skip_epochs:
        res["epoch"] = epochs(dev, args.clips, args.store_epochs)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
