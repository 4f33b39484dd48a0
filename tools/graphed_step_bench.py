"""Head step of BASELINE configs[4] (frozen encoder): eager launches vs one CUDA-graph replay.

    python tools/graphed_step_bench.py [--batch 64] [--iters 30] [--head fused] [--hs-dtype bfloat16]
    python tools/graphed_step_bench.py --head fused --memory 4096,16384,65536


hs is the encoder output the reference hands the head: (B, 25, 1024, 199) fp32 (1.3 GB at B = 64), synthetic; with
--hs-dtype bfloat16 it is the output of an encoder run in bf16 (0.65 GB), which the fused head reads as it is.
The head has the shape/ops of the reference's compression head (compression_module.py:35-67): layer mean,
Dropout(0.1), LeakyReLU, Linear(1024 -> 256) per frame.  Step = stage1_utils.py:121-130 without the encoder.
Times are CUDA events on the launching stream, median of --iters steps after warm-up; hs is far larger than the L2,
so every pass reads it from HBM.  Rates are over algorithmic bytes: hs read once by the forward; hs read once and d hs
(K copies of the (B, F, T) gradient) written once by the backward.  The card's name and power limit are read in the
same run and printed with the times.

--memory M,...: the step with MemorySupConLoss (cross-batch memory of M rows) instead, for fp32 z and for bf16 z with
unit rows, alpha 0 and 0.5: one graph replay with the memory full, one while it fills (reset to empty before the
timed window, which enqueues fewer than M rows), the eager step with the memory full, and the graphed step with
SupConBinaryLoss on the same batch.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


class LayerMeanHead(nn.Module):
    def __init__(self, feat=1024, dim=256, p=0.1):
        super().__init__()
        self.drop, self.act, self.proj = nn.Dropout(p), nn.LeakyReLU(), nn.Linear(feat, dim)

    def forward(self, hs):                      # (B, K, F, T) -> (B, dim, T)
        x = self.act(self.drop(hs.mean(dim=1)))
        return self.proj(x.transpose(1, 2)).transpose(1, 2)


def median_ms(fn, iters):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    torch.cuda.synchronize()
    for s, e in ev:
        s.record()
        fn()
        e.record()
    torch.cuda.synchronize()
    return statistics.median(s.elapsed_time(e) for s, e in ev)


def card():
    """name and power limit of device 0 (the limit is part of any time measured on it)"""
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def memory_steps(args, hs, y, sizes):
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    dev, B, res = hs.device, hs.size(0), []
    for z_dtype in (torch.float32, torch.bfloat16):
        normalize = (lambda x: Fn.l2_normalize(x, torch.bfloat16)) if z_dtype == torch.bfloat16 else None
        for alpha in (0.0, 0.5):
            def make(loss_fn):
                head = (FusedCompressionHead() if args.head == "fused" else LayerMeanHead()).to(dev).train()
                opt = torch.optim.AdamW(head.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
                return head, opt, S.GraphedHeadStep(head, loss_fn, opt, hs, y, topk_neg=15, normalize=normalize)

            _, _, plain = make(SupConBinaryLoss(temperature=0.07, similarity="cosine"))
            t_plain = median_ms(lambda: plain(plain.hs, plain.labels, alpha), args.iters)
            del plain
            for m in sizes:
                loss_fn = MemorySupConLoss(0.07, "cosine", memory_size=m)
                head, opt, step = make(loss_fn)
                mem = loss_fn.memory
                g = torch.Generator(device=dev).manual_seed(m)
                fill = _unit_rows(torch.randn(m, 256, device=dev, generator=g)).to(z_dtype)
                mem.enqueue(fill, torch.randint(0, 2, (m,), device=dev, generator=g), unit_rows=True)
                t_full = median_ms(lambda: step(step.hs, step.labels, alpha), args.iters)
                mem.reset()
                t_fill = median_ms(lambda: step(step.hs, step.labels, alpha), args.iters)
                filled_after = mem.filled

                def eager_step():
                    z = S.embed(head, hs, normalize)
                    loss = loss_fn(z, y, topk_neg=15, alpha=alpha)
                    opt.zero_grad(set_to_none=True)
                    loss.backward()
                    torch.nn.utils.clip_grad_norm_(head.parameters(), 5.0)
                    opt.step()

                mem.enqueue(fill, torch.randint(0, 2, (m,), device=dev, generator=g), unit_rows=True)
                t_eager = median_ms(eager_step, args.iters)
                res.append({"z_dtype": str(z_dtype).replace("torch.", ""), "alpha": alpha, "memory_size": m,
                            "graphed_memory_full_ms": t_full, "graphed_memory_filling_ms": t_fill,
                            "filling_window_ends_at_rows": filled_after, "eager_memory_full_ms": t_eager,
                            "graphed_without_memory_ms": t_plain})
                print(json.dumps(res[-1]), file=sys.stderr, flush=True)
                del step, head, opt, loss_fn, mem, fill
    return res


def _unit_rows(x):
    return torch.nn.functional.normalize(x, dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--frames", type=int, default=199)
    ap.add_argument("--head", choices=("torch", "fused"), default="torch",
                    help="torch: the reference's op chain; fused: FusedCompressionHead (csrc/supcon_head.cu)")
    ap.add_argument("--hs-dtype", choices=("float32", "bfloat16"), default="float32",
                    help="element type of the encoder output hs (bfloat16 needs --head fused)")
    ap.add_argument("--memory", default="", help="comma-separated memory sizes: time the cross-batch memory step")
    args = ap.parse_args()
    if args.hs_dtype == "bfloat16" and args.head != "fused":
        ap.error("--hs-dtype bfloat16 needs --head fused (the torch op chain's Linear layer is fp32)")
    from wav2vec_contr_loss_b200 import build
    build.build()
    from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss, layer_time_pool
    from wav2vec_contr_loss_b200 import stage1 as S

    dev = torch.device("cuda", 0)
    torch.manual_seed(1337)
    B = args.batch
    hs = torch.randn(B, 25, 1024, args.frames, device=dev, dtype=getattr(torch, args.hs_dtype))
    y = (torch.arange(B, device=dev) % 2).long()
    loss_fn = SupConBinaryLoss(temperature=0.07, similarity="cosine", uniformity_weight=0.0)
    hs_bytes = hs.numel() * hs.element_size()
    out = {"batch": B, "hs_shape": list(hs.shape), "hs_dtype": args.hs_dtype, "hs_GB": hs_bytes / 1e9,
           "iters": args.iters, "head": args.head, "card": card()}
    if args.memory:
        out["memory"] = memory_steps(args, hs, y, [int(m) for m in args.memory.split(",")])
        print(json.dumps(out))
        return
    if args.head == "fused":
        rng = torch.tensor([1337, 0], dtype=torch.int64, device=dev)
        with torch.no_grad():
            t_eval = median_ms(lambda: layer_time_pool(hs, 0.0, 0.01, None), args.iters)
            t_drop = median_ms(lambda: layer_time_pool(hs, 0.1, 0.01, rng), args.iters)
        kern = {"eval_ms": t_eval, "dropout_ms": t_drop,
                "eval_GBps": hs_bytes / 1e6 / t_eval, "dropout_GBps": hs_bytes / 1e6 / t_drop}
        # the backward (encoder fine-tuned), dropout on: d hs in hs's dtype
        x = hs.detach().requires_grad_(True)
        pooled = layer_time_pool(x, 0.1, 0.01, rng)
        up = torch.randn_like(pooled)
        t_bwd = median_ms(lambda: torch.autograd.grad(pooled, x, up, retain_graph=True), args.iters)
        kern.update(backward_ms=t_bwd, backward_GBps=2 * hs_bytes / 1e6 / t_bwd)
        if hs.dtype != torch.float32:
            # the route without a kernel for hs's dtype: an fp32 copy of hs, the fp32 kernel, and in the backward the
            # fp32 d hs converted back to hs's dtype
            with torch.no_grad():
                t_up = median_ms(lambda: layer_time_pool(hs.float(), 0.0, 0.01, None), args.iters)
            pooled_up = layer_time_pool(x.float(), 0.1, 0.01, rng)
            t_up_bwd = median_ms(lambda: torch.autograd.grad(pooled_up, x, up, retain_graph=True), args.iters)
            del pooled_up
            kern.update(upcast_route_eval_ms=t_up, upcast_route_backward_ms=t_up_bwd)
        del x, pooled
        out["head_pool_kernel"] = kern

    for alpha in (0.0, 0.5):
        head = (FusedCompressionHead() if args.head == "fused" else LayerMeanHead()).to(dev).train()
        opt = torch.optim.AdamW(head.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)

        def eager_step():
            z = S.embed(head, hs)
            loss = loss_fn(z, y, topk_neg=15, alpha=alpha)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(head.parameters(), 5.0)
            opt.step()
            return loss

        t_eager = median_ms(eager_step, args.iters)
        step = S.GraphedHeadStep(head, loss_fn, opt, hs, y, topk_neg=15)
        t_graph_copy = median_ms(lambda: step(hs, y, alpha), args.iters)             # + 1.3 GB input copy
        t_graph = median_ms(lambda: step(step.hs, step.labels, alpha), args.iters)  # producer writes in place

        z = S.embed(head, hs).detach()

        def loss_only():
            zz = z.clone().requires_grad_(True)
            loss_fn(zz, y, topk_neg=15, alpha=alpha).backward()

        t_loss = median_ms(loss_only, args.iters)
        with torch.no_grad():
            t_mean = median_ms(lambda: hs.mean(dim=1), args.iters)
        out[f"alpha_{alpha}"] = {"eager_step_ms": t_eager, "graphed_step_ms": t_graph,
                                 "graphed_step_with_input_copy_ms": t_graph_copy,
                                 "loss_fwd_bwd_eager_ms": t_loss, "layer_mean_only_ms": t_mean,
                                 "layer_mean_GBps": hs_bytes / 1e6 / t_mean}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
