#!/usr/bin/env python
"""Step time and peak memory of ``CachedBatchStep`` for a global batch of k micro-batches of B = 64, k in
{1, 4, 16, 64}, frozen and fine-tuned encoder.

The encoder is synthetic with the Stage-1 output shape: a strided conv (hop 320) of a 63680-sample waveform to
F = 1024 channels, dropout, tanh, and a learned scale per layer that expands it to hs = (64, 25, 1024, 199) fp32
(1.3 GB per micro-batch, the size of the XLS-R output the fused head reads).  Head: ``FusedCompressionHead(1024, 256,
0.1)`` in train mode; z in bf16 with unit rows (the tensor-core loss path from N = 256 on); ``SupConBinaryLoss``
cosine, tau 0.07, K 15, alpha 0; SGD.  Per configuration:

* ``step_ms``: one ``step(...)`` call (both passes, loss, clip, optimizer), CUDA events, median over the timed steps;
* ``peak_mb``: ``max_memory_allocated`` during one step, above what was allocated before it (inputs, weights,
  gradients and optimizer state of the previous step);
* ``loss_ms``: ``call_loss`` + ``autograd.grad`` alone on a bf16 z of the step's k B rows, and ``loss_share`` =
  loss_ms / step_ms;
* ``encoder_fwd_ms``: one encoder forward without a graph on one micro-batch (what the fine-tuned route and the
  frozen torch-head route pay a second time per micro-batch).

The card's name and power limit are read in the same run.  Writes one JSON document to ``--out``.

    python tools/cached_batch_bench.py [--steps 5] [--warmup 2] [--out profiles/r05_cached_batch_step.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from wav2vec_contr_loss_b200 import FusedCompressionHead, SupConBinaryLoss  # noqa: E402
from wav2vec_contr_loss_b200 import functional as Fn  # noqa: E402
from wav2vec_contr_loss_b200.cached_batch import CachedBatchStep  # noqa: E402
from wav2vec_contr_loss_b200.stage1 import call_loss  # noqa: E402

B, LAYERS, FEAT, FRAMES, HOP, D = 64, 25, 1024, 199, 320, 256


class SyntheticEncoder(nn.Module):
    """(B, 63680) waveforms -> (B, 25, 1024, 199)"""

    def __init__(self):
        super().__init__()
        self.conv = nn.Conv1d(1, FEAT, HOP, stride=HOP)
        self.drop = nn.Dropout(0.1)
        self.scale = nn.Parameter(torch.linspace(0.5, 1.5, LAYERS))

    def forward(self, waveforms, attention_mask=None):
        x = (waveforms * attention_mask.to(waveforms.dtype)).unsqueeze(1)
        h = torch.tanh(self.drop(self.conv(x)))                                   # (B, F, T)
        return h.unsqueeze(1) * self.scale.view(1, LAYERS, 1, 1)


def card():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"not read: {exc}"
    return info


def events_ms(fn, steps, warmup):
    times = []
    for it in range(warmup + steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if it >= warmup:
            times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def run(k, finetune, micro, steps, warmup):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    enc = SyntheticEncoder().to(dev).train(finetune)
    head = FusedCompressionHead(FEAT, D, 0.1).to(dev).train()
    params = list(head.parameters()) + (list(enc.parameters()) if finetune else [])
    opt = torch.optim.SGD(params, lr=1e-3, momentum=0.9)
    loss_fn = SupConBinaryLoss(0.07, "cosine")
    step = CachedBatchStep(enc, head, loss_fn, opt, micro_batches=k, finetune_encoder=finetune,
                           normalize=lambda x: Fn.l2_normalize(x, torch.bfloat16))
    batch = micro[:k]
    step_ms = events_ms(lambda: step(batch, 15, 0.0), steps, warmup)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    loss = step(batch, 15, 0.0)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    assert torch.isfinite(loss).item()

    g = torch.Generator(device=dev).manual_seed(1)
    z = Fn.l2_normalize(torch.randn(k * B, D, device=dev, generator=g), torch.bfloat16)
    z.requires_grad_(True)
    labels = torch.cat([y for _, y in batch])

    def loss_only():
        torch.autograd.grad(call_loss(loss_fn, z, labels, 15, 0.0), z)

    loss_ms = events_ms(loss_only, 20, 5)
    with torch.no_grad():
        w = batch[0][0]
        enc_ms = events_ms(lambda: enc(w, attention_mask=(w != 0.0).long()), 10, 3)
    return {"k": k, "B": B, "N": k * B, "encoder": "finetuned" if finetune else "frozen",
            "step_ms": round(step_ms, 3), "step_ms_per_micro_batch": round(step_ms / k, 3),
            "peak_mb": round(peak / 2 ** 20, 1), "loss_ms": round(loss_ms, 4),
            "loss_share": round(loss_ms / step_ms, 4), "encoder_fwd_ms": round(enc_ms, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ks", default="1,4,16,64")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_cached_batch_step.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cached_batch_bench needs a CUDA device")
    ks = [int(v) for v in args.ks.split(",")]
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    micro = []
    for _ in range(max(ks)):
        y = (torch.randperm(B, device=dev, generator=g) % 2)
        micro.append((torch.randn(B, FRAMES * HOP, device=dev, generator=g) + 0.3 * (2.0 * y.view(-1, 1) - 1.0), y))
    doc = {"card": card(), "hs": [B, LAYERS, FEAT, FRAMES], "z": "bf16 unit rows", "loss": "SupConBinaryLoss cosine "
           "tau 0.07 K 15 alpha 0", "head": "FusedCompressionHead(1024, 256, 0.1)", "results": []}
    print(json.dumps(doc["card"]), flush=True)
    for finetune in (False, True):
        for k in ks:
            rec = run(k, finetune, micro, args.steps, args.warmup)
            print(json.dumps(rec), flush=True)
            doc["results"].append(rec)
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
