#!/usr/bin/env python
"""fwd+bwd time of MemorySupConLoss at the Stage-1 batch size: B = 64 anchors, d = 256, against a full memory of M
embeddings, M in {4096, 16384, 65536}, fp32 (exact path) and bf16 with unit rows (tensor-core path).

Each timed step is what a training step does with the loss: the module's forward (stage the batch, forward kernels)
and loss.backward() (backward kernels, enqueue of the batch), so the memory stays full and n_total = B + M.  Device
time per step from CUDA events around each step (median and min over the timed steps).  The memory (up to 64 MB of
fp32 z) stays in the 126 MB L2 between steps here; in training the encoder runs in between.  The card's name and
power limit are read in the same run.  One JSON line per configuration; --out also writes them to a file.

    python tools/memory_bench.py [--steps 50] [--warmup 10] [--out memory_bench.jsonl]
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
import torch.nn.functional as F  # noqa: E402

from wav2vec_contr_loss_b200.memory import MemorySupConLoss  # noqa: E402

B, D = 64, 256


def card():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        info["nvidia_smi"] = out
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def time_steps(m, dtype, alpha, steps, warmup):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1337)
    mod = MemorySupConLoss(0.07, "cosine", 0.2, 2.0, memory_size=m)
    mod.assume_unit_rows = dtype == torch.bfloat16
    fill = F.normalize(torch.randn(m, D, generator=g), dim=1).to(dev, dtype)
    mod.memory.enqueue(fill, torch.randint(0, 2, (m,), generator=g).to(dev), unit_rows=True)
    batches = [(F.normalize(torch.randn(B, D, generator=g), dim=1).to(dev, dtype).requires_grad_(True),
                (torch.arange(B) % 2).to(dev)) for _ in range(4)]
    times = []
    for it in range(warmup + steps):
        z, y = batches[it % len(batches)]
        z.grad = None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = mod(z, y, topk_neg=15, alpha=alpha)
        loss.backward()
        e1.record()
        torch.cuda.synchronize()
        if it >= warmup:
            times.append(e0.elapsed_time(e1))
    assert mod.memory.filled == m and torch.isfinite(loss).item()
    return statistics.median(times), min(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("memory_bench needs a CUDA device")
    info = card()
    print(json.dumps(info), flush=True)
    lines = [info]
    for dtype in (torch.float32, torch.bfloat16):
        for m in (4096, 16384, 65536):
            for alpha in (0.0, 0.5):
                med, best = time_steps(m, dtype, alpha, args.steps, args.warmup)
                rec = {"B": B, "d": D, "M": m, "dtype": str(dtype)[6:], "alpha": alpha, "topk": 15, "lambda": 0.2,
                       "step_ms_median": round(med, 4), "step_ms_min": round(best, 4),
                       "tflops": round(6 * B * (B + m) * D / (med * 1e-3) / 1e12, 2)}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(json.dumps(r) for r in lines) + "\n")


if __name__ == "__main__":
    main()
