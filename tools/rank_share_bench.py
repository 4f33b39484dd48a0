#!/usr/bin/env python
"""Time one rank's share of the row-sharded problem on a single GPU:
rows [0, N/R) against all N columns (what each of R ranks runs between collectives)."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from wav2vec_contr_loss_b200 import functional as Fn
n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
ranks = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1,2,4,8").split(",")]
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(1337)
z = torch.nn.functional.normalize(torch.randn(n, 256, generator=g), dim=1).to(dev).to(torch.bfloat16)
y = (torch.rand(n, generator=g) < 0.5).to(torch.int32).to(dev)
for R in ranks:
    nl = n // R
    prob = Fn.make_problem(n, 256, 1, tau=0.07, similarity=0, topk=15, alpha=0.0, row_offset=0, n_rows=nl, flags=32)
    whole = Fn.make_problem(n, 256, 1, tau=0.07, similarity=0, topk=15, alpha=0.0, flags=32)
    stats_all = torch.zeros(n, 8, device=dev)
    for _ in range(3):
        stats, partials, _ = Fn.forward_rows(z, y, prob, want_loss=False)
        stats_all[:nl] = stats
        if R > 1:
            stats_all[nl:] = stats.repeat(R - 1, 1)
            partials = partials * R
        dz = Fn.backward_rows(z, y, stats_all, partials, None, prob, out_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    fw = bw = 0.0
    iters = 20
    for _ in range(iters):
        e[0].record(); stats, partials2, _ = Fn.forward_rows(z, y, prob, want_loss=False)
        e[1].record(); dz = Fn.backward_rows(z, y, stats_all, partials, None, prob, out_dtype=torch.bfloat16)
        e[2].record(); torch.cuda.synchronize()
        fw += e[0].elapsed_time(e[1]); bw += e[1].elapsed_time(e[2])
    fw /= iters; bw /= iters
    # whole rank step as one CUDA graph (no host launch gaps)
    gms = None
    try:
        gr = torch.cuda.CUDAGraph(); side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        def both():
            st_, pa_, _ = Fn.forward_rows(z, y, prob, want_loss=False)
            return Fn.backward_rows(z, y, stats_all, partials, None, prob, out_dtype=torch.bfloat16)
        with torch.cuda.stream(side):
            both(); torch.cuda.synchronize()
            with torch.cuda.graph(gr, stream=side):
                both()
        torch.cuda.synchronize()
        for _ in range(3): gr.replay()
        e[0].record()
        for _ in range(iters): gr.replay()
        e[1].record(); torch.cuda.synchronize()
        gms = e[0].elapsed_time(e[1]) / iters
    except Exception as ex:  # noqa: BLE001
        gms = str(ex)
    fl = 6.0 * n * nl * 256
    print(json.dumps(dict(N=n, R=R, rows=nl, fwd_ms=round(fw, 4), bwd_ms=round(bw, 4), graph_ms=(round(gms, 4) if isinstance(gms, float) else gms), graph_tflops=(round(fl / gms / 1e9, 1) if isinstance(gms, float) else None), tflops=round(fl / (fw + bw) / 1e9, 1))), flush=True)
