#!/usr/bin/env python
"""Benchmark of the SupCon hot path (BASELINE.json metric: fwd+bwd sim-pairs/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--batch-n 65536] [--d 256] [--dtype bf16|f32] [--similarity cosine]
                    [--dump-outputs DIR]

One "step" = one forward + backward of the loss over one batch of synthetic
unit-norm embeddings (value = N^2 / t).  Default workload = BASELINE.json
configs[3], the largest single-GPU configuration the metric is quoted on:
cosine SupCon, tau 0.07, N = 65536, d = 256, bf16 z / fp32-or-bf16 dz.  With
--gpus R > 1 (launched by torchrun) the N rows are sharded over the ranks
(strong scaling at fixed N, the BASELINE config): rows and labels pushed into
every peer's buffer (or all-gathered) beside the forward over the rank's own
columns -> the other columns -> exchange of row statistics and partial sums ->
backward.  The same run then measures the step once more at WEAK scaling
(N = batch-n * sqrt(R), the per-GPU pair count of the single-GPU workload: the
north_star's 8-GPU target is a weak-scaling one) and reports it under "weak".
The timed call is the drop-in module itself (SupConBinaryLoss / ShardedSupConLoss
called as stage1_utils.py:125-128 calls the reference's) + autograd.

Prints ONE JSON line (rank 0).  `--impl reference` times the reference's own CPU
implementation -- the UNMODIFIED loss.py behind F.normalize, from the verbatim
copies oracle/build_ref.py stages under oracle/_ref (they ship with the gpurun
snapshot; /root/reference does not exist on the GPU box) -- on a bounded sample
of the same workload, and adds the N x threads table of BASELINE.md section 3.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "supcon_fwd_bwd_sim_pairs_per_s"
UNIT = "pairs/s"
DUMP_DZ_BYTES = 32 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-n", dest="n", type=int, default=65536)
    ap.add_argument("--d", type=int, default=256)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--similarity", default="cosine")
    ap.add_argument("--tau", type=float, default=0.07)
    ap.add_argument("--lambda-uni", type=float, default=0.0)
    ap.add_argument("--topk", type=int, default=15)
    ap.add_argument("--alpha", type=float, default=0.0)
    ap.add_argument("--cpu-sample-n", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-table", action="store_true",
                    help="--impl reference: skip the N x threads table of BASELINE.md section 3")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: N fixed (BASELINE configs[3] as named); weak: per-GPU pair count fixed, "
                         "N = batch-n * sqrt(gpus)")
    ap.add_argument("--workload", default="loss", choices=["loss", "stage1"],
                    help="loss: the SupCon hot path (default, BASELINE configs[3]); stage1: one Stage-1 training step "
                         "around it (BASELINE configs[4]) reporting the loss's share of the step")
    ap.add_argument("--stage1-batch", type=int, default=64)
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="several ranks: how rows and row statistics travel -- peer = this library's kernels store "
                         "into the peers' buffers over NVLink (symmetric memory), nccl = torch.distributed all-gathers")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the N = 64 / 1024 / mined side measurements (one GPU only)")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every step from Python instead of replaying a CUDA graph")
    ap.add_argument("--no-weak-leg", action="store_true",
                    help="several ranks, strong scaling: skip the additional weak-scaling measurement (per-GPU pair "
                         "count of the single-GPU workload, N = batch-n * sqrt(gpus)) reported under \"weak\"")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as float32 DIR/<name>.npy: "
                         "loss.npy and dz.npy = d loss / d z of the whole batch (all ranks' rows), all rows or a "
                         "fixed, seeded sample of them "
                         f"(at most {DUMP_DZ_BYTES >> 20} MiB); the inputs are seeded, so two builds compare file "
                         "for file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "loss"):
        ap.error("--dump-outputs writes the outputs of --impl ours --workload loss only")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(tflops=float(p["bf16_tflops"]), tflops_sustained=float(p.get("bf16_tflops_sustained", 0)),
                    hbm_gbs=float(p["hbm_gbs"]), source="measured")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nme, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def traffic_bytes(kernel, args, world):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/), when the
    workload is the one that was profiled; None otherwise."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not (os.path.isfile(path) and world == 1 and args.n == 65536 and args.d == 256 and args.dtype == "bf16"
            and args.similarity == "cosine" and args.alpha == 0.0 and args.lambda_uni == 0.0):
        return None
    with open(path) as f:
        return json.load(f).get(kernel, {}).get("dram_bytes")


def synth(n, d, dtype, seed=1337):
    """Unit-norm embeddings + balanced binary labels (SURVEY 8d), generated on the host."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    z = torch.nn.functional.normalize(x, dim=1).to(dtype)
    y = torch.zeros(n, dtype=torch.int64)
    y[torch.randperm(n, generator=g)[: n // 2]] = 1
    return z, y


def dump_outputs(out_dir, loss, dz):
    """Write the loss and d loss / d z of one step as float32 .npy files.  dz keeps all its rows when they fit
    DUMP_DZ_BYTES, else a sample of rows that depends only on the shape (fixed seed, ascending order)."""
    import numpy as np
    import torch
    rows, cols = dz.shape
    keep = max(1, DUMP_DZ_BYTES // (4 * cols))
    if rows > keep:
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        dz = dz[idx.to(dz.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "dz.npy"), dz.detach().float().cpu().numpy())


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_loss(args):
    """The CPU implementation that stands for the reference: the UNMODIFIED loss.py when it is reachable
    (oracle/_ref staged by oracle/build_ref.py, or /root/reference in the build container; kind "reference"),
    else the oracle's per-anchor port of it (kind "port").  Returns (callable(z, y) -> loss, kind, description)."""
    from oracle import ref_loader as R
    if R.reference_available():
        mod = R.load_reference_module("loss")
        fn = mod.SupConBinaryLoss(temperature=args.tau, similarity=args.similarity,
                                  uniformity_weight=args.lambda_uni, uniformity_t=2.0)
        return (lambda z, y: fn(z, y, topk_neg=args.topk, alpha=args.alpha)), "reference", \
            f"unmodified loss.py:110-153 ({R.reference_kind()})"
    from oracle import supcon_oracle as O
    return (lambda z, y: O.anchor_loop_loss(z, y, temperature=args.tau, similarity=args.similarity,
                                            uniformity_weight=args.lambda_uni, uniformity_t=2.0,
                                            topk_neg=args.topk, alpha=args.alpha)), "port", \
        "per-anchor loop port of loss.py (oracle/supcon_oracle.py)"


def cpu_ref_step(loss_fn, x, y):
    """One fwd+bwd as the reference's caller runs it (stage1_utils.py:123-128): F.normalize -> loss -> backward.
    Returns (fwd seconds, bwd seconds)."""
    import torch
    xx = x.clone().requires_grad_(True)
    t0 = time.perf_counter()
    loss = loss_fn(torch.nn.functional.normalize(xx, p=2, dim=1), y)
    t1 = time.perf_counter()
    loss.backward()
    return t1 - t0, time.perf_counter() - t1


def cpu_reference_table(args, loss_fn, budget_s=150.0):
    """BASELINE.md section 3: literal loss at N in {64, 256, 1024, 2048}, 1 thread and all cores, fwd / bwd split,
    median of the timed runs after one warm-up; rows are dropped once the time budget is spent."""
    import torch
    cores = os.cpu_count() or 1
    rows, t_start = [], time.perf_counter()
    for n, reps in ((64, 5), (256, 5), (1024, 3), (2048, 1)):
        g = torch.Generator().manual_seed(1337)
        x = torch.randn(n, args.d, generator=g)
        y = torch.zeros(n, dtype=torch.int64)
        y[torch.randperm(n, generator=g)[: n // 2]] = 1
        for threads in (1, cores):
            if time.perf_counter() - t_start > budget_s:
                return rows
            torch.set_num_threads(threads)
            if n <= 1024:
                cpu_ref_step(loss_fn, x, y)
            ts = [cpu_ref_step(loss_fn, x, y) for _ in range(reps)]
            f, b = statistics.median(t[0] for t in ts), statistics.median(t[1] for t in ts)
            rows.append({"N": n, "threads": threads, "fwd_ms": round(1e3 * f, 2), "bwd_ms": round(1e3 * b, 2),
                         "pairs_per_s": n * n / (f + b), "runs": reps, "warmup": 1 if n <= 1024 else 0})
    torch.set_num_threads(cores)
    return rows


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (unmodified loss.py behind
    F.normalize) on the box's host cores, all threads, each step one fwd+bwd over a bounded sample (the first
    cpu_sample_n rows/columns) of the workload; plus the BASELINE.md table (N, threads, fwd/bwd split)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    loss_fn, kind, what = cpu_reference_loss(args)
    n = min(args.cpu_sample_n, args.n)
    z, y = synth(n, args.d, torch.float32)
    for _ in range(args.warmup):
        cpu_ref_step(loss_fn, z, y)
    times = [cpu_ref_step(loss_fn, z, y) for _ in range(args.steps)]
    t = sum(a + b for a, b in times) / len(times)
    value = n * n / t
    sample = (f"first {n} rows/cols of the workload (N^2 = {n * n} pairs each step), fp32, F.normalize + {what}, "
              f"{cores} threads, fwd {1e3 * statistics.median(a for a, _ in times):.0f} ms + bwd "
              f"{1e3 * statistics.median(b for _, b in times):.0f} ms, torch {torch.__version__}, CPU {cpu_model()}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_model": cpu_model(), "host_cores": cores,
    }
    if not args.no_ref_table:
        line["cpu_table"] = cpu_reference_table(args, loss_fn)
    print(json.dumps(line), flush=True)


def workload_config(args, extra=None):
    cfg = {"workload": f"SupCon {args.similarity} tau={args.tau} N={args.n} d={args.d} {args.dtype} "
                       f"fwd+bwd (BASELINE configs[3])",
           "N": args.n, "d": args.d, "similarity": args.similarity, "tau": args.tau,
           "lambda_uni": args.lambda_uni, "topk": args.topk, "alpha": args.alpha,
           "parallelism": f"rows sharded over {args.gpus} rank(s)",
           "l2_flush": "256 MiB memset between timed iterations, outside the per-step CUDA events",
           "launch": "eager" if args.no_graph else "one CUDA-graph replay per step"}
    if extra:
        cfg.update(extra)
    return cfg


def run_stage1(args):
    """BASELINE configs[4] through the reference's UNCHANGED callers (oracle/_ref, staged verbatim by
    oracle/build_ref.py): encoder.Wav2Vec2Encoder (encoder.py:11-70) on a random-init XLS-R-300M saved locally
    (no checkpoints offline), compression_module.CompressionModule(1024, 256, 0.1) and
    stage1_utils.train_one_epoch (stage1_utils.py:102-134) over synthetic 4 s / 16 kHz audio, batch 64 per GPU,
    frozen encoder (CLI default finetune_encoder=0, stage1_config.py:30), AdamW on the head.  Several GPUs exactly as
    train_stage1.py:82-84 does it: nn.DataParallel over encoder and head in ONE process, so the loss sees the
    gathered batch (64 x n_gpus) on cuda:0.  The only thing that changes between the two timed runs is which
    object is passed as loss_fn: the reference's loss.py class or this repo's drop-in.  Reports ms/step and the
    loss's share of the step (loss fwd+bwd alone on the same embeddings, host-inclusive)."""
    import tempfile
    from types import SimpleNamespace
    import torch
    from transformers import Wav2Vec2Config, Wav2Vec2Model
    from wav2vec_contr_loss_b200 import build as _build
    _build.build()
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from oracle import ref_loader as R
    root = R.reference_root()
    if root is None:
        print(json.dumps({"workload": "stage1_step", "unavailable": "reference not staged (oracle/_ref missing)"}))
        return
    sys.path.insert(0, root)
    import compression_module as ref_head      # noqa: E402  (the reference's own files, unedited)
    import encoder as ref_encoder              # noqa: E402
    import stage1_utils as ref_utils           # noqa: E402
    ref_loss = R.load_reference_module("loss")

    ngpu = max(1, min(args.gpus, torch.cuda.device_count()))
    dev = torch.device("cuda")                  # as train_stage1.py:28
    ref_utils.set_seed(1337)
    cfg_m = Wav2Vec2Config(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                           feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True, conv_dim=(512,) * 7,
                           conv_stride=(5, 2, 2, 2, 2, 2, 2), conv_kernel=(10, 3, 3, 3, 3, 2, 2),
                           num_conv_pos_embeddings=128, num_conv_pos_embedding_groups=16, layerdrop=0.0)
    tmp = tempfile.mkdtemp(prefix="xlsr300m_random_")
    Wav2Vec2Model(cfg_m).save_pretrained(tmp)
    enc = ref_encoder.Wav2Vec2Encoder(model_name=tmp, freeze_encoder=True).to(dev)
    n_params = sum(p_.numel() for p_ in enc.parameters())
    B = args.stage1_batch * ngpu
    g = torch.Generator().manual_seed(1337)
    steps = args.steps
    batches = [(torch.randn(B, 64000, generator=g), (torch.arange(B) % 2).long()) for _ in range(steps)]
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=args.topk, warmup_epochs=0,
                          alpha_ramp_epochs=1, alpha_end=args.alpha)      # epoch 1 -> alpha = alpha_end

    def make_loss(kind):
        cls = ref_loss.SupConBinaryLoss if kind == "reference_loss_py" else SupConBinaryLoss
        return cls(temperature=args.tau, similarity=args.similarity, uniformity_weight=args.lambda_uni,
                   uniformity_t=2.0)

    result = {"workload": "stage1_step (BASELINE configs[4])", "n_gpus": ngpu, "batch_per_gpu": args.stage1_batch,
              "global_batch": B, "encoder": f"random-init XLS-R-300M ({n_params / 1e6:.1f} M params), frozen",
              "callers": "UNCHANGED reference files from oracle/_ref: encoder.Wav2Vec2Encoder, "
                         "compression_module.CompressionModule, stage1_utils.train_one_epoch"
                         + ("; nn.DataParallel over encoder and head as train_stage1.py:82-84" if ngpu > 1 else ""),
              "audio": "synthetic 4 s @ 16 kHz", "similarity": args.similarity, "tau": args.tau, "topk": args.topk,
              "alpha": cfg.alpha_end, "timed_steps": steps, "step_ms": {}, "loss_fwd_bwd_ms": {},
              "loss_share_of_step": {}, "epoch_mean_loss": {}}
    z_fixed = None
    for kind in ("b200_dropin", "reference_loss_py"):
        ref_utils.set_seed(1337)
        head = ref_head.CompressionModule(1024, 256, 0.1).to(dev)
        e_run, h_run = enc, head
        if ngpu > 1:
            e_run = torch.nn.DataParallel(enc, device_ids=list(range(ngpu)))
            h_run = torch.nn.DataParallel(head, device_ids=list(range(ngpu)))
        opt = torch.optim.AdamW([{"params": h_run.parameters(), "lr": 1e-4}], weight_decay=3e-3)
        loss_fn = make_loss(kind)
        ref_utils.train_one_epoch(e_run, h_run, loss_fn, batches[:2], opt, dev, 1, cfg)      # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        avg, _ = ref_utils.train_one_epoch(e_run, h_run, loss_fn, batches, opt, dev, 1, cfg)
        torch.cuda.synchronize()
        result["step_ms"][kind] = 1e3 * (time.perf_counter() - t0) / steps
        result["epoch_mean_loss"][kind] = avg
        if z_fixed is None:
            with torch.no_grad():
                w = batches[0][0].to(dev)
                hs = e_run(w, attention_mask=(w != 0.0).long())
                z_fixed = torch.nn.functional.normalize(h_run(hs).mean(dim=-1), p=2, dim=1).detach()
        y = batches[0][1].to(dev)

        def loss_only():
            zz = z_fixed.clone().requires_grad_(True)
            loss_fn(zz, y, topk_neg=cfg.topk_neg, alpha=cfg.alpha_end).backward()
        loss_only()
        torch.cuda.synchronize()
        reps = 20 if kind == "b200_dropin" else 3
        t0 = time.perf_counter()
        for _ in range(reps):
            loss_only()
        torch.cuda.synchronize()
        result["loss_fwd_bwd_ms"][kind] = 1e3 * (time.perf_counter() - t0) / reps
        result["loss_share_of_step"][kind] = result["loss_fwd_bwd_ms"][kind] / result["step_ms"][kind]
    print(json.dumps(result), flush=True)


def main():
    args = parse()
    if args.workload == "stage1":
        run_stage1(args)
        return
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from wav2vec_contr_loss_b200 import build as _build
    _build.build()
    from wav2vec_contr_loss_b200 import SupConBinaryLoss, _cabi
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss, exchange_stats, gather_inputs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    tdtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    if args.scaling == "weak" and world > 1:
        # per-GPU work (N^2 / R pairs) held at the single-GPU workload's: N grows like sqrt(R)
        unit = 256 * world
        args.n = int(round(args.n * (world ** 0.5) / unit)) * unit
    n, d = args.n, args.d
    assert n % world == 0
    n_local = n // world
    z_host, y_host = synth(n, d, tdtype)
    zl_host = z_host[rank * n_local:(rank + 1) * n_local].contiguous().pin_memory()
    yl_host = y_host[rank * n_local:(rank + 1) * n_local].to(torch.int32).contiguous().pin_memory()
    z_local = zl_host.to(dev)
    y_local = yl_host.to(dev)
    sim_id = Fn.similarity_id(args.similarity)
    flags = args.flags | _cabi.FLAG_UNIT_ROWS          # synth() L2-normalises the rows
    kw = dict(tau=args.tau, similarity=sim_id, lambda_uni=args.lambda_uni, uni_t=2.0, topk=args.topk,
              alpha=args.alpha, flags=flags)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # The timed step IS the drop-in boundary: the loss module called like stage1_utils.py:125-128 calls the
    # reference's -- loss = loss_fn(z, labels, topk_neg=..., alpha=...); loss.backward() -- on one GPU
    # SupConBinaryLoss, on several ShardedSupConLoss (same signature, rows of the global batch per rank).
    cls = ShardedSupConLoss if world > 1 else SupConBinaryLoss
    extra_kw = {"exchange": args.exchange} if world > 1 else {}
    loss_fn = cls(temperature=args.tau, similarity=args.similarity, uniformity_weight=args.lambda_uni, uniformity_t=2.0,
                  **extra_kw)
    loss_fn.kernel_flags = args.flags
    loss_fn.assume_unit_rows = True
    # kernels of libsupcon_b200.so per step on the tensor path.  One GPU: prep_fwd, label_table, class_sum,
    # class_reduce, tc_fwd (class-sum variant + its per-pair twin, one of which returns at once), merge,
    # prep_bwd, tc_bwd, reduce.  Several ranks: forward in two phases (prep + label_table + tc_fwd twice, merge),
    # finalize_sets, backward in two phases (prep_bwd + tc_bwd twice), reduce.
    # Peer exchange: push, forward in two phases (7), wait, push, wait, finalize_sets, backward (3), end_step = 16.
    # The single-phase backward of >= 2^30 pairs adds label_table, class_sum, class_reduce and its own twin.
    # (one GPU: the module hands the forward's workspace to the backward, which then only adds its twin.)
    class_sums = args.similarity == "cosine" and args.alpha == 0.0
    bwd_plin = class_sums and n_local * n >= (1 << 30)
    bwd_extra = 4 if bwd_plin else 0
    launches_per_step = (7 + (4 if bwd_plin else 0)) if world == 1 else 14   # fwd +3, bwd +1 (its twin)
    launches = {"count": 0}

    def step(z_loc, y_loc):
        """fwd + bwd through the module and autograd; returns (loss, d loss / d z_local)."""
        z = z_loc.detach().requires_grad_(True)
        loss = loss_fn(z, y_loc, topk_neg=args.topk, alpha=args.alpha)
        (dz,) = torch.autograd.grad(loss, z)
        launches["count"] += launches_per_step
        return loss, dz

    class Stepper:
        """One step = one CUDA-graph replay (captured once, NCCL collectives included) unless --no-graph."""

        def __init__(self, fn):
            self.fn, self.graph, self.out = fn, None, None
            if not args.no_graph:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    fn()
                    torch.cuda.synchronize()
                    if world > 1:
                        dist.barrier()
                    self.graph = torch.cuda.CUDAGraph()
                    n0 = launches["count"]
                    with torch.cuda.graph(self.graph, stream=side, capture_error_mode="thread_local"):
                        self.out = fn()
                    self.per_step = launches["count"] - n0
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()

        def __call__(self):
            if self.graph is None:
                return self.fn()
            self.graph.replay()
            launches["count"] += self.per_step
            return self.out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(z_local, y_local)
    barrier()
    exchange_used = "none"
    if world > 1:
        exchange_used = "peer" if any(v is not None for v in loss_fn._peers.values()) else "nccl"
        if exchange_used == "peer":
            launches_per_step = 16 + bwd_extra

    # ---- host-inclusive time of the same call issued eagerly from Python (SURVEY 8d: both figures) ----
    def eager_ms(fn, reps):
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0) / reps
    eager_step_ms = eager_ms(lambda: step(z_local, y_local), min(args.steps, 10))

    resident = Stepper(lambda: step(z_local, y_local))

    def e2e_step():
        zl = zl_host.to(dev, non_blocking=True)
        yl = yl_host.to(dev, non_blocking=True)
        loss, dz = step(zl, yl)
        loss_host.copy_(loss.float(), non_blocking=True)
        return loss, dz

    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    e2e = Stepper(e2e_step)
    for _ in range(2):
        resident(); e2e()
    barrier()

    # ---- device-resident timing: K steps, per-step CUDA events, L2 flushed between steps ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches["count"] = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in ev:
        flush.zero_()
        s.record()
        loss, dz = resident()
        e.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    n_launch = launches["count"]
    ms = [s.elapsed_time(e) for s, e in ev]
    t_local = sum(ms) / len(ms)
    tt = torch.tensor([t_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_per_step = float(tt)
    if args.dump_outputs:
        dz_all = dz
        if world > 1:       # the row shards in rank order: dz of the whole batch, whatever the number of ranks
            parts = [torch.empty_like(dz) for _ in range(world)]
            dist.all_gather(parts, dz.contiguous())
            dz_all = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, loss, dz_all)

    # ---- end-to-end: pinned host inputs -> H2D -> fwd+bwd -> loss D2H, every step ----
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in ev2:
        flush.zero_()
        s.record()
        e2e()
        e.record()
    barrier()
    t2 = torch.tensor([sum(s.elapsed_time(e) for s, e in ev2) / len(ev2)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_ms = float(t2)

    # ---- per-kernel durations for the roofline: forward-only and backward-only CUDA graphs over this rank's
    #      row block (direct C-ABI wrappers), CUDA events on the launching stream ----
    prob_t = Fn.make_problem(n, d, Fn._dtype_id(z_local), row_offset=rank * n_local, n_rows=n_local, **kw)
    if world > 1:
        z_all_t, y_all_t = gather_inputs(z_local, y_local)
    else:
        z_all_t, y_all_t = z_local, y_local
    stats_t, partials_t, _ = Fn.forward_rows(z_all_t, y_all_t, prob_t, want_loss=(world == 1))
    if world > 1:
        stats_all_t = exchange_stats(partials_t, stats_t)
    else:
        stats_all_t = stats_t
    barrier()
    fwd_only = Stepper(lambda: Fn.forward_rows(z_all_t, y_all_t, prob_t, want_loss=(world == 1)))
    bwd_only = Stepper(lambda: Fn.backward_rows(z_all_t, y_all_t, stats_all_t, partials_t, None, prob_t, out_dtype=tdtype))
    reps = min(args.steps, 10)

    def time_graph(stepper, reps=reps, do_flush=True):
        tot = 0.0
        for _ in range(reps):
            if do_flush:
                flush.zero_()
            s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_.record(); stepper(); e_.record()
            torch.cuda.synchronize()
            tot += s_.elapsed_time(e_)
        return tot / reps

    def graph_us_back_to_back(stepper, reps_):
        """device time per replay in steady state: reps_ replays between ONE pair of events (small batches: the
        per-replay event pair and sync of time_graph would add the graph-launch latency to a 25 us kernel)"""
        for _ in range(3):
            stepper()
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s_.record()
        for _ in range(reps_):
            stepper()
        e_.record()
        torch.cuda.synchronize()
        return 1e3 * s_.elapsed_time(e_) / reps_

    n_before = launches["count"]
    fwd_ms = time_graph(fwd_only)
    bwd_ms = time_graph(bwd_only)
    launches["count"] = n_before
    barrier()

    # ---- other configurations of BASELINE.json through the same module (one GPU only; reported, not the metric) ----
    extras = None
    if world == 1 and not args.no_extras:
        def module_case(nn_, dtype, similarity, lam, topk, alpha, reps_):
            zc, yc = synth(nn_, d, dtype)
            zc, yc = zc.to(dev), yc.to(dev)
            fn_ = SupConBinaryLoss(temperature=args.tau, similarity=similarity, uniformity_weight=lam, uniformity_t=2.0)
            fn_.assume_unit_rows = True

            def one():
                zz = zc.detach().requires_grad_(True)
                ls = fn_(zz, yc, topk_neg=topk, alpha=alpha)
                torch.autograd.grad(ls, zz)
                return ls
            for _ in range(3):
                one()
            host_ms = eager_ms(one, reps_)
            return {"device_us": round(graph_us_back_to_back(Stepper(one), reps_), 2),
                    "host_inclusive_us": round(1e3 * host_ms, 2)}
        def cabi_case(nn_):     # supcon_loss_and_grad through the C-ABI wrapper: the kernel(s) alone, no autograd glue
            zc, yc = synth(nn_, d, torch.float32)
            zc, yc = zc.to(dev), yc.to(dev).to(torch.int32)
            pr = Fn.make_problem(nn_, d, _cabi.F32, tau=args.tau, similarity=sim_id, topk=15, alpha=0.0)
            one = lambda: Fn.loss_and_grad(zc, yc, pr, want_grad=True)
            for _ in range(3):
                one()
            return round(graph_us_back_to_back(Stepper(one), 50), 2)
        extras = {
            "n64_cabi_single_launch_us": cabi_case(64),      # the <30 us target of the north_star: one cluster launch
            "n256_cabi_single_launch_us": cabi_case(256),    # the reference's default batch (stage1_config.py:22), fp32
            "n64_fwd_bwd_us": module_case(64, torch.float32, "cosine", 0.0, 15, 0.0, 50),               # configs[0]
            "n64_geodesic_uniformity_us": module_case(64, torch.float32, "geodesic", 0.05, 15, 0.0, 50),  # configs[1]
            "n1024_mined_f32_us": module_case(1024, torch.float32, "cosine", 0.0, 15, 0.5, 20),           # configs[2]
            "n1024_mined_bf16_us": module_case(1024, torch.bfloat16, "cosine", 0.0, 15, 0.5, 20),
            "n65536_mined_bf16_us": module_case(65536, torch.bfloat16, "cosine", 0.0, 15, 0.5, 5),
            "note": "fwd+bwd through SupConBinaryLoss + autograd (label cast, the loss kernels, grad_out fill and "
                    "scaling); device_us = CUDA-graph replays back to back between one pair of CUDA events, "
                    "host_inclusive_us = eager Python call, wall clock incl. launch overhead; *_cabi_* = "
                    "supcon_loss_and_grad alone (one cluster launch at these sizes), graph replays back to back",
        }
        launches["count"] = n_before

    # ---- several ranks: the same step once more at WEAK scaling (the north_star's 8-GPU target is stated for weak
    #      scaling; BASELINE configs[3], the headline above, is the fixed N = 65536, i.e. strong) ----
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_weak_leg:
        try:
            unit = 256 * world
            n_w = int(round(args.n * (world ** 0.5) / unit)) * unit
            nl_w = n_w // world
            zw_host, yw_host = synth(n_w, d, tdtype)
            zw = zw_host[rank * nl_w:(rank + 1) * nl_w].contiguous().to(dev)
            yw = yw_host[rank * nl_w:(rank + 1) * nl_w].to(torch.int32).contiguous().to(dev)
            del zw_host, yw_host
            loss_w = cls(temperature=args.tau, similarity=args.similarity, uniformity_weight=args.lambda_uni,
                         uniformity_t=2.0, **extra_kw)
            loss_w.kernel_flags = args.flags
            loss_w.assume_unit_rows = True

            def step_w():
                zz = zw.detach().requires_grad_(True)
                ls = loss_w(zz, yw, topk_neg=args.topk, alpha=args.alpha)
                (g_,) = torch.autograd.grad(ls, zz)
                return ls, g_
            for _ in range(3):
                step_w()
            barrier()
            weak_step = Stepper(step_w)
            for _ in range(2):
                weak_step()
            barrier()
            k_w = max(3, min(args.steps, 10))
            evw = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k_w)]
            for s_, e_ in evw:
                flush.zero_()
                s_.record()
                loss_weak, _ = weak_step()
                e_.record()
            barrier()
            tw = torch.tensor([sum(s_.elapsed_time(e_) for s_, e_ in evw) / k_w], device=dev, dtype=torch.float64)
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
            weak = {"N": n_w, "rows_per_gpu": nl_w, "steps": k_w, "ms_per_step": float(tw),
                    "value": float(n_w) * float(n_w) / (float(tw) * 1e-3), "unit": UNIT,
                    "pairs_per_gpu_vs_single_gpu_workload": float(n_w) * float(n_w) / world / (float(args.n) ** 2),
                    "loss": float(loss_weak),
                    "note": "same module call, exchange, graph replay, L2 flush and max-over-ranks timing as the "
                            "headline, at N = batch-n * sqrt(n_gpus) so that every GPU computes the single-GPU "
                            "workload's number of pairs; weak-scaling efficiency = value / (n_gpus * the 1-GPU value)"}
        except Exception as exc:  # noqa: BLE001  (reported, never fatal for the headline measurement)
            weak = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        pk = peaks()
        pairs = float(n) * float(n)
        flop_per_pair_bwd = (4 + (2 if args.lambda_uni > 0 else 0)) * d   # dz = (G + G^T) z  (+ W z)
        flop_per_pair_fwd = 2 * d
        bwd_tflops = pairs / world * flop_per_pair_bwd / (bwd_ms * 1e-3) / 1e12
        fwd_tflops = pairs / world * flop_per_pair_fwd / (fwd_ms * 1e-3) / 1e12
        total_tflops = pairs * (flop_per_pair_bwd + flop_per_pair_fwd) / (ms_per_step * 1e-3) / 1e12
        cfg = workload_config(args)
        cfg["exchange"] = {"none": "single GPU", "nccl": "NCCL all-gathers (torch.distributed) overlapped with the "
                           "own-column phases of forward and backward",
                           "peer": "peer-memory stores over NVLink by this library's kernels (symmetric memory), "
                                   "rows pushed beside the own-column forward"}[exchange_used]
        cfg["api"] = (f"{cls.__name__}(temperature, similarity, ...)(z, labels, topk_neg, alpha) + autograd backward "
                      f"(the reference's call, stage1_utils.py:125-128); assume_unit_rows=True")
        line = {
            "metric": METRIC, "value": pairs / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": cfg,
            "clocks": clocks,
            "e2e": {"value": pairs / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(zl_host.numel() * zl_host.element_size() + yl_host.numel() * 4),
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms,
                    "dz": f"device-resident ({args.dtype}: autograd returns the gradient in z's dtype; it feeds the "
                          f"normalisation backward on the device, only the scalar loss goes back to the host)"},
            "boundary": {"graph_replay_ms": ms_per_step, "eager_host_inclusive_ms": eager_step_ms,
                         "note": "same module call; eager = issued from Python every step, wall clock with a final sync, "
                                 "no L2 flush between iterations (the graph figure flushes L2 before every step)"},
            "gpu_launches": n_launch,
            "roofline": {"bound": "tensor", "kernel": "tc_bwd_kernel + its O(N) kernels (class sums, prep, reduce): recompute S, dz = (G+G^T) z",
                         "achieved": bwd_tflops, "peak": pk["tflops"], "unit": "TFLOP/s",
                         "frac": bwd_tflops / pk["tflops"], "traffic": traffic_bytes("tc_bwd_kernel", args, world),
                         "peak_source": pk["source"],
                         "launch_ms": bwd_ms,
                         "algorithmic_flops_per_launch": pairs / world * flop_per_pair_bwd},
            "roofline_fwd": {"bound": "tensor", "achieved": fwd_tflops, "peak": pk["tflops"], "unit": "TFLOP/s",
                             "frac": fwd_tflops / pk["tflops"], "launch_ms": fwd_ms},
            "step_tflops": total_tflops, "step_frac_of_bf16_peak": total_tflops / pk["tflops"] / world,
            "loss": float(loss),
        }
        if extras is not None:
            line["extras"] = extras
        if weak is not None:
            line["weak"] = weak
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            loss_ref, kind, what = cpu_reference_loss(args)
            ns = min(args.cpu_sample_n, n)
            g = torch.Generator().manual_seed(1337)
            xc, yc = torch.randn(ns, d, generator=g), y_host[:ns]
            cpu_ref_step(loss_ref, xc, yc)
            tcs = [sum(cpu_ref_step(loss_ref, xc, yc)) for _ in range(3)]
            tc = statistics.median(tcs)
            line["cpu_baseline"] = {"value": ns * ns / tc, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"{ns} rows/cols (N^2 pairs per fwd+bwd), fp32, F.normalize + {what}, "
                                              f"median of 3, {tc:.2f} s per fwd+bwd, CPU {cpu_model()}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tearing the process group down while captured NCCL graphs are alive can block; every rank has
        # finished its work, so synchronise and leave without running the destructors.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
