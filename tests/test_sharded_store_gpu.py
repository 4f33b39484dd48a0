"""GPU: the layer-mean store sharded over the GPUs of a node (feature_store.ShardedLayerMeanStore,
head_sharded_store_pool_fwd_kernel in csrc/supcon_head.cu).

One GPU: the kernel reads R shards through its device table of base addresses wherever they are; here R
allocations on the same GPU stand for R ranks' shards.  Its pooled rows must equal those of the single-store
kernel bit for bit for every index pattern.  A process group of one rank runs the whole Python path on symmetric
memory: the build, the epochs and the graphed step equal those from a LayerMeanStore bit for bit.

Two GPUs (skipped below 2, mp.spawn as in test_multi_gpu.py): each rank builds its shard and reads the other's over
NVLink; pooled rows equal a single-GPU LayerMeanStore's bit for bit, and three epochs with ShardedSupConLoss + GradSync
follow one process training on the merged global batches within the bars of
test_multi_gpu.py::test_two_ranks_nccl_train_like_one_process_on_the_global_batch."""
import copy
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

CFG = dict(finetune_encoder=False, use_rawboost=False, topk_neg=3, warmup_epochs=1, alpha_ramp_epochs=2,
           alpha_end=1.0)


def sharded_pool(bases, ranks, n, feat, frames, idx, p=0.0, rng=None):
    """supcon_head_sharded_store_pool_forward on the shards at the device addresses ``bases``"""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200 import functional as Fn
    pooled = torch.empty((idx.shape[0], feat), dtype=torch.float32, device=idx.device)
    _cabi.check(_cabi.load().supcon_head_sharded_store_pool_forward(
        Fn._p(bases), ranks, n, feat, frames, Fn._p(idx), idx.shape[0], p, 0.01, Fn._p(rng), Fn._p(pooled),
        Fn._stream(idx.device)), "supcon_head_sharded_store_pool_forward")
    return pooled


def shard(rows, ranks):
    """R shard tensors of ceil(n / R) rows (the padding rows NaN) and the device table of their addresses"""
    n, f, t = rows.shape
    local = -(-n // ranks)
    shards = []
    for r in range(ranks):
        s = torch.full((local, f, t), float("nan"), device=rows.device)
        s[: len(range(r, n, ranks))] = rows[r::ranks]
        shards.append(s)
    return shards, torch.tensor([s.data_ptr() for s in shards], dtype=torch.int64, device=rows.device)


def single_store(rows):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    store = LayerMeanStore(rows.shape[0], rows.shape[1], rows.shape[2], rows.device)
    store.rows.copy_(rows)
    store.filled = rows.shape[0]
    return store


def index_patterns(n, ranks, rank, b, g):
    """rows of `rank`'s own shard, of the others', both mixed, repeated, permuted"""
    own = torch.tensor([i for i in range(n) if i % ranks == rank])
    other = torch.tensor([i for i in range(n) if i % ranks != rank]) if ranks > 1 else own
    return {"local": own[torch.randint(0, len(own), (b,), generator=g)],
            "remote": other[torch.randint(0, len(other), (b,), generator=g)],
            "mixed": torch.randperm(n, generator=g)[:b],
            "repeated": torch.full((b,), n - 1).index_put_((torch.arange(0, b, 3),), torch.tensor(0)),
            "permuted": torch.arange(n).flip(0)}


@pytest.mark.parametrize("ranks", [1, 2, 3, 8])
@pytest.mark.parametrize("shape", [(20, 1024, 199), (23, 7, 13), (17, 40, 50), (9, 18, 199)],
                         ids=lambda s: "x".join(map(str, s)))
def test_sharded_pool_equals_single_store(cuda_device, shape, ranks):
    """eval and dropout 0.1, every index pattern seen from every rank: the same bits as the single-store kernel.
    (7, 13) and (18, 199) have runs that are not a multiple of four floats: the scalar path."""
    n, f, t = shape
    if n < ranks:
        pytest.skip("fewer clips than ranks")
    rows = torch.randn(n, f, t, generator=torch.Generator().manual_seed(n + f)).to(cuda_device)
    ref = single_store(rows)
    shards, bases = shard(rows, ranks)
    g = torch.Generator().manual_seed(7)
    rng = torch.tensor([1234, 5], dtype=torch.int64, device=cuda_device)
    for rank in range(ranks):
        for name, idx in index_patterns(n, ranks, rank, 12, g).items():
            idx = idx.to(cuda_device)
            assert torch.equal(sharded_pool(bases, ranks, n, f, t, idx), ref.pool(idx)), (rank, name)
            assert torch.equal(sharded_pool(bases, ranks, n, f, t, idx, 0.1, rng), ref.pool(idx, 0.1, 0.01, rng)), \
                (rank, name)


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_sharded_out_of_range_index_gives_nan_row(cuda_device, p):
    n, f, t = 9, 40, 50
    rows = torch.randn(n, f, t, device=cuda_device)
    shards, bases = shard(rows, 4)
    idx = torch.tensor([0, 9, 5, -1, 2 ** 40, 8, 11, 3], device=cuda_device)   # 11: a padding row of shard 3
    rng = torch.tensor([99, 4], dtype=torch.int64, device=cuda_device)
    got = sharded_pool(bases, 4, n, f, t, idx, p, rng if p else None)
    want = single_store(rows).pool(idx.clamp(0, n - 1), p, 0.01, rng if p else None)
    bad = torch.tensor([False, True, False, True, True, False, True, False], device=cuda_device)
    assert bool(got[bad].isnan().all())
    assert torch.equal(got[~bad], want[~bad])


def test_sharded_offsets_past_32_bits(cuda_device):
    """two shards of 10540 rows of (1024, 199): local rows from 10539 on start past 2^31 elements of their shard"""
    from wav2vec_contr_loss_b200.head import layer_time_pool
    f, t = 1024, 199
    first_high = 2 ** 31 // (f * t) + 1
    local = first_high + 1
    n = 2 * local
    shards = [torch.empty(local, f, t, device=cuda_device) for _ in range(2)]
    assert shards[0].numel() > 2 ** 31
    bases = torch.tensor([s.data_ptr() for s in shards], dtype=torch.int64, device=cuda_device)
    slots = [n - 1, 2 * first_high, 3, 2 * first_high - 1, 0, n - 2, 2 * first_high + 1, 2 * (first_high - 1)]
    torch.manual_seed(5)
    for i in slots:
        shards[i % 2][i // 2].normal_()
    idx = torch.tensor(slots, device=cuda_device)
    hs = torch.stack([shards[i % 2][i // 2] for i in slots]).unsqueeze(1)        # K = 1: the row is the layer mean
    rng = torch.tensor([31, 2], dtype=torch.int64, device=cuda_device)
    assert torch.equal(sharded_pool(bases, 2, n, f, t, idx), layer_time_pool(hs))
    assert torch.equal(sharded_pool(bases, 2, n, f, t, idx, 0.1, rng), layer_time_pool(hs, 0.1, 0.01, rng))


def test_sharded_pool_graph_takes_new_indices(cuda_device):
    n, f, t, b = 30, 64, 20, 16
    rows = torch.randn(n, f, t, device=cuda_device)
    shards, bases = shard(rows, 3)
    ref = single_store(rows)
    g = torch.Generator().manual_seed(1)
    idx = torch.randperm(n, generator=g)[:b].to(cuda_device)
    sharded_pool(bases, 3, n, f, t, idx)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = sharded_pool(bases, 3, n, f, t, idx)
    for _ in range(3):
        idx.copy_(torch.randint(0, n, (b,), generator=g))
        graph.replay()
        assert torch.equal(out, ref.pool(idx))


# ------------------------------------------------------------ the Python path on a process group of one rank

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _init(rank, world, port):
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    return dev


class Identity(torch.nn.Module):
    def forward(self, x, attention_mask=None):
        return x


def clips(n, k, f, t, seed=3):
    g = torch.Generator().manual_seed(seed)
    y = torch.arange(n) % 2
    hs = torch.randn(n, k, f, t, generator=g) + 0.5 * (2.0 * y.view(-1, 1, 1, 1) - 1.0)
    return hs, y, SimpleNamespace(data=[(f"utt{i}", int(v)) for i, v in enumerate(y)])


def loader_of(hs, y, slots, batch=10):
    slots = list(slots)
    return [(hs[slots[s:s + batch]], y[slots[s:s + batch]]) for s in range(0, len(slots), batch)]


def make_head(feat, p, dev, seed=4):
    from wav2vec_contr_loss_b200 import FusedCompressionHead
    torch.manual_seed(seed)
    return FusedCompressionHead(feat, 16, p).to(dev)


def weights(head):
    return torch.cat([p.detach().reshape(-1) for p in head.parameters()]).double().cpu()


def _one_rank(rank, world, port, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import (ShardedLayerMeanStore, build_layer_mean_store,
                                                       build_sharded_layer_mean_store, shard_slots)
    from wav2vec_contr_loss_b200.head import layer_time_pool
    dev = _init(rank, world, port)
    try:
        res = {}
        n, k, f, t = 96, 3, 16, 12
        hs, y, ds = clips(n, k, f, t)
        sharded = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, shard_slots(n, 0, 1)), dev, n=n)
        single = build_layer_mean_store(Identity(), loader_of(hs, y, range(n), batch=20), dev, n=n)
        res["build"] = (sharded.filled, sharded.n, torch.equal(sharded.rows, single.rows),
                        torch.equal(sharded.labels, single.labels))
        # three epochs (dropout 0.1) and evaluations from each store: the same bits
        cfg = SimpleNamespace(**CFG)
        heads = [make_head(f, 0.1, dev), None]
        heads[1] = copy.deepcopy(heads[0])
        opts = [torch.optim.AdamW(h.parameters(), lr=5e-3, weight_decay=3e-3) for h in heads]
        losses = [SupConBinaryLoss(0.1, "cosine", 0.05, 2.0) for _ in heads]
        samplers = [S.BalancedBatchSampler(ds, 16, seed=13) for _ in heads]
        dev_batches = [list(range(i, i + 12)) for i in range(0, 36, 12)]
        hist = [[], []]
        for epoch in (1, 2, 3):
            for j, store in enumerate((single, sharded)):
                samplers[j].set_epoch(epoch)
                sync = S.GradSync(heads[j].parameters()) if j else None
                tr = S.train_one_epoch_from_store(heads[j], losses[j], store, list(samplers[j]), opts[j], dev, epoch,
                                                  cfg, grad_sync=sync)
                ev = S.evaluate_from_store(heads[j], losses[j], store, dev_batches, dev, cfg)
                hist[j].append((tr, ev))
        res["epochs"] = (hist[0] == hist[1], torch.equal(weights(heads[0]), weights(heads[1])))
        # graphed steps from the sharded store follow the eager ones
        res["graphed"] = _graphed_vs_eager(sharded, f, dev, grad_sync=False)
        sharded.close()
        try:
            sharded.pool(torch.zeros(1, dtype=torch.int64, device=dev))
            res["closed"] = "no error"
        except RuntimeError as exc:
            res["closed"] = str(exc)
        # a symmetric allocation of 20 GB: 25 k clips of (1024, 199)
        big = ShardedLayerMeanStore(25000, 1024, 199, dev)
        slots = torch.tensor([24999, 0, 12345, 24998], device=dev)
        torch.manual_seed(9)
        for i in slots.tolist():
            big.rows[i].normal_()
        big.filled = 25000
        res["big"] = (big.rows.numel() * 4 / 1e9,
                      torch.equal(big.pool(slots), layer_time_pool(big.rows[slots].unsqueeze(1))))
        big.close()
        out[rank] = res
    finally:
        dist.destroy_process_group()


def _graphed_vs_eager(store, feat, dev, grad_sync):
    """five steps (dropout 0.1, alpha 0 / 0.5) eagerly and as GraphedHeadStep(store=) replays, on this rank's own
    batches; returns (eager losses, graphed losses, eager weights, graphed weights, equal dropout streams)"""
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss
    g = torch.Generator().manual_seed(5)
    idx = [torch.randperm(store.n, generator=g)[:32].to(dev) for _ in range(5)]
    alphas = [0.0, 0.0, 0.5, 0.5, 0.0]
    head_e = make_head(feat, 0.1, dev).train()
    head_g = copy.deepcopy(head_e)
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    opt_g = torch.optim.AdamW(head_g.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    loss_e, loss_g = ShardedSupConLoss(0.1, "cosine", 0.05, 2.0), ShardedSupConLoss(0.1, "cosine", 0.05, 2.0)
    sync_e = S.GradSync(head_e.parameters()) if grad_sync else None
    eager = []
    for s, alpha in enumerate(alphas):
        z = Fn.l2_normalize(head_e.pooled_embedding_from_store(store, idx[s]))
        loss = loss_e(z, store.labels_of(idx[s]), topk_neg=7, alpha=alpha)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        if sync_e is not None:
            sync_e()
        torch.nn.utils.clip_grad_norm_(head_e.parameters(), 5.0)
        opt_e.step()
        eager.append(float(loss))
    step = S.GraphedHeadStep(head_g, loss_g, opt_g, idx[0], topk_neg=7, store=store,
                             grad_sync=S.GradSync(head_g.parameters()) if grad_sync else None)
    graphed = [float(step(idx[s], alpha=alpha)) for s, alpha in enumerate(alphas)]
    torch.cuda.synchronize()
    return eager, graphed, weights(head_e), weights(head_g), head_e.rng_state.tolist() == head_g.rng_state.tolist()


def _check_graphed(res):
    eager, graphed, w_e, w_g, same_stream = res
    assert same_stream
    assert graphed == pytest.approx(eager, rel=1e-5)
    assert torch.allclose(w_g, w_e, rtol=1e-4, atol=1e-6)


def test_one_rank_store_on_symmetric_memory(cuda_device):
    """world size 1: the build, three epochs + evaluations and the graphed step from a ShardedLayerMeanStore equal
    those from a LayerMeanStore; a 20 GB symmetric shard allocates and pools; a closed store refuses to pool"""
    out = mp.Manager().dict()
    mp.spawn(_one_rank, args=(1, _free_port(), out), nprocs=1, join=True)
    res = out[0]
    assert res["build"] == (96, 96, True, True)
    assert res["epochs"] == (True, True)
    _check_graphed(res["graphed"])
    assert res["closed"] == "the sharded store is closed"
    assert res["big"][0] > 20 and res["big"][1]


# --------------------------------------------------------------------------------------------- two ranks

WORLD = 2


def _need_two_gpus():
    if torch.cuda.device_count() < WORLD:
        pytest.skip(f"needs {WORLD} GPUs (have {torch.cuda.device_count()})")


def _two_ranks(rank, world, port, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss
    from wav2vec_contr_loss_b200.feature_store import ShardedLayerMeanStore, build_sharded_layer_mean_store, shard_slots
    from wav2vec_contr_loss_b200.head import layer_time_pool
    dev = _init(rank, world, port)
    try:
        res = {}
        # pooled rows against a single-GPU LayerMeanStore of the same hs, built on every rank
        for (n, k, f, t) in [(21, 3, 1024, 199), (23, 2, 7, 13), (18, 3, 40, 50)]:
            hs, y, _ = clips(n, k, f, t, seed=n)
            sharded = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, shard_slots(n, rank, world), 4),
                                                     dev, n=n)
            single = single_store_of(hs.to(dev), y.to(dev))
            ok = [sharded.filled == n, torch.equal(sharded.labels, single.labels)]
            g = torch.Generator().manual_seed(7)
            rng = torch.tensor([77, 3], dtype=torch.int64, device=dev)
            for idx in index_patterns(n, world, rank, 12, g).values():
                idx = idx.to(dev)
                ok.append(torch.equal(sharded.pool(idx), single.pool(idx)))
                ok.append(torch.equal(sharded.pool(idx, 0.1, 0.01, rng), single.pool(idx, 0.1, 0.01, rng)))
                ok.append(torch.equal(sharded.labels_of(idx), single.labels_of(idx)))
            bad = torch.tensor([0, n, 1, -1, 2 ** 40, n - 1], device=dev)
            got = sharded.pool(bad, 0.1, 0.01, rng)
            want = single.pool(bad.clamp(0, n - 1), 0.1, 0.01, rng)
            keep = torch.tensor([True, False, True, False, False, True], device=dev)
            ok += [bool(got[~keep].isnan().all()), torch.equal(got[keep], want[keep])]
            res[f"pool/{f}x{t}"] = ok
            sharded.close()
        # a peer offset past 2^31 elements: shards of 10540 rows of (1024, 199)
        f, t = 1024, 199
        local = 2 ** 31 // (f * t) + 2
        n = world * local
        big = ShardedLayerMeanStore(n, f, t, dev)
        slots = [n - 1, n - 2, world * (local - 2) + 1, 0, 1, world * (local - 1)]
        for i in slots:
            gen = torch.Generator(device=dev).manual_seed(1000 + i)
            row = torch.randn(f, t, generator=gen, device=dev)
            if i % world == rank:
                big.rows[i // world].copy_(row)
        torch.cuda.synchronize(dev)
        dist.barrier()
        big.filled = n
        hs = torch.stack([torch.randn(f, t, generator=torch.Generator(device=dev).manual_seed(1000 + i), device=dev)
                          for i in slots]).unsqueeze(1)
        idx = torch.tensor(slots, device=dev)
        rng = torch.tensor([5, 1], dtype=torch.int64, device=dev)
        res["past_2^31"] = [torch.equal(big.pool(idx), layer_time_pool(hs)),
                            torch.equal(big.pool(idx, 0.1, 0.01, rng), layer_time_pool(hs, 0.1, 0.01, rng))]
        big.close()
        # three epochs, dropout 0, global-batch loss from the sharded store
        n, k, f, t = 96, 3, 16, 12
        hs, y, ds = clips(n, k, f, t)
        store = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, shard_slots(n, rank, world)), dev, n=n)
        head = make_head(f, 0.0, dev)
        opt = torch.optim.AdamW(head.parameters(), lr=5e-3, weight_decay=3e-3)
        loss_fn = ShardedSupConLoss(0.1, "cosine", 0.05, 2.0)
        sampler = S.BalancedBatchSampler(ds, 8, seed=5, rank=rank, world_size=world)
        dev_batches = [list(range(i + 6 * rank, i + 6 * rank + 6)) for i in range(0, 36, 12)]
        history = []
        for epoch in (1, 2, 3):
            sampler.set_epoch(epoch)
            batches = list(sampler)
            tr = S.train_one_epoch_from_store(head, loss_fn, store, batches, opt, dev, epoch, SimpleNamespace(**CFG),
                                              grad_sync=S.GradSync(head.parameters()))
            ev = S.evaluate_from_store(head, loss_fn, store, dev_batches, dev, SimpleNamespace(**CFG))
            history.append((len(batches), tr, ev))
        res["epochs"] = (history, weights(head))
        res["graphed"] = _graphed_vs_eager(store, f, dev, grad_sync=True)
        store.close()
        out[rank] = res
    finally:
        dist.destroy_process_group()


def single_store_of(hs, y):
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    return build_layer_mean_store(Identity(), loader_of(hs, y, range(hs.shape[0]), 7), hs.device, n=hs.shape[0])


def test_two_ranks_sharded_store(cuda_device):
    _need_two_gpus()
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    out = mp.Manager().dict()
    mp.spawn(_two_ranks, args=(WORLD, _free_port(), out), nprocs=WORLD, join=True)
    for rank in range(WORLD):
        for key, ok in out[rank].items():
            if key.startswith("pool/") or key == "past_2^31":
                assert all(ok), (rank, key, ok)
        _check_graphed(out[rank]["graphed"])

    # one process, one single-GPU store, the merged global batches
    n, k, f, t = 96, 3, 16, 12
    hs, y, ds = clips(n, k, f, t)
    store = single_store_of(hs.to(cuda_device), y.to(cuda_device))
    head = make_head(f, 0.0, cuda_device)
    opt = torch.optim.AdamW(head.parameters(), lr=5e-3, weight_decay=3e-3)
    loss_fn = SupConBinaryLoss(0.1, "cosine", 0.05, 2.0)
    sampler = S.BalancedBatchSampler(ds, 8, seed=5)
    dev_batches = [list(range(i, i + 12)) for i in range(0, 36, 12)]
    want = []
    for epoch in (1, 2, 3):
        sampler.set_epoch(epoch)
        batches = list(sampler)
        steps = len(batches) // WORLD
        merged = [sum((batches[s * WORLD + r] for r in range(WORLD)), []) for s in range(steps)]
        tr = S.train_one_epoch_from_store(head, loss_fn, store, merged, opt, cuda_device, epoch, SimpleNamespace(**CFG))
        ev = S.evaluate_from_store(head, loss_fn, store, dev_batches, cuda_device, SimpleNamespace(**CFG))
        want.append((steps, tr, ev))
    for rank in range(WORLD):
        history, got_w = out[rank]["epochs"]
        for (steps, (avg, alpha), ev), (w_steps, (w_avg, w_alpha), w_ev) in zip(history, want):
            assert steps == w_steps and alpha == w_alpha
            assert avg == pytest.approx(w_avg, rel=1e-5) and ev == pytest.approx(w_ev, rel=1e-5)
        assert torch.allclose(got_w, weights(head), rtol=1e-4, atol=1e-6)
    assert torch.equal(out[0]["epochs"][1], out[1]["epochs"][1])          # the replicas stay identical
