"""GPU: the layer-mean store kept in fp16 (feature_store ``dtype=torch.float16``, head_store_pool_fwd_kernel<__half>
and head_sharded_store_pool_fwd_kernel<__half> in csrc/supcon_head.cu).

The contract: pooling an fp16 store gives bit for bit what pooling an fp32 store gives when that fp32 store holds the
same fp16 values widened (``LayerMeanStore.from_arrays(rows16.float())``): the kernel widens each element exactly and
runs the fp32 body after the load.  An fp16 store's rows are the fp32 build's rows rounded to nearest even
(``.half()``).  Against the fp32 store of the same clips the pooled values differ only by that rounding, within the
bound stated in test_pooled_error_within_bound_of_fp32_store.  Sharded fp16 stores (R allocations on one GPU standing
for R ranks' shards) pool like the single fp16 store, and the Stage-1 epoch functions and GraphedHeadStep take an
fp16 store unchanged."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from torch.utils.data import DataLoader

from test_feature_store_gpu import FEAT, N_CLIPS, Clips, StandInEncoder, make_loss
from test_sharded_store_gpu import (CFG, Identity, _free_port, _init, clips, index_patterns, loader_of, make_head,
                                    weights)

pytestmark = pytest.mark.gpu

F16 = torch.float16


def store_with(rows, labels=None, dtype=None):
    """a filled LayerMeanStore of ``dtype`` (default: rows' dtype) holding ``rows`` (converted by torch's copy_)"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    n, f, t = rows.shape
    store = LayerMeanStore(n, f, t, rows.device, dtype or rows.dtype)
    store.rows.copy_(rows)
    if labels is not None:
        store.labels.copy_(labels)
    store.filled = n
    return store


def same_bits(a, b):
    return a.dtype == b.dtype and torch.equal(a.view(torch.int16 if a.element_size() == 2 else torch.int32),
                                              b.view(torch.int16 if b.element_size() == 2 else torch.int32))


def sharded_pool16(bases, ranks, n, feat, frames, idx, p=0.0, rng=None):
    """supcon_head_sharded_store_pool_forward_typed (SUPCON_F16) on the shards at the device addresses ``bases``"""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200 import functional as Fn
    pooled = torch.empty((idx.shape[0], feat), dtype=torch.float32, device=idx.device)
    _cabi.check(_cabi.load().supcon_head_sharded_store_pool_forward_typed(
        Fn._p(bases), ranks, _cabi.F16, n, feat, frames, Fn._p(idx), idx.shape[0], p, 0.01, Fn._p(rng),
        Fn._p(pooled), Fn._stream(idx.device)), "supcon_head_sharded_store_pool_forward_typed")
    return pooled


def shard16(rows16, ranks):
    n, f, t = rows16.shape
    local = -(-n // ranks)
    shards = []
    for r in range(ranks):
        s = torch.full((local, f, t), float("nan"), dtype=F16, device=rows16.device)
        s[: len(range(r, n, ranks))] = rows16[r::ranks]
        shards.append(s)
    return shards, torch.tensor([s.data_ptr() for s in shards], dtype=torch.int64, device=rows16.device)


SHAPES = [(20, 1024, 199), (23, 7, 13), (17, 40, 50), (9, 18, 199), (12, 64, 1000)]
ids = ["x".join(map(str, s)) for s in SHAPES]


# ----------------------------------------------------------------------------------------------- the build

@pytest.mark.parametrize("hs_dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(10, 3, 1024, 199), (7, 2, 7, 13), (9, 4, 40, 50)],
                         ids=["1024x199", "7x13", "40x50"])
def test_fp16_build_rows_are_fp32_build_rows_rounded(cuda_device, shape, hs_dtype):
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    b, k, f, t = shape
    g = torch.Generator().manual_seed(b * f + t)
    hs = (torch.randn(2 * b, k, f, t, generator=g) * 30).to(hs_dtype)
    hs[0, :, 0, :3] = 1e-6                                                   # means in fp16's subnormal range
    y = torch.arange(2 * b)
    batches = loader_of(hs, y, range(2 * b), batch=b)
    s32 = build_layer_mean_store(Identity(), batches, cuda_device, n=2 * b)
    s16 = build_layer_mean_store(Identity(), batches, cuda_device, n=2 * b, dtype=F16)
    assert s16.dtype == F16 and s16.filled == 2 * b
    assert same_bits(s16.rows, s32.rows.half())
    assert torch.equal(s16.labels, s32.labels)


def test_mean_beyond_fp16_range_raises_naming_the_slot(cuda_device, tmp_path):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore, build_layer_mean_store
    hs = torch.randn(8, 3, 16, 12)
    hs[5, :, 4, 7] = 70000.0                                                 # the mean of slot 5 is 70000
    hs[6, :, 0, 0] = 65519.0                                                 # rounds to 65504: fine
    batches = loader_of(hs, torch.arange(8), range(8), batch=4)
    with pytest.raises(ValueError, match="slot 5: a finite layer mean rounds to inf in fp16"):
        build_layer_mean_store(Identity(), batches, cuda_device, n=8, dtype=F16)
    assert build_layer_mean_store(Identity(), batches, cuda_device, n=8).rows[5, 4, 7] == 70000.0    # fp32: fine
    store = LayerMeanStore(8, 16, 12, cuda_device, dtype=F16)
    for x, y in batches:
        store.append(x.to(cuda_device), y.to(cuda_device))
    with pytest.raises(ValueError, match="slot 5: .* not saved"):
        store.save(tmp_path / "store")
    assert os.listdir(tmp_path) == []
    # non-finite hidden states are carried into the rows, not an overflow (the loss turns NaN, as with fp32)
    hs[5, :, 4, 7] = float("inf")
    inf = build_layer_mean_store(Identity(), loader_of(hs, torch.arange(8), range(8)), cuda_device, n=8, dtype=F16)
    assert bool(inf.rows[5, 4, 7].isinf())


# ------------------------------------------------------------------------------- the gather: the main oracle

@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("shape", SHAPES, ids=ids)
def test_fp16_pool_equals_pool_of_widened_fp32_store(cuda_device, shape, p):
    """eval and dropout 0.1; random, repeated and permuted indices.  (7, 13), (18, 199) and (40, 50) have runs that
    are not a multiple of eight fp16: the scalar path; (64, 1000) has 8 rows per block where fp32 has 12."""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    n, f, t = shape
    g = torch.Generator().manual_seed(n + f + t)
    rows16 = (torch.randn(n, f, t, generator=g) * 4).half().to(cuda_device)
    s16 = store_with(rows16)
    s32 = LayerMeanStore.from_arrays(rows16.float().cpu(), np.arange(n), cuda_device)
    rng = torch.tensor([1234, 5], dtype=torch.int64, device=cuda_device)
    for name, idx in index_patterns(n, 1, 0, 12, g).items():
        idx = idx.to(cuda_device)
        got = s16.pool(idx, p, 0.01, rng if p else None)
        assert torch.equal(got, s32.pool(idx, p, 0.01, rng if p else None)), name
        assert not bool(got.isnan().any())


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_fp16_out_of_range_index_gives_nan_row(cuda_device, p):
    n, f, t = 9, 40, 56
    rows16 = torch.randn(n, f, t, device=cuda_device).half()
    s16, s32 = store_with(rows16), store_with(rows16.float())
    idx = torch.tensor([0, 9, 5, -1, 2 ** 40, 8], device=cuda_device)
    rng = torch.tensor([99, 4], dtype=torch.int64, device=cuda_device)
    got = s16.pool(idx, p, 0.01, rng if p else None)
    want = s32.pool(idx.clamp(0, n - 1), p, 0.01, rng if p else None)
    bad = torch.tensor([False, True, False, True, True, False], device=cuda_device)
    assert bool(got[bad].isnan().all())
    assert torch.equal(got[~bad], want[~bad])


def test_fp16_store_past_32_bit_offsets(cuda_device):
    """10541 clips of (1024, 199) fp16 = 4.3 GB: rows from 10538 on start past 2^31 elements"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    from wav2vec_contr_loss_b200.head import layer_time_pool
    f, t = 1024, 199
    first_high = 2 ** 31 // (f * t) + 1
    n = first_high + 3
    store = LayerMeanStore(n, f, t, cuda_device, dtype=F16)
    assert store.rows.numel() > 2 ** 31 and store.rows.nbytes > 4.29e9
    slots = [n - 1, first_high, 3, first_high - 1, 0, n - 2]
    torch.manual_seed(5)
    for i in slots:
        store.rows[i].normal_()
    store.filled = n
    idx = torch.tensor(slots, device=cuda_device)
    hs = store.rows[idx].float().unsqueeze(1)                                # K = 1: the widened row is the mean
    rng = torch.tensor([31, 2], dtype=torch.int64, device=cuda_device)
    assert torch.equal(store.pool(idx), layer_time_pool(hs))
    assert torch.equal(store.pool(idx, 0.1, 0.01, rng), layer_time_pool(hs, 0.1, 0.01, rng))


def test_fp16_pool_graph_takes_new_indices(cuda_device):
    n, f, t, b = 30, 64, 20, 16
    rows16 = torch.randn(n, f, t, device=cuda_device).half()
    s16, s32 = store_with(rows16), store_with(rows16.float())
    g = torch.Generator().manual_seed(1)
    idx = torch.randperm(n, generator=g)[:b].to(cuda_device)
    rng = torch.tensor([7, 0], dtype=torch.int64, device=cuda_device)
    s16.pool(idx, 0.1, 0.01, rng)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = s16.pool(idx, 0.1, 0.01, rng)
    for r in range(3):
        idx.copy_(torch.randint(0, n, (b,), generator=g))
        rng[1] = r + 1
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, s32.pool(idx, 0.1, 0.01, rng)), r


@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("shape", [(40, 1024, 199), (23, 7, 13)], ids=["1024x199", "7x13"])
def test_pooled_error_within_bound_of_fp32_store(cuda_device, shape, p):
    """|p16 - p32| <= 2^-11 mean_t|a_t| + 2T 2^-24 mean_t|a_t| + s 2^-25 per pooled element, a = the fp32 store's
    activated value LeakyReLU(Dropout(m)), s = 1 / (1 - p): half an fp16 ulp relative (the rounding of each mean,
    carried through Dropout and LeakyReLU, which scale it), the two fp32 time sums (T terms each), and the absolute
    rounding floor of fp16's subnormals (half of 2^-24) times the dropout scale.  mean_t|a_t| is pooled from an fp32
    store of |LeakyReLU(m)| with the same mask (Dropout's multiplier is not negative)."""
    n, f, t = shape
    g = torch.Generator().manual_seed(f + t)
    rows = torch.randn(n, f, t, generator=g) * torch.logspace(-7, 3, n).view(-1, 1, 1)    # 1e-7 .. 1e3: subnormals
    rows = rows.to(cuda_device)
    s32, s16 = store_with(rows), store_with(rows, dtype=F16)
    mag = store_with(torch.where(rows > 0, rows, rows * 0.01).abs())
    rng = torch.tensor([55, 3], dtype=torch.int64, device=cuda_device) if p else None
    idx = torch.arange(n, device=cuda_device)
    p16, p32, m = (s.pool(idx, p, 0.01, rng).double() for s in (s16, s32, mag))
    s = 1.0 / (1.0 - p)
    bound = (2.0 ** -11 + 2 * t * 2.0 ** -24) * m * (1 + 1e-5) + s * 2.0 ** -25
    err = (p16 - p32).abs()
    assert bool((err <= bound).all()), float((err / bound).max())
    assert float(err.max()) > 0                                               # the rounding is visible


# ---------------------------------------------------------------------------------------------- sharded

@pytest.mark.parametrize("ranks", [1, 2, 3, 8])
@pytest.mark.parametrize("shape", [(20, 1024, 199), (23, 7, 13), (17, 40, 50)], ids=lambda s: "x".join(map(str, s)))
def test_sharded_fp16_pool_equals_single_fp16_store(cuda_device, shape, ranks):
    n, f, t = shape
    rows16 = torch.randn(n, f, t, generator=torch.Generator().manual_seed(n + f)).half().to(cuda_device)
    ref = store_with(rows16)
    shards, bases = shard16(rows16, ranks)
    g = torch.Generator().manual_seed(7)
    rng = torch.tensor([1234, 5], dtype=torch.int64, device=cuda_device)
    for rank in range(ranks):
        for name, idx in index_patterns(n, ranks, rank, 12, g).items():
            idx = idx.to(cuda_device)
            assert torch.equal(sharded_pool16(bases, ranks, n, f, t, idx), ref.pool(idx)), (rank, name)
            assert torch.equal(sharded_pool16(bases, ranks, n, f, t, idx, 0.1, rng),
                               ref.pool(idx, 0.1, 0.01, rng)), (rank, name)
    idx = torch.tensor([0, n, -1, n - 1], device=cuda_device)
    got = sharded_pool16(bases, ranks, n, f, t, idx)
    assert bool(got[1:3].isnan().all()) and torch.equal(got[[0, 3]], ref.pool(idx[[0, 3]]))


def _one_rank(rank, world, port, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store, build_sharded_layer_mean_store
    dev = _init(rank, world, port)
    try:
        res = {}
        n, k, f, t = 96, 3, 16, 12
        hs, y, ds = clips(n, k, f, t)
        sharded = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, range(n)), dev, n=n, dtype=F16)
        single = build_layer_mean_store(Identity(), loader_of(hs, y, range(n), batch=20), dev, n=n, dtype=F16)
        res["build"] = (sharded.dtype == F16, sharded.rows.dtype == F16, same_bits(sharded.rows, single.rows),
                        torch.equal(sharded.labels, single.labels))
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
        res["graphed"] = _graphed_vs_eager(sharded, f, dev)
        sharded.close()
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_one_rank_fp16_store_on_symmetric_memory(cuda_device):
    out = mp.Manager().dict()
    mp.spawn(_one_rank, args=(1, _free_port(), out), nprocs=1, join=True)
    res = out[0]
    assert res["build"] == (True, True, True, True)
    assert res["epochs"] == (True, True)
    _check_graphed(res["graphed"])


def _two_ranks(rank, world, port, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store, build_sharded_layer_mean_store
    from wav2vec_contr_loss_b200.feature_store import shard_slots
    dev = _init(rank, world, port)
    try:
        n, k, f, t = 41, 2, 1024, 199
        hs, y, _ = clips(n, k, f, t)
        store = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, shard_slots(n, rank, world), batch=8),
                                               dev, n=n, dtype=F16)
        single = build_layer_mean_store(Identity(), loader_of(hs, y, range(n), batch=8), dev, n=n, dtype=F16)
        rng = torch.tensor([77, 1], dtype=torch.int64, device=dev)
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(rank))[:32].to(dev)
        out[rank] = (torch.equal(store.pool(idx), single.pool(idx)),
                     torch.equal(store.pool(idx, 0.1, 0.01, rng), single.pool(idx, 0.1, 0.01, rng)))
        store.close()
    finally:
        dist.destroy_process_group()


def test_two_ranks_fp16_sharded_store(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = mp.Manager().dict()
    mp.spawn(_two_ranks, args=(2, _free_port(), out), nprocs=2, join=True)
    assert out[0] == out[1] == (True, True)


# ---------------------------------------------------------------------------------------------- training

@pytest.mark.parametrize("kind", ["binary", "multiclass", "memory"])
def test_epochs_from_fp16_store_equal_epochs_from_widened_store(cuda_device, kind):
    """three epochs (alpha 0 -> 0.5 -> 1, dropout 0.1) with evaluations: the fp16 store and the fp32 store of its
    widened rows give identical losses and head weights; against the plain fp32 store, the first step's loss agrees
    to 1e-3 relative"""
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    label_index = 2 if kind == "multiclass" else 1
    ds = Clips()
    enc = StandInEncoder().to(cuda_device)
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=3, warmup_epochs=1,
                          alpha_ramp_epochs=2, alpha_end=1.0)
    loader = DataLoader(ds, batch_size=20, shuffle=False)
    s16 = build_layer_mean_store(enc, loader, cuda_device, label_index=label_index, dtype=F16)
    s32 = build_layer_mean_store(enc, loader, cuda_device, label_index=label_index)
    wide = store_with(s16.rows.float(), s16.labels)
    assert s16.filled == N_CLIPS and torch.equal(s16.labels, s32.labels)

    heads = [make_head(FEAT, 0.1, cuda_device, seed=4)]
    heads.append(copy.deepcopy(heads[0]))
    first = []
    for store in (s16, s32):
        idx = torch.arange(16, device=cuda_device)
        with torch.no_grad():
            z = Fn.l2_normalize(copy.deepcopy(heads[0]).eval().pooled_embedding_from_store(store, idx))
            first.append(float(S.call_loss(make_loss(kind), z, store.labels_of(idx), 3, 0.0)))
    assert first[0] == pytest.approx(first[1], rel=1e-3)

    opts = [torch.optim.AdamW(h.parameters(), lr=5e-3, weight_decay=3e-3) for h in heads]
    losses = [make_loss(kind), make_loss(kind)]
    samplers = [S.BalancedBatchSampler(ds, 16, seed=13) for _ in heads]
    dev_batches = [list(range(i, i + 12)) for i in range(0, 36, 12)]
    for epoch in (1, 2, 3):
        got = []
        for j, store in enumerate((s16, wide)):
            samplers[j].set_epoch(epoch)
            tr = S.train_one_epoch_from_store(heads[j], losses[j], store, list(samplers[j]), opts[j], cuda_device,
                                              epoch, cfg)
            got.append((tr, S.evaluate_from_store(heads[j], losses[j], store, dev_batches, cuda_device, cfg)))
        assert got[0] == got[1], epoch
    for pa, pb in zip(*(h.parameters() for h in heads)):
        assert torch.equal(pa, pb)


def _graphed_vs_eager(store, feat, dev):
    """five steps (dropout 0.1, alpha 0 / 0.5) eagerly and as GraphedHeadStep(store=) replays"""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    g = torch.Generator().manual_seed(5)
    idx = [torch.randperm(store.n, generator=g)[:32].to(dev) for _ in range(5)]
    alphas = [0.0, 0.0, 0.5, 0.5, 0.0]
    head_e = make_head(feat, 0.1, dev).train()
    head_g = copy.deepcopy(head_e)
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    opt_g = torch.optim.AdamW(head_g.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    loss_e, loss_g = SupConBinaryLoss(0.1, "cosine", 0.05, 2.0), SupConBinaryLoss(0.1, "cosine", 0.05, 2.0)
    eager = []
    for s, alpha in enumerate(alphas):
        z = Fn.l2_normalize(head_e.pooled_embedding_from_store(store, idx[s]))
        loss = loss_e(z, store.labels_of(idx[s]), topk_neg=7, alpha=alpha)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(head_e.parameters(), 5.0)
        opt_e.step()
        eager.append(float(loss))
    step = S.GraphedHeadStep(head_g, loss_g, opt_g, idx[0], topk_neg=7, store=store)
    graphed = [float(step(idx[s], alpha=alpha)) for s, alpha in enumerate(alphas)]
    torch.cuda.synchronize()
    return eager, graphed, weights(head_e), weights(head_g), head_e.rng_state.tolist() == head_g.rng_state.tolist()


def _check_graphed(res):
    eager, graphed, w_e, w_g, same_stream = res
    assert same_stream
    assert graphed == pytest.approx(eager, rel=1e-5)
    assert torch.allclose(w_g, w_e, rtol=1e-4, atol=1e-6)


def test_graphed_step_from_fp16_store_follows_eager_steps(cuda_device):
    n, f, t = 200, 64, 20
    g = torch.Generator().manual_seed(5)
    y = torch.arange(n) % 2
    rows = torch.randn(n, f, t, generator=g) + 0.5 * (2.0 * y.view(-1, 1, 1) - 1.0)
    store = store_with(rows.to(cuda_device), y.to(cuda_device), dtype=F16)
    _check_graphed(_graphed_vs_eager(store, f, cuda_device))


# -------------------------------------------------------------------------------------------- save and load

@pytest.mark.parametrize("stage_bytes", [None, 4000], ids=["stage_64MiB", "stage_4000B"])
def test_fp16_save_load_round_trip_on_the_gpu(cuda_device, tmp_path, monkeypatch, stage_bytes):
    from wav2vec_contr_loss_b200 import feature_store as FS
    if stage_bytes:
        monkeypatch.setattr(FS, "STAGE_BYTES", stage_bytes)
    n, f, t = 24, 40, 50
    rows = torch.randn(n, f, t, generator=torch.Generator().manual_seed(2)).to(cuda_device) * 100
    s16 = store_with(rows, torch.arange(n, device=cuda_device) % 3, dtype=F16)
    s16.save(tmp_path / "s16")
    assert np.load(tmp_path / "s16" / "rows.npy", mmap_mode="r").dtype == np.float16
    back = FS.load_layer_mean_store(tmp_path / "s16", cuda_device, dtype=F16)
    assert same_bits(back.rows, s16.rows) and torch.equal(back.labels, s16.labels)
    idx = torch.randperm(n, device=cuda_device)
    rng = torch.tensor([3, 9], dtype=torch.int64, device=cuda_device)
    assert torch.equal(back.pool(idx, 0.1, 0.01, rng), s16.pool(idx, 0.1, 0.01, rng))
    # an fp32 file loaded into an fp16 store is rounded on the device: .half(), chunk edges included
    store_with(rows).save(tmp_path / "s32")
    rounded = FS.load_layer_mean_store(tmp_path / "s32", cuda_device, dtype=F16)
    assert same_bits(rounded.rows, rows.half())
    rows[13, 7, 9] = 1e6
    store_with(rows).save(tmp_path / "hot")
    with pytest.raises(ValueError, match=r"hot/rows\.npy: slot 13: a finite layer mean rounds to inf"):
        FS.load_layer_mean_store(tmp_path / "hot", cuda_device, dtype=F16)
