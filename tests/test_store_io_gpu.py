"""GPU: the layer-mean store saved to disk and loaded back (feature_store: LayerMeanStore.save / from_arrays,
load_layer_mean_store, ShardedLayerMeanStore.save, load_sharded_layer_mean_store).

A load must give back the store that was saved, bit for bit: the rows (compared as int32), the labels, and so
everything trained from it -- pooled rows, three epochs of train_one_epoch_from_store, graphed steps.  Files do not
depend on the number of ranks: a sharded store saves what a single store of the same clips saves, and a single
store's file loads into R ranks.  The two-rank cases are skipped below two GPUs."""
import copy
import os
import shutil
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from torch.utils.data import DataLoader

from test_feature_store_gpu import FEAT, N_CLIPS, Clips, StandInEncoder, make_head, make_loss
from test_sharded_store_gpu import Identity, _free_port, _init, clips, index_patterns, loader_of, single_store_of

pytestmark = pytest.mark.gpu

CFG = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=3, warmup_epochs=1, alpha_ramp_epochs=2,
                      alpha_end=1.0)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.fixture(scope="module")
def built(cuda_device):
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    return build_layer_mean_store(StandInEncoder().to(cuda_device), DataLoader(Clips(), batch_size=20), cuda_device)


@pytest.mark.parametrize("stage_bytes", [None, 4000], ids=["stage_64MiB", "stage_4000B"])
def test_round_trip_rows_labels_and_pool(cuda_device, built, tmp_path, monkeypatch, stage_bytes):
    """4000-byte staging: chunks of 1000 elements split the rows of 192, and both buffers are reused many times"""
    from wav2vec_contr_loss_b200 import feature_store as FS
    if stage_bytes:
        monkeypatch.setattr(FS, "STAGE_BYTES", stage_bytes)
    assert built.save(tmp_path / "store") == N_CLIPS
    loaded = FS.load_layer_mean_store(tmp_path / "store", cuda_device)
    assert (loaded.n, loaded.filled, loaded.device) == (N_CLIPS, N_CLIPS, built.device)
    assert same_bits(loaded.rows, built.rows)
    assert torch.equal(loaded.labels, built.labels)
    g = torch.Generator().manual_seed(3)
    rng = torch.tensor([41, 6], dtype=torch.int64, device=cuda_device)
    for idx in (torch.randperm(N_CLIPS, generator=g)[:24], torch.randint(0, N_CLIPS, (24,), generator=g),
                torch.arange(N_CLIPS).flip(0)):
        idx = idx.to(cuda_device)
        assert torch.equal(loaded.pool(idx), built.pool(idx))
        assert torch.equal(loaded.pool(idx, 0.1, 0.01, rng), built.pool(idx, 0.1, 0.01, rng))
        assert torch.equal(loaded.labels_of(idx), built.labels_of(idx))


@pytest.mark.parametrize("kind", ["binary", "memory"])
def test_epochs_from_loaded_store_equal_epochs_from_built_store(cuda_device, built, tmp_path, kind):
    """three epochs (dropout 0.1, alpha 0 -> 0.5 -> 1) and evaluations: identical losses, dropout streams and weights"""
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import load_layer_mean_store
    built.save(tmp_path / "store")
    loaded = load_layer_mean_store(tmp_path / "store", cuda_device)
    ds = Clips()
    heads = [make_head(FEAT, 0.1, cuda_device, seed=4)]
    heads.append(copy.deepcopy(heads[0]))
    opts = [torch.optim.AdamW(h.parameters(), lr=5e-3, weight_decay=3e-3) for h in heads]
    losses = [make_loss(kind), make_loss(kind)]
    samplers = [S.BalancedBatchSampler(ds, 16, seed=13) for _ in heads]
    dev_batches = [list(range(i, i + 12)) for i in range(0, 36, 12)]
    hist = [[], []]
    for epoch in (1, 2, 3):
        for j, store in enumerate((built, loaded)):
            samplers[j].set_epoch(epoch)
            tr = S.train_one_epoch_from_store(heads[j], losses[j], store, list(samplers[j]), opts[j], cuda_device,
                                              epoch, CFG)
            hist[j].append((tr, S.evaluate_from_store(heads[j], losses[j], store, dev_batches, cuda_device, CFG)))
    assert hist[0] == hist[1]
    assert heads[0].rng_state.tolist() == heads[1].rng_state.tolist()
    for pa, pb in zip(heads[0].parameters(), heads[1].parameters()):
        assert torch.equal(pa, pb)


def test_graphed_step_from_loaded_store_equals_eager_steps(cuda_device, built, tmp_path):
    """GraphedHeadStep(store=loaded) replays against the same steps run eagerly from the built store (the tolerance of
    test_feature_store_gpu.py::test_graphed_store_step_equals_eager_store_steps)"""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import load_layer_mean_store
    built.save(tmp_path / "store")
    loaded = load_layer_mean_store(tmp_path / "store", cuda_device)
    g = torch.Generator().manual_seed(5)
    idx = [torch.randperm(N_CLIPS, generator=g)[:32].to(cuda_device) for _ in range(5)]
    alphas = [0.0, 0.0, 0.5, 0.5, 0.0]
    loss_fn = SupConBinaryLoss(temperature=0.1, similarity="cosine", uniformity_weight=0.05)
    head_e = make_head(FEAT, 0.1, cuda_device).train()
    head_g = copy.deepcopy(head_e)
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    opt_g = torch.optim.AdamW(head_g.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    eager = []
    for s, alpha in enumerate(alphas):
        z = S.Fn.l2_normalize(head_e.pooled_embedding_from_store(built, idx[s]))
        loss = loss_fn(z, built.labels_of(idx[s]), topk_neg=7, alpha=alpha)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(head_e.parameters(), 5.0)
        opt_e.step()
        eager.append(float(loss))
    step = S.GraphedHeadStep(head_g, loss_fn, opt_g, idx[0], topk_neg=7, store=loaded)
    graphed = [float(step(idx[s], alpha=alpha)) for s, alpha in enumerate(alphas)]
    assert head_g.rng_state.tolist() == head_e.rng_state.tolist()
    assert graphed == pytest.approx(eager, rel=1e-5)
    for pg, pe in zip(head_g.parameters(), head_e.parameters()):
        assert torch.allclose(pg, pe, rtol=1e-4, atol=1e-6)


def test_float16_rows_are_widened_exactly(cuda_device, tmp_path):
    """from an array and from a float16 .npy file (the file path reads with readinto and widens on the host)"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore, load_layer_mean_store
    a = (np.random.default_rng(4).standard_normal((9, 40, 50)) * 500).astype(np.float16)
    a.reshape(-1)[:6] = [np.inf, -np.inf, np.nan, 6e-8, -0.0, 65504]
    want = torch.from_numpy(a).float()
    store = LayerMeanStore.from_arrays(a, np.arange(9), cuda_device)
    assert same_bits(store.rows.cpu(), want)
    os.makedirs(tmp_path / "fp16")
    np.save(tmp_path / "fp16" / "rows.npy", a)
    np.save(tmp_path / "fp16" / "labels.npy", np.arange(9, dtype=np.int32))
    loaded = load_layer_mean_store(tmp_path / "fp16", cuda_device)
    assert same_bits(loaded.rows.cpu(), want) and loaded.labels.tolist() == list(range(9))


def test_round_trip_past_4_GiB(cuda_device, tmp_path):
    """5300 clips of (1024, 199): a 4.32 GB rows.npy, so file offsets pass 2^32 bytes"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore, load_layer_mean_store
    n, f, t = 5300, 1024, 199
    need = n * f * t * 4
    assert need > 2 ** 32
    if shutil.disk_usage(tmp_path).free < need + (1 << 30):
        pytest.skip(f"{need / 1e9:.1f} GB of free space needed in {tmp_path}")
    store = LayerMeanStore(n, f, t, cuda_device)
    store.rows.normal_(generator=torch.Generator(device=cuda_device).manual_seed(8))
    store.labels.copy_(torch.arange(n, device=cuda_device) % 2)
    store.filled = n
    assert store.save(tmp_path / "big") == n
    assert os.path.getsize(tmp_path / "big" / "rows.npy") > 2 ** 32
    loaded = load_layer_mean_store(tmp_path / "big", cuda_device)
    assert same_bits(loaded.rows, store.rows) and torch.equal(loaded.labels, store.labels)
    high = 2 ** 32 // (f * t * 4) + 1                             # the first clip that starts past 2^32 bytes
    idx = torch.tensor([n - 1, high, 0, high - 1], device=cuda_device)
    assert torch.equal(loaded.pool(idx), store.pool(idx))


# ------------------------------------------------------------------------------ process groups

def _one_rank(rank, world, port, root, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200.feature_store import load_layer_mean_store, load_sharded_layer_mean_store
    dev = _init(rank, world, port)
    try:
        n, k, f, t = 23, 3, 40, 50
        hs, y, _ = clips(n, k, f, t)
        single = single_store_of(hs.to(dev), y.to(dev))
        single.save(os.path.join(root, "single"))
        sharded = load_sharded_layer_mean_store(os.path.join(root, "single"), dev)
        ok = [sharded.filled == n, same_bits(sharded.rows, single.rows), torch.equal(sharded.labels, single.labels)]
        rng = torch.tensor([77, 3], dtype=torch.int64, device=dev)
        for idx in index_patterns(n, 1, 0, 12, torch.Generator().manual_seed(7)).values():
            idx = idx.to(dev)
            ok += [torch.equal(sharded.pool(idx), single.pool(idx)),
                   torch.equal(sharded.pool(idx, 0.1, 0.01, rng), single.pool(idx, 0.1, 0.01, rng))]
        ok.append(sharded.save(os.path.join(root, "sharded")) == n)
        sharded.close()
        again = load_layer_mean_store(os.path.join(root, "sharded"), dev)
        ok += [same_bits(again.rows, single.rows), torch.equal(again.labels, single.labels)]
        out[rank] = ok
    finally:
        dist.destroy_process_group()


def test_one_rank_sharded_load_equals_single_load(cuda_device, tmp_path):
    """a process group of one rank on symmetric memory: a single store's file loads into a sharded store with the
    same rows and pools, and the sharded store's save loads back as the single store"""
    out = mp.Manager().dict()
    mp.spawn(_one_rank, args=(1, _free_port(), str(tmp_path), out), nprocs=1, join=True)
    assert all(out[0]), out[0]


WORLD = 2
N2, K2, F2, T2 = 23, 2, 40, 50


def _two_ranks(rank, world, port, root, out):
    import torch.distributed as dist
    from wav2vec_contr_loss_b200.feature_store import (build_sharded_layer_mean_store, load_sharded_layer_mean_store,
                                                       shard_slots)
    dev = _init(rank, world, port)
    try:
        hs, y, _ = clips(N2, K2, F2, T2)
        sharded = build_sharded_layer_mean_store(Identity(), loader_of(hs, y, shard_slots(N2, rank, world), 4), dev,
                                                 n=N2)
        ok = [sharded.save(os.path.join(root, "sharded")) == N2]
        sharded.close()
        # the file of a single-GPU store, loaded into R = 2: pools what the single store pools
        single = single_store_of(hs.to(dev), y.to(dev))
        loaded = load_sharded_layer_mean_store(os.path.join(root, "single"), dev)
        ok += [loaded.filled == N2, torch.equal(loaded.labels, single.labels)]
        rng = torch.tensor([77, 3], dtype=torch.int64, device=dev)
        for idx in index_patterns(N2, world, rank, 12, torch.Generator().manual_seed(7)).values():
            idx = idx.to(dev)
            ok += [torch.equal(loaded.pool(idx), single.pool(idx)),
                   torch.equal(loaded.pool(idx, 0.1, 0.01, rng), single.pool(idx, 0.1, 0.01, rng))]
        loaded.close()
        out[rank] = ok
    finally:
        dist.destroy_process_group()


def test_two_ranks_save_and_load(cuda_device, tmp_path):
    if torch.cuda.device_count() < WORLD:
        pytest.skip(f"needs {WORLD} GPUs (have {torch.cuda.device_count()})")
    from wav2vec_contr_loss_b200.feature_store import load_layer_mean_store
    hs, y, _ = clips(N2, K2, F2, T2)
    single = single_store_of(hs.to(cuda_device), y.to(cuda_device))
    single.save(tmp_path / "single")
    out = mp.Manager().dict()
    mp.spawn(_two_ranks, args=(WORLD, _free_port(), str(tmp_path), out), nprocs=WORLD, join=True)
    for rank in range(WORLD):
        assert all(out[rank]), (rank, out[rank])
    # the sharded build's file, loaded on one GPU, is the single-GPU build
    loaded = load_layer_mean_store(tmp_path / "sharded", cuda_device)
    assert same_bits(loaded.rows, single.rows) and torch.equal(loaded.labels, single.labels)
