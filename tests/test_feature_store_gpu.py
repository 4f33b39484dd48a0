"""GPU: the layer-mean store (wav2vec_contr_loss_b200.feature_store, head_layer_mean_kernel and
head_store_pool_fwd_kernel in csrc/supcon_head.cu) and the Stage-1 epochs trained from it.

Everything here is compared bit for bit: the store's rows are the fp32 product (sum_k hs[k]) * (1/K) that the fused
head computes internally, and the gather-pool draws the dropout masks of the batch position, so pooling from the
store and pooling the same clips' hs give the same bits.  The one tolerance is the graphed step's, taken from
test_stage1_gpu.py::test_graphed_step_equals_eager_steps."""
import copy

import pytest
import torch
from torch.utils.data import DataLoader, Dataset

pytestmark = pytest.mark.gpu

SHAPES = [          # batch, layers, feat, frames (those of test_head_gpu.py, and the reference's full batch)
    (64, 25, 1024, 199),
    (3, 25, 256, 199),
    (2, 3, 7, 13),
    (2, 2, 18, 199),
    (2, 5, 40, 50),
    (1, 2, 6, 3000),
]
ids = lambda s: "x".join(map(str, s))     # noqa: E731


def sequential_mean(hs):
    """fp32 sum over k = 0..K-1 in order, then times the fp32 1/K"""
    k = hs.shape[1]
    s = torch.zeros_like(hs[:, 0], dtype=torch.float32)
    for i in range(k):
        s = s + hs[:, i].float()
    inv_k = (torch.ones(1, dtype=torch.float32) / torch.full((1,), float(k), dtype=torch.float32)).to(hs.device)
    return s * inv_k


def store_of(hs, labels=None, splits=2):
    """a store holding hs's clips in order, written in `splits` appends (slot offsets other than 0)"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    n = hs.shape[0]
    store = LayerMeanStore(n, hs.shape[2], hs.shape[3], hs.device)
    labels = torch.arange(n, device=hs.device) if labels is None else labels
    for part, lab in zip(hs.chunk(splits), labels.chunk(splits)):
        store.append(part, lab)
    assert store.filled == n
    return store


def make_head(feat, p, device, seed=0):
    from wav2vec_contr_loss_b200 import FusedCompressionHead
    torch.manual_seed(seed)
    return FusedCompressionHead(feat, 16, p).to(device)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", SHAPES, ids=ids)
def test_layer_mean_rows_equal_sequential_sum(cuda_device, shape, dtype):
    hs = torch.randn(*shape, generator=torch.Generator().manual_seed(7)).to(cuda_device, dtype)
    store = store_of(hs)
    assert torch.equal(store.rows, sequential_mean(hs))
    assert store.labels.tolist() == list(range(shape[0]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", SHAPES[1:], ids=ids)
def test_pooled_from_store_equals_pooled_features(cuda_device, shape, dtype):
    """eval and train (p = 0.1, the same rng_state), repeated and permuted indices: the same bits as the fused head on
    the gathered hs, and the dropout stream advances by one per call either way"""
    b, k, f, t = shape
    n = b + 5
    hs_all = torch.randn(n, k, f, t, generator=torch.Generator().manual_seed(3)).to(cuda_device, dtype)
    store = store_of(hs_all, splits=3)
    g = torch.Generator().manual_seed(11)
    picks = [torch.randperm(n, generator=g)[:b], torch.randint(0, n, (b,), generator=g),
             torch.full((b,), n - 1), torch.arange(n).flip(0)]
    head = make_head(f, 0.1, cuda_device)
    for idx in picks:
        idx = idx.to(cuda_device)
        hs = hs_all[idx]
        head.eval()
        assert torch.equal(head.pooled_features_from_store(store, idx), head.pooled_features(hs))
        head.train()
        start = head.rng_state.clone()
        want = head.pooled_features(hs)
        head.rng_state.copy_(start)
        got = head.pooled_features_from_store(store, idx)
        assert head.rng_state.tolist() == [start[0].item(), start[1].item() + 1]
        assert torch.equal(got, want)
        # the embedding is the same Linear on the same features
        head.rng_state.copy_(start)
        e_hs = head.pooled_embedding(hs)
        head.rng_state.copy_(start)
        assert torch.equal(head.pooled_embedding_from_store(store, idx), e_hs)


def test_store_beyond_32_bit_offsets(cuda_device):
    """a store of more than 2^31 elements (8.6 GB): rows past 2^31 / (F T) are written and gathered at their own
    64-bit offsets"""
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    f, t = 1024, 199
    first_high = 2 ** 31 // (f * t) + 1                       # 10539: the first row starting past 2^31 elements
    n = first_high + 64
    store = LayerMeanStore(n, f, t, cuda_device)
    assert store.rows.numel() > 2 ** 31
    torch.manual_seed(5)
    store.rows[: n - 4].normal_()
    store.labels[: n - 4] = torch.arange(n - 4, device=cuda_device) % 2
    store.filled = n - 4
    hs_tail = torch.randn(4, 3, f, t, device=cuda_device)
    assert store.append(hs_tail, torch.ones(4, device=cuda_device)) == n - 4
    assert torch.equal(store.rows[n - 4:], sequential_mean(hs_tail))
    idx = torch.tensor([n - 1, first_high, 3, first_high - 1, n - 4, first_high + 40, 0, n - 1], device=cuda_device)
    hs = store.rows[idx].unsqueeze(1)                           # K = 1: the layer mean is the row itself
    head = make_head(f, 0.1, cuda_device)
    head.eval()
    assert torch.equal(head.pooled_features_from_store(store, idx), head.pooled_features(hs))
    head.train()
    start = head.rng_state.clone()
    want = head.pooled_features(hs)
    head.rng_state.copy_(start)
    assert torch.equal(head.pooled_features_from_store(store, idx), want)


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_out_of_range_index_gives_nan_row(cuda_device, p):
    from wav2vec_contr_loss_b200.head import layer_time_pool
    b, k, f, t = 6, 3, 40, 50
    hs_all = torch.randn(8, k, f, t, device=cuda_device)
    store = store_of(hs_all)
    idx = torch.tensor([0, 8, 5, -1, 2 ** 40, 7], device=cuda_device)
    rng = torch.tensor([99, 4], dtype=torch.int64, device=cuda_device)
    got = store.pool(idx, p, 0.01, rng if p else None)
    want = layer_time_pool(hs_all[idx.clamp(0, 7)], p, 0.01, rng if p else None)
    bad = torch.tensor([False, True, False, True, True, False], device=cuda_device)
    assert bool(got[bad].isnan().all())
    assert torch.equal(got[~bad], want[~bad])
    # a store filled short of its size: the unwritten slots count as outside it
    short = store_of(hs_all)
    short.filled = 5
    assert bool(short.pool(torch.tensor([5], device=cuda_device))[0].isnan().all())
    assert short.labels_of(torch.tensor([5, 9], device=cuda_device)).tolist() == [4, 4]


# ------------------------------------------------------------------------- epochs: hs against the store

HOP, K, FEAT, FRAMES, N_CLIPS = 8, 4, 16, 12, 96


class StandInEncoder(torch.nn.Module):
    """(B, FRAMES * HOP) waveforms -> (B, K, FEAT, FRAMES) by elementwise ops only: a clip's output does not depend
    on its batch mates, to the bit (the condition under which the store reproduces train_one_epoch exactly)."""

    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(21)
        self.register_buffer("gain", torch.randn(1, K, 1, 1, generator=g))
        self.register_buffer("shift", torch.randn(1, 1, FEAT, 1, generator=g))

    def forward(self, waveforms, attention_mask=None):
        b = waveforms.shape[0]
        x = (waveforms * attention_mask.to(waveforms.dtype)).view(b, FRAMES, HOP).transpose(1, 2)   # (B, HOP, T)
        x = x.repeat(1, FEAT // HOP, 1)                                                             # (B, F, T)
        return torch.sin(self.gain * x[:, None] + self.shift).contiguous()


class Clips(Dataset):
    """N_CLIPS synthetic clips; data[i] = (name, bonafide/spoof label) as BalancedBatchSampler reads it, and a
    multi-class id as the third item of each sample (train_multiclass_con.py's layout)"""

    def __init__(self, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.y = torch.arange(N_CLIPS) % 2
        self.cls = torch.randint(0, 5, (N_CLIPS,), generator=g) * 2 + self.y
        self.wave = torch.randn(N_CLIPS, FRAMES * HOP, generator=g) + 0.7 * (2.0 * self.y.view(-1, 1) - 1.0)
        self.wave[::3, -HOP * 3:] = 0.0                                                 # padded clips
        self.data = [(f"utt{i}", int(self.y[i])) for i in range(N_CLIPS)]

    def __len__(self):
        return N_CLIPS

    def __getitem__(self, i):
        return self.wave[i], self.y[i], self.cls[i]


def make_loss(kind):
    from wav2vec_contr_loss_b200 import MemorySupConLoss, SupConBinaryLoss, SupConMultiClassLoss
    if kind == "binary":
        return SupConBinaryLoss(0.1, "cosine", 0.05, 2.0)
    if kind == "multiclass":
        return SupConMultiClassLoss(0.1)
    return MemorySupConLoss(0.1, "cosine", 0.05, 2.0, memory_size=48)


@pytest.mark.parametrize("kind", ["binary", "multiclass", "memory"])
def test_epochs_from_store_equal_epochs_from_encoder(cuda_device, kind):
    """three epochs (alpha 0 -> 0.5 -> 1) of train_one_epoch with the frozen stand-in encoder and the fused head
    (dropout 0.1) against build_layer_mean_store + train_one_epoch_from_store, the same sampler seed, the same head
    and dropout stream: identical epoch losses, evaluation losses and head weights"""
    from types import SimpleNamespace
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store
    label_index = 2 if kind == "multiclass" else 1
    ds = Clips()
    enc = StandInEncoder().to(cuda_device)
    cfg = SimpleNamespace(finetune_encoder=False, use_rawboost=False, topk_neg=3, warmup_epochs=1,
                          alpha_ramp_epochs=2, alpha_end=1.0)
    head_a = make_head(FEAT, 0.1, cuda_device, seed=4)
    head_b = copy.deepcopy(head_a)
    opt_a = torch.optim.AdamW(head_a.parameters(), lr=5e-3, weight_decay=3e-3)
    opt_b = torch.optim.AdamW(head_b.parameters(), lr=5e-3, weight_decay=3e-3)
    loss_a, loss_b = make_loss(kind), make_loss(kind)
    sampler_a = S.BalancedBatchSampler(ds, 16, seed=13)
    sampler_b = S.BalancedBatchSampler(ds, 16, seed=13)
    loader_a = DataLoader(ds, batch_sampler=sampler_a)
    dev_batches = [list(range(i, i + 12)) for i in range(0, 36, 12)]
    dev_loader = [ds[b[0]:b[-1] + 1] for b in dev_batches]

    store = build_layer_mean_store(enc, DataLoader(ds, batch_size=20, shuffle=False), cuda_device,
                                   label_index=label_index)
    assert store.filled == store.n == N_CLIPS
    assert store.labels.tolist() == (ds.cls if label_index == 2 else ds.y).tolist()

    for epoch in (1, 2, 3):
        sampler_a.set_epoch(epoch)
        sampler_b.set_epoch(epoch)
        ta, alpha_a = S.train_one_epoch(enc, head_a, loss_a, loader_a, opt_a, cuda_device, epoch, cfg,
                                        label_index=label_index)
        tb, alpha_b = S.train_one_epoch_from_store(head_b, loss_b, store, list(sampler_b), opt_b, cuda_device,
                                                   epoch, cfg)
        assert (ta, alpha_a) == (tb, alpha_b)
        da = S.evaluate(enc, head_a, loss_a, dev_loader, cuda_device, cfg, label_index=label_index)
        db = S.evaluate_from_store(head_b, loss_b, store, dev_batches, cuda_device, cfg)
        assert da == db
        assert head_a.rng_state.tolist() == head_b.rng_state.tolist()
    for pa, pb in zip(head_a.parameters(), head_b.parameters()):
        assert torch.equal(pa, pb)
    assert head_a.rng_state.tolist()[1] == 3 * len(sampler_a)


def test_build_store_refuses_a_clip_of_another_shape(cuda_device):
    from wav2vec_contr_loss_b200.feature_store import build_layer_mean_store

    class Ragged(StandInEncoder):
        def forward(self, waveforms, attention_mask=None):
            hs = super().forward(waveforms, attention_mask)
            return hs if waveforms.shape[0] == 20 else hs[..., :-1].contiguous()

    with pytest.raises(ValueError, match=r"\(F, T\) = \(16, 11\), the store holds \(16, 12\)"):
        build_layer_mean_store(Ragged().to(cuda_device), DataLoader(Clips(), batch_size=20), cuda_device)


def test_graphed_store_step_equals_eager_store_steps(cuda_device):
    """GraphedHeadStep(store=...) replays walk the trajectory of the same steps run eagerly from the store (dropout
    on, one offset per step); capture does not train"""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    f, t, n, b = 64, 20, 200, 64
    g = torch.Generator().manual_seed(5)
    y = torch.arange(n) % 2
    hs = torch.randn(n, 3, f, t, generator=g) + 0.5 * (2.0 * y.view(-1, 1, 1, 1) - 1.0)
    store = store_of(hs.to(cuda_device), y.to(cuda_device))
    idx = [torch.randperm(n, generator=g)[:b].to(cuda_device) for _ in range(5)]
    alphas = [0.0, 0.0, 0.5, 0.5, 0.0]
    loss_fn = SupConBinaryLoss(temperature=0.1, similarity="cosine", uniformity_weight=0.05)

    head_e = make_head(f, 0.1, cuda_device).train()
    head_g = copy.deepcopy(head_e)
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    eager = []
    for s, alpha in enumerate(alphas):
        z = S.Fn.l2_normalize(head_e.pooled_embedding_from_store(store, idx[s]))
        loss = loss_fn(z, store.labels_of(idx[s]), topk_neg=7, alpha=alpha)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(head_e.parameters(), 5.0)
        opt_e.step()
        eager.append(float(loss))

    opt_g = torch.optim.AdamW(head_g.parameters(), lr=5e-3, weight_decay=3e-3, capturable=True)
    with pytest.raises(ValueError, match="no labels_example"):
        S.GraphedHeadStep(head_g, loss_fn, opt_g, idx[0], store.labels[:b], store=store)
    step = S.GraphedHeadStep(head_g, loss_fn, opt_g, idx[0], topk_neg=7, store=store)
    start = torch.cat([p.detach().reshape(-1) for p in head_g.parameters()]).clone()
    graphed = []
    for s, alpha in enumerate(alphas):
        if s == 0:
            step._graphs[float(alpha)] = step._capture(float(alpha))
            assert torch.equal(torch.cat([p.detach().reshape(-1) for p in head_g.parameters()]), start)
            assert head_g.rng_state.tolist()[1] == 0
        graphed.append(float(step(idx[s], alpha=alpha)))
    assert len(step._graphs) == 2
    assert head_g.rng_state.tolist() == head_e.rng_state.tolist()
    assert graphed == pytest.approx(eager, rel=1e-5)
    for pg, pe in zip(head_g.parameters(), head_e.parameters()):
        assert torch.allclose(pg, pe, rtol=1e-4, atol=1e-6)
    with pytest.raises(ValueError, match="store rows"):
        step(idx[0][:8], alpha=0.0)
