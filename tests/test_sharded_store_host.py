"""CPU: the layer-mean store sharded over the GPUs of a node (feature_store.ShardedLayerMeanStore,
supcon_head_sharded_store_pool_forward): the declaration and export, argument checks that return before any CUDA
work, the slot layout, and the build's bookkeeping under gloo with two ranks.  There the shard allocation is a CPU
stand-in (as test_distributed_cpu.py stands in for the kernels): every check that can fail on one rank must raise on
both, and the label all-gather must return slot order."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from wav2vec_contr_loss_b200 import _cabi

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "supcon_b200.h")
NAME = "supcon_head_sharded_store_pool_forward"


def test_entry_declared_exported_and_abi_unchanged(lib_built):
    assert f"int {NAME}(" in open(HEADER).read()
    assert NAME in _cabi.EXPORTS
    lib = _cabi.load()
    assert hasattr(lib, NAME)
    assert lib.supcon_abi_version() == _cabi.ABI_VERSION == 3


def test_sharded_pool_rejects_bad_arguments(lib_built):
    lib = _cabi.load()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    fn = getattr(lib, NAME)
    who = NAME.encode()
    #        bases, R, n, F, T, idx, B, p, slope, rng, pooled, stream
    assert fn(None, 2, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    assert fn(p, 2, 10, 4, 5, p, 2, 0.0, 0.01, None, None, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    assert fn(p, 2, 10, 4, 5, None, 2, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL idx passed to " + who
    for ranks in (0, -1):
        assert fn(p, ranks, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad rank count %d" % ranks
    for n, ranks in ((1, 2), (0, 1), (7, 8)):
        assert fn(p, ranks, n, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad store size %d for %d ranks" % (n, ranks)
    assert fn(p, 2, 10, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"
    assert fn(p, 2, 10, 0, 5, p, 2, 0.0, 0.01, None, p, None) == -1 and b"bad shape" in lib.supcon_last_error()
    assert fn(p, 2, 10, 4, 0, p, 2, 0.0, 0.01, None, p, None) == -1 and b"bad shape" in lib.supcon_last_error()
    for bad_p in (1.0, -0.1, float("nan")):
        assert fn(p, 2, 10, 4, 5, p, 2, bad_p, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": dropout_p must be in [0, 1)"
    assert fn(p, 2, 10, 4, 5, p, 70000, 0.0, 0.01, None, p, None) == -2 and b"65535" in lib.supcon_last_error()
    assert fn(p, 2, 10, 4, 12289, p, 2, 0.0, 0.01, None, p, None) == -2 and b"frames" in lib.supcon_last_error()
    # n_store is 64-bit: a count past 2^31 passes the size check and stops at the next one
    assert fn(p, 8, 2 ** 33, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"


@pytest.mark.parametrize("n", [1, 2, 7, 8, 9, 64, 1001])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_shard_slots_cover_every_slot_once(n, world):
    from wav2vec_contr_loss_b200.feature_store import shard_slots
    seen = []
    for rank in range(world):
        slots = list(shard_slots(n, rank, world))
        assert all(i % world == rank for i in slots)
        assert [i // world for i in slots] == list(range(len(slots)))      # local rows in order, from 0
        assert len(slots) <= -(-n // world)                                 # every shard fits ceil(n / R) rows
        seen += slots
    assert sorted(seen) == list(range(n))


# ---------------------------------------------------------------------------------- the build under gloo

K, FEAT, FRAMES = 2, 4, 3


class CpuShard:
    """stand-in for the symmetric allocation: a CPU tensor, and the layer mean written by torch"""

    def __init__(self, rows, feat, frames, device, group):
        self.rows = torch.full((rows, feat, frames), float("nan"))
        self.bases = [0] * dist.get_world_size(group)

    def write(self, row0, hs):
        self.rows[row0:row0 + hs.shape[0]] = hs.float().mean(1)

    def close(self):
        self.rows = None


class Identity(torch.nn.Module):
    def forward(self, x, attention_mask=None):
        return x


def clip(i, frames=FRAMES):
    return torch.randn(K, FEAT, frames, generator=torch.Generator().manual_seed(100 + i))


def loader(slots, batch=2, frames_of=lambda i: FRAMES):
    """(hs as the 'waveforms' of an identity encoder, labels 10 i) in batches of `batch`"""
    slots = list(slots)
    return [(torch.stack([clip(i, frames_of(i)) for i in slots[s:s + batch]]),
             torch.tensor([10 * i for i in slots[s:s + batch]]))
            for s in range(0, len(slots), batch)]


def _outcome(fn):
    try:
        return "ok", fn()
    except (ValueError, MemoryError, RuntimeError) as exc:
        return type(exc).__name__, str(exc)


def _worker(rank, world, port, out):
    from wav2vec_contr_loss_b200.feature_store import build_sharded_layer_mean_store, shard_slots
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        def build(n, slots, **kw):
            return build_sharded_layer_mean_store(Identity(), loader(slots, **kw), "cpu", n=n, allocate=CpuShard)

        res = {}
        n = 7
        mine = list(shard_slots(n, rank, world))

        def good():
            store = build(n, mine)
            got = (store.filled, store.n, store.local_rows, store.labels.tolist(), store.rows.clone(),
                   store.labels_of(torch.tensor([6, 0, 3, -2, 9])).tolist())
            store.close()
            assert store.rows is None
            return got
        res["good"] = _outcome(good)
        # every failure below happens on ONE rank; both must raise (a hang would time the test out)
        res["first_shape"] = _outcome(lambda: build(n, mine, frames_of=lambda i: FRAMES + (rank == 1)))
        res["later_shape"] = _outcome(lambda: build(n, mine, frames_of=lambda i: FRAMES + (i == 5)))
        res["short"] = _outcome(lambda: build(n, mine[:-1] if rank == 1 else mine))
        res["long"] = _outcome(lambda: build(n, mine + [mine[0]] if rank == 0 else mine))
        res["empty"] = _outcome(lambda: build(n, [] if rank == 1 else mine))
        res["n_below_world"] = _outcome(lambda: build(1, [0] if rank == 0 else []))
        res["n_disagrees"] = _outcome(lambda: build(n + 2 * rank, mine))
        res["after"] = _outcome(lambda: build(n, mine).filled)      # the group still works after all of that
        out[rank] = res
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_two_rank_build_bookkeeping_under_gloo():
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    for rank in (0, 1):
        res = out[rank]
        kind, (filled, n, local_rows, labels, rows, picked) = res["good"]
        assert kind == "ok" and (filled, n, local_rows) == (7, 7, 4)
        assert labels == [10 * i for i in range(7)]                                # slot order
        assert picked == [60, 0, 30, 0, 60]                                        # clamped into [0, filled)
        for j, i in enumerate(range(rank, 7, 2)):                                  # row j = slot 2 j + rank
            assert torch.equal(rows[j], clip(i).mean(0))
        if rank == 1:
            assert bool(rows[3].isnan().all())                                     # the padding row is never written

        def raised(case, *fragments):
            kind, msg = res[case]
            assert kind == "ValueError", (rank, case, kind, msg)
            for f in fragments:
                assert f in msg, (rank, case, msg)
        raised("first_shape", "disagree on the store's (n, F, T)", "rank 0 (7, 4, 3)", "rank 1 (7, 4, 4)")
        raised("later_shape", "rank 1: clips 2..2: hidden states of (F, T) = (4, 4), the store holds (4, 3)")
        raised("short", "rank 1: the loader yielded 2 clips, this rank's share of 7 is 3")
        raised("long", "rank 0: the loader yields more than this rank's 4 clips of 7")
        raised("empty", "rank 1 (7, 0, 0)")
        raised("n_below_world", "needs at least 2 clips, got 1")
        raised("n_disagrees", "rank 0 (7, 4, 3)", "rank 1 (9, 4, 3)")
        assert res["after"] == ("ok", 7)
