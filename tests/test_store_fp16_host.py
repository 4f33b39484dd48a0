"""CPU: the layer-mean store kept in fp16 (feature_store ``dtype=torch.float16``,
supcon_head_store_pool_forward_typed / supcon_head_sharded_store_pool_forward_typed): the declarations and exports,
argument checks that return before any CUDA work, the bookkeeping of fp16 stores, their files (``<f2``) and the
loads into them, and the sharded build, save and load under gloo with two ranks.  The stores live on the CPU; where
a layer mean is written, torch's mean stands in for the kernel (the GPU tests cover the kernel)."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharded_store_host import FRAMES, FEAT, CpuShard, Identity, _free_port, _outcome, clip, loader
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import feature_store as FS

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "supcon_b200.h")
NEW = ("supcon_head_store_pool_forward_typed", "supcon_head_sharded_store_pool_forward_typed")


def torch_layer_means(rows, slot0, hs):
    """CPU stand-in of ``feature_store.write_layer_means`` (the kernel needs a GPU)"""
    rows[slot0:slot0 + hs.shape[0]] = hs.float().mean(1)


class CpuShard16:
    """stand-in for the symmetric allocation of an fp16 shard: ``dtype`` arrives as a keyword"""

    def __init__(self, rows, feat, frames, device, group, *, dtype):
        self.rows = torch.full((rows, feat, frames), float("nan"), dtype=dtype)
        self.bases = [0] * dist.get_world_size(group)

    def close(self):
        self.rows = None


def bits16(x):
    return torch.from_numpy(np.ascontiguousarray(x)).view(torch.int16)


def test_entries_declared_exported_and_abi_unchanged(lib_built):
    text = open(HEADER).read()
    assert "#define SUPCON_F16 2" in text and _cabi.F16 == 2
    lib = _cabi.load()
    for name in NEW:
        assert f"int {name}(" in text
        assert name in _cabi.EXPORTS
        assert hasattr(lib, name)
    assert lib.supcon_abi_version() == _cabi.ABI_VERSION == 3


def test_hs_entries_still_reject_f16(lib_built):
    lib = _cabi.load()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.supcon_head_layer_mean_typed(p, _cabi.F16, 2, 3, 4, 5, p, None) == -1
    assert b"hs_dtype 2" in lib.supcon_last_error()
    assert lib.supcon_head_pool_forward_typed(p, _cabi.F16, 2, 3, 4, 5, 0.0, 0.01, None, p, None) == -1
    assert b"hs_dtype 2" in lib.supcon_last_error()


def test_typed_store_pool_rejects_bad_arguments(lib_built):
    lib = _cabi.load()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    fn = lib.supcon_head_store_pool_forward_typed
    who = b"supcon_head_store_pool_forward_typed"
    #        store, dtype, n_store, F, T, idx, B, p, slope, rng, pooled, stream
    for dtype in (-1, _cabi.BF16, 3):
        assert fn(p, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": unknown store_dtype %d (SUPCON_F32 or SUPCON_F16)" % dtype
    for dtype in (_cabi.F32, _cabi.F16):
        assert fn(None, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == b"NULL buffer passed to " + who
        assert fn(p, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, None, None) == -1
        assert lib.supcon_last_error() == b"NULL buffer passed to " + who
        assert fn(p, dtype, 10, 4, 5, None, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == b"NULL idx passed to " + who
        assert fn(p, dtype, 0, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad store size 0"
        assert fn(p, dtype, 10, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"
        for bad_p in (1.0, -0.1, float("nan")):
            assert fn(p, dtype, 10, 4, 5, p, 2, bad_p, 0.01, None, p, None) == -1
            assert lib.supcon_last_error() == who + b": dropout_p must be in [0, 1)"
        assert fn(p, dtype, 10, 4, 5, p, 70000, 0.0, 0.01, None, p, None) == -2
        assert fn(p, dtype, 10, 4, 12289, p, 2, 0.0, 0.01, None, p, None) == -2
        assert b"frames" in lib.supcon_last_error()
        assert fn(p, dtype, 2 ** 33, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1      # 64-bit n_store
        assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"


def test_typed_sharded_store_pool_rejects_bad_arguments(lib_built):
    lib = _cabi.load()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    fn = lib.supcon_head_sharded_store_pool_forward_typed
    who = b"supcon_head_sharded_store_pool_forward_typed"
    #        bases, R, dtype, n, F, T, idx, B, p, slope, rng, pooled, stream
    for dtype in (-1, _cabi.BF16, 3):
        assert fn(p, 2, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": unknown store_dtype %d (SUPCON_F32 or SUPCON_F16)" % dtype
    for dtype in (_cabi.F32, _cabi.F16):
        assert fn(None, 2, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == b"NULL buffer passed to " + who
        assert fn(p, 2, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, None, None) == -1
        assert lib.supcon_last_error() == b"NULL buffer passed to " + who
        assert fn(p, 2, dtype, 10, 4, 5, None, 2, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == b"NULL idx passed to " + who
        for ranks in (0, -1):
            assert fn(p, ranks, dtype, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
            assert lib.supcon_last_error() == who + b": bad rank count %d" % ranks
        for n, ranks in ((1, 2), (0, 1), (7, 8)):
            assert fn(p, ranks, dtype, n, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
            assert lib.supcon_last_error() == who + b": bad store size %d for %d ranks" % (n, ranks)
        assert fn(p, 2, dtype, 10, 0, 5, p, 2, 0.0, 0.01, None, p, None) == -1
        assert b"bad shape" in lib.supcon_last_error()
        assert fn(p, 2, dtype, 10, 4, 5, p, 2, 1.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": dropout_p must be in [0, 1)"
        assert fn(p, 2, dtype, 10, 4, 5, p, 70000, 0.0, 0.01, None, p, None) == -2
        assert fn(p, 8, dtype, 2 ** 33, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"


def test_fp16_store_bookkeeping():
    store = FS.LayerMeanStore(6, 8, 5, "cpu", dtype=torch.float16)
    assert store.dtype == store.rows.dtype == torch.float16 and store.rows.shape == (6, 8, 5)
    assert (store.n, store.feat, store.frames, store.filled) == (6, 8, 5, 0)
    assert store.labels.dtype == torch.int64 and store.labels.tolist() == [-1] * 6
    assert FS.LayerMeanStore(6, 8, 5, "cpu").dtype == torch.float32                # the default
    assert FS.store_bytes(6, 8, 5, torch.float16) == 6 * 8 * 5 * 2 + 6 * 8
    assert FS.store_bytes(6, 8, 5, torch.float32) == FS.store_bytes(6, 8, 5) == 6 * 8 * 5 * 4 + 6 * 8
    assert FS.store_bytes(2 ** 20, 1024, 199, torch.float16) == 2 ** 21 * 1024 * 199 + 2 ** 23    # 64-bit
    for bad in (torch.bfloat16, torch.float64, np.float16, "float16"):
        with pytest.raises(ValueError, match="store dtype must be torch.float32 or torch.float16"):
            FS.LayerMeanStore(6, 8, 5, "cpu", dtype=bad)
        with pytest.raises(ValueError, match="store dtype"):
            FS.store_bytes(6, 8, 5, bad)


def test_fit_error_names_the_dtype(monkeypatch):
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (10 ** 9, 2 * 10 ** 9))
    need = FS.store_bytes(25000, 1024, 199, torch.float16)
    msg = FS._fit_error(25000, 1024, 199, torch.device("cuda:0"), need, torch.float16)
    assert msg == "a store of 25000 clips x (1024, 199) fp16 takes 10.19 GB; 1.00 GB are free on cuda:0"


def fp16_cpu_store(n, feat, frames, seed=0):
    store = FS.LayerMeanStore(n, feat, frames, "cpu", dtype=torch.float16)
    g = torch.Generator().manual_seed(seed)
    store.rows.copy_(torch.randn(n, feat, frames, generator=g) * 100)
    store.labels.copy_(torch.arange(n) * 3 - 7)
    store.filled = n
    return store


def test_fp16_save_opens_as_float16_and_loads_bit_for_bit(tmp_path):
    store = fp16_cpu_store(9, 7, 13)
    store.rows[0, 0, :4] = torch.tensor([float("inf"), float("nan"), 6e-8, -0.0])   # carried as they are
    path = tmp_path / "store"
    assert store.save(path) == 9
    rows = np.load(path / "rows.npy")
    assert rows.dtype == np.float16 and rows.shape == (9, 7, 13)
    assert os.path.getsize(path / "rows.npy") - 128 == 9 * 7 * 13 * 2
    assert torch.equal(bits16(rows), store.rows.view(torch.int16))
    loaded = FS.load_layer_mean_store(path, "cpu", dtype=torch.float16)             # fp16 file -> fp16 store
    assert loaded.dtype == torch.float16 and loaded.filled == 9
    assert torch.equal(loaded.rows.view(torch.int16), store.rows.view(torch.int16))
    assert torch.equal(loaded.labels, store.labels)
    widened = FS.load_layer_mean_store(path, "cpu")                                 # fp16 file -> default store
    assert widened.dtype == torch.float32
    assert torch.equal(widened.rows.view(torch.int32), store.rows.float().view(torch.int32))
    loaded.save(tmp_path / "again")                                                # and saved again, the same
    assert (tmp_path / "again" / "rows.npy").read_bytes() == (path / "rows.npy").read_bytes()


def test_fp32_source_rounds_to_nearest_even(tmp_path):
    g = np.random.default_rng(3)
    a = (g.standard_normal((6, 5, 11)) * 1000).astype(np.float32)
    # halfway cases, the edges of the range, subnormals, and non-finite values (carried, not an error)
    a.reshape(-1)[:10] = [65504, 65519.99, -65519.99, 1 + 2 ** -11, 1 + 3 * 2 ** -11, 2 ** -25, 2 ** -26,
                          np.inf, np.nan, -np.inf]
    want = torch.from_numpy(a).half().view(torch.int16)
    np.save(tmp_path / "rows.npy", a)
    np.save(tmp_path / "labels.npy", np.arange(6))
    for rows in (np.load(tmp_path / "rows.npy", mmap_mode="r"), a, torch.from_numpy(a)):
        store = FS.LayerMeanStore.from_arrays(rows, np.arange(6), "cpu", dtype=torch.float16)
        assert store.dtype == torch.float16
        assert torch.equal(store.rows.view(torch.int16), want), type(rows)
    store = FS.load_layer_mean_store(tmp_path, "cpu", dtype=torch.float16)
    assert torch.equal(store.rows.view(torch.int16), want)


@pytest.mark.parametrize("value", [65520.0, -70000.0, 3e38])
def test_overflowing_fp32_source_raises_naming_file_and_slot(tmp_path, value):
    a = np.ones((5, 3, 7), np.float32)
    a[3, 2, 6] = value
    a[4, 0, 0] = value                                           # a later slot: the first one is named
    np.save(tmp_path / "rows.npy", a)
    np.save(tmp_path / "labels.npy", np.arange(5))
    with pytest.raises(ValueError, match=r"rows\.npy: slot 3: a finite layer mean rounds to inf in fp16") as err:
        FS.load_layer_mean_store(tmp_path, "cpu", dtype=torch.float16)
    assert str(tmp_path) in str(err.value)
    with pytest.raises(ValueError, match="^rows: slot 3: "):
        FS.LayerMeanStore.from_arrays(a, np.arange(5), "cpu", dtype=torch.float16)
    assert FS.load_layer_mean_store(tmp_path, "cpu").rows[3, 2, 6] == value      # an fp32 store takes it


def test_fp16_append_overflow_refuses_save(tmp_path, monkeypatch):
    monkeypatch.setattr(FS, "write_layer_means", torch_layer_means)
    store = FS.LayerMeanStore(6, 3, 4, "cpu", dtype=torch.float16)
    hs = torch.randn(4, 2, 3, 4)
    store.append(hs, torch.arange(4))
    assert torch.equal(store.rows[:4].view(torch.int16), hs.mean(1).half().view(torch.int16))
    big = torch.randn(2, 2, 3, 4)
    big[1, :, 1, 2] = 1e5
    store.append(big, torch.arange(2))                           # no error yet: the flag is on the device
    assert store.filled == 6 and bool(store.rows[5, 1, 2].isinf())
    with pytest.raises(ValueError, match="slot 5: a finite layer mean rounds to inf in fp16.*not saved"):
        store.save(tmp_path / "store")
    assert os.listdir(tmp_path) == []
    # non-finite hidden states are carried into the rows, as in an fp32 store: not an overflow
    nan = FS.LayerMeanStore(2, 3, 4, "cpu", dtype=torch.float16)
    nan.append(torch.full((2, 2, 3, 4), float("inf")), torch.arange(2))
    assert nan.save(tmp_path / "inf") == 2


@pytest.mark.parametrize("src_dtype", [np.float16, np.float32])
@pytest.mark.parametrize("shape", [(9, 7, 13), (5, 37, 41)], ids=["rows_smaller_than_a_chunk", "rows_over_a_chunk"])
def test_chunks_split_fp16_rows(tmp_path, monkeypatch, shape, src_dtype):
    """4 KiB staging: 2048 fp16 elements (or 1024 fp32 of a source being rounded); rows of 91 elements straddle
    chunk edges, rows of 1517 span two chunks (of fp32).  Every kind of source, and a save through the same chunks."""
    monkeypatch.setattr(FS, "STAGE_BYTES", 4096)
    n = shape[0]
    a = (np.random.default_rng(4).standard_normal((n, shape[1], 2 * shape[2])) * 50).astype(src_dtype)
    strided = a[:, :, ::2]
    dense = np.ascontiguousarray(strided)
    want = torch.from_numpy(dense).half().view(torch.int16)
    np.save(tmp_path / "rows.npy", dense)
    np.save(tmp_path / "labels.npy", np.arange(n))
    mm = np.load(tmp_path / "rows.npy", mmap_mode="r")
    for rows in (mm, dense, strided, torch.from_numpy(dense)):
        store = FS.LayerMeanStore.from_arrays(rows, np.arange(n), "cpu", dtype=torch.float16)
        assert torch.equal(store.rows.view(torch.int16), want), type(rows)
    tail = FS.LayerMeanStore.from_arrays(mm[1:], np.arange(n - 1), "cpu", dtype=torch.float16)
    assert torch.equal(tail.rows.view(torch.int16), want[1:])
    store.save(tmp_path / "again")
    assert torch.equal(bits16(np.load(tmp_path / "again" / "rows.npy")), want)


# ------------------------------------------------------------------------------ sharded fp16 stores under gloo

def _worker(rank, world, port, root, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    FS.STAGE_BYTES = 40                        # 20 fp16 or 10 fp32 elements: chunks split the rows of 12
    FS.write_layer_means = torch_layer_means
    f16 = torch.float16
    try:
        res = {}
        n = 7
        mine = list(FS.shard_slots(n, rank, world))

        def build(batches, **kw):
            return FS.build_sharded_layer_mean_store(Identity(), batches, "cpu", n=n, allocate=CpuShard16,
                                                     dtype=f16, **kw)

        def built():
            store = build(loader(mine))
            got = (store.dtype, store.filled, store.labels.tolist(), store.rows.clone(),
                   store.save(os.path.join(root, "sharded")))
            store.close()
            return got
        res["built"] = _outcome(built)
        dist.barrier()
        if rank == 0:                                             # R = 1 writes an fp32 file that R = 2 rounds
            means = torch.stack([clip(i).mean(0) for i in range(n)])
            FS.LayerMeanStore.from_arrays(-means, 10 * np.arange(n), "cpu").save(os.path.join(root, "single"))
        dist.barrier()

        def load(name, **kw):
            store = FS.load_sharded_layer_mean_store(os.path.join(root, name), "cpu", **kw)
            got = (store.dtype, store.filled, store.labels.tolist(), store.rows.clone())
            store.close()
            return got
        res["from_single"] = _outcome(lambda: load("single", allocate=CpuShard16, dtype=f16))
        res["from_sharded"] = _outcome(lambda: load("sharded", allocate=CpuShard16, dtype=f16))
        res["widened"] = _outcome(lambda: load("sharded", allocate=CpuShard))
        # each failure below happens on ONE rank; both must raise
        res["dtypes"] = _outcome(lambda: load("sharded", allocate=CpuShard16 if rank else CpuShard,
                                              **({"dtype": f16} if rank else {})))
        res["bf16"] = _outcome(lambda: FS.ShardedLayerMeanStore(n, FEAT, FRAMES, "cpu", allocate=CpuShard16,
                                                                dtype=torch.bfloat16))

        def hot(batches):                                         # slot 5 (rank 1's local row 2) overflows
            return [(x * torch.tensor([1e6 if label == 50 else 1.0 for label in y.tolist()]).view(-1, 1, 1, 1), y)
                    for x, y in batches]
        res["build_overflow"] = _outcome(lambda: build(hot(loader(mine))).filled)
        big = np.stack([clip(i).mean(0).numpy() for i in range(n)])
        big[5, 1, 1] = 1e6
        res["load_overflow"] = _outcome(lambda: FS.ShardedLayerMeanStore.from_arrays(
            big, np.arange(n), "cpu", allocate=CpuShard16, dtype=f16).filled)
        res["after"] = _outcome(lambda: load("sharded", allocate=CpuShard16, dtype=f16)[1])
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_two_rank_fp16_build_save_load_under_gloo(tmp_path):
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), out), nprocs=2, join=True)
    n = 7
    means = torch.stack([clip(i).mean(0) for i in range(n)])
    rows = np.load(tmp_path / "sharded" / "rows.npy")             # the sharded fp16 save: slot order, <f2
    assert rows.dtype == np.float16
    assert torch.equal(bits16(rows), means.half().view(torch.int16))
    one = FS.load_layer_mean_store(tmp_path / "sharded", "cpu", dtype=torch.float16)       # R' = 1
    assert torch.equal(one.rows.view(torch.int16), means.half().view(torch.int16))
    for rank in (0, 1):
        res = out[rank]
        kind, (dtype, filled, labels, shard, saved) = res["built"]
        assert kind == "ok" and (dtype, filled, saved) == (torch.float16, n, n)
        assert labels == [10 * i for i in range(n)]
        for j, i in enumerate(range(rank, n, 2)):
            assert torch.equal(shard[j].view(torch.int16), means[i].half().view(torch.int16))
        for case, want, wdtype in (("from_single", (-means).half(), torch.float16),
                                   ("from_sharded", means.half(), torch.float16),
                                   ("widened", means.half().float(), torch.float32)):
            kind, (dtype, filled, labels, shard) = res[case]
            assert kind == "ok" and (dtype, filled) == (wdtype, n), (rank, case)
            assert labels == [10 * i for i in range(n)]
            for j, i in enumerate(range(rank, n, 2)):
                assert torch.equal(shard[j], want[i]), (rank, case, j)

        def raised(case, *fragments):
            kind, msg = res[case]
            assert kind == "ValueError", (rank, case, kind, msg)
            for f in fragments:
                assert f in msg, (rank, case, msg)
        raised("dtypes", "disagree on the store dtype", "rank 0 torch.float32", "rank 1 torch.float16")
        raised("bf16", "store dtype must be torch.float32 or torch.float16, got torch.bfloat16")
        raised("build_overflow", "rank 1: slot 5: a finite layer mean rounds to inf in fp16")
        raised("load_overflow", "rank 1: rows: slot 5: a finite layer mean rounds to inf in fp16")
        assert "rank 0" not in res["build_overflow"][1] and "rank 0" not in res["load_overflow"][1]
        assert res["after"] == ("ok", n)
