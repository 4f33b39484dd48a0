"""CPU: the layer-mean store on disk (feature_store: LayerMeanStore.save / from_arrays, load_layer_mean_store,
ShardedLayerMeanStore.save / from_arrays, load_sharded_layer_mean_store).  The stores here live on the CPU, which
runs the same chunked copy as a GPU store with a synchronous copy in place of the side stream's: the file format,
the partial directory, the checks, chunks that split rows, and the slot order of a sharded save and load under gloo
with two ranks (the shard allocation stood in for by test_sharded_store_host.CpuShard)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharded_store_host import CpuShard, Identity, _free_port, _outcome, clip, loader
from wav2vec_contr_loss_b200 import feature_store as FS


def cpu_store(n, feat, frames, filled=None, seed=0):
    store = FS.LayerMeanStore(n, feat, frames, "cpu")
    g = torch.Generator().manual_seed(seed)
    store.rows.copy_(torch.randn(n, feat, frames, generator=g))
    store.labels.copy_(torch.arange(n) * 3 - 7)
    store.filled = n if filled is None else filled
    return store


def bits(x):
    return torch.from_numpy(np.array(x)).view(torch.int32)


@pytest.mark.parametrize("filled", [5, 9])
def test_format_opens_with_plain_np_load(tmp_path, filled):
    store = cpu_store(9, 7, 13, filled=filled)
    path = tmp_path / "store"
    assert store.save(path) == filled
    assert sorted(os.listdir(path)) == ["labels.npy", "rows.npy"]
    rows = np.load(path / "rows.npy", mmap_mode="r")
    assert rows.dtype == np.float32 and rows.shape == (filled, 7, 13) and rows.flags.c_contiguous
    assert torch.equal(bits(rows), store.rows[:filled].view(torch.int32))
    labels = np.load(path / "labels.npy")
    assert labels.dtype == np.int64 and labels.tolist() == store.labels[:filled].tolist()
    loaded = FS.load_layer_mean_store(path, "cpu")
    assert (loaded.n, loaded.filled, loaded.feat, loaded.frames) == (filled, filled, 7, 13)
    assert torch.equal(loaded.rows.view(torch.int32), store.rows[:filled].view(torch.int32))
    assert torch.equal(loaded.labels, store.labels[:filled])
    assert not os.path.exists(str(path) + ".partial")


def test_existing_path_kept_unless_overwrite(tmp_path):
    path = tmp_path / "store"
    a, b = cpu_store(4, 3, 5, seed=1), cpu_store(6, 3, 5, seed=2)
    assert a.save(path) == 4
    assert b.save(path) is None                                           # kept
    assert torch.equal(FS.load_layer_mean_store(path, "cpu").rows, a.rows)
    assert b.save(path, overwrite=True) == 6
    assert torch.equal(FS.load_layer_mean_store(path, "cpu").rows, b.rows)
    assert sorted(os.listdir(tmp_path)) == ["store"]                      # no .partial, no .old left


def test_failed_save_leaves_no_partial_directory(tmp_path, monkeypatch):
    path = tmp_path / "store"
    store = cpu_store(5, 4, 3)
    real = os.fsync
    calls = []

    def dying_fsync(fd):
        calls.append(fd)
        if len(calls) == 2:                                               # the labels file's: after rows.npy
            raise OSError(28, "No space left on device")
        real(fd)
    monkeypatch.setattr(FS.os, "fsync", dying_fsync)
    with pytest.raises(OSError, match="No space left"):
        store.save(path)
    assert os.listdir(tmp_path) == []
    monkeypatch.setattr(FS.os, "fsync", real)
    # a save killed earlier left its partial directory: the next save replaces it, and it never loads
    (tmp_path / "store.partial").mkdir()
    (tmp_path / "store.partial" / "rows.npy").write_bytes(b"junk")
    with pytest.raises(FileNotFoundError, match="no layer-mean store"):
        FS.load_layer_mean_store(path, "cpu")
    assert store.save(path) == 5
    assert sorted(os.listdir(tmp_path)) == ["store"]
    # an overwrite that fails keeps the old store
    monkeypatch.setattr(FS, "_write_rows", lambda *a: (_ for _ in ()).throw(OSError(5, "I/O error")))
    with pytest.raises(OSError, match="I/O error"):
        cpu_store(2, 4, 3, seed=9).save(path, overwrite=True)
    assert sorted(os.listdir(tmp_path)) == ["store"]
    assert torch.equal(FS.load_layer_mean_store(path, "cpu").rows, store.rows)


def test_empty_store_refuses_to_save(tmp_path):
    with pytest.raises(ValueError, match="empty"):
        cpu_store(3, 2, 2, filled=0).save(tmp_path / "store")
    assert os.listdir(tmp_path) == []


@pytest.mark.parametrize("name", ["rows.npy", "labels.npy"])
def test_truncated_file_is_refused_by_name(tmp_path, name):
    path = tmp_path / "store"
    cpu_store(6, 5, 7).save(path)
    file = path / name
    with open(file, "r+b") as fh:
        fh.truncate(os.path.getsize(file) - 4)
    with pytest.raises(ValueError, match=name):
        FS.load_layer_mean_store(path, "cpu")
    os.remove(file)
    with pytest.raises(FileNotFoundError, match=name):
        FS.load_layer_mean_store(path, "cpu")
    with pytest.raises(FileNotFoundError, match="no layer-mean store"):
        FS.load_layer_mean_store(tmp_path / "nowhere", "cpu")


def test_dtype_rank_and_label_checks():
    a = np.random.default_rng(0).standard_normal((4, 3, 5)).astype(np.float32)
    y = np.arange(4)
    for bad in (a.astype(np.float64), a.astype(np.int32), torch.from_numpy(a).bfloat16(), a.astype(">f4")):
        with pytest.raises(ValueError, match="float32 or float16"):
            FS.LayerMeanStore.from_arrays(bad, y, "cpu")
    for bad in (a[0], a[None]):
        with pytest.raises(ValueError, match=r"must be \(n, F, T\)"):
            FS.LayerMeanStore.from_arrays(bad, y, "cpu")
    with pytest.raises(ValueError, match="numpy array or a CPU tensor"):
        FS.LayerMeanStore.from_arrays(a.tolist(), y, "cpu")
    for bad in (y[:3], y.reshape(2, 2), y.astype(np.float32), np.ones(4, bool), torch.ones(4)):
        with pytest.raises(ValueError, match=r"labels must be \(4,\) integers"):
            FS.LayerMeanStore.from_arrays(a, bad, "cpu")
    for y_ok in (y.astype(np.int32), y.astype(np.uint8), torch.arange(4, dtype=torch.int16)):
        assert FS.LayerMeanStore.from_arrays(a, y_ok, "cpu").labels.tolist() == [0, 1, 2, 3]


def test_float16_is_widened_exactly():
    g = np.random.default_rng(1)
    a = (g.standard_normal((5, 7, 11)) * 300).astype(np.float16)
    a.reshape(-1)[:6] = [np.inf, -np.inf, np.nan, 6e-8, -0.0, 65504]           # specials and a subnormal
    want = torch.from_numpy(a).float().view(torch.int32)
    for rows in (a, torch.from_numpy(a)):
        store = FS.LayerMeanStore.from_arrays(rows, np.arange(5), "cpu")
        assert torch.equal(store.rows.view(torch.int32), want)


@pytest.mark.parametrize("dtype", [np.float32, np.float16])
@pytest.mark.parametrize("shape", [(9, 7, 13), (5, 37, 41)], ids=["rows_smaller_than_a_chunk", "rows_over_a_chunk"])
def test_chunks_that_split_rows(tmp_path, monkeypatch, shape, dtype):
    """4 KiB staging (1024 fp32 elements): rows of 91 elements straddle chunk edges, rows of 1517 span two chunks.
    Every kind of source: the file (readinto), a memmap slice, a plain array, a strided array, a CPU tensor."""
    monkeypatch.setattr(FS, "STAGE_BYTES", 4096)
    n = shape[0]
    a = np.random.default_rng(2).standard_normal((n, shape[1], 2 * shape[2])).astype(dtype)
    strided = a[:, :, ::2]
    dense = np.ascontiguousarray(strided)
    want = torch.from_numpy(dense).float().view(torch.int32)
    np.save(tmp_path / "rows.npy", dense)
    np.save(tmp_path / "labels.npy", np.arange(n))
    mm = np.load(tmp_path / "rows.npy", mmap_mode="r")
    whole = FS._RowSource(mm)
    assert whole.file is not None and FS._RowSource(mm[1:]).file is None
    for rows in (mm, dense, strided, torch.from_numpy(dense)):
        store = FS.LayerMeanStore.from_arrays(rows, np.arange(n), "cpu")
        assert torch.equal(store.rows.view(torch.int32), want), type(rows)
    tail = FS.LayerMeanStore.from_arrays(mm[1:], np.arange(n - 1), "cpu")
    assert torch.equal(tail.rows.view(torch.int32), want[1:])
    if dtype == np.float32:                                       # save through the same chunks, load it back
        store = FS.load_layer_mean_store(tmp_path, "cpu")
        store.save(tmp_path / "again")
        assert torch.equal(bits(np.load(tmp_path / "again" / "rows.npy")), want)


def test_chunks_cover_the_slots_in_order():
    for slots, row, chunk in [(range(7), 5, 3), (range(1, 9, 3), 4, 6), (range(0, 5, 2), 10, 4), (range(2, 2), 3, 4)]:
        got = list(FS._chunks(slots, row, chunk))
        d = 0
        flat = []
        for d0, pieces in got:
            assert d0 == d and 0 < sum(k for _, k in pieces) <= chunk
            d += sum(k for _, k in pieces)
            flat += [f for f0, k in pieces for f in range(f0, f0 + k)]
        assert flat == [s * row + e for s in slots for e in range(row)]


# ------------------------------------------------------------------------------ sharded save / load under gloo

K, FEAT, FRAMES = 2, 4, 3          # test_sharded_store_host's clip shape


def _worker(rank, world, port, root, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    FS.STAGE_BYTES = 40                                           # 10 elements: chunks split the rows of 12
    try:
        res = {}
        n = 7
        mine = list(FS.shard_slots(n, rank, world))
        built = FS.build_sharded_layer_mean_store(Identity(), loader(mine), "cpu", n=n, allocate=CpuShard)
        res["saved"] = _outcome(lambda: built.save(os.path.join(root, "sharded")))
        res["kept"] = _outcome(lambda: built.save(os.path.join(root, "sharded")))
        built.close()
        dist.barrier()
        if rank == 0:                                             # R = 1 writes a file that R = 2 loads
            means = torch.stack([clip(i).mean(0) for i in range(n)])
            FS.LayerMeanStore.from_arrays(-means, 10 * np.arange(n), "cpu").save(os.path.join(root, "single"))
        dist.barrier()

        def load(name, **kw):
            store = FS.load_sharded_layer_mean_store(os.path.join(root, name), "cpu", allocate=CpuShard, **kw)
            got = (store.filled, store.local_rows, store.labels.tolist(), store.rows.clone())
            store.close()
            return got
        res["from_single"] = _outcome(lambda: load("single"))
        res["from_sharded"] = _outcome(lambda: load("sharded"))
        # each failure below happens on ONE rank; both must raise
        res["missing"] = _outcome(lambda: load("sharded" if rank == 0 else "nowhere"))
        res["shapes"] = _outcome(lambda: FS.ShardedLayerMeanStore.from_arrays(
            np.zeros((n, FEAT, FRAMES + rank), np.float32), np.arange(n), "cpu", allocate=CpuShard))
        res["dtypes"] = _outcome(lambda: FS.ShardedLayerMeanStore.from_arrays(
            np.zeros((n, FEAT, FRAMES), np.float16 if rank else np.float32), np.arange(n), "cpu",
            allocate=CpuShard))
        res["labels"] = _outcome(lambda: FS.ShardedLayerMeanStore.from_arrays(
            np.zeros((n, FEAT, FRAMES), np.float32), np.arange(n - rank), "cpu", allocate=CpuShard))
        res["after"] = _outcome(lambda: load("single")[0])          # the group still works after all of that
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_two_rank_save_and_load_under_gloo(tmp_path):
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), out), nprocs=2, join=True)
    n = 7
    means = torch.stack([clip(i).mean(0) for i in range(n)])
    # the sharded save wrote slot order, which R' = 1 loads
    rows = np.load(tmp_path / "sharded" / "rows.npy")
    assert torch.equal(torch.from_numpy(rows), means)
    assert np.load(tmp_path / "sharded" / "labels.npy").tolist() == [10 * i for i in range(n)]
    one = FS.load_layer_mean_store(tmp_path / "sharded", "cpu")
    assert torch.equal(one.rows, means) and one.filled == n
    assert sorted(os.listdir(tmp_path)) == ["sharded", "single"]
    for rank in (0, 1):
        res = out[rank]
        assert res["saved"] == ("ok", n) and res["kept"] == ("ok", None)
        for case, want in (("from_single", -means), ("from_sharded", means)):
            kind, (filled, local_rows, labels, shard) = res[case]
            assert kind == "ok" and (filled, local_rows) == (n, 4), (rank, case)
            assert labels == [10 * i for i in range(n)]
            for j, i in enumerate(range(rank, n, 2)):                        # local row j = slot rank + 2 j
                assert torch.equal(shard[j], want[i]), (rank, case, j)
            if rank == 1:
                assert bool(shard[3].isnan().all())                          # the padding row is never written

        def raised(case, *fragments):
            kind, msg = res[case]
            assert kind == "ValueError", (rank, case, kind, msg)
            for f in fragments:
                assert f in msg, (rank, case, msg)
        raised("missing", "rank 1: no layer-mean store at", "nowhere")
        raised("shapes", "disagree on the store's (n, F, T)", "rank 0 (7, 4, 3)", "rank 1 (7, 4, 4)")
        raised("dtypes", "disagree on the rows' dtype", "rank 0 float32", "rank 1 float16")
        raised("labels", "rank 1: labels must be (7,) integers")
        assert res["after"] == ("ok", n)
