"""The layer-mean store on disk: what a build costs against a save and a load of the same store, in one process:

    python tools/store_io_bench.py [--clips 4096] [--dir /tmp] [--out profiles/r08_store_io_bench.json]

* build: --clips synthetic 4 s clips through a random-init XLS-R-300M (tools/store_step_bench.py's encoder), frozen,
  fp32, batch 64, with build_layer_mean_store, after one warm-up batch (as tools/sharded_store_bench.py builds).
* save: LayerMeanStore.save into a fresh directory under --dir, fsyncs and rename included.
* load: load_layer_mean_store of that directory, --loads times; each loaded store is checked bit for bit against
  the built one.

Times are host clocks around work that ends in a device synchronise; rates are rows.npy's bytes over them.  Host
memory: the peak growth of this process's resident set over each step, sampled every millisecond from
/proc/self/statm.  Page cache: the share of rows.npy's pages resident just before each load, from mincore(2).
Caches are not dropped, so a load right after the save reads from memory, not from the disk; the record says so.
The store directory is removed at the end.
"""
import argparse
import ctypes
import json
import os
import shutil
import sys
import tempfile
import threading
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from sharded_store_bench import card  # noqa: E402

B, F, T = 64, 1024, 199
PAGE = os.sysconf("SC_PAGE_SIZE")


class PeakRss:
    """peak growth of this process's resident set while the block runs (sampled every millisecond)"""

    def __enter__(self):
        self.start = self.peak = self._rss()
        self.stop = threading.Event()
        self.thread = threading.Thread(target=self._watch, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.thread.join()
        self.peak = max(self.peak, self._rss())
        self.growth_MB = (self.peak - self.start) / 1e6

    def _watch(self):
        while not self.stop.wait(0.001):
            self.peak = max(self.peak, self._rss())

    @staticmethod
    def _rss():
        with open("/proc/self/statm") as fh:
            return int(fh.read().split()[1]) * PAGE


def resident_share(file):
    """share of ``file``'s pages in the page cache (mincore of an untouched read-only mapping), or None"""
    libc = ctypes.CDLL(None, use_errno=True)
    libc.mmap.restype = ctypes.c_void_p
    libc.mmap.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_long]
    libc.munmap.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    libc.mincore.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    size = os.path.getsize(file)
    fd = os.open(file, os.O_RDONLY)
    try:
        addr = libc.mmap(None, size, 1, 1, fd, 0)                       # PROT_READ, MAP_SHARED
        if addr in (None, ctypes.c_void_p(-1).value):
            return None
        vec = np.zeros(-(-size // PAGE), np.uint8)
        rc = libc.mincore(addr, size, vec.ctypes.data)
        libc.munmap(addr, size)
        return None if rc != 0 else float((vec & 1).mean())
    finally:
        os.close(fd)


def timed(dev, fn):
    torch.cuda.synchronize(dev)
    with PeakRss() as rss:
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize(dev)
        s = time.perf_counter() - t0
    return out, s, rss.growth_MB


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--clips", type=int, default=4096)
    ap.add_argument("--dir", default=tempfile.gettempdir(), help="where the store is written (and removed)")
    ap.add_argument("--loads", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    from torch.utils.data import DataLoader
    from store_step_bench import Clips, XlsrStandIn
    from wav2vec_contr_loss_b200 import build
    from wav2vec_contr_loss_b200 import feature_store as FS
    build.build()
    rows_bytes = args.clips * F * T * 4
    free = shutil.disk_usage(args.dir).free
    if free < rows_bytes * 1.1 + (1 << 30):
        raise SystemExit(f"{args.dir} has {free / 1e9:.1f} GB free; the store takes {rows_bytes / 1e9:.2f} GB")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card(dev), "clips": args.clips, "rows_GB": rows_bytes / 1e9, "dir": args.dir,
           "disk_free_GB_before": free / 1e9, "stage_bytes": FS.STAGE_BYTES,
           "encoder": "random-init XLS-R-300M, frozen, fp32, batch 64"}
    torch.manual_seed(1337)
    enc = XlsrStandIn().to(dev).eval()
    ds = Clips(args.clips)
    with torch.no_grad():                                      # warm-up: cuDNN / cuBLAS choices for the shapes used
        w = ds.wave[:B].to(dev)
        enc(w, attention_mask=(w != 0).long())
    store, res["build_s"], res["build_rss_growth_MB"] = timed(
        dev, lambda: FS.build_layer_mean_store(enc, DataLoader(ds, batch_size=B), dev))
    del enc, ds
    torch.cuda.empty_cache()
    path = os.path.join(tempfile.mkdtemp(dir=args.dir, prefix="store_io_bench_"), "store")
    try:
        n, res["save_s"], res["save_rss_growth_MB"] = timed(dev, lambda: store.save(path))
        assert n == args.clips
        res["save_GB_per_s"] = rows_bytes / res["save_s"] / 1e9
        res["loads"] = []
        for _ in range(args.loads):
            cached = resident_share(os.path.join(path, FS.ROWS_FILE))
            loaded, s, grow = timed(dev, lambda: FS.load_layer_mean_store(path, dev))
            same = bool(torch.equal(loaded.rows.view(torch.int32), store.rows.view(torch.int32))
                        and torch.equal(loaded.labels, store.labels))
            res["loads"].append({"load_s": s, "GB_per_s": rows_bytes / s / 1e9, "rss_growth_MB": grow,
                                 "rows_file_share_in_page_cache_before": cached, "equal_to_built_bit_for_bit": same})
            del loaded
            torch.cuda.empty_cache()
        best = min(x["load_s"] for x in res["loads"])
        res["build_over_load"] = res["build_s"] / best
        res["page_cache_note"] = ("caches were not dropped: each load read rows.npy from the page cache as far as "
                                  "rows_file_share_in_page_cache_before says, not from the disk; the save's time "
                                  "includes its fsync, so the data reached the disk")
    finally:
        shutil.rmtree(os.path.dirname(path), ignore_errors=True)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
