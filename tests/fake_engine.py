"""TEST INFRASTRUCTURE: a stand-in for `lantern_b200.api` that answers through the CPU oracle (oracle/portlib.py).

tests/test_bench_dryrun.py uses it to walk bench.py's `run_ours` glue (argument plumbing, the JSON line, the
cpu_baseline / parity / sharding branches) on a machine without a GPU.  It mirrors the few entry points bench.py calls,
with the same signatures (raw pointers in, results written through raw pointers).  The oracle also stands in for the
compiled reference (`oracle.reflib`) that cpu_baseline and the `--impl reference` arm (tests/test_bench_contract.py) drive,
so that neither walk needs a reference build.  Nothing here is a product path."""
import ctypes as C
import time
import types

import numpy as np

from oracle import portlib

LAUNCHES = [0]


class HostEvent:
    def __init__(self, enable_timing=True):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return 1e3 * (other.t - self.t)


class HostStream:
    cuda_stream = 0


TINY = {
    "tiny": dict(n=3000, dim=32, metric="l2sq", M=8, efc=32, ef=16, batch=8, k=10, recall_1gpu=0.9,
                 desc="tiny: dry run on the CPU stand-in"),
    "tinybits": dict(n=2000, dim=128, kind="b1", metric="hamming", M=8, efc=32, ef=16, batch=8, k=10,
                     desc="tinybits: dry run on the CPU stand-in"),
}


def install(bench, setattr_=setattr, setitem=None):
    """Point bench.py at this module and at host stand-ins for torch.cuda's stream/event calls.  `setattr_` / `setitem` let
    pytest's monkeypatch undo it; the 2-rank runner (tests/dryrun_rank.py) patches for the life of its process."""
    import sys

    import torch

    import lantern_b200
    import oracle.reflib
    if setitem is None:
        def setitem(d, k, v):
            d[k] = v
    me = sys.modules[__name__]
    setitem(sys.modules, "lantern_b200.api", me)
    setattr_(lantern_b200, "api", me)
    setitem(sys.modules, "oracle.reflib", REFLIB)
    setattr_(oracle, "reflib", REFLIB)
    setattr_(torch.cuda, "set_device", lambda d: None)
    setattr_(torch.cuda, "synchronize", lambda *a: None)
    setattr_(torch.cuda, "current_stream", lambda *a: HostStream())
    setattr_(torch.cuda, "empty_cache", lambda: None)
    setattr_(torch.cuda, "Event", HostEvent)
    setattr_(torch.Tensor, "pin_memory", lambda self: self)
    import torch.distributed as dist

    def gather_into(out, inp):  # gloo wants out.shape == (world * inp.shape[0], ...); NCCL (the real run) takes [world, ...]
        dist.all_gather(list(out.unbind(0)), inp)
    setattr_(dist, "all_gather_into_tensor", gather_into)
    setattr_(bench, "DEVICE_TYPE", "cpu")
    setattr_(bench, "DIST_BACKEND", "gloo")
    for name, wl in TINY.items():
        setitem(bench.WORKLOADS, name, dict(wl))


def view(ptr, shape, dtype):
    ptr = getattr(ptr, "value", ptr)
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    return np.frombuffer((C.c_char * n).from_address(int(ptr)), dtype=dtype).reshape(shape)


def lib():
    return None


def kernel_launches():
    return LAUNCHES[0]


class Index:
    def __init__(self, dim, metric="l2sq", quant="f32", M=16, efc=128, ef=64, **kw):
        assert not kw.get("pq"), "the stand-in covers the non-pq workloads"
        self.dim, self.kind, self.ef = dim, quant, ef
        self.p = portlib.PortIndex(dim, metric, quant, M=M, efc=efc, ef=ef)
        self.stats = dict(queries=0, computed_distances=0, base_pops=0, upper_hops=0, algorithmic_bytes=0, kernel_ms=0.0)
        self.row = dim // 8 if quant == "b1" else dim * 4
        self.M = M

    def reserve(self, n):
        self.p.reserve(n)

    def _rows(self, ptr, n, stride):
        assert stride == self.row
        return view(ptr, (n, self.dim // 8), np.uint8) if self.kind == "b1" else view(ptr, (n, self.dim), np.float32)

    def add_batch_device(self, keys, dptr, n, stride, kind="f32"):
        rows = self._rows(dptr, n, stride)
        for key, row in zip(keys, rows):
            self.p.add(int(key), row)

    def build(self):
        pass

    def last_build_stats(self):
        return dict(vectors=0, computed_distances=0, algorithmic_bytes=0, device_ms=0.0)

    def set_option(self, name, value):
        pass

    def _search(self, qptr, nq, stride, k, ef):
        t0 = time.perf_counter()
        keys, dists, counts, tot = self.p.search_batch(self._rows(qptr, nq, stride), k, ef)
        LAUNCHES[0] += 2  # cast + search, as the engine counts them
        alg = tot["computed_distances"] * self.row + tot["base_pops"] * (4 + 8 * self.M) + tot["upper_hops"] * (4 + 4 * self.M) + nq * self.row
        self.stats = dict(queries=nq, computed_distances=tot["computed_distances"], base_pops=tot["base_pops"],
                          upper_hops=tot["upper_hops"], algorithmic_bytes=alg, kernel_ms=1e3 * (time.perf_counter() - t0))
        return keys, dists, counts

    def search_batch_device(self, qptr, nq, stride, kind, k, ef, keys_ptr, dists_ptr, counts_ptr, stream=0):
        keys, dists, counts = self._search(qptr, nq, stride, k, ef)
        view(keys_ptr, (nq, k), np.uint64)[:] = keys
        view(dists_ptr, (nq, k), np.float32)[:] = dists
        if counts_ptr:
            view(counts_ptr, (nq,), np.int32)[:] = counts

    def search_batch_raw(self, qptr, nq, stride, kind, k, ef, keys_ptr, dists_ptr, counts_ptr):
        keys, dists, counts = self._search(qptr, nq, stride, k, ef)
        view(keys_ptr, (nq, k), np.uint64)[:] = keys
        view(dists_ptr, (nq, k), np.float32)[:] = dists
        view(counts_ptr, (nq,), np.int64)[:] = counts

    def last_stats(self):
        return dict(self.stats)

    def save_buffer(self):
        return self.p.save_buffer()

    def close(self):
        self.p = None


def exact_search_device(d_data, n, d_stride, d_queries, nq, q_stride, k, d_keys, d_dists, metric="l2sq", quant="f32", dims=None,
                        stream=0):
    width, dt = (dims // 8, np.uint8) if quant == "b1" else (dims, np.float32)
    assert d_stride == width * np.dtype(dt).itemsize and q_stride == d_stride
    keys, dists = portlib.exact_search(view(d_data, (n, width), dt), view(d_queries, (nq, width), dt), k, metric, quant, dims)
    view(d_keys, (nq, k), np.uint64)[:] = keys
    view(d_dists, (nq, k), np.float32)[:] = dists
    LAUNCHES[0] += 2


def merge_shards_device(d_keys, d_dists, shards, nq, k, d_out_keys, d_out_dists, stream=0):
    keys = view(d_keys, (shards, nq, k), np.uint64).transpose(1, 0, 2).reshape(nq, shards * k)
    dists = view(d_dists, (shards, nq, k), np.float32).transpose(1, 0, 2).reshape(nq, shards * k)
    order = np.argsort(dists, axis=1, kind="stable")[:, :k]
    view(d_out_keys, (nq, k), np.uint64)[:] = np.take_along_axis(keys, order, 1)
    view(d_out_dists, (nq, k), np.float32)[:] = np.take_along_axis(dists, order, 1)
    LAUNCHES[0] += 1


class RefIndex:
    """The reference's index as bench.py drives it: build over rows (--impl reference) or load the engine's index file
    (cpu_baseline), then search query batches."""

    def __init__(self, dim, metric="l2sq", quant="f32", M=16, efc=128, ef=64, threads=1):
        self.p = portlib.PortIndex(dim, metric, quant, M=M, efc=efc, ef=ef)

    def reserve(self, n):
        self.p.reserve(n)

    def add_batch(self, keys, vecs, threads=None):
        for key, row in zip(keys, vecs):
            self.p.add(int(key), row)

    def load_buffer(self, buf):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self.p.reserve(int(buf[80:88].view(np.uint64)[0]))  # node count of the file header
        self.p.load_buffer(buf)

    def search_batch(self, queries, k, threads=None):
        keys, dists, counts, tot = self.p.search_batch(queries, k)
        return keys, dists, counts, tot["computed_distances"], tot["visited_members"]


REFLIB = types.SimpleNamespace(available=lambda: True, lib=lambda: types.SimpleNamespace(refx_hardware_threads=lambda: 1),
                               RefIndex=RefIndex)
