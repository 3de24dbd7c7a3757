"""Host-side checks that need no GPU: the C-ABI library loads, exports every declared symbol (and the reference's own
names), fails loudly without a device, and the sharding helpers work across two gloo ranks."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "lantern_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"LB200_EXPORT[^;(]*?\b(lb200_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from lantern_b200 import api
    L = api.lib()  # raises if the library is missing: there is no fallback path
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(L, n), n
        assert n in api.SIGNATURES, "ctypes signature missing for " + n
    # the reference's own entry points (U/c/usearch.h) resolve to the same library
    for n in ("usearch_init", "usearch_free", "usearch_add", "usearch_search_ef", "usearch_search", "usearch_reserve",
              "usearch_size", "usearch_capacity", "usearch_dimensions", "usearch_connectivity", "usearch_save",
              "usearch_load", "usearch_view", "usearch_save_buffer", "usearch_load_buffer", "usearch_view_buffer",
              "usearch_serialized_length", "usearch_metadata_buffer", "usearch_index_metadata", "usearch_distance",
              "usearch_exact_search", "usearch_cast", "usearch_header_get_entry_slot", "usearch_header_set_entry_slot"):
        assert hasattr(L, n), n


def test_struct_layout_matches_usearch_header():
    """usearch_init_options_t (U/c/usearch.h:74-117): 15 fields; x86-64 SysV layout."""
    from lantern_b200 import api
    assert C.sizeof(api.InitOptions) == 120  # == sizeof(usearch_init_options_t), checked with gcc
    assert api.InitOptions.dimensions.offset == 24 and api.InitOptions.num_subvectors.offset == 112
    assert api.InitOptions.pq.offset == 96 and api.InitOptions.multi.offset == 56
    assert C.sizeof(api.IndexMetadata) == 184


def test_header_entry_slot_helpers():
    from lantern_b200 import api
    buf = (C.c_char * 136)()
    api.lib().lb200_header_set_entry_slot(buf, 0x0000_1234_5678_9ABC)
    assert api.lib().lb200_header_get_entry_slot(buf) == 0x1234_5678_9ABC
    raw = bytes(buf)
    assert raw[112:118] == (0x123456789ABC).to_bytes(6, "little")  # index_serialized_header_t::entry_slot at 80+32


def test_no_device_fails_loudly():
    from lantern_b200 import api
    if api.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(api.EngineError, match="CUDA device unavailable"):
        api.Index(8, "l2sq")
    with pytest.raises(api.EngineError, match="CUDA device unavailable"):
        api.distance(np.zeros(4, np.float32), np.zeros(4, np.float32), "l2sq")


def test_product_never_touches_the_oracle():
    """Nothing under lantern_b200/ (the product) may import, link or load anything from oracle/."""
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "lantern_b200")):
        if "build" in dirpath:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc", "Makefile")):
                if "oracle" in open(os.path.join(dirpath, f), errors="ignore").read():
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_row_ranges_and_merge():
    from lantern_b200 import shard
    n = 1003
    ranges = [shard.row_range(n, r, 8) for r in range(8)]
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
    assert max(h - l for l, h in ranges) - min(h - l for l, h in ranges) <= 1
    rng = np.random.default_rng(0)
    d = np.sort(rng.random((3, 5, 4)).astype(np.float32), axis=2)
    k = rng.permutation(60).reshape(3, 5, 4).astype(np.uint64)
    mk, md = shard.merge_topk_host(k, d)
    for q in range(5):
        allp = sorted(zip(d[:, q].ravel(), k[:, q].ravel()))[:4]
        assert [p[1] for p in allp] == list(mk[q]) and np.allclose([p[0] for p in allp], md[q])


WORKER = r'''
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch, torch.distributed as dist
from lantern_b200 import shard
from oracle import portlib
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
rank = dist.get_rank()
rng = np.random.default_rng(7)
X = rng.standard_normal((600, 16)).astype(np.float32)
Q = rng.standard_normal((20, 16)).astype(np.float32)
lo, hi = shard.row_range(len(X), rank, 2)
# per-shard top-k on this rank's rows (CPU oracle stands in for the per-GPU search), keys stay global
ek, ed = portlib.exact_search(X[lo:hi], Q, 5, "l2sq")
keys = torch.from_numpy((ek + lo + 1).astype(np.int64)); dists = torch.from_numpy(ed)
gk = [torch.empty_like(keys) for _ in range(2)]; gd = [torch.empty_like(dists) for _ in range(2)]
dist.all_gather(gk, keys); dist.all_gather(gd, dists)      # the one exchange step
mk, md = shard.merge_topk_host(torch.stack(gk).numpy().astype(np.uint64), torch.stack(gd).numpy())
fk, fd = portlib.exact_search(X, Q, 5, "l2sq")            # unsharded truth
assert np.array_equal(mk, fk + 1), (mk, fk)
assert np.allclose(md, fd)
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_sharded_search_two_ranks_gloo(tmp_path):
    """world_size=2, gloo, CPU: row-range shards -> per-shard top-k -> all_gather -> merge == unsharded result."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29541", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


GROUP_WORKER = '''
import os, sys
sys.path.insert(0, {root!r})
import torch.distributed as dist
from lantern_b200 import api
rank, world = int(os.environ["RANK"]), 2
dist.init_process_group("gloo", rank=rank, world_size=world)
def allgather(send):
    outs = [None] * world
    dist.all_gather_object(outs, send)
    return b"".join(outs)
# the bootstrap collective of a multi-process group, driven through the C ABI (no device needed for this part)
assert api.Group.selftest_exchange(rank, world, allgather) == 0
# ... and a broken collective is noticed
assert api.Group.selftest_exchange(rank, world, lambda send: send * world) == (0 if False else 2)
if api.device_count() == 0:  # the group itself has no CPU fallback
    try:
        api.Group.ranked(rank, world, allgather)
        raise SystemExit("a group was created without a CUDA device")
    except api.EngineError as e:
        assert "CUDA device unavailable" in str(e), e
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_group_bootstrap_two_ranks_gloo(tmp_path):
    """world_size=2, gloo, CPU: the all-gather callback a multi-process search group is bootstrapped with (lb200_group_create)
    round-trips rank-stamped blobs through the C ABI; without a device the group refuses to exist."""
    script = tmp_path / "group_worker.py"
    script.write_text(GROUP_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29547", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_group_plan_invariants():
    """Host logic of the multi-GPU search: how the resident warps of a GPU are split into owners and helpers.  Invariants: whole
    CTAs; owners + helpers fit; every query a rank owns gets an owner slot when the warps allow it; no more helpers than
    mailboxes and at most 32 mailboxes per helper; one GPU needs no helpers."""
    from lantern_b200 import api
    for world in (1, 2, 3, 4, 8):
        for nq in (1, 3, 61, 300, 1024, 4096, 5000, 20000):
            for W in (16 * world, 592, 2368, 3552, 4144):
                W -= W % (4 * world)
                omax = min(W, -(-(-(-max(nq, 1) // world)) // 4) * 4)
                ok, O, H = api.Group.plan(world, nq, W, omax)
                if not ok:
                    assert world > 1 and (world - 1) * O > 32 * (W - O)
                    continue
                assert O % 4 == 0 and H % 4 == 0 and 0 < O and O + H <= W
                owned = -(-nq // world)
                if world == 1:
                    assert H == 0 and O == min(-(-nq // 4) * 4, W)
                else:
                    M = (world - 1) * O
                    assert O == min(-(-owned // 4) * 4, omax, (W - W // 4) & ~3)
                    assert 0 < H <= max(-(-M // 4) * 4, 4) and M <= 32 * H
    # the metric's configuration: 4096 queries, 8 GPUs, 3552 resident warps -> every owned query has its owner, 3040 helpers
    assert api.Group.plan(8, 4096, 3552, 512) == (True, 512, 3040)
    assert api.Group.plan(2, 4096, 3552, 2048) == (True, 2048, 1504)


REF_HEADER_DIR = "/root/reference/lantern_hnsw/third_party/usearch/c"


def test_source_level_drop_in_with_the_reference_header(tmp_path):
    """A C caller written against the reference's own usearch.h compiles unchanged and links against liblantern_b200.so
    (what replacing U/c/lib.cpp in lantern.so amounts to, INTEGRATION.md 1).  Runs the cube when a GPU is present;
    without one the library must report that through the usearch error convention (exit code 3)."""
    if not os.path.exists(os.path.join(REF_HEADER_DIR, "usearch.h")):
        pytest.skip("reference header not available on this machine")
    exe = tmp_path / "dropin"
    lib_dir = os.path.join(ROOT, "lantern_b200")
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-I", REF_HEADER_DIR, os.path.join(ROOT, "tests", "c", "dropin_usearch_h.c"),
                           "-o", str(exe), "-L", lib_dir, "-llantern_b200", "-Wl,-rpath," + lib_dir])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    from lantern_b200 import api
    assert r.returncode == (0 if api.device_count() > 0 else 3), (r.returncode, r.stdout, r.stderr)


def test_metadata_of_reference_written_files():
    """usearch_metadata_buffer (U/c/lib.cpp:315-333) needs no device: metric / scalar kind / dimensions of the golden index
    files written by the reference."""
    from lantern_b200 import api
    G = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))
    L = api.lib()
    for name, metric, scalar, dims in (("cube_l2sq_file", 3, 1, 3), ("cube_cos_file", 1, 1, 3), ("lattice_f16_file", 3, 3, 3),
                                       ("lattice_i8_file", 3, 4, 3), ("rand_cos_file", 1, 1, 12)):
        buf = np.ascontiguousarray(G[name])
        o = api.InitOptions()
        err = C.c_char_p()
        L.lb200_metadata_buffer(buf.ctypes.data, len(buf), C.byref(o), C.byref(err))
        assert not err.value
        assert (o.metric_kind, o.quantization, o.dimensions) == (metric, scalar, dims), name
    err = C.c_char_p()
    L.lb200_metadata_buffer(np.zeros(100, np.uint8).ctypes.data, 100, C.byref(api.InitOptions()), C.byref(err))
    assert err.value and b"magic" in err.value


def test_metadata_from_path(tmp_path):
    """usearch_metadata (U/c/lib.cpp:268-284): the same answer from a file on disk; errors through the usual convention."""
    from lantern_b200 import api
    G = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))
    L = api.lib()
    path = tmp_path / "lattice_f16.usearch"
    path.write_bytes(bytes(np.ascontiguousarray(G["lattice_f16_file"])))
    for fn in (L.lb200_metadata, L.usearch_metadata):
        fn.restype, fn.argtypes = None, [C.c_char_p, C.POINTER(api.InitOptions), C.POINTER(C.c_char_p)]
        o, err = api.InitOptions(), C.c_char_p()
        fn(str(path).encode(), C.byref(o), C.byref(err))
        assert not err.value
        assert (o.metric_kind, o.quantization, o.dimensions, o.connectivity) == (3, 3, 3, 0)
        err = C.c_char_p()
        fn(str(tmp_path / "missing").encode(), C.byref(api.InitOptions()), C.byref(err))
        assert err.value and b"open" in err.value
    short = tmp_path / "short"
    short.write_bytes(b"usearch")
    err = C.c_char_p()
    L.lb200_metadata(str(short).encode(), C.byref(api.InitOptions()), C.byref(err))
    assert err.value and b"truncated" in err.value


def reference_header_symbols():
    """The function names U/c/usearch.h declares, as recorded in the golden fixture (tests/golden/make_oracle_ref.py)."""
    return list(np.load(os.path.join(ROOT, "tests", "golden", "oracle_ref_v1.npz"))["usearch_h_entry_points"])


def test_every_entry_point_of_the_reference_header_is_exported():
    """A binary built against U/c/usearch.h must link against this library unchanged."""
    from lantern_b200 import api
    L = api.lib()
    names = reference_header_symbols()
    assert len(names) >= 35
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_page_storage_entry_points_explain_themselves():
    """The reference's in-Postgres page storage / label bookkeeping entry points are exported but cannot work on a graph in
    HBM: they must say so through usearch_error_t (never crash, never pretend), with or without a device."""
    from lantern_b200 import api
    L = api.lib()
    P = C.POINTER(C.c_char_p)
    calls = {
        "usearch_view_mem_lazy": ([C.c_void_p, C.c_void_p, P], (None, None)),
        "usearch_set_node_retriever": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, P], (None, None, None, None)),
        "usearch_add_external": ([C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_int16, C.c_uint64, P],
                                 (None, 1, None, None, 1, 0, 0)),
        "usearch_newnode_level": ([C.c_void_p, P], (None,)),
        "usearch_get": ([C.c_void_p, C.c_uint64, C.c_size_t, C.c_void_p, C.c_int, P], (None, 1, 1, None, 1)),
        "usearch_remove": ([C.c_void_p, C.c_uint64, P], (None, 1)),
        "usearch_rename": ([C.c_void_p, C.c_uint64, C.c_uint64, P], (None, 1, 2)),
    }
    for name, (argtypes, args) in calls.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = None if name in ("usearch_view_mem_lazy", "usearch_set_node_retriever", "usearch_add_external") else C.c_size_t
        err = C.c_char_p()
        r = fn(*args, C.byref(err))
        assert err.value and name.encode() in err.value, name
        assert not r
    # and the ones that need an index report a null handle instead of dereferencing it
    for name, args in (("lb200_count", (None, 5)), ("lb200_update_header", (None, None))):
        fn = getattr(L, name)
        fn.restype, fn.argtypes = api.SIGNATURES[name]
        err = C.c_char_p()
        fn(*args, C.byref(err))
        assert err.value and b"null" in err.value


def test_ctypes_signatures_agree_with_the_header():
    """lantern_b200/api.py binds by hand: every prototype's parameter count (and 'returns a value or not') must match the
    declaration in include/lantern_b200.h, or calls would silently shift arguments."""
    from lantern_b200 import api
    text = open(os.path.join(ROOT, "include", "lantern_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = re.findall(r"LB200_EXPORT\s+([^;(]*?)\b(lb200_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert len(protos) >= 40
    for ret, name, params in protos:
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        restype, argtypes = api.SIGNATURES[name]
        assert len(argtypes) == n, (name, n, len(argtypes))
        returns_value = ret.strip() not in ("void",)
        assert (restype is not None) == returns_value, (name, ret)
