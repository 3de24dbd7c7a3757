"""Generates tests/golden/oracle_ref_v1.npz from the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref refpq`).

    python tests/golden/make_oracle_ref.py [OUT.npz]

Every input below is the one a test of tests/test_oracle_ref.py (or tests/test_abi_host.py) feeds the plain-C restatement;
everything stored is what the compiled reference answered for it: index-file digests (SHA-256 of the trimmed file),
keys, distances, work counters, k-means codebooks, and the entry points its usearch.h declares.  The property tests of
test_oracle_ref.py run on the fixed, seeded configurations drawn here.
"""
import ctypes as C
import hashlib
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from oracle import reflib  # noqa: E402
from util import scalar_kind_inputs, with_vectors  # noqa: E402

METRICS = ("l2sq", "cos")
VARIANTS = ("f16", "i8", "b1", "pq")
NO_KEY = np.iinfo(np.uint64).max


def trim(buf, stored_bytes=None):
    """The reference's save_buffer may leave slack after the last node; pq nodes carry `num_subvectors` code bytes instead
    of the header's vector_size_bytes."""
    n, M, M0 = struct.unpack_from("<QQQ", buf, 80)
    vsz, = struct.unpack_from("<Q", buf, 120)
    if stored_bytes is not None:
        vsz = stored_bytes
    off, b = 136, bytes(buf)
    for _ in range(n):
        lvl, = struct.unpack_from("<h", b, off + 8)
        off += 10 + 4 + 6 * M0 + lvl * (4 + 6 * M) + vsz
    return np.array(buf[:off])


def digest(buf):
    return np.frombuffer(hashlib.sha256(bytes(buf)).digest(), np.uint8)


def graph_only(buf):
    """An index file without its vector payloads: header, then key, level and adjacency lists node by node
    (tests/util.py::with_vectors puts the vectors back)."""
    b = bytes(buf)
    n, M, M0 = struct.unpack_from("<QQQ", b, 80)
    vsz, = struct.unpack_from("<Q", b, 120)
    out, off = [b[:136]], 136
    for _ in range(n):
        lvl, = struct.unpack_from("<h", b, off + 8)
        size = 10 + 4 + 6 * M0 + lvl * (4 + 6 * M)
        out.append(b[off:off + size])
        off += size + vsz
    return np.frombuffer(b"".join(out), np.uint8)


def searches(idx, Q, ks):
    """One query at a time (usearch_search_ef); row i holds the ks[i] results, padded with NO_KEY / +inf."""
    kmax = max(ks)
    keys = np.full((len(Q), kmax), NO_KEY, np.uint64)
    dists = np.full((len(Q), kmax), np.inf, np.float32)
    for i, (q, k) in enumerate(zip(Q, ks)):
        kk, dd = idx.search(q, k)
        keys[i, :len(kk)], dists[i, :len(kk)] = kk, dd
    return keys, dists


def build(d, metric, X, quant="f32", **kw):
    r = reflib.RefIndex(d, metric, quant, **kw)
    r.reserve(len(X))
    for i in range(len(X)):
        r.add(i + 1, X[i])
    return r


out = {}

# --- test_build_and_search_byte_exact_on_integer_data ---
for n, d, M, efc, ef, metric in ((1500, 32, 16, 128, 64, "l2sq"), (2000, 24, 6, 40, 20, "l2sq"), (1200, 48, 16, 96, 50, "cos")):
    rng = np.random.default_rng(n)
    X = rng.integers(-8, 9, (n, d)).astype(np.float32)
    Q = rng.integers(-8, 9, (150, d)).astype(np.float32)
    r = build(d, metric, X, M=M, efc=efc, ef=ef)
    name = "int_%s_n%d" % (metric, n)
    out[name + "_file_sha256"] = digest(trim(r.save_buffer()))
    out[name + "_keys"], out[name + "_dists"] = searches(r, Q, [10] * len(Q))

# --- test_counters_match_reference: computed_distances / visited_members per query ---
rng = np.random.default_rng(5)
X = rng.integers(-8, 9, (2000, 32)).astype(np.float32)
r = build(32, "l2sq", X, M=16, efc=128, ef=64)
comps, viss = [], []
for q in rng.integers(-8, 9, (50, 32)).astype(np.float32):
    keys, dists = np.zeros(10, np.uint64), np.zeros(10, np.float32)
    comp, vis = C.c_uint64(), C.c_uint64()
    reflib.lib().refx_search_stats(r.h, q.ctypes.data, 10, keys.ctypes.data, dists.ctypes.data, C.byref(comp), C.byref(vis))
    comps.append(comp.value)
    viss.append(vis.value)
out["counters_computed_distances"], out["counters_visited_members"] = np.array(comps, np.uint64), np.array(viss, np.uint64)

# --- test_float_data_ids_and_tolerance: the reference's graph over float data, and its answers on it ---
rng = np.random.default_rng(11)
X = rng.standard_normal((1500, 64)).astype(np.float32)
r = build(64, "cos", X, M=16, efc=128, ef=64)
f = trim(r.save_buffer())
g = graph_only(f)
assert np.array_equal(with_vectors(g, X), f), "the stored vectors are not the rows as added"
out["float_cos_graph"] = g
out["float_cos_keys"], out["float_cos_dists"] = searches(r, rng.standard_normal((200, 64)).astype(np.float32), [10] * 200)

# --- test_pq_128_centroid_quirk: ef = N search over a pq index with 256 centroids ---
rng = np.random.default_rng(2)
d, nsub, ncent = 16, 4, 256
cb = rng.standard_normal((ncent, d)).astype(np.float32)
X = rng.standard_normal((300, d)).astype(np.float32)
r = build(d, "l2sq", X, M=8, efc=32, ef=300, pq=True, num_centroids=ncent, num_subvectors=nsub, codebook=cb)
out["pq256_keys"], out["pq256_dists"] = r.search(rng.standard_normal(d).astype(np.float32), 300)

# --- test_property_port_equals_reference_on_random_small_configs ---
# rows: n, d, M, efc, ef, metric (index into METRICS), seed; the smallest and largest configuration, then 24 random draws
cfg_rng = np.random.default_rng(2145)
cfgs = np.array([[2, 1, 2, 4, 1, 0, 0], [2, 1, 2, 4, 1, 1, 1], [300, 20, 16, 64, 48, 0, 2], [300, 20, 16, 64, 48, 1, 3]] +
                [[cfg_rng.integers(2, 301), cfg_rng.integers(1, 21), cfg_rng.choice([2, 3, 4, 8, 16]), cfg_rng.integers(4, 65),
                  cfg_rng.integers(1, 49), cfg_rng.integers(0, 2), cfg_rng.integers(0, 10_001)] for _ in range(24)], np.int64)
files, keys, dists = [], [], []
for n, d, M, efc, ef, metric, seed in cfgs:
    rng = np.random.default_rng(seed)
    X = rng.integers(-5, 6, (n, d)).astype(np.float32)
    r = build(int(d), METRICS[metric], X, M=int(M), efc=int(efc), ef=int(ef))
    files.append(digest(trim(r.save_buffer())))
    Q = rng.integers(-5, 6, (10, d)).astype(np.float32)
    kq, dq = searches(r, Q, [int(rng.integers(1, 12)) for _ in Q])
    keys.append(np.pad(kq, ((0, 0), (0, 11 - kq.shape[1])), constant_values=NO_KEY))
    dists.append(np.pad(dq, ((0, 0), (0, 11 - dq.shape[1])), constant_values=np.inf))
out["prop_configs"], out["prop_file_sha256"], out["prop_keys"], out["prop_dists"] = cfgs, np.stack(files), np.stack(keys), np.stack(dists)

# --- test_property_scalar_kinds_bits_and_pq: every (variant, metric) pair, three random draws each ---
# rows: n, subvectors, M, efc, ef, variant (index into VARIANTS), metric (index into METRICS), seed
cfg_rng = np.random.default_rng(2146)
cfgs = np.array([[cfg_rng.integers(2, 201), cfg_rng.integers(1, 7), cfg_rng.choice([2, 4, 8]), cfg_rng.integers(4, 49),
                  cfg_rng.integers(1, 33), v, m, cfg_rng.integers(0, 10_001)]
                 for v in range(len(VARIANTS)) for m in range(len(METRICS)) for _ in range(3)], np.int64)
files, keys, dists = [], [], []
for n, sub, M, efc, ef, v, m, seed in cfgs:
    rng, X, Q, d, metric, quant, kw = scalar_kind_inputs(int(n), int(sub), VARIANTS[v], METRICS[m], int(seed))
    r = build(d, metric, X, quant, M=int(M), efc=int(efc), ef=int(ef), **kw)
    files.append(digest(trim(r.save_buffer(), int(sub) if VARIANTS[v] == "pq" else None)))
    kq, dq = searches(r, Q, [int(rng.integers(1, 10)) for _ in Q])
    keys.append(np.pad(kq, ((0, 0), (0, 9 - kq.shape[1])), constant_values=NO_KEY))
    dists.append(np.pad(dq, ((0, 0), (0, 9 - dq.shape[1])), constant_values=np.inf))
out["kinds_configs"], out["kinds_file_sha256"], out["kinds_keys"], out["kinds_dists"] = cfgs, np.stack(files), np.stack(keys), np.stack(dists)

# --- test_kmeans_restatement_equals_the_reference: the reference's product_quantization() codebooks ---
for metric, scale in (("l2sq", 3.0), ("l2sq", 8.0), ("cos", 3.0)):
    rng = np.random.default_rng(6)
    n, d, nsub, ncent = 3000, 24, 4, 16
    centers = rng.standard_normal((ncent, d)).astype(np.float32) * scale
    X = (centers[rng.integers(0, ncent, n)] + rng.standard_normal((n, d))).astype(np.float32)
    init = np.stack([rng.choice(n, ncent, replace=False) for _ in range(nsub)]).astype(np.uint32)
    name = "kmeans_%s_%g" % (metric, scale)
    for it in (1, 3, 25):
        out["%s_it%d" % (name, it)] = reflib.ref_kmeans(X, nsub, ncent, init, metric, it)
    Xc = np.repeat((np.arange(10) * 0.1).astype(np.float32)[:, None], 16, axis=1)
    perm = np.stack([rng.permutation(10) for _ in range(4)]).astype(np.uint32)
    out[name + "_fixture"] = reflib.ref_kmeans(Xc, 4, 10, perm, "l2sq", 20)

# --- the function names U/c/usearch.h declares (oracle/Makefile extracts them next to the compiled reference) ---
with open(os.path.join(ROOT, "oracle", "_ref", "usearch_h_entry_points.txt")) as fh:
    out["usearch_h_entry_points"] = np.array(sorted(fh.read().split()))

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_ref_v1.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes;", len(out), "arrays")
