"""The plain-C restatement against the compiled reference itself.

tests/golden/oracle_ref_v1.npz holds what the UNMODIFIED reference (oracle/_ref) answered for exactly these inputs; it is
written by tests/golden/make_oracle_ref.py, and test_golden.py checks that it still reproduces from oracle/_ref wherever
that is built.  Index files are compared through their SHA-256 digests."""
import hashlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(__file__))
from util import scalar_kind_inputs, with_vectors  # noqa: E402

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "oracle_ref_v1.npz"))
METRICS = ("l2sq", "cos")
VARIANTS = ("f16", "i8", "b1", "pq")
NO_KEY = np.iinfo(np.uint64).max


def same_file(buf, want_sha256):
    return hashlib.sha256(bytes(buf)).digest() == bytes(want_sha256)


def searches(idx, Q, ks, width):
    """One query at a time; row i holds the ks[i] results, padded to `width` with NO_KEY / +inf (the fixture's layout)."""
    keys = np.full((len(Q), width), NO_KEY, np.uint64)
    dists = np.full((len(Q), width), np.inf, np.float32)
    for i, (q, k) in enumerate(zip(Q, ks)):
        kk, dd, _ = idx.search(q, k)
        keys[i, :len(kk)], dists[i, :len(kk)] = kk, dd
    return keys, dists


@pytest.mark.parametrize("n,d,M,efc,ef,metric", [(1500, 32, 16, 128, 64, "l2sq"), (2000, 24, 6, 40, 20, "l2sq"), (1200, 48, 16, 96, 50, "cos")])
def test_build_and_search_byte_exact_on_integer_data(port, n, d, M, efc, ef, metric):
    rng = np.random.default_rng(n)
    X = rng.integers(-8, 9, (n, d)).astype(np.float32)
    Q = rng.integers(-8, 9, (150, d)).astype(np.float32)
    p = port.PortIndex(d, metric, M=M, efc=efc, ef=ef)
    p.reserve(n)
    for i in range(n):
        p.add(i + 1, X[i])
    name = "int_%s_n%d" % (metric, n)
    assert same_file(p.save_buffer(), G[name + "_file_sha256"])
    pk, pd = searches(p, Q, [10] * len(Q), 10)
    assert np.array_equal(G[name + "_keys"], pk) and np.array_equal(G[name + "_dists"], pd)


def test_counters_match_reference(port):
    """computed_distances / visited_members (index.hpp:2726-2727) -- the quantity the roofline's algorithmic bytes use."""
    rng = np.random.default_rng(5)
    X = rng.integers(-8, 9, (2000, 32)).astype(np.float32)
    p = port.PortIndex(32, "l2sq", M=16, efc=128, ef=64)
    p.reserve(2000)
    for i in range(2000):
        p.add(i + 1, X[i])
    Q = rng.integers(-8, 9, (50, 32)).astype(np.float32)
    for q, comp, vis in zip(Q, G["counters_computed_distances"], G["counters_visited_members"]):
        pk, pd, st = p.search(q, 10)
        assert st.computed_distances == comp and st.visited_members == vis


def test_float_data_ids_and_tolerance(port):
    rng = np.random.default_rng(11)
    X = rng.standard_normal((1500, 64)).astype(np.float32)
    p = port.PortIndex(64, "cos", M=16, efc=128, ef=64)
    p.reserve(1500)
    p.load_buffer(with_vectors(G["float_cos_graph"], X))  # same graph, the reference's own bytes
    same = 0
    for q, rk, rd in zip(rng.standard_normal((200, 64)).astype(np.float32), G["float_cos_keys"], G["float_cos_dists"]):
        pk, pd, _ = p.search(q, 10)
        assert np.allclose(rd, pd, rtol=1e-5, atol=1e-6)
        same += np.array_equal(rk, pk)
    assert same >= 198


def test_pq_128_centroid_quirk(port):
    """codebook_t::compress never picks centroids >= 128 (signed char loop, lantern_storage.hpp:123)."""
    rng = np.random.default_rng(2)
    d, nsub, ncent = 16, 4, 256
    cb = rng.standard_normal((ncent, d)).astype(np.float32)
    X = rng.standard_normal((300, d)).astype(np.float32)
    codes = port.pq_compress(cb, X, nsub, compat128=True)
    assert codes.max() < 128
    dec = port.pq_decompress(cb, codes)
    q = rng.standard_normal(d).astype(np.float32)
    # the reference's pq index over X with ef = N answers (almost) every node for q; its distances are raw query vs decoded
    # candidate
    rk, rd = G["pq256_keys"], G["pq256_dists"]
    mine = ((dec[rk.astype(int) - 1] - q) ** 2).sum(1)
    assert np.allclose(mine, rd, rtol=1e-5, atol=1e-6)
    full = port.pq_compress(cb, X, nsub, compat128=False)
    assert (full >= 128).any()


def test_engine_tie_order_mode_equals_reference_without_ties(port):
    """The oracle's model of the CUDA engine's queue discipline is the reference's algorithm whenever distances are distinct
    (ids AND work counters identical); with exact ties only equal-distance order may differ (same distance profile)."""
    import sys, os
    sys.path.insert(0, os.path.dirname(__file__))
    from util import build_port_index, structured
    X, Q = structured(2500, 24, seed=3), structured(150, 24, seed=4)
    p = build_port_index(port, X, "cos", "f32", M=12, efc=64, ef=40)
    k1, d1, c1, t1 = p.search_batch(Q, 10)
    p.set_engine_order(True)
    k2, d2, c2, t2 = p.search_batch(Q, 10)
    assert np.array_equal(k1, k2) and np.array_equal(d1, d2) and t1 == t2
    rng = np.random.default_rng(9)
    Xi = rng.integers(-3, 4, (2000, 12)).astype(np.float32)  # integer data: ties everywhere
    Qi = rng.integers(-3, 4, (100, 12)).astype(np.float32)
    p = build_port_index(port, Xi, "l2sq", "f32", M=8, efc=48, ef=24)
    k1, d1, _, _ = p.search_batch(Qi, 10)
    p.set_engine_order(True)
    k2, d2, _, _ = p.search_batch(Qi, 10)
    assert np.mean(d1 == d2) > 0.97


def test_property_port_equals_reference_on_random_small_configs(port):
    """Property test over the 28 seeded configurations (N, d, M, ef_construction, ef, metric) of the fixture -- the smallest
    and largest of the ranges, then random draws: on integer-valued data the restatement writes the reference's index
    file and returns its ids and distances."""
    for cfg, want_file, want_k, want_d in zip(G["prop_configs"], G["prop_file_sha256"], G["prop_keys"], G["prop_dists"]):
        n, d, M, efc, ef, metric, seed = (int(v) for v in cfg)
        rng = np.random.default_rng(seed)
        X = rng.integers(-5, 6, (n, d)).astype(np.float32)
        p = port.PortIndex(d, METRICS[metric], M=M, efc=efc, ef=ef)
        p.reserve(n)
        for i in range(n):
            p.add(i + 1, X[i])
        assert same_file(p.save_buffer(), want_file), cfg
        Q = rng.integers(-5, 6, (10, d)).astype(np.float32)
        pk, pd = searches(p, Q, [int(rng.integers(1, 12)) for _ in Q], want_k.shape[1])
        assert np.array_equal(want_k, pk) and np.array_equal(want_d, pd), cfg


def test_property_scalar_kinds_bits_and_pq(port):
    """Same property for the storage variants (tests/util.py::scalar_kind_inputs), three seeded configurations for every
    (variant, metric) pair: f16 / i8 scalar quantisation (f32 in, cast on add), packed bits with the hamming metric, and
    pq storage with a random codebook (stored side decoded, value side raw)."""
    for cfg, want_file, want_k, want_d in zip(G["kinds_configs"], G["kinds_file_sha256"], G["kinds_keys"], G["kinds_dists"]):
        n, sub, M, efc, ef, variant, metric, seed = (int(v) for v in cfg)
        rng, X, Q, d, metric, quant, kw = scalar_kind_inputs(n, sub, VARIANTS[variant], METRICS[metric], seed)
        p = port.PortIndex(d, metric, quant, M=M, efc=efc, ef=ef, **kw)
        p.reserve(n)
        for i in range(n):
            p.add(i + 1, X[i])
        assert same_file(p.save_buffer(), want_file), cfg
        pk, pd = searches(p, Q, [int(rng.integers(1, 10)) for _ in Q], want_k.shape[1])
        assert np.array_equal(want_k, pk) and np.array_equal(want_d, pd), cfg


@pytest.mark.parametrize("metric,quant", [("l2sq", "f32"), ("cos", "f32"), ("hamming", "b1")])
def test_batched_build_model_with_batches_of_one_is_sequential_insertion(port, metric, quant):
    """ora_add_batch_engine models the CUDA engine's two-phase batched build on top of the reference procedures
    (hnsw_oracle.c).  With batch_cap = 1 it must BE the reference's sequential insertion: byte-identical index file."""
    rng = np.random.default_rng(23)
    n = 1500
    if quant == "b1":
        X, dim = rng.integers(0, 256, (n, 24), dtype=np.uint8), 192
    else:
        X, dim = rng.integers(-8, 9, (n, 24)).astype(np.float32), 24
    keys = np.arange(1, n + 1, dtype=np.uint64)
    a = port.PortIndex(dim, metric, quant, M=8, efc=48, ef=32)
    a.reserve(n)
    for k, v in zip(keys, X):
        a.add(int(k), v)
    b = port.PortIndex(dim, metric, quant, M=8, efc=48, ef=32)
    b.reserve(n)
    b.add_batch_engine(keys[:700], X[:700], 1)   # two calls: the level generator carries over like in ora_add
    b.add_batch_engine(keys[700:], X[700:], 1)
    assert np.array_equal(a.save_buffer(), b.save_buffer())


def test_batched_build_model_is_deterministic_and_as_good_as_sequential(port):
    rng = np.random.default_rng(29)
    n, d = 4000, 24
    X = rng.integers(-8, 9, (n, d)).astype(np.float32)
    Q = rng.integers(-8, 9, (300, d)).astype(np.float32)
    keys = np.arange(1, n + 1, dtype=np.uint64)
    truth, _ = port.exact_search(X, Q, 10)

    def rec(idx):
        k, _, _, _ = idx.search_batch(Q, 10)
        return float(np.mean([len(set(a.tolist()) & set((t + 1).tolist())) / 10.0 for a, t in zip(k, truth)]))

    seq = port.PortIndex(d, "l2sq", "f32", M=8, efc=48, ef=32)
    seq.reserve(n)
    for k, v in zip(keys, X):
        seq.add(int(k), v)
    files = []
    for _ in range(2):
        b = port.PortIndex(d, "l2sq", "f32", M=8, efc=48, ef=32)
        b.reserve(n)
        b.add_batch_engine(keys, X, 64, 64)
        files.append(b.save_buffer())
    assert np.array_equal(files[0], files[1])
    assert len(files[0]) == len(seq.save_buffer())  # same level draws -> same file size
    assert abs(rec(b) - rec(seq)) < 0.02
    # every link of the batched graph points to a node that exists on that level (what lb200_load_buffer verifies)
    for slot in range(0, n, 97):
        for level in range(b.level(slot) + 1):
            for nb in b.neighbors(slot, level):
                assert b.level(int(nb)) >= level


@pytest.mark.parametrize("metric,scale", [("l2sq", 3.0), ("l2sq", 8.0), ("cos", 3.0)])
def test_kmeans_restatement_equals_the_reference(port, metric, scale):
    """PQ codebook training: the UNMODIFIED reference k-means (lantern_hnsw/src/hnsw/product_quantization.c compiled against
    the stand-in postgres.h of oracle/pg_shim/, PRNG scripted so that both sides start from the same rows) against the
    plain-C restatement ora_kmeans -- bit for bit, for 1, 3 and up to 25 Lloyd rounds, which pins row (f4) of SURVEY 8."""
    rng = np.random.default_rng(6)
    n, d, nsub, ncent = 3000, 24, 4, 16
    centers = rng.standard_normal((ncent, d)).astype(np.float32) * scale
    X = (centers[rng.integers(0, ncent, n)] + rng.standard_normal((n, d))).astype(np.float32)
    init = np.stack([rng.choice(n, ncent, replace=False) for _ in range(nsub)]).astype(np.uint32)
    seen_rounds = set()
    name = "kmeans_%s_%g" % (metric, scale)
    for it in (1, 3, 25):
        rcb = G["%s_it%d" % (name, it)]
        pcb, rounds = port.kmeans(X, nsub, ncent, init, metric, it)
        assert np.array_equal(rcb.view(np.uint32), pcb.view(np.uint32)), np.abs(rcb - pcb).max()
        seen_rounds.add(rounds)
    if metric == "l2sq":
        assert max(seen_rounds) > 3  # the stop rule (mean centre shift <= 0.1) was exercised beyond the early rounds
    # the hnsw_pq_index.sql fixture geometry: k == n, every init is a permutation, one round moves nothing
    Xc = np.repeat((np.arange(10) * 0.1).astype(np.float32)[:, None], 16, axis=1)
    perm = np.stack([rng.permutation(10) for _ in range(4)]).astype(np.uint32)
    assert np.array_equal(G[name + "_fixture"], port.kmeans(Xc, 4, 10, perm, "l2sq", 20)[0])
