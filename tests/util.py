"""Shared helpers for the parity tests."""
import numpy as np


def structured(n, d, seed, latent=32, noise=0.05):
    """Low-intrinsic-dimension synthetic vectors (SURVEY.md 8d): x = z P + noise * eps."""
    rng = np.random.default_rng(seed)
    P = (np.random.default_rng(1234).standard_normal((latent, d)) / np.sqrt(latent)).astype(np.float32)
    z = rng.standard_normal((n, latent)).astype(np.float32)
    return (z @ P + noise * rng.standard_normal((n, d)).astype(np.float32)).astype(np.float32)


def build_port_index(portlib, X, metric="l2sq", quant="f32", M=16, efc=128, ef=64, keys=None, **kw):
    n = len(X)
    dim = X.shape[1] * 8 if X.dtype == np.uint8 else X.shape[1]
    idx = portlib.PortIndex(dim, metric, quant, M=M, efc=efc, ef=ef, **kw)
    idx.reserve(n)
    keys = np.arange(1, n + 1, dtype=np.uint64) if keys is None else keys
    for i in range(n):
        idx.add(keys[i], X[i])
    return idx


def compare_results(keys_a, dists_a, keys_b, dists_b, rtol=1e-5, atol=1e-6):
    """Position-wise id equality, tolerating permutations inside groups of (near-)equal distances.
    Returns (n_exact_rows, n_rows_ok)."""
    nq = len(keys_a)
    exact = ok = 0
    for q in range(nq):
        ka, kb, da, db = keys_a[q], keys_b[q], dists_a[q], dists_b[q]
        if np.array_equal(ka, kb):
            exact += 1
            ok += 1
            continue
        # distances must agree position-wise within tolerance and differing ids must sit in near-tie groups
        if not np.allclose(da, db, rtol=rtol * 10, atol=atol * 10):
            continue
        good = True
        for i in np.nonzero(ka != kb)[0]:
            # id kb[i] must appear in ka at a position whose distance is within tolerance of da[i]
            pos = np.nonzero(ka == kb[i])[0]
            if len(pos) == 0:
                # allowed only at the tail boundary: distance equal to the last one
                if not np.isclose(db[i], da[-1], rtol=rtol * 10, atol=atol * 10):
                    good = False
            elif not np.isclose(da[pos[0]], db[i], rtol=rtol * 10, atol=atol * 10):
                good = False
        ok += good
    return exact, ok


def recall(found, truth):
    hits = 0
    for f, t in zip(found, truth):
        hits += len(set(f.tolist()) & set(t.tolist()))
    return hits / truth.size


def adjacency_lists(buf, M, stored_bytes):
    """Parse a usearch/lantern index file (SURVEY App. B) into {(node, level): tuple(neighbour ids)} plus the level array.
    Vectors and keys are skipped: comparisons through this helper look at the graph only."""
    b = np.asarray(buf, dtype=np.uint8).tobytes()
    n = int(np.frombuffer(b, np.uint64, 1, 80)[0])
    M0 = 2 * M
    lists, levels = {}, np.zeros(n, np.int16)
    p = 136
    for i in range(n):
        lvl = int(np.frombuffer(b, np.int16, 1, p + 8)[0])
        levels[i] = lvl
        p += 10
        for l in range(lvl + 1):
            width = M0 if l == 0 else M
            cnt = int(np.frombuffer(b, np.uint32, 1, p)[0])
            raw = np.frombuffer(b, np.uint8, 6 * width, p + 4).reshape(width, 6)[:cnt]
            ids = raw[:, :4].copy().view(np.uint32)[:, 0]
            lists[(i, l)] = tuple(int(x) for x in ids)
            p += 4 + 6 * width
        p += stored_bytes
    assert p == len(b), (p, len(b))
    return lists, levels


def graph_agreement(buf_a, buf_b, M, stored_bytes):
    """Fraction of (node, level) adjacency lists that are identical (same ids, same order) in two index files."""
    la, lva = adjacency_lists(buf_a, M, stored_bytes)
    lb, lvb = adjacency_lists(buf_b, M, stored_bytes)
    assert np.array_equal(lva, lvb), "level draws differ"
    assert la.keys() == lb.keys()
    same = sum(1 for k in la if la[k] == lb[k])
    return same / max(1, len(la))


def with_vectors(graph, X):
    """An index file from its vector-free form (tests/golden/make_oracle_ref.py::graph_only) and the rows in slot order."""
    g = np.asarray(graph, dtype=np.uint8).tobytes()
    n, M, M0 = (int(v) for v in np.frombuffer(g, np.uint64, 3, 80))
    vsz = int(np.frombuffer(g, np.uint64, 1, 120)[0])
    X = np.ascontiguousarray(X)
    assert len(X) == n and X[0].nbytes == vsz, (len(X), n, X[0].nbytes, vsz)
    out, off = [g[:136]], 136
    for i in range(n):
        lvl = int(np.frombuffer(g, np.int16, 1, off + 8)[0])
        size = 10 + 4 + 6 * M0 + lvl * (4 + 6 * M)
        out += [g[off:off + size], X[i].tobytes()]
        off += size
    assert off == len(g), (off, len(g))
    return np.frombuffer(b"".join(out), np.uint8)


def scalar_kind_inputs(n, sub, variant, metric, seed):
    """Inputs of one configuration of tests/test_oracle_ref.py::test_property_scalar_kinds_bits_and_pq: f16 / i8 scalar
    quantisation (f32 in, cast on add), packed bits with the hamming metric, or pq storage with a random codebook.  Small
    multiples of 1/4: exact in f16, and |x| * 100 stays an integer below the i8 clamp for the small ones.  Returns the rng
    (the test draws each query's k from it next), rows, queries, dimensions, metric, scalar kind and the pq arguments."""
    rng = np.random.default_rng(seed)
    kw, quant, d = {}, "f32", 4 * sub
    if variant == "b1":
        metric, quant, d = "hamming", "b1", 32 * sub
        X = rng.integers(0, 256, (n, d // 8), dtype=np.uint8)
        Q = rng.integers(0, 256, (8, d // 8), dtype=np.uint8)
    else:
        X = (rng.integers(-4, 5, (n, d)) / 4.0).astype(np.float32)
        Q = (rng.integers(-4, 5, (8, d)) / 4.0).astype(np.float32)
        if variant == "pq":
            ncent = int(rng.integers(2, 9))
            kw = dict(pq=True, num_centroids=ncent, num_subvectors=sub,
                      codebook=(rng.integers(-4, 5, (ncent, d)) / 4.0).astype(np.float32))
        else:
            quant = variant
    return rng, X, Q, d, metric, quant, kw
