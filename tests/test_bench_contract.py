"""bench.py contract checks that need no GPU: the reference arm runs on the host cores and prints one JSON line with the
keys a reader of the benchmark relies on; the workload table is self-consistent."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line(monkeypatch, capsys):
    """The arm's glue, with the oracle standing in for the compiled reference (tests/fake_engine.py)."""
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    import bench
    import fake_engine
    fake_engine.install(bench, monkeypatch.setattr, monkeypatch.setitem)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--workload", "cfg2s", "--steps", "2", "--warmup", "3",
                                      "--ref-rows", "3000", "--ref-seconds", "1"])
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "queries/s" and line["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["value"] > 0 and line["config"]["workload"].startswith("cfg2s")


def test_workload_table():
    sys.path.insert(0, ROOT)
    import bench
    assert set(bench.WORKLOADS) >= {"cfg2", "cfg3", "cfg4", "cfg5"}
    cfg2 = bench.WORKLOADS["cfg2"]
    assert (cfg2["n"], cfg2["dim"], cfg2["M"], cfg2["efc"], cfg2["ef"], cfg2["batch"], cfg2["k"]) == (1_000_000, 768, 16, 128, 64, 1024, 10)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.METRIC_NAME == base["metric"]
    X = bench.structured_np(1000, 16, 42)
    assert X.shape == (1000, 16) and abs(float(X.mean())) < 0.2
    b = bench.bits_np(100, 64, 1)
    assert b.shape == (100, 8) and b.dtype.name == "uint8"


def test_parity_block_is_tie_aware_and_usable_cores_is_sane():
    """The same-graph parity block of the bench line: position-wise identity, and the tie-aware row test that lets ids swap
    inside groups of equal distances (hamming) but nowhere else."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    d = np.array([[1.0, 2.0, 2.0, 3.0], [0.5, 0.6, 0.7, 0.8]], np.float32)
    k = np.array([[10, 11, 12, 13], [20, 21, 22, 23]], np.uint64)
    same = bench.parity_block(k, d, k.copy(), d.copy())
    assert same["identical_id_rows"] == 1.0 and same["rows_identical_up_to_distance_ties"] == 1.0 and same["max_rel_dist_err"] == 0.0
    swapped = k.copy()
    swapped[0, 1], swapped[0, 2] = 12, 11  # inside the tie group of row 0
    p = bench.parity_block(k, d, swapped, d.copy())
    assert p["identical_id_rows"] == 0.5 and p["rows_identical_up_to_distance_ties"] == 1.0
    wrong = k.copy()
    wrong[1, 0], wrong[1, 1] = 21, 20  # distinct distances: a real difference
    p = bench.parity_block(k, d, wrong, d.copy())
    assert p["rows_identical_up_to_distance_ties"] == 0.5
    assert 1 <= bench.usable_cores() <= (os.cpu_count() or 1)
