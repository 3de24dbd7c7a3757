"""bench.py's own arm walked end to end on the CPU: the engine is replaced by tests/fake_engine.py (the oracle behind the
same entry points) and torch.cuda's stream/event calls by host stand-ins, so that every line of the N=1 glue -- data
generation, build calls, timed loops, roofline block, e2e loop, cpu_baseline over the reference (the oracle stands in for
it as well), parity block, the JSON line -- executes here before it is trusted on a GPU box.  No number printed by this test
means anything."""
import json
import os
import sys
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTRACT_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline")


@pytest.fixture
def host_bench(monkeypatch):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bench
    import fake_engine
    fake_engine.install(bench, monkeypatch.setattr, monkeypatch.setitem)
    return bench


def run(bench, monkeypatch, capsys, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + list(argv))
    bench.main()
    out = capsys.readouterr()
    return json.loads(out.out.strip().splitlines()[-1]), out.err


@pytest.mark.parametrize("big", [False, True])
def test_single_gpu_glue_runs_and_prints_the_contract_line(host_bench, monkeypatch, capsys, big):
    bench = host_bench
    if big:  # the branch the 10M-row default takes: prefix graph for the reference, recorded recall for shards
        monkeypatch.setattr(bench, "BIG_CORPUS_BYTES", 1e4)
    line, err = run(bench, monkeypatch, capsys, "--workload", "tiny", "--steps", "4", "--warmup", "1", "--cpu-seconds", "0.5",
                    "--cpu-prefix-rows", "1000")
    for key in CONTRACT_KEYS:
        assert key in line, key
    assert line["cpu_baseline_note"] is None, (line["cpu_baseline_note"], err)
    assert line["n_gpus"] == 1 and line["steps"] == 4 and line["warmup"] == 3  # warm-up clamped to the timing rules' minimum
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["gpu_launches"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 8 * 32 * 4 and line["e2e"]["d2h_bytes_per_step"] == 8 * 10 * 12 + 8 * 4
    assert 0.5 < line["recall_at_10"] <= 1.0
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["achieved"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    c = line["cpu_baseline"]
    assert c["kind"] == "reference" and c["cores"] >= 1 and c["value"] > 0
    assert ("first 1000 of the 3000" in c["sample"]) == big
    p = line["parity"]  # the stand-in IS the oracle, and the reference loads its file: identical by construction
    assert p["graph_rows"] == (1000 if big else 3000)
    assert p["identical_id_rows"] == 1.0 and p["reference_computed_distances"] == p["engine_computed_distances"]
    assert p["reference_recall_at_10"] == p["engine_recall_at_10"]


def test_binary_workload_glue(host_bench, monkeypatch, capsys):
    line, err = run(host_bench, monkeypatch, capsys, "--workload", "tinybits", "--steps", "3", "--warmup", "3", "--cpu-seconds", "0.3")
    assert line["cpu_baseline_note"] is None, (line["cpu_baseline_note"], err)
    assert line["dtype"].startswith("u8") and line["e2e"]["h2d_bytes_per_step"] == 8 * 16
    assert line["parity"]["reference_computed_distances"] > 0 and line["cpu_baseline"]["value"] > 0


def test_default_workload_is_the_one_the_metric_names(host_bench):
    bench = host_bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "10M vectors, batch 4096" in base["metric"]
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'os.environ.get("LB200_WORKLOAD", "cfg3")' in src
    w = bench.WORKLOADS["cfg3"]
    assert (w["n"], w["dim"], w["batch"], w["k"], w["metric"], w["M"], w["ef"]) == (10_000_000, 768, 4096, 10, "cos", 32, 128)
    assert w["n"] * w["dim"] * 4 < 180e9  # fits one B200


@pytest.mark.parametrize("big", [False, True])
def test_two_rank_glue_over_gloo(big):
    """The sharded path (row-range shards, all-gather of per-shard top-k, merge, recall-matched per-shard ef, max-over-ranks
    timing) on two CPU ranks over gloo; `big` = the branch the 10M-row default takes (recorded 1-GPU recall as the target)."""
    env = dict(os.environ, DRYRUN_BIG="1" if big else "", MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(29731 + int(big)), os.path.join(ROOT, "tests", "dryrun_rank.py"), "--gpus", "2", "--workload", "tiny",
           "--steps", "3", "--warmup", "3", "--shard-mode", "graphs"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout  # rank 0 alone prints
    line = json.loads(lines[0])
    for key in CONTRACT_KEYS:
        assert key in line, key
    assert line["n_gpus"] == 2 and line["scaling"] == "strong" and line["config"]["rows_per_gpu"] == 1500
    sh = line["sharding"]
    assert 10 <= sh["ef_per_shard"] <= 16 and sh["sweep_merged_recall_by_ef"]
    assert ("recorded" in sh["recall_target_source"]) == big
    assert ("replicated_comparison" in sh) == (not big)
    assert line["e2e"]["h2d_bytes_per_step"] == 2 * 8 * 32 * 4 and line["value"] > 0 and 0.5 < line["recall_at_10"] <= 1.0


def test_dump_outputs_are_the_last_timed_step(host_bench, monkeypatch, capsys, tmp_path):
    """--dump-outputs: the arrays the timed path returned in its last step, as float npy files, identical across runs with the
    same arguments."""
    import numpy as np
    dumps = []
    for run_dir in ("a", "b"):
        line, err = run(host_bench, monkeypatch, capsys, "--workload", "tiny", "--steps", "5", "--warmup", "3", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path / run_dir))
        assert line["steps"] == 5
        dumps.append({n: np.load(tmp_path / run_dir / (n + ".npy")) for n in ("keys", "distances", "counts")})
    a, b = dumps
    assert a["keys"].shape == a["distances"].shape == (8, 10) and a["counts"].shape == (8,)
    assert a["keys"].dtype == np.float64 and a["distances"].dtype == np.float32 and a["counts"].dtype == np.float64
    assert all(np.array_equal(a[n], b[n]) for n in a)
    # step s searches query batch s % pool: the last timed step (s = 7, pool 8) is the last batch of the query pool
    bench = host_bench
    X = bench.structured_torch(3000, 32, bench.SEED_CORPUS, "cpu").numpy()
    Q = bench.structured_torch(8 * 8, 32, bench.SEED_QUERY, "cpu").numpy()[7 * 8:]
    d = ((Q[:, None, :] - X[a["keys"].astype(np.int64) - 1]) ** 2).sum(-1)
    assert np.allclose(d, a["distances"], rtol=1e-4, atol=1e-4)
