"""bench.py's N=1 line assembled on a CPU box: the measuring legs are replaced by canned results (they need a GPU), everything
else — argument handling, secondary legs, failure isolation of the secondary legs, the one JSON line the driver parses — runs
for real."""
import json
import sys

import numpy as np
import pytest

import bench

ROOF = {"bound": "hbm", "achieved": 6000.0, "peak": 6566.7, "unit": "GB/s", "frac": 0.91, "traffic": None, "kernel": "K1", "kernel_ms": 4.6}
CLOCKS = {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": [], "samples": 9}


def fake_search(a, rank, local_rank, world, full=True):
    res = {"value": 2.0e6, "ms_per_step": 5.0, "recall_at_10": 0.97 if a.data == "sift" else 0.32, "ef_search": a.ef, "gpu_launches": 2 * a.steps,
           "clocks": CLOCKS, "retried_per_launch": 0, "roofline": dict(ROOF)}
    if full:
        res["e2e"] = {"value": 1.9e6, "unit": "queries/s", "h2d_bytes_per_step": a.batch * a.dim * 4, "d2h_bytes_per_step": a.batch * 84,
                      "callers": a.callers}
        res["cpu_baseline"] = {"value": 1.0e4, "unit": "queries/s", "cores": 16, "kind": "port", "sample": "canned"}
    return res


def fake_sharded(a, rank, local_rank, world, full=True):
    return {"value": 2.5e5, "unit": "queries/s", "n_gpus": world, "ms_per_step": 400.0, "recall_at_10": 0.989, "merged_eq_protocol": True,
            "gpu_launches": 380, "clocks": CLOCKS, "roofline": dict(ROOF), "build_s_per_rank": 20.0}


def fake_build(a, local_rank):
    assert (a.n, a.dim, a.M, a.efc) == (2_000_000, 300, 24, 200)  # BASELINE configs[2]
    return {"metric": "GPU Builder::build throughput", "value": 1.7e5, "unit": "points/s", "seconds": [11.7], "recall_at_10_of_built_graph": 0.89,
            "ef_search": 100, "config": {"workload": "canned"}, "search": {"value": 5.0e5}, "cpu_baseline": {"value": 8.9e3}}


@pytest.fixture
def cpu_bench(monkeypatch):
    import torch
    from instant_distance_b200 import _abi

    class FakeLib:
        def idb_device_count(self):
            return 1

    monkeypatch.setattr(_abi, "lib", lambda: FakeLib())
    monkeypatch.setattr(torch.cuda, "set_device", lambda *_: None)
    monkeypatch.setattr(bench, "leg_search", fake_search)
    monkeypatch.setattr(bench, "leg_sharded", fake_sharded)
    monkeypatch.setattr(bench, "leg_build", fake_build)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)

    def run(argv, capsys):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        bench.main()
        out = capsys.readouterr().out.strip().splitlines()
        assert len(out) == 1, "exactly ONE line on stdout"
        return json.loads(out[0])

    return run


def test_default_line_has_every_contract_key(cpu_bench, capsys):
    line = cpu_bench(["--steps", "7", "--warmup", "1"], capsys)
    assert line["metric"].startswith("batched QPS at recall@10") and line["unit"] == "queries/s" and line["n_gpus"] == 1
    assert line["steps"] == 7 and line["warmup"] == 3  # timing rule: at least 3 warm-up steps
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["dtype"] == "f32" and line["data"] == "synthetic"
    for key in ("value", "ms_per_step", "scaling", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "recall_at_10"):
        assert key in line, key
    assert {"h2d_bytes_per_step", "d2h_bytes_per_step", "value", "unit"} <= set(line["e2e"])
    assert "workload" in line["config"] and "model" not in line["config"]
    assert line["sharded"]["merged_eq_protocol"] is True and line["uniform"]["recall_at_10"] == 0.32
    assert line["build"]["unit"] == "points/s" and "search" in line["build"] and "cpu_baseline" in line["build"]


def test_a_failing_secondary_leg_does_not_take_the_headline_down(cpu_bench, capsys, monkeypatch):
    def boom(a, local_rank):
        raise RuntimeError("out of memory (canned)")

    monkeypatch.setattr(bench, "leg_build", boom)
    line = cpu_bench([], capsys)
    assert line["value"] == 2.0e6 and "error" in line["build"] and "canned" in line["build"]["error"]
    assert "error" not in line["sharded"] and "error" not in line["uniform"]


def test_skip_secondary_prints_the_headline_only(cpu_bench, capsys):
    line = cpu_bench(["--skip-secondary"], capsys)
    assert "sharded" not in line and "uniform" not in line and "build" not in line and line["roofline"]["bound"] == "hbm"


def test_dump_outputs_writes_the_last_steps_results(cpu_bench, capsys, monkeypatch, tmp_path):
    rng = np.random.default_rng(1)
    ids = rng.integers(0, 1 << 20, (1000, 10)).astype(np.uint32)
    ids[3, 7:] = 0xFFFFFFFF
    outs = {"ids": ids, "distances": rng.random((1000, 10), dtype=np.float32), "lengths": np.full(1000, 10, np.uint32)}
    monkeypatch.setattr(bench, "leg_search", lambda *a_, **k_: {**fake_search(*a_, **k_), "outputs": outs})
    cpu_bench(["--skip-secondary", "--dump-outputs", str(tmp_path / "all")], capsys)
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in outs}
    assert got["ids"].dtype == np.float64 and (got["ids"] == ids).all() and got["ids"][3, 9] == 0xFFFFFFFF
    assert got["distances"].dtype == np.float32 and got["distances"].tobytes() == outs["distances"].tobytes()
    assert got["lengths"].dtype == np.float64 and (got["lengths"] == 10).all()
    assert not (tmp_path / "all" / "rows.npy").exists()

    monkeypatch.setattr(bench, "DUMP_BYTES", 20_000)  # over the cap: the same seeded sample of rows on every run
    for d in ("s1", "s2"):
        cpu_bench(["--skip-secondary", "--dump-outputs", str(tmp_path / d)], capsys)
    rows = np.load(tmp_path / "s1" / "rows.npy")
    assert (rows == np.load(tmp_path / "s2" / "rows.npy")).all() and 0 < len(rows) < 1000
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) <= 20_000
    assert (np.load(tmp_path / "s1" / "ids.npy") == ids[rows.astype(np.int64)]).all()


def test_dump_outputs_is_refused_where_there_is_no_search_step(cpu_bench, capsys, tmp_path):
    with pytest.raises(SystemExit):
        cpu_bench(["--mode", "build", "--dump-outputs", str(tmp_path)], capsys)


@pytest.fixture
def oracle_graphs(monkeypatch, oracle):
    """bench.obtain_graph replaced by a single-threaded oracle build, remembered by data seed for the expected results."""
    graphs = {}

    def obtain(pts, n, dim, data, data_seed, M, efc, ef, seed, *_, **__):
        ix, ids = oracle.build(pts, M=M, ef_construction=efc, ef_search=ef, seed=seed, threads=1)
        g = ix.export()
        graphs[data_seed] = g, ids
        return g.points, g.zero, g.upper, ids

    monkeypatch.setattr(bench, "obtain_graph", obtain)
    return graphs


@pytest.mark.parametrize("world", [1, 2])
def test_reference_arm_dumps_its_last_timed_batch(cpu_bench, capsys, monkeypatch, tmp_path, oracle, oracle_graphs, world):
    """World 1: the configs[1] path, one graph.  World 2: the configs[4] path, every query on all sub-indexes, merged on the host."""
    from instant_distance_b200.sharded import merge_keys, pack_keys
    from tests import datagen

    monkeypatch.setenv("WORLD_SIZE", str(world))
    argv = ["--impl", "reference", "--n", "1500", "--dim", "12", "--batch", "90", "--shard-n", "400", "--ref-sample-sharded", "70",
            "--steps", "2", "--warmup", "3", "--dump-outputs", str(tmp_path)]
    line = cpu_bench(argv, capsys)
    got = [np.load(tmp_path / f"{k}.npy") for k in ("ids", "distances", "lengths")]
    search = lambda g, q: oracle.from_graph(oracle.Graph(g.points, g.zero, g.upper, 32, 100)).search(q, ef_search=100, k=10)
    if world == 1:
        want = search(oracle_graphs[1][0], datagen.sift_shaped(90, 12, 5000 + 4))  # (3 warm + 2 timed: batch 4 is the last)
    else:
        q, keys = datagen.sift_shaped(70, 12, 7000 + 4), []
        for s in range(bench.N_SUB):
            g, ids = oracle_graphs[1000 + s]
            i_, d_, l_ = search(g, q)
            gid = np.empty(400, dtype=np.uint32)  # PointId -> global row number of the sub-index's input range
            gid[ids] = np.arange(400 * s, 400 * (s + 1))
            keys.append(pack_keys(d_, gid[np.minimum(i_, 399)], l_))
        want = merge_keys(np.stack(keys), 10)
    assert line["steps"] == 2 and got[1].tobytes() == want[1].tobytes()
    assert (got[0] == want[0]).all() and (got[2] == want[2]).all()
