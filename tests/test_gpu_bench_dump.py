"""bench.py --dump-outputs on the GPU: the dump is the result of the last TIMED step — the lane the device-resident arm issued it on,
and the sharded leg's merged result before its isolated K1 launch reuses the buffers — checked against a fresh search of that batch."""
import argparse
import json
import sys

import numpy as np
import pytest

import bench
from tests import datagen

pytestmark = pytest.mark.gpu

SEED = 20260923  # bench.py's default --seed


def _bench(monkeypatch, capsys, argv):
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    bench.main()
    return json.loads(capsys.readouterr().out.strip().splitlines()[-1])


def _assert_dump_is(d, want):
    ids, dist, lens = (np.load(d / f"{k}.npy") for k in ("ids", "distances", "lengths"))
    assert dist.tobytes() == np.asarray(want[1], dtype=np.float32).tobytes()
    assert (ids == want[0]).all() and (lens == want[2]).all()


@pytest.mark.parametrize("lanes", [2, 3])
def test_headline_dump_is_the_last_timed_step(monkeypatch, capsys, tmp_path, lanes):
    from instant_distance_b200 import _abi

    line = _bench(monkeypatch, capsys, ["--mode", "headline", "--n", "20000", "--dim", "32", "--batch", "3000", "--steps", "3", "--warmup", "3",
                                        "--lanes", str(lanes), "--callers", "1", "--no-cache", "--skip-cpu-baseline", "--recall-sample", "200",
                                        "--dump-outputs", str(tmp_path)])
    p, zero, upper, _ = bench.obtain_graph(datagen.sift_shaped(20000, 32, 1), 20000, 32, "sift", 1, 32, 100, 100, SEED, 0, use_abi=True,
                                           no_cache=True)
    ix = _abi.Index.from_graph(p, zero, upper, 32, 100)
    want = ix.search(datagen.sift_shaped(3000, 32, 5000 + 5), ef_search=line["ef_search"], k=10)  # 3 warm + 3 timed: batch 5 is the last
    ix.close()
    _assert_dump_is(tmp_path, want)


def test_sharded_dump_is_the_last_timed_step(monkeypatch, capsys, tmp_path):
    from instant_distance_b200 import _abi, sharded

    _bench(monkeypatch, capsys, ["--mode", "sharded", "--dim", "32", "--shard-n", "3000", "--shard-batch", "1500", "--steps", "3", "--warmup", "3",
                                 "--skip-cpu-baseline", "--recall-sample", "100", "--dump-outputs", str(tmp_path)])
    shards = []
    for s in range(bench.N_SUB):
        ix, ids = _abi.Index.build(bench.shard_points(argparse.Namespace(shard_n=3000, dim=32), s), M=32, ef_construction=100, ef_search=100,
                                   seed=SEED + s)
        ix.set_id_map(sharded.global_id_map(ids, s * 3000))
        shards.append(ix)
    comm = _abi.Comm(_abi.comm_unique_id(), 0, 1, 0)
    want = _abi.sharded_search_multi(shards, comm, datagen.sift_shaped(1500, 32, 7000 + 5), ef_search=100, k=10)  # step 5 is the last
    comm.close()
    [s_.close() for s_ in shards]
    _assert_dump_is(tmp_path, want)
