"""Sharded search on >= 2 GPUs (SURVEY §8e): runs scripts/sharded_check.py under torchrun, one rank per GPU.
Checks (inside the script): every shard's GPU search == the oracle on that shard's graph; the fused path (K1 epilogue
pack -> ONE ncclAllGather -> merge kernel) == the host statement of the protocol; identical results on all ranks."""
import json
import os
import subprocess
import sys

import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu


def _gpu_count():
    from instant_distance_b200 import _abi

    return _abi.lib().idb_device_count()


@pytest.mark.parametrize("k,ef", [(10, 100), (100, 100)])
def test_sharded_search_world_of_one_three_shards(oracle, k, ef):
    """The whole fused path on ONE GPU: three PointId-range shards on the device, a world-size-1 NCCL communicator.
    per-shard K1 (keys epilogue) -> pre-merge kernel -> ncclAllGather -> merge kernel; checked against (a) the oracle on every
    shard's graph and (b) the host statement of the protocol.  k = ef = 100 exercises the widest merge (3 x 100 keys per query)."""
    import numpy as np

    from instant_distance_b200 import _abi, sharded
    from tests import datagen

    n_sh, per, dim = 3, 9000, 48
    q = datagen.sift_shaped(1200, dim, 77)
    shards, keys = [], []
    for s in range(n_sh):
        rows = datagen.sift_shaped(per, dim, 200 + s)
        ix, ids = _abi.Index.build(rows, seed=40 + s)
        gmap = sharded.global_id_map(ids, s * per)
        p, zero, upper = ix.export_graph()
        ox = oracle.from_graph(oracle.Graph(p, zero, upper, 32, ef))
        o_ids, o_dist, o_len = ox.search(q, ef_search=ef, k=k, threads=8)
        l_ids, l_dist, l_len = ix.search(q, ef_search=ef, k=k)  # (a) local search == oracle on this shard's graph
        assert (o_ids == l_ids).all() and o_dist.tobytes() == l_dist.tobytes() and (o_len == l_len).all()
        gids = np.where(o_ids == 0xFFFFFFFF, 0, gmap[np.minimum(o_ids, per - 1)])
        keys.append(sharded.pack_keys(o_dist, gids, np.minimum(o_len, k)))
        ix.set_id_map(gmap)
        shards.append(ix)
    comm = _abi.Comm(_abi.comm_unique_id(), 0, 1, 0)
    ids, dist, lens = _abi.sharded_search_multi(shards, comm, q, ef_search=ef, k=k)
    w_ids, w_dist, w_len = sharded.merge_keys(np.stack(keys), k)  # (b) host statement of the protocol
    assert (ids == w_ids).all() and dist.tobytes() == w_dist.tobytes() and (lens == w_len).all()
    one = shards[0].sharded_search(comm, q, ef_search=ef, k=k)  # a single shard: K1 -> all-gather -> merge
    o_ids, o_dist, o_len = sharded.merge_keys(keys[0][None], k)
    assert (one[0] == o_ids).all() and one[1].tobytes() == o_dist.tobytes() and (one[2] == o_len).all()
    comm.close()
    [s_.close() for s_ in shards]


@pytest.mark.skipif("_gpu_count() < 2", reason="needs >= 2 GPUs")
def test_sharded_search_two_ranks():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "scripts", "sharded_check.py"), "--points", "60000", "--queries", "3000"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res["local_eq_oracle"] and res["fused_eq_protocol"] and res["world"] == 2
