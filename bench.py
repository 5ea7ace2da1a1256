#!/usr/bin/env python
"""bench.py — batched HNSW search QPS at recall@10 >= 0.95 on B200 (BASELINE.json metric), with roofline and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, through the C ABI)
  python bench.py --impl reference [...]                         reference arm: the CPU path on the box's host cores
  python bench.py --mode build|sharded|headline [...]            one leg only (default --mode auto, below)
  python bench.py --dump-outputs DIR [...]                       also write the last timed search step's results as DIR/*.npy

A "step" = one pass of the hot path (Hnsw::search, lib.rs:352-383) over one batch of synthetic queries.

--gpus 1 (auto): BASELINE.json configs[1] — 1M x 128 f32 "SIFT-shaped" synthetic points, M=32, ef_construction=100, ef_search=100
  (raised only if recall@10 < 0.95), batch = 10k queries.  `value` = queries/s with queries + outputs resident in HBM (batches
  issued alternately on two submission lanes, so consecutive launches overlap at the batch boundary); `e2e` = the same through
  idb_search_batch_f32 with pinned HOST buffers (H2D + D2H inside the timed region, three caller threads).  The line also carries
  `sharded` (BASELINE configs[4] on ONE GPU: 10M x 128 in 8 sub-indexes by contiguous input range, batch 100k — the denominator of
  the 1 -> 8 GPU figure north_star asks for), `uniform` (the same headline kernel on uniform-random data) and `build` (BASELINE
  configs[2]: GPU Builder::build of 2M x 300, M=24, ef_construction=200, then batch=10k search on that graph, next to the threaded CPU
  build of the reference algorithm on a prefix).
--gpus N > 1 (auto): BASELINE.json configs[4] — the same 8 sub-indexes spread over the N GPUs (8/N each), every query searched on
  every sub-index, per-rank pre-merge, ONE ncclAllGather of the per-rank top-k, merge kernel (idb_sharded_search_batch_*_multi).
  `value` = queries/s of the whole job ("scaling": "strong"); `one_gpu_same_layout` = the same 8 sub-indexes on ONE GPU, measured by
  rank 0 in the same run (the denominator of the 1 -> N speed-up, SURVEY 8e; it is also `sharded` of the --gpus 1 line);
  `replicas` carries the configs[1] replica figure (queries sharded over N copies of the 1M index, no collective) as a secondary field.
--impl reference: the reference algorithm's CPU path (oracle/ restatement; the Rust crate cannot be built here) with all host
  threads, on the same config: N=1 -> configs[1]; N>1 -> configs[4] (rank 0 only; the other ranks exit).  It never loads the CUDA
  library: the graph both arms search is built in an untimed setup step by lib/idb_build_graph (a C++ program over the C ABI).

The indexes (>= 512 MB points + 308 MB adjacency) are far larger than the 126 MB L2 and every step uses a different query batch,
so no L2 flush is needed between iterations.  torch is plumbing only: device buffers, CUDA events, torch.distributed, brute force.
"""
import argparse
import ctypes as C
import functools
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "instant-distance_b200", "python"))

from tests import datagen  # noqa: E402  (seeded synthetic data shared with the tests)

TOOL = os.path.join(ROOT, "instant-distance_b200", "lib", "idb_build_graph")
K = 10  # results per query (recall@10)
N_SUB = 8  # sub-indexes of the sharded config


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def host_threads():
    n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE K1 launch at the headline config, from the committed ncu --set full
    capture of the current kernel (profiles/k1_ncu_traffic.json names the capture it was read from)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "k1_ncu_traffic.json")))
        return float(d["dram_bytes_per_launch"]), d["source"]
    except Exception:  # noqa: BLE001
        return None, None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md), via NVML every ~10 ms."""

    def __init__(self, gpu_index):
        self.rows, self.gpu, self._stop, self.th, self.h, self.nv = [], gpu_index, False, None, None, None

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            self.h, self.nv = nv.nvmlDeviceGetHandleByIndex(idx), nv
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
        except Exception as e:  # noqa: BLE001
            log("clock sampler unavailable:", e)

    def _run(self):
        nv = self.nv
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.rows.append((time.time(), sm, r, pw))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.01)

    def window(self, t0, t1):
        out = [r for r in self.rows if t0 <= r[0] <= t1]
        return out or [r for r in self.rows if t0 - 0.05 <= r[0] <= t1 + 0.05] or self.rows[-3:]

    def stop(self):
        self._stop = True

    def summarize(self, rows):
        if not rows or self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted({k for k, bit in names.items() for r in rows if r[2] & bit})
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": float(self.max_sm), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(r[3] for r in rows)}


# ---------------------------------------------------------------------------------------------------------------------
# workloads and graphs (setup; never timed)
# ---------------------------------------------------------------------------------------------------------------------
def generator(data):
    return datagen.sift_shaped if data == "sift" else datagen.uniform


def permute_points(pts, ids):
    p = np.empty_like(pts)
    p[ids] = pts  # points[pid] = rows[orig]   (lib.rs:262-270)
    return p


def cache_dir():
    """IDB_CACHE, else a per-user directory under the system temp dir: the tree bench.py runs from may be read-only."""
    d = os.environ.get("IDB_CACHE") or os.path.join(tempfile.gettempdir(), f"idb_bench_cache_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


@functools.lru_cache(maxsize=None)
def file_digest(path):
    h = hashlib.sha1()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 22), b""):
            h.update(block)
    return h.hexdigest()


def graph_cache_path(n, dim, data, data_seed, M, efc, seed, builder):
    """`builder` is the binary that builds the graph (the CUDA library, or the oracle's for --graph oracle).  Its digest is part of
    the key, so a cached graph is only reused by the same build of the code that made it, whichever checkout runs bench.py."""
    key = f"{n}-{dim}-{data}-{data_seed}-{M}-{efc}-{seed}-{os.path.basename(builder)}-{file_digest(builder)}-v4"
    return os.path.join(cache_dir(), "graph_" + hashlib.sha1(key.encode()).hexdigest()[:16] + ".npz")


def build_graph_with_tool(pts, M, efc, ef, seed, device):
    """Graph of `pts` by the GPU Builder::build, through lib/idb_build_graph (a separate C++ process over the C ABI).
    Returns (ids, zero, upper list, build seconds)."""
    n, dim = pts.shape
    base = os.path.join(cache_dir(), f"tool_{os.getpid()}")
    raw = base + ".points.f32"
    np.ascontiguousarray(pts, dtype=np.float32).tofile(raw)
    try:
        r = subprocess.run([TOOL, raw, str(n), str(dim), str(M), str(efc), str(ef), str(seed), str(device), base],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"idb_build_graph failed: {r.stderr.strip()[-400:]}")
        meta = open(base + ".meta").read().split()
        n_layers = int(meta[3])
        layer_n = [int(x) for x in meta[4:4 + n_layers]]
        ids = np.fromfile(base + ".ids.u32", dtype=np.uint32)
        zero = np.fromfile(base + ".zero.u32", dtype=np.uint32).reshape(n, 2 * M)
        upper = [np.fromfile(f"{base}.upper{l}.u32", dtype=np.uint32).reshape(layer_n[l], M) for l in range(1, n_layers)]
        return ids, zero, upper, float(meta[4 + n_layers])
    finally:
        for f in os.listdir(cache_dir()):
            if f.startswith(os.path.basename(base) + "."):
                os.remove(os.path.join(cache_dir(), f))


def obtain_graph(pts, n, dim, data, data_seed, M, efc, ef, seed, device, use_abi, no_cache=False, by="gpu"):
    """(points in PointId order, zero, upper, ids).  The graph is the GPU Builder::build's (deterministic in the seed): built
    in-process when the caller is the CUDA arm (use_abi), else by the C++ tool; cached under cache_dir() (graph_cache_path).
    by="oracle" (--graph oracle): the reference algorithm's own threaded CPU build (lib.rs:313-318) instead — BASELINE configs[1]'s
    "reference-built graph" to the letter; minutes of host time at 1M points, so it is not the default."""
    if by == "oracle":
        from oracle import oracle as O

        builder = O.build_lib()
        use_abi = False
    elif use_abi:
        from instant_distance_b200 import _abi

        builder = _abi.LIB_PATH
    else:
        builder = os.path.join(os.path.dirname(TOOL), "libinstant_distance_b200.so")  # the library the tool loads
    cp = graph_cache_path(n, dim, data, data_seed, M, efc, seed, builder) if os.path.exists(builder) else None
    if cp and os.path.exists(cp) and not no_cache:
        try:
            z = np.load(cp)
            got = permute_points(pts, z["ids"]), z["zero"], [z[f"u{i}"] for i in range(int(z["n_upper"]))], z["ids"]
            log(f"graph loaded from cache {os.path.basename(cp)}")
            if by == "oracle":
                GRAPH_HOW["by"] = "oracle (reference algorithm, threaded CPU build, lib.rs:313-318), searched by both arms"
            return got
        except Exception as e:  # noqa: BLE001  (a truncated file from an interrupted run: rebuild)
            log(f"graph cache {os.path.basename(cp)} unreadable ({e!r}); rebuilding")
    t = time.time()
    if use_abi:
        from instant_distance_b200 import _abi

        ix, ids = _abi.Index.build(pts, M=M, ef_construction=efc, ef_search=ef, seed=seed, device=device)
        _, zero, upper = ix.export_graph()
        ix.close()
    elif by == "oracle":
        ids = None
    elif os.path.exists(TOOL):
        try:
            ids, zero, upper, _ = build_graph_with_tool(pts, M, efc, ef, seed, device)
        except Exception as e:  # noqa: BLE001  (no GPU on this box: the reference algorithm builds it on the CPU)
            log("GPU graph tool unavailable:", e)
            ids = None
    else:
        ids = None
    stand_in = ids is None and by != "oracle"  # the oracle builds in place of the GPU build: not cached under the library's key
    if ids is None:
        from oracle import oracle as O

        ix, ids = O.build(pts, M=M, ef_construction=efc, ef_search=ef, seed=seed, threads=host_threads())
        g = ix.export()
        zero, upper = g.zero, g.upper
        if by == "oracle":
            GRAPH_HOW["by"] = "oracle (reference algorithm, threaded CPU build, lib.rs:313-318), searched by both arms"
        else:
            GRAPH_HOW["by"] = GRAPH_HOW["sharded"] = "oracle (reference algorithm, threaded CPU build): no GPU was available to this arm"
        log("graph built by the oracle (CPU) — NOT the GPU build's graph")
    log(f"graph built in {time.time() - t:.1f}s (setup, untimed)")
    if cp and not no_cache and not stand_in:
        try:
            tmp = cp[:-4] + f".{os.getpid()}.tmp.npz"  # written whole, then renamed: a reader never sees a partial file
            np.savez(tmp, ids=ids, zero=zero, n_upper=len(upper), **{f"u{i}": u for i, u in enumerate(upper)})
            os.replace(tmp, cp)
        except Exception as e:  # cache is best effort
            log("cache write failed:", e)
    return permute_points(pts, ids), zero, upper, ids


GRAPH_NOTE = "GPU Builder::build of this library (deterministic in the seed; untimed setup), searched by both arms"
GRAPH_HOW = {"by": GRAPH_NOTE, "sharded": GRAPH_NOTE}  # replaced when a graph had to be built by the oracle on the CPU (no GPU on the box)


def search_config(a, world, mode):
    par = "1 GPU" if world == 1 else f"replica x{world}, queries sharded, no collective"
    return {"workload": f"{a.n} x {a.dim} f32 {a.data}-shaped synthetic, M={a.M}, ef_construction={a.efc}, ef_search={a.ef}, "
                        f"batch={a.batch} queries/step, k={K}",
            "graph": GRAPH_HOW["by"], "l2": "index >> 126 MB L2 and a fresh query batch per step (no flush needed)", "parallelism": par}


def sharded_config(a, world):
    return {"workload": f"{N_SUB} x {a.shard_n} = {N_SUB * a.shard_n} x {a.dim} f32 sift-shaped synthetic in {N_SUB} sub-indexes by contiguous "
                        f"input range, M={a.M}, ef_construction={a.efc}, ef_search={a.ef}, batch={a.shard_batch} queries/step, k={K}",
            "graph": GRAPH_HOW["sharded"], "l2": "every sub-index >> 126 MB L2 and a fresh query batch per step (no flush needed)",
            "parallelism": f"{N_SUB} sub-indexes over {world} GPU(s) ({N_SUB // world} per GPU), per-rank pre-merge + ONE ncclAllGather + merge"}


def brute_force_topk_torch(points_dev, queries, k):
    import torch

    q = torch.from_numpy(queries).to(points_dev.device)
    pn = (points_dev * points_dev).sum(1)
    ids, ds = [], []
    for s in range(0, q.shape[0], 256):
        qq = q[s:s + 256]
        d = pn[None, :] - 2.0 * (qq @ points_dev.T) + (qq * qq).sum(1)[:, None]
        t = torch.topk(d, k, dim=1, largest=False)
        ids.append(t.indices.cpu())
        ds.append(t.values.cpu())
    return torch.cat(ids).numpy(), torch.cat(ds).numpy()


def recall_at_k(ids, truth, k=10):
    hit = 0
    for a, b in zip(ids[:, :k], truth[:, :k]):
        hit += len(set(a.tolist()) & set(b.tolist()))
    return hit / (k * len(ids))


def algorithmic_bytes(counters, dim, M, k, elem=4):
    """SURVEY §8d: B(q) = vec + sum_layers[n_expand_l * row_bytes_l + n_dist_l * vec] + k*8."""
    vec = dim * elem
    c = counters.astype(np.float64)
    per_q = dim * 4 + c[:, 0] * (M * 4) + c[:, 1] * vec + c[:, 2] * (2 * M * 4) + c[:, 3] * vec + k * 8
    return per_q


def cpu_qps(search_fn, batches, warm, timed):
    """The ONE CPU-baseline protocol (in-arm leg and reference arm): `warm` untimed passes, then `timed` passes."""
    for b in batches[:warm]:
        search_fn(b)
    t0 = time.perf_counter()
    for b in batches[warm:warm + timed]:
        search_fn(b)
    dt = time.perf_counter() - t0
    return sum(len(b) for b in batches[warm:warm + timed]) / dt, dt


DUMP_BYTES = 64_000_000  # all files of one dump, .npy headers included
NPY_HEADER = 128  # bytes of an .npy (v1.0) header for these shapes


def dump_outputs(d, outputs):
    """--dump-outputs: the last timed step's results (one row per query) as d/<name>.npy — ids and lengths as float64 (exact),
    distances as float32 — so that two builds can be compared output for output.  Beyond DUMP_BYTES in all, a fixed seeded
    sample of rows is written instead, with the sampled row numbers as rows.npy."""
    out = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in outputs.items()}
    n = len(out["ids"])
    row_bytes = sum(v.nbytes for v in out.values()) // n
    if n * row_bytes + NPY_HEADER * len(out) > DUMP_BYTES:
        m = (DUMP_BYTES - NPY_HEADER * (len(out) + 1)) // (row_bytes + 8)  # (+ 8: the row number in rows.npy)
        rows = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        out = {**{k: v[rows] for k, v in out.items()}, "rows": rows.astype(np.float64)}
    os.makedirs(d, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), v)


def pinned(nbytes, dtype, shape):
    from instant_distance_b200 import _abi

    p = C.c_void_p()
    _abi.check(_abi.lib().idb_host_alloc(nbytes, C.byref(p)))
    buf = (C.c_char * nbytes).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


def reduce_max(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist

    t = torch.tensor([x], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()


# ---------------------------------------------------------------------------------------------------------------------
# leg: one index per rank, queries sharded over ranks (BASELINE configs[1] at N = 1)
# ---------------------------------------------------------------------------------------------------------------------
def leg_search(a, rank, local_rank, world, full=True):
    import torch

    from instant_distance_b200 import _abi

    gen = generator(a.data)
    pts = gen(a.n, a.dim, 1)
    p, zero, upper, _ = obtain_graph(pts, a.n, a.dim, a.data, 1, a.M, a.efc, a.ef, a.seed, local_rank, use_abi=True,
                                     no_cache=a.no_cache or world > 1, by=a.graph)
    del pts
    ix = _abi.Index.from_graph(p, zero, upper, a.M, a.ef, device=local_rank)
    ix.set_profiling(True)

    # ---- recall gate: raise ef_search until recall@10 >= 0.95 on a sample --------------------------------------
    pdev = torch.from_numpy(p).cuda()
    rq = gen(a.recall_sample, a.dim, 999)
    truth, _ = brute_force_topk_torch(pdev, rq, K)
    del pdev
    torch.cuda.empty_cache()
    ef, recall = a.ef, 0.0
    for cand in [a.ef, 128, 160, 200, 256, 320, 400, 512, 768, 1024]:
        if cand < a.ef:
            continue
        ids, _, _ = ix.search(rq, ef_search=cand, k=K)
        ef, recall = cand, recall_at_k(ids, truth)
        log(f"[{a.data}] recall@10 = {recall:.4f} at ef_search = {cand}")
        if recall >= 0.95 or not full:  # the secondary (uniform-data) line stays at the config's ef_search
            break
    else:
        log("WARNING: recall@10 < 0.95 even at ef_search = 1024")

    # ---- device-resident arm ("value"): batches alternate over two submission lanes ----------------------------------
    total = a.warmup + a.steps
    nq = a.batch
    host_q = [gen(nq, a.dim, 5000 + 977 * rank + s) for s in range(total)]
    dq = [torch.from_numpy(q).cuda() for q in host_q]
    max_lanes = 4
    d_ids = [torch.empty((nq, K), dtype=torch.int32, device="cuda") for _ in range(max_lanes)]
    d_dist = [torch.empty((nq, K), dtype=torch.float32, device="cuda") for _ in range(max_lanes)]
    d_len = [torch.empty((nq,), dtype=torch.int32, device="cuda") for _ in range(max_lanes)]
    streams = [torch.cuda.ExternalStream(ix.lane_stream(l), device=local_rank) for l in range(max_lanes)]
    torch.cuda.synchronize()

    def step(s, lane):
        ix.search_device(dq[s].data_ptr(), nq, ef, K, d_ids[lane].data_ptr(), d_dist[lane].data_ptr(), d_len[lane].data_ptr(), lane=lane)

    def device_arm(lanes):
        """W warm steps, then exactly K timed steps issued round-robin over `lanes` submission lanes; device time, max over ranks."""
        for s in range(a.warmup):
            step(s, s % lanes)
        ix.sync()
        sampler = ClockSampler(local_rank)
        sampler.start()
        time.sleep(0.3)
        barrier(world)
        torch.cuda.synchronize()
        ev0 = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(lanes)]
        t_wall0 = time.time()
        ev0.record(streams[0])
        for l in range(1, lanes):
            streams[l].wait_event(ev0)
        n_launch = 0
        for s in range(a.warmup, total):
            step(s, s % lanes)
            n_launch += 2  # K1 search_kernel + its (normally idle) overflow-retry launch; the control-block memset is not a kernel
        for l in range(lanes):
            ends[l].record(streams[l])
        for l in range(lanes):
            ends[l].synchronize()
        torch.cuda.synchronize()
        t_wall1 = time.time()
        barrier(world)
        ms = reduce_max(max(ev0.elapsed_time(e) for e in ends), world)
        ck = sampler.summarize(sampler.window(t_wall0, t_wall1))
        sampler.stop()
        return ms, ck, n_launch

    lanes = a.lanes
    dev_ms, clocks, launches = device_arm(lanes)
    last = (total - 1) % lanes  # the last timed step's results, before the sweep and the isolated launches reuse the buffers
    outputs = {"ids": d_ids[last].cpu().numpy().view(np.uint32), "distances": d_dist[last].cpu().numpy(),
               "lengths": d_len[last].cpu().numpy().view(np.uint32)}
    qps = world * nq * a.steps / (dev_ms / 1e3)
    sweep = None
    if a.sweep and full:
        sweep = {"lanes_ms_per_step": {str(l): device_arm(l)[0] / a.steps for l in (1, 2, 3, 4)}}

    # isolated launches (one lane, event-bracketed per launch, back to back), then the algorithmic bytes of the same batches
    iso_ms, alg_bytes = [], []
    for s in range(a.warmup, total):
        step(s, 0)
        ms, _ = ix.last_kernel_ms()
        iso_ms.append(ms)
    for s in range(a.warmup, total):
        step(s, 0)
        alg_bytes.append(float(algorithmic_bytes(ix.last_counters(nq), a.dim, a.M, K).sum()))
    assert ix.last_failures(0) == 0
    retried = ix.last_retried(0)
    alg = float(np.mean(alg_bytes))
    peak, peak_src = measured_peaks()
    k_ms = dev_ms / a.steps
    res = {
        "value": qps, "ms_per_step": dev_ms / a.steps, "recall_at_10": recall, "ef_search": ef, "gpu_launches": launches, "clocks": clocks,
        "retried_per_launch": retried,
        "roofline": {"bound": "hbm", "achieved": alg / (k_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": alg / (k_ms / 1e3) / 1e9 / peak, "traffic": None, "kernel": "search_kernel (K1 search_layer)",
                     "kernel_ms": k_ms, "kernel_ms_note": f"timed region / launches, {lanes} launches in flight (successive launches overlap at the batch boundary)",
                     "kernel_ms_isolated": float(np.mean(iso_ms)), "frac_isolated": alg / (float(np.mean(iso_ms)) / 1e3) / 1e9 / peak,
                     "algorithmic_bytes_per_launch": alg, "peak_source": peak_src},
        "outputs": outputs,
    }
    if a.n == 1_000_000 and a.dim == 128 and a.batch == 10_000 and a.data == "sift":
        res["roofline"]["traffic"], res["roofline"]["traffic_source"] = ncu_traffic()
    if not full:
        ix.close()
        return res

    # ---- e2e arm: public host API, pinned host buffers, H2D + D2H inside the timed region, two caller threads --------------
    L = _abi.lib()
    hqs = []
    for s_ in range(total):
        h = pinned(nq * a.dim * 4, np.float32, (nq, a.dim))
        h[...] = host_q[s_]
        hqs.append(h)
    max_callers = 4
    hid = [pinned(nq * K * 4, np.uint32, (nq, K)) for _ in range(max_callers)]
    hds = [pinned(nq * K * 4, np.float32, (nq, K)) for _ in range(max_callers)]
    hln = [pinned(nq * 4, np.uint32, (nq,)) for _ in range(max_callers)]
    last_ids = {}

    def e2e_step(s, t):
        _abi.check(L.idb_search_batch_f32(ix._h, _abi.ptr(hqs[s], C.c_float), nq, ef, K, _abi.ptr(hid[t], C.c_uint32),
                                          _abi.ptr(hds[t], C.c_float), _abi.ptr(hln[t], C.c_uint32)))

    def e2e_run(lo, hi, callers):
        def work(t):
            for s in range(lo + t, hi, callers):
                e2e_step(s, t)
                if s == total - 1:
                    last_ids["ids"], last_ids["dist"], last_ids["len"] = hid[t].copy(), hds[t].copy(), hln[t].copy()
        th = [threading.Thread(target=work, args=(t,)) for t in range(callers)]
        [x.start() for x in th]
        [x.join() for x in th]

    def e2e_arm(callers):
        e2e_run(0, a.warmup, callers)
        barrier(world)
        t0 = time.perf_counter()
        e2e_run(a.warmup, total, callers)
        return reduce_max(time.perf_counter() - t0, world)

    callers = a.callers
    if sweep is not None:
        sweep["e2e_callers_qps"] = {str(c): world * nq * a.steps / e2e_arm(c) for c in (1, 2, 3, 4) if c != callers}
    e2e_s = e2e_arm(callers)  # (last: the parity leg below compares the final batch's results)
    res["e2e"] = {"value": world * nq * a.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": nq * a.dim * 4,
                  "d2h_bytes_per_step": nq * K * 8 + nq * 4, "callers": callers}
    if sweep is not None:
        sweep["e2e_callers_qps"][str(callers)] = res["e2e"]["value"]
        res["sweep"] = sweep

    # ---- CPU baseline (rank 0, N=1 leg only) + parity against it: ids, distances, lengths AND traversal counters -------------
    res["cpu_baseline"] = None
    if rank == 0 and world == 1 and not a.skip_cpu_baseline:
        from oracle import oracle as O

        T = host_threads()
        ox = O.from_graph(O.Graph(p, zero, upper, a.M, ef))
        sample = min(nq, a.ref_sample)
        o_ids, o_dist, o_len, o_cnt = ox.search(host_q[total - 1][:sample], ef_search=ef, k=K, threads=T, counters=True)
        ix.search(host_q[total - 1][:sample], ef_search=ef, k=K)
        g_cnt = ix.last_counters(sample)
        same = bool((o_ids == last_ids["ids"][:sample]).all() and o_dist.tobytes() == last_ids["dist"][:sample].tobytes()
                    and (o_len == last_ids["len"][:sample]).all() and (o_cnt == g_cnt).all())
        if not same:
            log("PARITY FAILURE: GPU results differ from the oracle on the same graph")
        batches = [q[:sample] for q in host_q]
        v, dt = cpu_qps(lambda b: ox.search(b, ef_search=ef, k=K, threads=T), batches, a.warmup, a.steps)
        res["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": T, "kind": "port",
                               "sample": f"{a.steps} passes of {sample} queries after {a.warmup} warm passes ({dt:.1f} s), same graph, ef_search={ef}, "
                                         f"{T} threads (one Search per thread); GPU ids/distances/lengths/counters identical to the oracle's: {same}"}
        res["parity_ok"] = same
    ix.close()
    return res


# ---------------------------------------------------------------------------------------------------------------------
# leg: BASELINE configs[4] — 8 sub-indexes by contiguous input range over `world` GPUs, one all-gather per batch
# ---------------------------------------------------------------------------------------------------------------------
def shard_points(a, s):
    return datagen.sift_shaped(a.shard_n, a.dim, 1000 + s)


def leg_sharded(a, rank, local_rank, world, full=True):
    import torch
    import torch.distributed as dist

    from instant_distance_b200 import _abi
    from instant_distance_b200 import sharded as SH

    assert N_SUB % world == 0, "the sharded config needs 1, 2, 4 or 8 GPUs"
    per = N_SUB // world
    mine = list(range(rank * per, (rank + 1) * per))
    gen = datagen.sift_shaped
    shards, gmaps, t_build = [], [], 0.0
    rq = gen(a.recall_sample, a.dim, 999)
    truth_local = []
    for s in mine:
        pts = shard_points(a, s)
        t = time.time()
        ix, ids = _abi.Index.build(pts, M=a.M, ef_construction=a.efc, ef_search=a.ef, seed=a.seed + s, device=local_rank)
        t_build += time.time() - t
        gmaps.append(SH.global_id_map(ids, s * a.shard_n))
        ix.set_id_map(gmaps[-1])
        shards.append(ix)
        pdev = torch.from_numpy(pts).cuda()  # exact top-10 of the sample queries on this sub-index (for recall)
        ti, td = brute_force_topk_torch(pdev, rq, K)
        truth_local.append((td, ti.astype(np.int64) + s * a.shard_n))
        del pdev, pts
        torch.cuda.empty_cache()
    log(f"rank {rank}: built sub-indexes {mine} in {t_build:.1f}s (Builder::build on the GPU, setup)")
    uid = _abi.comm_unique_id() if rank == 0 else None
    if world > 1:
        box = [uid]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
    sys.stdout.flush()
    saved = os.dup(1)  # NCCL prints its version banner on stdout when NCCL_DEBUG is set: keep stdout to the ONE JSON line
    os.dup2(2, 1)
    try:
        comm = _abi.Comm(uid, rank, world, local_rank)
    finally:
        os.dup2(saved, 1)
        os.close(saved)
    shards[0].set_profiling(True)

    total = a.warmup + a.steps
    nq = a.shard_batch
    dq_pool = [torch.from_numpy(gen(nq, a.dim, 7000 + s)).cuda() for s in range(min(total, 6))]  # identical on every rank
    d_ids = torch.empty((nq, K), dtype=torch.int32, device="cuda")
    d_dist = torch.empty((nq, K), dtype=torch.float32, device="cuda")
    d_len = torch.empty((nq,), dtype=torch.int32, device="cuda")
    main = torch.cuda.ExternalStream(shards[0].stream, device=local_rank)
    torch.cuda.synchronize()

    def step(s):
        _abi.sharded_search_multi_device(shards, comm, dq_pool[s % len(dq_pool)].data_ptr(), nq, a.ef, K, d_ids.data_ptr(), d_dist.data_ptr(),
                                         d_len.data_ptr())

    for s in range(a.warmup):
        step(s)
    for ix in shards:
        ix.sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.2)
    barrier(world)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record(main)
    for s in range(a.warmup, total):
        step(s)
    ev1.record(main)
    ev1.synchronize()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    barrier(world)
    dev_ms = reduce_max(ev0.elapsed_time(ev1), world)
    clocks = sampler.summarize(sampler.window(t_wall0, t_wall1))
    sampler.stop()
    qps = nq * a.steps / (dev_ms / 1e3)
    launches = a.steps * (2 * per + (1 if per > 1 else 0) + 2)  # per shard K1 + retry; pre-merge; all-gather; merge
    outputs = {"ids": d_ids.cpu().numpy().view(np.uint32), "distances": d_dist.cpu().numpy(), "lengths": d_len.cpu().numpy().view(np.uint32)}

    # K1 of the rank's first sub-index, isolated, for the roofline of the dominant kernel
    shards[0].search_device(dq_pool[0].data_ptr(), nq, a.ef, K, d_ids.data_ptr(), d_dist.data_ptr(), d_len.data_ptr())
    k_ms, _ = shards[0].last_kernel_ms()
    alg = float(algorithmic_bytes(shards[0].last_counters(nq), a.dim, a.M, K).sum())
    peak, peak_src = measured_peaks()

    # ---- recall@10 of the merged result against the exact top-10 over all N_SUB sub-indexes; protocol + parity checks --------
    td = np.concatenate([t[0] for t in truth_local], axis=1)
    ti = np.concatenate([t[1] for t in truth_local], axis=1)
    sample = a.recall_sample
    loc = [ix.search(rq, ef_search=a.ef, k=K) for ix in shards]  # per sub-index results (global ids) of the sample
    keys_loc = np.stack([SH.pack_keys(d_, i_, l_) for (i_, d_, l_) in loc])
    if world > 1:
        gt, gk = [None] * world, [None] * world
        dist.all_gather_object(gt, (td, ti))
        dist.all_gather_object(gk, keys_loc)
        td, ti = np.concatenate([g[0] for g in gt], axis=1), np.concatenate([g[1] for g in gt], axis=1)
        keys_all = np.concatenate(gk, axis=0)
    else:
        keys_all = keys_loc
    order = np.argsort(td, axis=1, kind="stable")[:, :K]
    truth = np.take_along_axis(ti, order, axis=1)
    m_ids, m_dist, m_len = _abi.sharded_search_multi(shards, comm, rq, ef_search=a.ef, k=K)  # collective, host buffers
    recall = recall_at_k(m_ids.astype(np.int64), truth)
    want_ids, want_dist, want_len = SH.merge_keys(keys_all, K)
    protocol_ok = bool((m_ids == want_ids).all() and m_dist.tobytes() == want_dist.tobytes() and (m_len == want_len).all())
    res = {
        "value": qps, "unit": "queries/s", "n_gpus": world, "ms_per_step": dev_ms / a.steps, "recall_at_10": recall,
        "merged_eq_protocol": protocol_ok, "gpu_launches": launches, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": alg / (k_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (k_ms / 1e3) / 1e9 / peak,
                     "traffic": None, "kernel": "search_kernel (K1) of one sub-index, isolated launch", "kernel_ms": k_ms,
                     "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                     "share_of_step": per * k_ms / (dev_ms / a.steps)},
        "build_s_per_rank": t_build, "outputs": outputs,
    }
    if not protocol_ok:
        log("PROTOCOL FAILURE: the fused sharded search differs from the host statement of the protocol")
    if full:
        # e2e: the host-buffer collective, H2D of the batch + D2H of the result inside the timed region
        hq = [pinned(nq * a.dim * 4, np.float32, (nq, a.dim)) for _ in range(2)]
        for i, h in enumerate(hq):
            h[...] = gen(nq, a.dim, 7000 + i)
        hid, hds, hln = pinned(nq * K * 4, np.uint32, (nq, K)), pinned(nq * K * 4, np.float32, (nq, K)), pinned(nq * 4, np.uint32, (nq,))
        L = _abi.lib()
        hs = _abi._handles(shards)

        def e2e_step(s):
            _abi.check(L.idb_sharded_search_batch_f32_multi(hs, len(shards), comm._h, _abi.ptr(hq[s % 2], C.c_float), nq, a.ef, K,
                                                            _abi.ptr(hid, C.c_uint32), _abi.ptr(hds, C.c_float), _abi.ptr(hln, C.c_uint32)))

        for s in range(a.warmup):
            e2e_step(s)
        barrier(world)
        t0 = time.perf_counter()
        for s in range(a.steps):
            e2e_step(s)
        e2e_s = reduce_max(time.perf_counter() - t0, world)
        res["e2e"] = {"value": nq * a.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": nq * a.dim * 4,
                      "d2h_bytes_per_step": nq * K * 8 + nq * 4, "steps": a.steps}
        # parity of one sub-index against the oracle on that sub-index's graph (rank 0's first)
        if rank == 0 and not a.skip_cpu_baseline:
            from oracle import oracle as O

            pp, zz, uu = shards[0].export_graph()
            ox = O.from_graph(O.Graph(pp, zz, uu, a.M, a.ef))
            o_ids, o_dist, o_len = ox.search(rq, ef_search=a.ef, k=K, threads=host_threads())
            l_ids, l_dist, l_len = loc[0]  # the GPU returns global ids (id map): map the oracle's PointIds the same way
            o_gids = np.where(o_ids == 0xFFFFFFFF, np.uint32(0xFFFFFFFF), gmaps[0][np.minimum(o_ids, a.shard_n - 1)])
            res["shard0_eq_oracle"] = bool((o_gids == l_ids).all() and (o_len == l_len).all() and o_dist.tobytes() == l_dist.tobytes())
            if not res["shard0_eq_oracle"]:
                log("PARITY FAILURE: sub-index 0 on the GPU differs from the oracle on the same graph")
    for ix in shards:
        ix.close()
    comm.close()
    return res


# ---------------------------------------------------------------------------------------------------------------------
# leg: BASELINE configs[2] — GPU Builder::build (points/s) next to the threaded CPU build of the reference algorithm
# ---------------------------------------------------------------------------------------------------------------------
def leg_build(a, local_rank):
    import torch

    from instant_distance_b200 import _abi

    gen = generator(a.data)
    pts = gen(a.n, a.dim, 1)
    times = []
    ix = None
    for rep in range(a.build_reps):
        if ix is not None:
            ix.close()
        t = time.perf_counter()
        ix, ids = _abi.Index.build(pts, M=a.M, ef_construction=a.efc, ef_search=a.ef, seed=a.seed, device=local_rank)
        times.append(time.perf_counter() - t)
        log(f"GPU Builder::build {a.n} x {a.dim}, M={a.M}, ef_construction={a.efc}: {times[-1]:.2f}s")
    rq = gen(a.recall_sample, a.dim, 999)
    pdev = torch.from_numpy(pts).cuda()
    truth, _ = brute_force_topk_torch(pdev, rq, K)
    del pdev
    inv = np.empty(a.n, dtype=np.int64)
    inv[ids] = np.arange(a.n)
    g_ids, _, _ = ix.search(rq, ef_search=a.ef, k=K)
    recall = recall_at_k(inv[np.minimum(g_ids, a.n - 1)], truth)
    res = {"metric": "GPU Builder::build throughput", "value": a.n / min(times), "unit": "points/s", "seconds": times,
           "recall_at_10_of_built_graph": recall, "ef_search": a.ef,
           "config": {"workload": f"{a.n} x {a.dim} f32 {a.data}-shaped synthetic, M={a.M}, ef_construction={a.efc}"}}
    # batched search on the graph just built (configs[2]: "GPU Builder::build + batch=10k search"): ef_search raised until recall@10 >= 0.95
    ef_s, rec_s = a.ef, recall
    for cand in [128, 160, 200, 256, 320, 400, 512]:
        if rec_s >= 0.95:
            break
        if cand <= ef_s:
            continue
        g_ids, _, _ = ix.search(rq, ef_search=cand, k=K)
        ef_s, rec_s = cand, recall_at_k(inv[np.minimum(g_ids, a.n - 1)], truth)
    nq = a.batch
    dq = [torch.from_numpy(gen(nq, a.dim, 5000 + s)).cuda() for s in range(4)]
    d_ids = torch.empty((nq, K), dtype=torch.int32, device="cuda")
    d_dist = torch.empty((nq, K), dtype=torch.float32, device="cuda")
    d_len = torch.empty((nq,), dtype=torch.int32, device="cuda")
    ix.set_profiling(True)
    k_ms, alg = [], []
    for s in range(a.warmup + a.steps):
        ix.search_device(dq[s % 4].data_ptr(), nq, ef_s, K, d_ids.data_ptr(), d_dist.data_ptr(), d_len.data_ptr())
        ms, _ = ix.last_kernel_ms()
        if s >= a.warmup:
            k_ms.append(ms)
            alg.append(float(algorithmic_bytes(ix.last_counters(nq), a.dim, a.M, K).sum()))
    peak, _ = measured_peaks()
    res["search"] = {"value": nq / (float(np.mean(k_ms)) / 1e3), "unit": "queries/s", "batch": nq, "ef_search": ef_s, "recall_at_10": rec_s,
                     "kernel_ms": float(np.mean(k_ms)), "k1_frac": float(np.mean(alg)) / (float(np.mean(k_ms)) / 1e3) / 1e9 / peak,
                     "what": f"K1 launches of one {nq}-query batch each (device-resident, isolated, {a.steps} timed after {a.warmup} warm), "
                             "on the graph built above"}
    del dq, d_ids, d_dist, d_len
    if not a.skip_cpu_baseline:
        from oracle import oracle as O

        T = host_threads()
        sub = min(a.n, a.build_cpu_sample)
        t = time.perf_counter()
        ox, o_ids = O.build(pts[:sub], M=a.M, ef_construction=a.efc, ef_search=a.ef, seed=a.seed, threads=T)
        dt = time.perf_counter() - t
        truth_s, _ = O.bruteforce(pts[:sub], rq[:200], K, threads=T)
        oi, _, _ = ox.search(rq[:200], ef_search=a.ef, k=K, threads=T)
        inv_s = np.empty(sub, dtype=np.int64)
        inv_s[o_ids] = np.arange(sub)
        # the same subset built on the GPU: is the batched GPU graph as good as the reference algorithm's (recall within noise)?
        gx, g_ids = _abi.Index.build(pts[:sub], M=a.M, ef_construction=a.efc, ef_search=a.ef, seed=a.seed, device=local_rank)
        gi, _, _ = gx.search(rq[:200], ef_search=a.ef, k=K)
        inv_g = np.empty(sub, dtype=np.int64)
        inv_g[g_ids] = np.arange(sub)
        res["recall_at_10_subset_gpu_graph"] = recall_at_k(inv_g[np.minimum(gi, sub - 1)], truth_s)
        gx.close()
        res["cpu_baseline"] = {"value": sub / dt, "unit": "points/s", "cores": T, "kind": "port",
                               "sample": f"threaded build (lib.rs:313-318: top layer sequential, the rest parallel with per-row locks) of the first "
                                         f"{sub} points in {dt:.1f}s; HNSW insert cost grows ~log N, so the full-size rate is lower",
                               "recall_at_10": recall_at_k(inv_s[oi], truth_s)}
    ix.close()
    return res


# ---------------------------------------------------------------------------------------------------------------------
# reference arm (CPU only; never imports the CUDA binding)
# ---------------------------------------------------------------------------------------------------------------------
def run_reference(a, rank, world):
    if rank != 0:
        return
    from oracle import oracle as O

    T = host_threads()
    if world == 1 or a.mode == "headline":
        gen = generator(a.data)
        pts = gen(a.n, a.dim, 1)
        p, zero, upper, _ = obtain_graph(pts, a.n, a.dim, a.data, 1, a.M, a.efc, a.ef, a.seed, 0, use_abi=False, no_cache=a.no_cache, by=a.graph)
        ix = O.from_graph(O.Graph(p, zero, upper, a.M, a.ef))
        sample = min(a.batch, a.ref_sample)
        batches = [gen(sample, a.dim, 5000 + s)[:sample] for s in range(a.warmup + a.steps)]
        last = []
        qps, dt = cpu_qps(lambda b: last.append(ix.search(b, ef_search=a.ef, k=K, threads=T)), batches, a.warmup, a.steps)
        outputs = dict(zip(("ids", "distances", "lengths"), last[-1]))
        cfg = search_config(a, 1, "headline")
        metric = "batched QPS at recall@10>=0.95 (1M x 128 f32)"
        desc = f"{sample} queries per step x {a.steps} steps after {a.warmup} warm steps, same graph/ef, {T} threads, one Search per thread"
        scaling = "weak"
    else:
        subs = []
        for s in range(N_SUB):
            pts = shard_points(a, s)
            p, zero, upper, ids = obtain_graph(pts, a.shard_n, a.dim, "sift", 1000 + s, a.M, a.efc, a.ef, a.seed + s, 0, use_abi=False,
                                               no_cache=a.no_cache)
            gid = np.empty(a.shard_n, dtype=np.uint32)
            gid[ids] = np.arange(s * a.shard_n, (s + 1) * a.shard_n, dtype=np.uint32)
            subs.append((O.from_graph(O.Graph(p, zero, upper, a.M, a.ef)), gid))
        sample = min(a.shard_batch, a.ref_sample_sharded)
        batches = [datagen.sift_shaped(sample, a.dim, 7000 + s) for s in range(a.warmup + a.steps)]

        def search_all(b):  # every query on every sub-index, then the k smallest (distance, global id) of the union
            keys = []
            for ox, gid in subs:
                i_, d_, l_ = ox.search(b, ef_search=a.ef, k=K, threads=T)
                g_ = gid[np.minimum(i_, a.shard_n - 1)]
                kk = (d_.view(np.uint32).astype(np.uint64) << np.uint64(32)) | g_.astype(np.uint64)
                kk[np.arange(K)[None, :] >= l_[:, None]] = np.uint64(0xFFFFFFFFFFFFFFFF)
                keys.append(kk)
            return np.sort(np.concatenate(keys, axis=1), axis=1)[:, :K]

        last = []
        qps, dt = cpu_qps(lambda b: last.append(search_all(b)), batches, a.warmup, a.steps)
        if a.dump_outputs:
            from instant_distance_b200.sharded import merge_keys  # (host code only: the CUDA library stays unloaded)

            outputs = dict(zip(("ids", "distances", "lengths"), merge_keys(last[-1][None], K)))
        cfg = sharded_config(a, world)
        metric = "batched QPS, 10M x 128 f32 in 8 PointId-range sub-indexes (BASELINE configs[4])"
        desc = (f"{sample} queries per step x {a.steps} steps after {a.warmup} warm steps, each searched on all {N_SUB} sub-indexes and merged on the "
                f"host, {T} threads")
        scaling = "strong"
    line = {
        "impl": "reference", "metric": metric, "value": qps, "unit": "queries/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg, "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": T, "kind": "port", "sample": desc},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="auto", choices=["auto", "headline", "sharded", "build"])
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--batch", type=int, default=10_000)
    ap.add_argument("--ef", type=int, default=100)
    ap.add_argument("--efc", type=int, default=100)
    ap.add_argument("--M", type=int, default=32)
    ap.add_argument("--seed", type=int, default=20260923)
    ap.add_argument("--data", default="sift", choices=["sift", "uniform"])
    ap.add_argument("--no-cache", action="store_true")
    ap.add_argument("--graph", default="gpu", choices=["gpu", "oracle"],
                    help="headline leg: who builds the graph both arms search — this library's GPU Builder::build (default) or the reference "
                         "algorithm's threaded CPU build (the oracle; minutes at 1M points)")
    ap.add_argument("--recall-sample", type=int, default=1000)
    ap.add_argument("--ref-sample", type=int, default=10_000)
    ap.add_argument("--ref-sample-sharded", type=int, default=2_000)
    ap.add_argument("--shard-n", type=int, default=1_250_000)
    ap.add_argument("--shard-batch", type=int, default=100_000)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true", help="N=1: headline only (no sharded / uniform legs)")
    ap.add_argument("--lanes", type=int, default=2, choices=[1, 2, 3, 4], help="submission lanes the device-resident arm alternates over")
    ap.add_argument("--callers", type=int, default=3, choices=[1, 2, 3, 4], help="host threads calling idb_search_batch_f32 in the e2e arm")
    ap.add_argument("--sweep", action="store_true", help="also time 1..4 lanes / callers (reported under `sweep`)")
    ap.add_argument("--build-reps", type=int, default=2)
    ap.add_argument("--build-cpu-sample", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ids, distances and lengths of the last timed search step as DIR/<name>.npy")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)  # timing rule: at least 3 untimed warm-up steps
    if a.dump_outputs and a.impl == "ours" and a.mode == "build":
        ap.error("--dump-outputs needs a search mode (--mode auto, headline or sharded)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        return run_reference(a, rank, world)

    import torch
    import torch.distributed as dist

    from instant_distance_b200 import _abi

    if _abi.lib().idb_device_count() < 1:
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(minutes=30))
    mode = a.mode if a.mode != "auto" else ("headline" if world == 1 else "sharded")
    common = {"n_gpus": world, "steps": a.steps, "warmup": a.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "f32",
              "data": "synthetic"}

    out = outputs = None
    if mode == "build":
        res = leg_build(a, local_rank)
        out = {**res, **common, "scaling": "weak"}
    elif mode == "headline":
        t_leg = time.time()
        h = leg_search(a, rank, local_rank, world)
        outputs = h.get("outputs")
        log(f"headline leg took {time.time() - t_leg:.1f}s")
        line = {"metric": "batched QPS at recall@10>=0.95 (1M x 128 f32)", "value": h["value"], "unit": "queries/s", **common,
                "ms_per_step": h["ms_per_step"], "scaling": "weak"}
        secondary = world == 1 and a.mode == "auto" and not a.skip_secondary

        def secondary_leg(key, what, fn):
            """A secondary leg of the N=1 line: its failure is reported under its key and never takes the headline down with it."""
            t_leg = time.time()
            try:
                line[key] = {"what": what, **fn()}
            except Exception as e:  # noqa: BLE001
                log(f"{key} leg FAILED: {e!r}")
                line[key] = {"what": what, "error": repr(e)[:300]}
                try:
                    torch.cuda.empty_cache()
                except Exception:  # noqa: BLE001
                    pass
            log(f"{key} leg took {time.time() - t_leg:.1f}s")

        def sharded_leg():
            s = leg_sharded(a, rank, local_rank, world, full=False)
            return {"value": s["value"], "unit": "queries/s", "ms_per_step": s["ms_per_step"], "recall_at_10": s["recall_at_10"],
                    "merged_eq_protocol": s["merged_eq_protocol"], "gpu_launches": s["gpu_launches"], "k1_frac": s["roofline"]["frac"]}

        if secondary:
            secondary_leg("sharded", f"BASELINE configs[4] on ONE GPU ({N_SUB} sub-indexes x {a.shard_n}, batch {a.shard_batch}): the 1-GPU point of "
                                     f"the strong-scaling curve `--gpus N` reports", sharded_leg)
        line.update({"config": search_config(a, world, mode), "recall_at_10": h["recall_at_10"], "ef_search": h["ef_search"], "e2e": h.get("e2e"),
                     "gpu_launches": h["gpu_launches"], "retried_per_launch": h["retried_per_launch"], "roofline": h["roofline"],
                     **({"sweep": h["sweep"]} if "sweep" in h else {}),
                     "cpu_baseline": h.get("cpu_baseline"), "clocks": h["clocks"]})

        def uniform_leg():
            ua = argparse.Namespace(**{**vars(a), "data": "uniform", "graph": "gpu"})
            u = leg_search(ua, rank, local_rank, world, full=False)
            return {"value": u["value"], "unit": "queries/s", "recall_at_10": u["recall_at_10"], "ef_search": u["ef_search"],
                    "k1_frac": u["roofline"]["frac"]}

        def build_leg():
            ba = argparse.Namespace(**{**vars(a), "n": 2_000_000, "dim": 300, "M": 24, "efc": 200, "ef": 100, "data": "sift", "batch": 10_000,
                                       "build_reps": 1})
            b = leg_build(ba, local_rank)
            return {k_: b[k_] for k_ in ("value", "unit", "seconds", "recall_at_10_of_built_graph", "ef_search", "config", "search",
                                         "recall_at_10_subset_gpu_graph", "cpu_baseline") if k_ in b}

        if secondary:
            secondary_leg("uniform", "the same kernel on uniform-random 1M x 128 (north_star's wording): no neighbourhood structure, recall@10 stays far "
                                     "below 0.95 at any practical ef", uniform_leg)
            secondary_leg("build", "BASELINE configs[2]: GPU Builder::build of 2M x 300 f32 (M=24, ef_construction=200) + batch=10k search on the graph it "
                                   "built; cpu_baseline = the reference algorithm's threaded build of a prefix on this box's host threads", build_leg)
        out = line
    else:  # sharded
        s = leg_sharded(a, rank, local_rank, world)
        outputs = s.get("outputs")
        line = {"metric": "batched QPS, 10M x 128 f32 in 8 PointId-range sub-indexes (BASELINE configs[4])", "value": s["value"], "unit": "queries/s",
                **common, "ms_per_step": s["ms_per_step"], "scaling": "strong",
                "strong_scaling_note": "the 1-GPU point of this curve is `sharded.value` of the --gpus 1 line (same 8 sub-indexes on one GPU); that line's "
                                       "primary value is configs[1], as the bench contract requires at N=1"}
        if world > 1 and a.mode == "auto" and not a.skip_secondary:
            ra = argparse.Namespace(**{**vars(a), "graph": "gpu"})
            r = leg_search(ra, rank, local_rank, world, full=False)
            line["replicas"] = {"what": "configs[1] with the 1M index replicated per GPU and the queries sharded (no collective)", "value": r["value"],
                                "unit": "queries/s", "k1_frac": r["roofline"]["frac"], "recall_at_10": r["recall_at_10"]}
        if world > 1 and a.mode == "auto" and not a.skip_secondary:
            # the denominator of the 1 -> N figure (SURVEY 8e): the SAME 8 sub-indexes on ONE GPU, measured by rank 0 in this very run
            # (world-size-1 communicator; the other ranks wait at the barrier below)
            if rank == 0:
                what = (f"the same {N_SUB} sub-indexes x {a.shard_n}, batch {a.shard_batch}, on ONE GPU of this box (rank 0, world-size-1 "
                        "communicator), same run: the 1-GPU point of this strong-scaling curve")
                try:
                    o = leg_sharded(a, 0, local_rank, 1, full=False)
                    line["one_gpu_same_layout"] = {"what": what, "value": o["value"], "unit": "queries/s", "ms_per_step": o["ms_per_step"],
                                                   "recall_at_10": o["recall_at_10"], "merged_eq_protocol": o["merged_eq_protocol"],
                                                   "k1_frac": o["roofline"]["frac"]}
                except Exception as e:  # noqa: BLE001  (the other ranks are waiting at the barrier: never leave them there)
                    log(f"one_gpu_same_layout leg FAILED: {e!r}")
                    line["one_gpu_same_layout"] = {"what": what, "error": repr(e)[:300]}
            barrier(world)
        line.update({"config": sharded_config(a, world), "recall_at_10": s["recall_at_10"], "ef_search": a.ef, "e2e": s.get("e2e"),
                     "gpu_launches": s["gpu_launches"], "roofline": s["roofline"], "merged_eq_protocol": s["merged_eq_protocol"],
                     "shard0_eq_oracle": s.get("shard0_eq_oracle"), "cpu_baseline": None, "clocks": s["clocks"]})
        out = line
    if world > 1:
        dist.destroy_process_group()  # (before the JSON line: NCCL's own log lines may share stdout)
    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, outputs)
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
