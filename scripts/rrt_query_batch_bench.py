#!/usr/bin/env python
"""RRT* planning for R distinct queries in one device call: porrt_rrt_grow_queries + porrt_rrt_best_paths, the paths fetched, at the
config-1 parameters of rrt_grow_batch_bench.py (single-world stand-in map synth.rrt_map, bounds [-1, 1]^2, max_step 0.1,
search_radius 1.0, n_iter 2500 .. 10000) for R in 1, 8, 32, 64, 148.  Query k has its own start and goal centre (free space, drawn
with a fixed seed), goal radius 0.05 and sampler seed k.  The CPU baseline is the C++ restatements on the same queries
(tests/rrt_oracle.cpp's grow_tree, the tree's export, tests/rrt_best_oracle.cpp's best path), on one host thread and with one
process per query over all host cores.  Also alternates grow_queries on R identical rows with grow_batch on the same seeds, to show
what the per-query form costs.  Writes one JSON file.

    python scripts/rrt_query_batch_bench.py --out profiles/r3_rrt_query_batch_bench.json
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402

import po_rrt_b200 as P  # noqa: E402
from po_rrt_b200 import synth  # noqa: E402
from oracle import pyoracle as O  # noqa: E402
import porrt_testutil as util  # noqa: E402
import rrt_best_oracle as RB  # noqa: E402
import rrt_oracle as RO  # noqa: E402

CONFIG1 = dict(max_step=0.1, search_radius=1.0, n_min=2500, n_max=10000)
GOAL_R, REPS, QUERY_SEED = 0.05, 3, 2024
RS = (1, 8, 32, 64, 148)
OVERHEAD_R = 64

_W = {}


def queries(omap, n):
    """n (start, goal centre) pairs of free space in [-0.9, 0.9]^2 from a fixed seed"""
    rng, pts = np.random.default_rng(QUERY_SEED), []
    while len(pts) < 2 * n:
        p = rng.uniform(-0.9, 0.9, 2)
        if omap.state_validity([list(p)])[0] >= 0:
            pts.append((float(p[0]), float(p[1])))
    return pts[:n], pts[n:]


def _oracle_plan(omap, seed, start, centre):
    ref = RO.RRT(omap, util.LOW, util.UP, seed=seed)
    ref.grow_tree(start, O.SquareGoal([(centre, [1])], GOAL_R), CONFIG1["max_step"], CONFIG1["search_radius"], CONFIG1["n_min"],
                  CONFIG1["n_max"])
    return RB.best_path(ref.tree())


def _worker_init(starts, centres):
    _W.update(omap=O.GridMap(synth.rrt_map(), None, util.LOW, util.UP, P.DOOR, 0.3), starts=starts, centres=centres)


def _worker_plan(k):
    got = _oracle_plan(_W["omap"], k, _W["starts"][k], _W["centres"][k])
    return None if got is None else got[1]


def run(ctx, rs, procs):
    omap, pmap = util.make_pair(ctx, synth.rrt_map(), None, P.DOOR, 0.3)
    starts, centres = queries(omap, max(rs))
    ms_, sr, n_min, n_max = CONFIG1["max_step"], CONFIG1["search_radius"], CONFIG1["n_min"], CONFIG1["n_max"]
    # the oracle, one host thread, query after query
    t_query, ref_paths = [], []
    for k in range(max(rs)):
        t0 = time.perf_counter()
        ref_paths.append(_oracle_plan(omap, k, starts[k], centres[k]))
        t_query.append(1e3 * (time.perf_counter() - t0))
    # the oracle, one process per query over all host cores (pool started and its map built before the clock)
    with mp.get_context("fork").Pool(procs, initializer=_worker_init, initargs=(starts, centres)) as pool:
        pool.map(_worker_plan, range(procs))
        t_pool = {}
        for R in rs:
            t0 = time.perf_counter()
            pool.map(_worker_plan, range(R), chunksize=1)
            t_pool[R] = 1e3 * (time.perf_counter() - t0)
    out = {}
    for R in rs:
        dev = P.RRTBatch(pmap, util.LOW, util.UP, np.arange(R))
        goals = [P.SquareGoal([(c, [1])], GOAL_R) for c in centres[:R]]

        def plan():
            status = dev.grow_queries(starts[:R], goals, ms_, sr, n_min, n_max)
            return status, dev.best_paths()
        plan()                                                          # warm-up (module load, buffers)
        ts = []
        for _ in range(REPS):
            t0 = time.perf_counter()
            status, paths = plan()
            ts.append(1e3 * (time.perf_counter() - t0))
        ms = min(ts)
        exact = all((p is None and q is None) or (p is not None and q is not None and p[1] == q[1] and np.array_equal(p[0], q[0]))
                    for p, q in zip(paths, ref_paths[:R]))
        t_ref = float(sum(t_query[:R]))
        row = {"device_ms_per_call": ms, "device_queries_per_s": 1e3 * R / ms,
               "oracle_1_thread_ms": t_ref, "oracle_1_thread_queries_per_s": 1e3 * R / t_ref,
               "oracle_all_cores_ms": t_pool[R], "oracle_all_cores_queries_per_s": 1e3 * R / t_pool[R],
               "beats_oracle_1_thread": bool(ms < t_ref), "beats_oracle_all_cores": bool(ms < t_pool[R]),
               "iterations_mean": float(dev.n_it.mean()), "V_mean": float(dev.sizes[:, 1].mean()),
               "with_path": int(sum(p is not None for p in paths)), "path_states_total": int(sum(len(p[0]) for p in paths if p)),
               "windows_mean": float(dev.counters[:, 0].mean()), "paths_equal_oracle": bool(exact)}
        out["R=%d" % R] = row
        print("queries", R, json.dumps(row), flush=True)
    # per-query form against the seed batch on identical rows, alternated
    R = OVERHEAD_R
    start, goal = starts[0], P.SquareGoal([(centres[0], [1])], GOAL_R)
    a, b = P.RRTBatch(pmap, util.LOW, util.UP, np.arange(R)), P.RRTBatch(pmap, util.LOW, util.UP, np.arange(R))
    a.grow_tree(start, goal, ms_, sr, n_min, n_max)
    b.grow_queries([start] * R, [goal] * R, ms_, sr, n_min, n_max)
    t_batch, t_queries = [], []
    for _ in range(2 * REPS):
        t0 = time.perf_counter()
        a.grow_tree(start, goal, ms_, sr, n_min, n_max)
        t_batch.append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        b.grow_queries([start] * R, [goal] * R, ms_, sr, n_min, n_max)
        t_queries.append(1e3 * (time.perf_counter() - t0))
    same = bool(np.array_equal(a.sizes, b.sizes) and np.array_equal(a.counters, b.counters)
                and all(np.array_equal(x, y) for t in range(R) for x, y in zip(a.tree(t), b.tree(t))))
    out["identical_rows"] = {"R": R, "grow_batch_ms": t_batch, "grow_queries_ms": t_queries, "grow_batch_best_ms": min(t_batch),
                             "grow_queries_best_ms": min(t_queries), "trees_and_counters_equal": same}
    print("identical rows", json.dumps(out["identical_rows"]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rrt_query_batch_bench.json"))
    ap.add_argument("--rs", default=",".join(str(r) for r in RS))
    a = ap.parse_args()
    rs = [int(x) for x in a.rs.split(",")]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    procs = os.cpu_count()
    ctx = P.Context(0)
    res = {"gpu": gpu, "host_cores": procs, "reps": REPS, "queries": "starts and goal centres from free space, numpy seed %d; sampler "
                                                                       "seed k for query k" % QUERY_SEED,
           "shape": dict(CONFIG1, map="synth.rrt_map()", goal_max_dist=GOAL_R),
           "timing": "device: best of reps after a warm-up, host clock around grow_queries + best_paths (paths fetched; ends in a "
                     "device synchronise); oracle 1 thread: grow_tree + tree export + best path query after query, one pass; oracle "
                     "all cores: one pass of a process pool",
           "oracle_all_cores": "C++ restatement, %d processes -- not the reference" % procs}
    res["config1"] = run(ctx, rs, procs)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
