#!/usr/bin/env python
"""RRT* tree growth for a batch of seeds in one device call (porrt_rrt_grow_batch) at the config-1 shape (single-world stand-in map
synth.rrt_map, bounds [-1, 1]^2, max_step 0.1, search_radius 1.0, n_iter 2500 .. 10000, goal radius 0.05), seeds 0 .. R-1, against
the C++ restatement over the oracle (tests/rrt_oracle.py) growing the same R seeds one after another on one host thread and with
one process per seed over all host cores.  Writes one JSON file.

    python scripts/rrt_grow_batch_bench.py --out profiles/r3_rrt_grow_batch_bench.json
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
import rrt_oracle as RO  # noqa: E402

CONFIG1 = dict(max_step=0.1, search_radius=1.0, n_min=2500, n_max=10000)
START, GOAL, REPS = (-0.8, -0.8), [((0.8, 0.8), [1])], 3
RS = (1, 8, 32, 64, 148)
EXACT_R = 8

_W = {}


def _worker_init():
    _W.update(omap=O.GridMap(synth.rrt_map(), None, util.LOW, util.UP, P.DOOR, 0.3), goal=O.SquareGoal(GOAL, 0.05))


def _worker_grow(seed):
    ref = RO.RRT(_W["omap"], util.LOW, util.UP, seed=seed)
    return ref.grow_tree(START, _W["goal"], CONFIG1["max_step"], CONFIG1["search_radius"], CONFIG1["n_min"], CONFIG1["n_max"])


def run(ctx, rs, procs):
    occ = synth.rrt_map()
    omap, pmap = util.make_pair(ctx, occ, None, P.DOOR, 0.3)
    pgoal, ogoal = P.SquareGoal(GOAL, 0.05), O.SquareGoal(GOAL, 0.05)
    ms_, sr, n_min, n_max = CONFIG1["max_step"], CONFIG1["search_radius"], CONFIG1["n_min"], CONFIG1["n_max"]
    out = {}
    # the oracle, one host thread, seed after seed: per-seed times, summed over the first R seeds
    t_seed, refs = [], []
    for s in range(max(rs)):
        t0 = time.perf_counter()
        ref = RO.RRT(omap, util.LOW, util.UP, seed=s)
        rc = ref.grow_tree(START, ogoal, ms_, sr, n_min, n_max)
        t_seed.append(1e3 * (time.perf_counter() - t0))
        if s < EXACT_R:
            refs.append((ref, rc))
    # the oracle, one process per seed over all host cores (pool started and its map built before the clock)
    with mp.get_context("fork").Pool(procs, initializer=_worker_init) as pool:
        pool.map(_worker_grow, range(procs))
        t_pool = {}
        for R in rs:
            t0 = time.perf_counter()
            pool.map(_worker_grow, range(R), chunksize=1)
            t_pool[R] = 1e3 * (time.perf_counter() - t0)
    for R in rs:
        dev = P.RRTBatch(pmap, util.LOW, util.UP, np.arange(R))
        dev.grow_tree(START, pgoal, ms_, sr, n_min, n_max)              # warm-up (module load, buffers)
        ts = []
        for _ in range(REPS):
            t0 = time.perf_counter()
            status = dev.grow_tree(START, pgoal, ms_, sr, n_min, n_max)
            ts.append(1e3 * (time.perf_counter() - t0))
        ms = min(ts)
        t_ref = float(sum(t_seed[:R]))
        row = {"device_ms_per_call": ms, "device_trees_per_s": 1e3 * R / ms,
               "oracle_1_thread_ms": t_ref, "oracle_1_thread_trees_per_s": 1e3 * R / t_ref,
               "oracle_all_cores_ms": t_pool[R], "oracle_all_cores_trees_per_s": 1e3 * R / t_pool[R],
               "beats_oracle_1_thread": bool(ms < t_ref), "beats_oracle_all_cores": bool(ms < t_pool[R]),
               "iterations_mean": float(dev.n_it.mean()), "V_mean": float(dev.sizes[:, 1].mean()),
               "with_final": int((status == 0).sum()),
               "windows_mean": float(dev.counters[:, 0].mean())}
        if R >= EXACT_R:
            exact = True
            for t, (ref, rc) in enumerate(refs):
                exact &= (int(status[t]) == rc and int(dev.n_it[t]) == ref.n_it()
                          and all(np.array_equal(a, b) for a, b in zip(dev.tree(t), ref.tree())))
            row["bit_exact_first_%d_trees" % EXACT_R] = bool(exact)
        out["R=%d" % R] = row
        print("config1", R, json.dumps(row), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rrt_grow_batch_bench.json"))
    ap.add_argument("--rs", default=",".join(str(r) for r in RS))
    a = ap.parse_args()
    rs = [int(x) for x in a.rs.split(",")]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    procs = os.cpu_count()
    ctx = P.Context(0)
    res = {"gpu": gpu, "host_cores": procs, "reps": REPS, "seeds": "0 .. R-1", "shape": dict(CONFIG1, map="synth.rrt_map()", start=START,
                                                                                          goal=GOAL[0][0], goal_max_dist=0.05),
           "timing": "device: best of reps after a warm-up, host clock around porrt_rrt_grow_batch (ends in a device synchronise); "
                     "oracle 1 thread: the R seeds one after another, one pass; oracle all cores: one pass of a process pool",
           "oracle_all_cores": "C++ restatement, %d processes -- not the reference" % procs}
    res["config1"] = run(ctx, rs, procs)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
