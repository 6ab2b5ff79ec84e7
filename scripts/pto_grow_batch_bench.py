#!/usr/bin/env python
"""PTO roadmap growth for a batch of seeds in one device call (porrt_pto_grow_batch) at the config-3 and config-4 shapes (stand-in
shelf maps, as scripts/pto_grow_bench.py), seeds 0 .. R-1, against the oracle growing the same R seeds one after another on one
host thread and with one process per seed over all host cores.  Writes one JSON file.

    python scripts/pto_grow_batch_bench.py --out profiles/r3_pto_grow_batch_bench.json
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

SHAPES = {"config3": dict(Z=8, visibility=0.5, max_step=0.1, search_radius=2.0, n_min=5000),
          "config4": dict(Z=12, visibility=0.2, max_step=0.05, search_radius=5.0, n_min=5000)}
START, N_MAX, REPS = (0.0, -0.9), 100000, 3
RS = (1, 8, 32, 64, 148)
EXACT_R = 8


def shelf(Z, visibility):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return occ, zones, omap, goals


_W = {}


def _worker_init(shape):
    sh = SHAPES[shape]
    _, _, omap, goals = shelf(sh["Z"], sh["visibility"])
    _W.update(omap=omap, goal=O.SquareGoal(goals, 0.05), sh=sh)


def _worker_grow(seed):
    sh = _W["sh"]
    ref = O.PTO(_W["omap"], util.LOW, util.UP, seed=seed)
    return ref.grow_graph(START, _W["goal"], sh["max_step"], sh["search_radius"], sh["n_min"], N_MAX)


def run_shape(ctx, name, Z, visibility, max_step, search_radius, n_min, rs, procs):
    occ, zones, omap, goals = shelf(Z, visibility)
    pmap = P.MapShelfDomain(ctx, occ, util.LOW, util.UP)
    pmap.add_zones(zones, visibility)
    pgoal, ogoal = P.SquareGoal(goals, 0.05), O.SquareGoal(goals, 0.05)
    out = {}
    # the oracle, one host thread, seed after seed: per-seed times, summed over the first R seeds
    t_seed, refs = [], []
    for s in range(max(rs)):
        t0 = time.perf_counter()
        ref = O.PTO(omap, util.LOW, util.UP, seed=s)
        rc = ref.grow_graph(START, ogoal, max_step, search_radius, n_min, N_MAX)
        t_seed.append(1e3 * (time.perf_counter() - t0))
        if s < EXACT_R:
            refs.append((ref, rc))
    # the oracle, one process per seed over all host cores (pool started and its map built before the clock)
    with mp.get_context("fork").Pool(procs, initializer=_worker_init, initargs=(name,)) as pool:
        pool.map(_worker_grow, range(procs))
        t_pool = {}
        for R in rs:
            t0 = time.perf_counter()
            pool.map(_worker_grow, range(R), chunksize=1)
            t_pool[R] = 1e3 * (time.perf_counter() - t0)
    for R in rs:
        dev = P.PTOBatch(pmap, util.LOW, util.UP, np.arange(R))
        dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX)              # warm-up (module load, buffers)
        ts = []
        for _ in range(REPS):
            t0 = time.perf_counter()
            status = dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX)
            ts.append(1e3 * (time.perf_counter() - t0))
        ms = min(ts)
        t_ref = float(sum(t_seed[:R]))
        row = {"device_ms_per_call": ms, "device_roadmaps_per_s": 1e3 * R / ms,
               "oracle_1_thread_ms": t_ref, "oracle_1_thread_roadmaps_per_s": 1e3 * R / t_ref,
               "oracle_all_cores_ms": t_pool[R], "oracle_all_cores_roadmaps_per_s": 1e3 * R / t_pool[R],
               "beats_oracle_1_thread": bool(ms < t_ref), "beats_oracle_all_cores": bool(ms < t_pool[R]),
               "iterations_mean": float(dev.n_it.mean()), "V_mean": float(dev.sizes[:, 1].mean()),
               "complete": int((status == 0).sum()),
               "windows_mean": float(dev.counters[:, 0].mean())}
        if R == EXACT_R:
            exact = True
            for r, (ref, rc) in enumerate(refs):
                want = ref.graph.export(0)
                ids, masks = dev.finals(r)
                oids, obits = ref.reach.finals()
                exact &= (int(status[r]) == rc and int(dev.n_it[r]) == ref.n_it()
                          and all(np.array_equal(a, b) for a, b in zip(dev.graph_arrays(r), want))
                          and np.array_equal(dev.reach_masks(r), ref.reach.all(len(want[0]))) and np.array_equal(ids, oids)
                          and np.array_equal(masks, P.words_from_bits(obits)))
            row["bit_exact_every_roadmap"] = bool(exact)
        out["R=%d" % R] = row
        print(name, R, json.dumps(row), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pto_grow_batch_bench.json"))
    ap.add_argument("--shapes", default="config3,config4")
    ap.add_argument("--rs", default=",".join(str(r) for r in RS))
    a = ap.parse_args()
    rs = [int(x) for x in a.rs.split(",")]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    procs = os.cpu_count()
    ctx = P.Context(0)
    res = {"gpu": gpu, "host_cores": procs, "reps": REPS, "seeds": "0 .. R-1",
           "timing": "device: best of reps after a warm-up, host clock around porrt_pto_grow_batch (ends in a device synchronise); "
                     "oracle 1 thread: the R seeds one after another, one pass; oracle all cores: one pass of a process pool",
           "oracle_all_cores": "C++ restatement, %d processes -- not the reference" % procs}
    for name in a.shapes.split(","):
        res[name] = run_shape(ctx, name, rs=rs, procs=procs, **SHAPES[name])
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
