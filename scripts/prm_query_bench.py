#!/usr/bin/env python
"""PRM path queries on the device: porrt_prm_plan_paths (PRM.plan_paths) with every path fetched, on the PRM of bench.py's metric
line (the c5 door map, synth.door_map(8192, 6 zones, seed 1), max_step 0.1, search_radius 2.0) at V = 1e4, 1e5 and 1e6 nodes, for
Q = 1, 64, 1024 and 16384 queries whose goals are all distinct or 16 shared points.  Host clock around the call (it ends in a
synchronise and the copy of the paths), best of 3 after a warm-up.  The CPU baseline is the oracle's PRM::plan_path (a C++
restatement of prm.rs, not the reference) on the same roadmap, on one thread for up to 64 queries and, for V <= 1e5, on all host
cores as processes; every query the oracle answers must equal the device's bit for bit.  Writes one JSON file.

    python scripts/prm_query_bench.py --out profiles/r3_prm_query_bench.json
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

import numpy as np  # noqa: E402

import po_rrt_b200 as P  # noqa: E402
from po_rrt_b200 import synth  # noqa: E402
from oracle import pyoracle as O  # noqa: E402

LOW, UP = [-1.0, -1.0], [1.0, 1.0]
MS, SR, REPS = 0.1, 2.0, 3
VS = (10_000, 100_000, 1_000_000)
QS = (1, 64, 1024, 16384)
CPU_QUERIES = 64

_W = {}


def query_set(Q, shared, seed):
    rng = np.random.default_rng(seed)
    starts = rng.uniform(-1.0, 1.0, (Q, 2))
    goals = rng.uniform(-1.0, 1.0, (16, 2))[np.arange(Q) % 16] if shared else rng.uniform(-1.0, 1.0, (Q, 2))
    return np.ascontiguousarray(starts), np.ascontiguousarray(goals)


def _oracle_query(k):
    return _W["oprm"].plan_path(_W["starts"][k], _W["goals"][k])


def cpu_baseline(oprm, starts, goals, multi):
    """one thread over the queries (ms per query, paths), and all host cores as forked processes (queries/s) if multi"""
    paths, t0 = [], time.perf_counter()
    for s, g in zip(starts, goals):
        paths.append(oprm.plan_path(s, g))
    one = 1e3 * (time.perf_counter() - t0) / len(starts)
    procs = os.cpu_count() or 1
    qps = None
    if multi:
        _W.update(oprm=oprm, starts=starts, goals=goals)
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_oracle_query, range(min(procs, len(starts))))   # start-up out of the timing
            t0 = time.perf_counter()
            pool.map(_oracle_query, range(len(starts)), chunksize=1)
            qps = len(starts) / (time.perf_counter() - t0)
    return one, qps, procs, paths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_prm_query_bench.json"))
    ap.add_argument("--vs", default=",".join(str(v) for v in VS))
    ap.add_argument("--qs", default=",".join(str(q) for q in QS))
    args = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    ctx = P.Context(0)
    occ, zones = synth.door_map(size=8192, n_zones=6, seed=1)
    pmap = P.Map(ctx, occ, LOW, UP)
    pmap.add_zones(zones, 0.3)
    omap = O.GridMap(occ, zones, LOW, UP, O.DOOR, 0.3)
    res = {"gpu": gpu, "host_cores": os.cpu_count(), "map": "synth.door_map(8192, n_zones=6, seed=1), visibility 0.3",
           "prm": {"max_step": MS, "search_radius": SR, "samples": "synth.points(V, seed=10)"},
           "device": "porrt_prm_plan_paths, every path fetched; host clock, best of %d after a warm-up" % REPS,
           "cpu": "oracle PRM::plan_path (C++ restatement, not the reference), one thread on up to %d queries; V <= 1e5 also one "
                  "process per host core" % CPU_QUERIES, "rows": []}
    for V in (int(v) for v in args.vs.split(",")):
        pts = synth.points(V, seed=10)
        prm = P.PRM(pmap).grow_graph(pts, MS, SR, fetch_col=False)
        t0 = time.perf_counter()
        oprm = O.PRM(omap, LOW, UP, seed=0)
        oprm.add_samples(pts, MS, SR)
        print("V", V, "oracle PRM built in %.1f s" % (time.perf_counter() - t0), flush=True)
        for shared in (False, True):
            for Q in (int(q) for q in args.qs.split(",")):
                starts, goals = query_set(Q, shared, seed=100 + Q)
                out = prm.plan_paths(starts, goals)                   # warm-up
                best = None
                for _ in range(REPS):
                    t0 = time.perf_counter()
                    out = prm.plan_paths(starts, goals)
                    best = min(best or 1e30, time.perf_counter() - t0)
                row = {"V": V, "Q": Q, "goals": "16 shared" if shared else "distinct", "distinct_goal_nodes": int(len(np.unique(out[4]))),
                       "device_ms": 1e3 * best, "device_queries_per_s": Q / best, "path_states": int(sum(len(p) for p in out[0])),
                       "found": int((out[2] == P.PATH_FOUND).sum()), "none": int((out[2] == P.PATH_NONE).sum()),
                       "cycle": int((out[2] == P.PATH_CYCLE).sum())}
                if Q == 64:
                    # the oracle never returns from a CYCLE query: those are left out of the baseline
                    ks = [k for k in range(Q) if out[2][k] != P.PATH_CYCLE][:CPU_QUERIES if V < 1_000_000 else 8]
                    nq = len(ks)
                    one, qps, procs, paths = cpu_baseline(oprm, starts[ks], goals[ks], multi=V <= 100_000)
                    match = all(np.array_equal(p, out[0][k]) if out[2][k] == P.PATH_FOUND else len(p) == 0 for p, k in zip(paths, ks))
                    row.update({"cpu_queries": nq, "cpu_1thread_ms_per_query": one, "cpu_1thread_queries_per_s": 1e3 / one,
                                "cpu_processes": procs if qps else None, "cpu_processes_queries_per_s": qps,
                                "oracle_match": bool(match)})
                    assert match, row
                res["rows"].append(row)
                print(json.dumps(row), flush=True)
                with open(args.out, "w") as f:                       # after every row: a long run keeps what it measured
                    json.dump(res, f, indent=1)
        del oprm


if __name__ == "__main__":
    main()
