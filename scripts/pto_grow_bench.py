#!/usr/bin/env python
"""PTO roadmap growth on the device (porrt_pto_grow) against the oracle's single-thread growth, at the config-3 and config-4
shapes (stand-in shelf maps, tests/test_pto_grow_gpu.py), and the end-to-end planner built on each.  Writes one JSON file.

    python scripts/pto_grow_bench.py --out profiles/r3_pto_grow_bench.json
"""
import argparse
import json
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
START, N_MAX, REPS = (0.0, -0.9), 100000, 5


def best(f, reps=REPS):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = f()
        ts.append(1e3 * (time.perf_counter() - t0))
    return min(ts), out


def run_shape(ctx, Z, visibility, max_step, search_radius, n_min):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    b0 = [1.0 / Z] * Z
    pgoal, ogoal = P.SquareGoal(goals, 0.05), O.SquareGoal(goals, 0.05)
    dev = P.PTO(pmap, util.LOW, util.UP, seed=0)
    dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX)                       # warm-up (module load, buffers)
    t_dev, rc = best(lambda: dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX))

    def oracle_grow():
        ref = O.PTO(omap, util.LOW, util.UP, seed=0)
        return ref, ref.grow_graph(START, ogoal, max_step, search_radius, n_min, N_MAX)
    t_ref, (ref, ref_rc) = best(oracle_grow)
    got, want = dev.graph_arrays(), ref.graph.export(0)
    ids, masks = dev.finals()
    oids, obits = ref.reach.finals()
    exact = (rc == ref_rc and dev.n_it == ref.n_it() and all(np.array_equal(a, b) for a, b in zip(got, want))
             and np.array_equal(dev.reach_masks(), ref.reach.all(len(want[0]))) and np.array_equal(ids, oids)
             and np.array_equal(masks, P.words_from_bits(obits)))

    def device_planner():
        dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX)
        xy, nvid, rp, col, ev = dev.graph_arrays()
        fi, fm = dev.finals()
        return P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fi, fm, copy=None)
    device_planner()
    t_e2e_dev, _ = best(device_planner)

    def oracle_planner():
        ref2, _ = oracle_grow()
        ref2.build_belief_graph(b0)
        ref2.compute_expected_costs_to_goals()
        return ref2.extract_policy()
    t_e2e_ref, _ = best(oracle_planner, reps=2 if Z > 8 else REPS)
    return {"device_grow_ms": t_dev, "oracle_grow_ms": t_ref, "speedup_grow": t_ref / t_dev, "bit_exact": bool(exact),
            "iterations": dev.n_it, "V": dev.sizes[1], "E": dev.sizes[2], "finals": dev.sizes[3],
            "counters": dict(zip(("windows", "respeculated", "conflicts_nn", "conflicts_radius_kd"), dev.counters)),
            "e2e_device_ms": t_e2e_dev, "e2e_oracle_ms": t_e2e_ref}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pto_grow_bench.json"))
    ap.add_argument("--shapes", default="config3,config4")
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    ctx = P.Context(0)
    res = {"gpu": gpu, "reps": REPS, "timing": "best of reps, host clock around the call (ends in a device synchronise)"}
    for name in a.shapes.split(","):
        res[name] = run_shape(ctx, **SHAPES[name])
        print(name, json.dumps(res[name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
