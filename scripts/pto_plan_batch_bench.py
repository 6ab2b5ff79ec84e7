#!/usr/bin/env python
"""Belief-space planning of every roadmap of a PTO seed batch in one device call (porrt_pto_plan_batch, PTOBatch.plan_belief_space)
against the per-roadmap loop on the same context and the same grown batch (porrt_pto_fetch_roadmap + plan_belief_space(copy=None)
per roadmap), at the config-3 and config-4 shapes (stand-in shelf maps, as scripts/pto_grow_batch_bench.py), seeds 0 .. R-1.
The two are timed alternately in one run, best of REPS after a warm-up, each with a host clock around work that ends in a device
synchronise; every roadmap's policy and expected cost from the batch must equal the loop's.  Beside them: the oracle's
single-thread belief pipeline (build_belief_graph + compute_expected_costs_to_goals + extract_policy) on two config-3 seeds, per
plan.  Writes one JSON file.

    python scripts/pto_plan_batch_bench.py --out profiles/r3_pto_plan_batch_bench.json
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
START, N_MAX, REPS = (0.0, -0.9), 100000, 3
RS = (1, 8, 32, 64, 148)
ORACLE_SEEDS = (0, 1)


def shelf(Z, visibility):
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, P.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    return occ, zones, omap, goals


def loop(pmap, dev, b0, beliefs):
    """the single path, roadmap after roadmap -> [(policy arrays, expected cost)]"""
    out = []
    for r in range(len(dev)):
        xy, nvid, rp, col, ev = dev.graph_arrays(r)
        ids, masks = dev.finals(r)
        p = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, ids, masks, beliefs=beliefs, copy=None)
        out.append(((p.policy_node, p.policy_belief, p.policy_parent, p.policy_leaf), p.expected_cost))
    return out


def same(batch, single):
    return all(p.status == 0 and p.expected_cost == c and all(np.array_equal(a, b) for a, b in
               zip((p.policy_node, p.policy_belief, p.policy_parent, p.policy_leaf), arrs)) for p, (arrs, c) in zip(batch, single))


def run_shape(ctx, name, Z, visibility, max_step, search_radius, n_min, rs):
    occ, zones, omap, goals = shelf(Z, visibility)
    pmap = P.MapShelfDomain(ctx, occ, util.LOW, util.UP)
    pmap.add_zones(zones, visibility)
    pgoal = P.SquareGoal(goals, 0.05)
    b0 = [1.0 / Z] * Z
    beliefs = pmap.reachable_belief_states(b0)
    out = {"B": len(beliefs)}
    for R in rs:
        dev = P.PTOBatch(pmap, util.LOW, util.UP, np.arange(R))
        dev.grow_graph(START, pgoal, max_step, search_radius, n_min, N_MAX)
        dev.plan_belief_space(b0, beliefs)                                          # warm-up (module load, buffers)
        single = loop(pmap, dev, b0, beliefs)
        t_batch, t_loop, phases = [], [], []
        exact = True
        for _ in range(REPS):                                                       # alternating
            t0 = time.perf_counter()
            plans = dev.plan_belief_space(b0, beliefs)
            ctx.synchronize()
            t_batch.append(1e3 * (time.perf_counter() - t0))
            phases.append([float(x) for x in dev.plan_phase_ms])
            t0 = time.perf_counter()
            single = loop(pmap, dev, b0, beliefs)
            ctx.synchronize()
            t_loop.append(1e3 * (time.perf_counter() - t0))
            exact &= same(plans, single)
        k = int(np.argmin(t_batch))
        row = {"batch_ms": min(t_batch), "loop_ms": min(t_loop), "speedup": min(t_loop) / min(t_batch),
               "batch_plans_per_s": 1e3 * R / min(t_batch), "loop_plans_per_s": 1e3 * R / min(t_loop),
               "batch_phase_ms": dict(zip(("host_setup", "preparation", "levels_device", "walks"), phases[k])),
               "V_mean": float(dev.sizes[:, 1].mean()), "policy_nodes_mean": float(np.mean([len(p.policy_node) for p in plans])),
               "equal_to_loop_every_roadmap": bool(exact)}
        out["R=%d" % R] = row
        print(name, R, json.dumps(row), flush=True)
    return out, omap, goals


def oracle_pipeline(omap, goals, sh):
    """the oracle's single-thread belief pipeline on ORACLE_SEEDS (growth not timed) -> ms per plan"""
    ts = []
    for s in ORACLE_SEEDS:
        ref = O.PTO(omap, util.LOW, util.UP, seed=s)
        ref.grow_graph(START, O.SquareGoal(goals, 0.05), sh["max_step"], sh["search_radius"], sh["n_min"], N_MAX)
        t0 = time.perf_counter()
        ref.build_belief_graph([1.0 / sh["Z"]] * sh["Z"])
        ref.compute_expected_costs_to_goals()
        ref.extract_policy()
        ts.append(1e3 * (time.perf_counter() - t0))
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pto_plan_batch_bench.json"))
    ap.add_argument("--shapes", default="config3,config4")
    ap.add_argument("--rs", default=",".join(str(r) for r in RS))
    ap.add_argument("--rs-config4", default="1", help="config-4 batch sizes: seed 3's policy walk runs to the 64 V B guard on "
                    "both paths (minutes), so R > 3 is not timed by default")
    ap.add_argument("--no-oracle", action="store_true")
    a = ap.parse_args()
    rs = [int(x) for x in a.rs.split(",")]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    ctx = P.Context(0)
    res = {"gpu": gpu.splitlines()[0] if gpu else "not measured", "reps": REPS, "seeds": "0 .. R-1",
           "timing": "best of reps after a warm-up, batch and loop alternating, host clock around each ending in a device synchronise; "
                     "loop = porrt_pto_fetch_roadmap + plan_belief_space(copy=None) per roadmap on the same ctx and grown batch"}
    for name in a.shapes.split(","):
        sh = SHAPES[name]
        rs_shape = [int(x) for x in a.rs_config4.split(",")] if name == "config4" else rs
        res[name], omap, goals = run_shape(ctx, name, **{k: sh[k] for k in ("Z", "visibility", "max_step", "search_radius", "n_min")},
                                           rs=rs_shape)
        if name == "config3" and not a.no_oracle:
            ts = oracle_pipeline(omap, goals, sh)
            res["oracle_config3_belief_pipeline_ms_per_plan"] = {"seeds": list(ORACLE_SEEDS), "ms": ts, "mean": float(np.mean(ts)),
                                                                 "note": "C++ restatement of the reference, one host thread"}
            print("oracle", json.dumps(res["oracle_config3_belief_pipeline_ms_per_plan"]), flush=True)
    ctx.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
