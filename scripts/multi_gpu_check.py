"""N-GPU check of the sharded paths (SURVEY.md 8(e)); run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 \
        scripts/multi_gpu_check.py [--big] [--out gpurun_out/multi_gpu_check.json]

Every rank holds two contexts on its GPU: `ctx` with an NCCL communicator (sharded porrt_prm_build / porrt_sssp_worlds,
porrt_comm_all_gather_dev) and `solo` without one (the single-GPU result).  Checks, all bit-exact:
  1. sharded PRM build == single-GPU PRM build == the oracle's PRM (CSR in the reference's insertion order), on every rank
  2. sharded plan_qmdp dist rows == single-GPU == oracle, through both value-backup schedules (on chip / frontier)
  3. all-gathered per-shard edge validity ids / world masks == the whole batch evaluated on one GPU
  4. belief-space value backups with the columns of every level sharded over the ranks == single GPU == oracle, both schedules
--big adds timings at the c5 shape (8192^2 map, V = 1e6 PRM build) and prints them as JSON on rank 0.
The oracle is used here as the checker only.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import po_rrt_b200 as P                    # noqa: E402
from po_rrt_b200 import shard, synth       # noqa: E402


def build_prm(pmap, xy, max_step, search_radius):
    prm = P.PRM(pmap)
    prm.init(xy[:1])
    prm.grow_graph(xy[1:], max_step, search_radius)
    return prm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29531")
    torch.cuda.set_device(local)
    dist.init_process_group("nccl" if world > 1 else "gloo", rank=rank, world_size=world,
                            device_id=torch.device("cuda", local) if world > 1 else None)
    ctx, solo = P.Context(local), P.Context(local)
    shard.init_comm(ctx)
    r, w, ver = ctx.comm_info()
    assert (r, w) == (rank, world)
    report = {"world": world, "nccl_version": ver}

    from oracle import pyoracle as O
    occ, zones = synth.door_map(size=512, n_rects=4096, n_zones=3, seed=11)
    maps = []
    for c in (ctx, solo):
        m = P.Map(c, occ, [-1.0, -1.0], [1.0, 1.0])
        m.add_zones(zones, 0.3)
        maps.append(m)
    pmap, smap = maps
    omap = O.GridMap(occ, zones, [-1.0, -1.0], [1.0, 1.0], O.DOOR, 0.3)

    # ---- 1. PRM build, ragged shards (n not divisible by world)
    n = 6001
    xy = synth.points(n, seed=5)
    got, one = build_prm(pmap, xy, 0.1, 2.0), build_prm(smap, xy, 0.1, 2.0)
    np.testing.assert_array_equal(got.row_ptr, one.row_ptr)
    np.testing.assert_array_equal(got.col, one.col)
    oprm = O.PRM(omap, [-1.0, -1.0], [1.0, 1.0], seed=0)
    oprm.init(xy[0])
    oprm.add_samples(xy[1:], 0.1, 2.0)
    _, _, rp, col, _ = oprm.graph.export(0)
    np.testing.assert_array_equal(got.row_ptr, rp)
    np.testing.assert_array_equal(got.col, col)
    report["prm_edges"] = int(len(col))
    # tiny builds: more ranks than useful work, empty shards
    for n_small in (1, 2, 3, 17):
        a, b = build_prm(pmap, xy[:n_small], 0.1, 2.0), build_prm(smap, xy[:n_small], 0.1, 2.0)
        np.testing.assert_array_equal(a.row_ptr, b.row_ptr)
        np.testing.assert_array_equal(a.col, b.col)

    # ---- 2. plan_qmdp: worlds sharded, dist rows all-gathered (8 worlds over `world` ranks; also 3 worlds: ragged / empty)
    nvid = smap.state_validity(got.states)
    keep = nvid >= 0
    nvid = np.where(keep, nvid, 0).astype(np.int32)
    vw = smap.world_validities_words()
    for force, n_fin_worlds in ((f, k) for f in (0, 1) for k in (8, 3)):   # force: the sharded run on the frontier relaxation
        finals = [list(range(k, n, 97 + 13 * k))[:5] for k in range(n_fin_worlds)]
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, force)
        a, _ = P.dijkstra_worlds(ctx, got.row_ptr, got.col, got.states, nvid, vw, finals)
        b, _ = P.dijkstra_worlds(solo, got.row_ptr, got.col, got.states, nvid, vw, finals)
        np.testing.assert_array_equal(a, b)
        assert np.isfinite(a).any()
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    report["qmdp_worlds"] = 8

    # ---- 3. per-shard edge validity + device all-gather
    E = 200_003
    fa, fb = synth.edges(E, seed=2, max_len=0.1)
    lo, hi = shard.shard_range(E, rank, world)
    dev = torch.device("cuda", local)
    ta, tb = torch.from_numpy(fa[lo:hi].copy()).to(dev), torch.from_numpy(fb[lo:hi].copy()).to(dev)
    vid_all = torch.full((E,), -77, dtype=torch.int32, device=dev)
    mask_all = torch.zeros((E,), dtype=torch.int64, device=dev)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    ctx.check(ctx.lib.porrt_edge_validity_dev(ctx.h, ta.data_ptr(), tb.data_ptr(), hi - lo,
                                              vid_all[lo:].data_ptr(), mask_all[lo:].data_ptr()))
    ctx.all_gather_dev(None, vid_all.data_ptr(), E, 4)       # in place: this rank's rows already sit at [lo, hi)
    ctx.all_gather_dev(None, mask_all.data_ptr(), E, 8)
    torch.cuda.synchronize()
    ctx.set_stream(None)
    want_vid, want_mask = smap.transition_validator(fa, fb, want_masks=True)
    np.testing.assert_array_equal(vid_all.cpu().numpy(), want_vid)
    np.testing.assert_array_equal(mask_all.cpu().numpy().view(np.uint64), want_mask.reshape(-1))
    np.testing.assert_array_equal(want_vid, omap.edge_validity(fa, fb))
    report["gathered_edges"] = E

    # ---- 4. belief-space value backups: the columns of every belief level sharded over the ranks, all-gathered per level
    for Z, nmin in ((5, 1500), (3, 700)):          # 31 / 7 beliefs: levels with fewer columns than ranks included
        socc, szones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
        somap = O.GridMap(socc, szones, [-1.0, -1.0], [1.0, 1.0], O.SHELF, 0.5)
        zp = somap.zone_positions()
        goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
        pto = O.PTO(somap, [-1.0, -1.0], [1.0, 1.0], seed=0)
        assert pto.grow_graph((0.0, -0.9), O.SquareGoal(goals, 0.05), 0.1, 2.0, nmin, 100000) == 0
        bxy, bnvid, brp, bcol, bev = pto.graph.export(0)
        fin_ids, fin_bits = pto.reach.finals()
        bms = []
        for c in (ctx, solo):
            bm = P.MapShelfDomain(c, socc, [-1.0, -1.0], [1.0, 1.0])
            bm.add_zones(szones, 0.5)
            bms.append(bm)
        pto.build_belief_graph([1.0 / Z] * Z)
        for force in (0, 1):                       # the sharded run on chip, then on the frontier relaxation
            ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, force)
            plans = [P.plan_belief_space(bm, brp, bcol, bev, bxy, bnvid, [1.0 / Z] * Z, fin_ids, P.words_from_bits(fin_bits)) for bm in bms]
            np.testing.assert_array_equal(plans[0].dist, plans[1].dist)
            np.testing.assert_array_equal(plans[0].type, plans[1].type)
            np.testing.assert_array_equal(plans[0].policy_node, plans[1].policy_node)
            np.testing.assert_array_equal(plans[0].dist.reshape(-1), pto.compute_expected_costs_to_goals())
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    report["belief_vi_sharded_levels"] = True
    for m in (pmap, smap):      # the belief problems replaced the ctx maps
        m.add_zones(zones, 0.3)

    if args.big:
        occ, zones = synth.door_map(size=8192, n_rects=4096, n_zones=6, seed=1)
        for m in (pmap, smap):
            m.occ, m.zones = occ, zones
            m.add_zones(zones, 0.3)
        big = {}
        for V in (100_000, 1_000_000):
            xy = synth.points(V, seed=3)
            col_buf = np.empty(80_000_000, np.int32)
            res = {}
            for name, m in (("sharded", pmap), ("single", smap)):
                best, phases, xch = 1e30, None, None
                for _ in range(4):
                    dist.barrier()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    prm = P.PRM(m)
                    prm.init(xy[:1])
                    prm.grow_graph(xy[1:], 0.1, 2.0, col_out=col_buf)
                    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
                    if name == "sharded":
                        dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    if t.item() < best:
                        best, phases = t.item(), [round(float(x), 3) for x in prm.phase_ms[:7]]
                        xch = m.ctx.last_phase_ms()[:1] if name == "sharded" and world > 1 else None
                res[name] = {"ms": best * 1e3, "phase_ms[radii,bin,radius,kd_rank,order,edges,csr]": phases, "exchange_ms": xch,
                             "directed_edges": int(prm.row_ptr[-1])}
                if name == "sharded":
                    keep_rp, keep_col = prm.row_ptr.copy(), prm.col.copy()
                else:
                    np.testing.assert_array_equal(keep_rp, prm.row_ptr)
                    np.testing.assert_array_equal(keep_col, prm.col)
            big["V%d" % V] = res
        report["prm_build"] = big

    dist.barrier()
    if rank == 0:
        line = json.dumps(report)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    ctx.comm_destroy()
    ctx.close()
    solo.close()
    dist.destroy_process_group()
    if rank == 0:
        print("multi_gpu_check: ok", flush=True)


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        traceback.print_exc()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(1)          # no interpreter teardown: a failed rank must not sit in a collective while torchrun waits for it
