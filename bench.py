#!/usr/bin/env python
"""bench.py -- headline benchmark of the po-rrt hot path on B200 (BASELINE.json metric, config c5).

A "step" is one pass of batched edge-world validity over one batch of E synthetic edges against the synthetic
8192 x 8192 door map (6 zones => 64 worlds).  One process per GPU; ranks shard the edges (independent units, map
replicated, no data-path collective => weak scaling).

  value  : edge-world validity checks/s, inputs resident in HBM, kernel launched through porrt_edge_validity_dev
  e2e    : the same metric through the host-buffer C-ABI call porrt_edge_validity (pinned host buffers, H2D + D2H inside)
  --impl reference : the reference's CPU path (oracle restatement; the Rust crate cannot be built here) on host cores
  --dump-outputs DIR : the per-edge results of the last timed step as DIR/*.npy (dump_outputs), to compare two builds
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "edge_world_validity_checks_per_s"
UNIT = "edge-world checks/s"
N_WORLDS = 64


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--edges", type=int, default=1 << 24, help="edges per GPU per step")
    ap.add_argument("--map-size", type=int, default=8192)
    ap.add_argument("--cpu-sample", type=int, default=2_000_000, help="edges in the CPU-baseline sample")
    ap.add_argument("--no-extras", action="store_true", help="skip the kNN / PRM-build side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (rank 0's edges; "
                         "see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def workload_config(args):
    return {"workload": "c5: synthetic %dx%d occupancy grid, 6 door zones = 64 worlds, edges a->b with |ab| ~ U[0,0.1] in [-1,1]^2"
                        % (args.map_size, args.map_size),
            "edges_per_gpu_per_step": args.edges, "map_seed": 1, "edge_seed": "2+rank",
            "l2": "edge streams (32 B in + 12 B out per edge, %.0f MB per step) exceed L2; the 64 MiB fused grid is meant to stay L2-resident"
                  % (args.edges * 44 / 1e6)}


DUMP_EDGES = 1 << 20   # edges written by --dump-outputs: 4 B + 16 B each = 20 MiB


def dump_outputs(out_dir, vid, mask=None):
    """Writes the per-edge results of the timed path's last step, so that two builds can be compared output for output:
    validity_id.npy (float32, the validity id or panic code of each edge) and, where the path returns them, world_mask.npy
    (float64 [low 32 bits, high 32 bits] of each edge's 64-bit world mask; both halves are exact in float64).  Batches of more
    than DUMP_EDGES edges are sampled: the same ascending edge indices every run (numpy default_rng(0)) for a given batch size."""
    n = len(vid)
    idx = np.arange(n) if n <= DUMP_EDGES else np.sort(np.random.default_rng(0).choice(n, DUMP_EDGES, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "validity_id.npy"), np.asarray(vid)[idx].astype(np.float32))
    if mask is not None:
        m = np.ascontiguousarray(np.asarray(mask)[idx]).view(np.uint64)
        words = np.stack([m & np.uint64(0xFFFFFFFF), m >> np.uint64(32)], axis=1)
        np.save(os.path.join(out_dir, "world_mask.npy"), words.astype(np.float64))


def make_inputs(args, rank):
    from po_rrt_b200 import synth
    occ, zones = synth.door_map(size=args.map_size, n_zones=6, seed=1)
    a, b = synth.edges(args.edges, seed=2 + rank)
    return occ, zones, a, b


class ClockSampler:
    """SM clock / throttle reasons / power DURING the timed region (B200_PROFILING.md clocks line), polled in-process through
    NVML every ~2 ms from before the warm-up on, so that even a 14 ms timed region holds several samples; falls back to an
    `nvidia-smi -lms` child when NVML is not importable."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []          # (t, sm_mhz, max_mhz, power_w, [4 reason flags])
        self.stop_flag = False
        self.p = None
        self.source = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu_index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            float(pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM))   # a box whose NVML cannot be read goes to nvidia-smi below
            self.source = "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
        except Exception:
            try:
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                           "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.source = "nvidia-smi"
                self.t = threading.Thread(target=self._read_smi, daemon=True)
                self.t.start()
            except Exception:
                self.p = None

    def _poll_nvml(self):
        nv = self.nv
        masks = [nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                 nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap]
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:   # (one query failing must not cost the clock sample)
                    r = 0
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = 0.0
                self.rows.append((time.perf_counter(), sm, self.max_mhz, pw, [bool(r & m) for m in masks]))
            except Exception:
                pass
            time.sleep(0.002)

    def _read_smi(self):
        for line in self.p.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((time.perf_counter(), float(r[0]), float(r[1]), float(r[2]), [x.lower().startswith("active") for x in r[3:7]]))
            except Exception:
                pass

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.p:
            self.p.terminate()
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        if not self.rows:   # the poll never produced a row: one nvidia-smi query right after the region is better than no clock record
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
                r = [x.strip() for x in out.split(",")]
                self.rows.append((t1, float(r[0]), float(r[1]), float(r[2]), [x.lower().startswith("active") for x in r[3:7]]))
                self.source = "nvidia-smi (one query right after the timed region; the in-process poll returned nothing)"
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock poll returned nothing"], "samples": 0, "source": self.source}
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        in_region = len(rows)
        if not rows:    # nothing landed inside (should not happen with the 2 ms poll): nearest samples around the region
            rows = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:4]
        sm = sorted(r[1] for r in rows)
        reasons = sorted({self.NAMES[k] for r in rows for k in range(4) if r[4][k]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": rows[0][2] if rows else None, "reasons": reasons,
                "power_w_max": max((r[3] for r in rows), default=None), "samples": in_region, "samples_total": len(self.rows),
                "source": self.source}


def cpu_baseline(args, occ, zones, a, b, all_threads=True):
    """the reference's CPU path restated (oracle/), timed on a bounded sample of the same workload"""
    from oracle import pyoracle as O
    omap = O.GridMap(occ, zones, [-1.0, -1.0], [1.0, 1.0], O.DOOR, 0.3)
    n = min(args.cpu_sample, len(a))
    sa, sb = np.ascontiguousarray(a[:n]), np.ascontiguousarray(b[:n])
    threads = host_threads() if all_threads else 1
    omap.edge_validity_timed(sa[:100000], sb[:100000], threads)  # warm-up
    out, t = omap.edge_validity_timed(sa, sb, threads)
    n1 = min(n, 400_000)
    _, t1 = omap.edge_validity_timed(sa[:n1], sb[:n1], 1)
    return {"value": n * N_WORLDS / t, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d of the step's edges, oracle C++ restatement (-O3, OpenMP over edges); the Rust reference is single-threaded "
                      "and cannot be built here" % n,
            "value_1thread": n1 * N_WORLDS / t1, "edges_per_s": n / t}, out, omap


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    occ, zones, a, b = make_inputs(args, 0)
    from oracle import pyoracle as O
    omap = O.GridMap(occ, zones, [-1.0, -1.0], [1.0, 1.0], O.DOOR, 0.3)
    threads = host_threads()
    n = len(a)        # a step of the reference arm is the b200 arm's step: all edges_per_gpu_per_step edges (about 1 s on 16 cores)
    sa, sb = a, b
    for _ in range(max(1, min(args.warmup, 2))):
        omap.edge_validity_timed(sa[: n // 4], sb[: n // 4], threads)
    t = 0.0
    for _ in range(args.steps):
        out, dt = omap.edge_validity_timed(sa, sb, threads)
        t += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    value = n * N_WORLDS * args.steps / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "each step = all %d edges of the b200 arm's step through the oracle C++ restatement with OpenMP "
                                       "over edges (reference Rust crate not buildable here: no cargo/rustc; it is single-threaded)" % n},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)



def side_measurements(ctx, pmap, args):
    """kNN queries/s and PRM build ms of BASELINE.json's metric line: V = Q = 1e6 uniform points, radius =
    heuristic_radius(1e6, 0.1, 2.0, 2).  Device time = CUDA-event phases inside the library; e2e = host call with pinned
    outputs; cpu = the oracle's kd-tree / PRM on the box's cores (bounded samples)."""
    import torch
    import po_rrt_b200 as P
    from po_rrt_b200 import synth
    from oracle import pyoracle as O
    ex = {}
    try:
        V = Q = 1_000_000
        pts, qs = synth.points(V, seed=3), synth.points(Q, seed=4)
        r = 2.0 * (np.log(V) / V) ** 0.5
        tree = P.KdTree(ctx, pts, cell_size=r)
        pin_ids = torch.empty(64 * Q, dtype=torch.int32).pin_memory().numpy()
        tree.nearest_neighbors(qs[:1000], r)
        best = None
        for _ in range(3):
            t0 = time.perf_counter(); offs, ids = tree.nearest_neighbors(qs, r, cap=64 * Q, ids_out=pin_ids); t1 = time.perf_counter()
            ph = ctx.last_phase_ms()
            if best is None or t1 - t0 < best[0]:
                best = (t1 - t0, ph)
        ex["radius"] = {"vertices": V, "queries": Q, "radius": r, "hits_per_query": len(ids) / Q,
                        "device_ms": {"search_ids_ascending": best[1][0] + best[1][1], "d2h": best[1][2]},
                        "algorithmic_bytes": 16 * Q + 8 * Q + 4 * len(ids),
                        "algorithmic_gbs": (24 * Q + 4 * len(ids)) / ((best[1][0] + best[1][1]) * 1e-3) / 1e9,
                        "queries_per_s_device": Q / ((best[1][0] + best[1][1]) * 1e-3), "queries_per_s_e2e": Q / best[0],
                        "note": "one-pass tile kernel (merge scripts per cell, lists id-ascending out of the search) + placement copy; "
                                "round 1: 0.68 ms search + 0.68 ms segment sort"}
        best = None
        for _ in range(3):
            t0 = time.perf_counter(); tree.nearest_neighbor(qs); t1 = time.perf_counter()
            ph = ctx.last_phase_ms()
            if best is None or t1 - t0 < best[0]:
                best = (t1 - t0, ph)
        ex["nearest"] = {"queries": Q, "device_ms": best[1][0], "queries_per_s_device": Q / (best[1][0] * 1e-3), "queries_per_s_e2e": Q / best[0]}
        pin_k = torch.empty((Q, 16), dtype=torch.int32).pin_memory().numpy()
        pin_d = torch.empty((Q, 16), dtype=torch.float64).pin_memory().numpy()
        best = None
        for _ in range(2):
            t0 = time.perf_counter(); tree.knn(qs, 16, ids_out=pin_k, dist_out=pin_d); t1 = time.perf_counter()
            ph = ctx.last_phase_ms()
            if best is None or t1 - t0 < best[0]:
                best = (t1 - t0, ph)
        ex["knn16"] = {"queries": Q, "device_ms": best[1][0], "queries_per_s_device": Q / (best[1][0] * 1e-3), "queries_per_s_e2e": Q / best[0]}
        # CPU: the oracle's kd-tree (nearest_neighbor.rs restated) on a sample of the queries
        threads = host_threads()
        t0 = time.perf_counter()
        otree = O.KdTree(pts[0], 0)
        otree.add_batch(pts[1:], 1)
        t_build = time.perf_counter() - t0
        qn = 200_000
        t0 = time.perf_counter(); _, _, tot = otree.radius_batch(qs[:qn], r, cap=64 * qn, threads=threads); t1 = time.perf_counter()
        ex["radius"]["cpu_queries_per_s"] = qn / (t1 - t0)
        t0 = time.perf_counter(); otree.nearest_batch(qs[:qn], threads=threads); t2 = time.perf_counter()
        ex["nearest"]["cpu_queries_per_s"] = qn / (t2 - t0)
        ex["cpu_note"] = "oracle kd-tree (incremental insert %.2f s for 1e6 vertices), %d threads, %d-query sample" % (t_build, threads, qn)
        # PRM build (prm.rs grow_graph): total host call incl. H2D of the samples and D2H of the CSR into pinned memory
        ex["prm_build"] = {}
        pin_pts = torch.from_numpy(pts).pin_memory().numpy()      # e2e from pinned host memory, like the edge arm
        for n_nodes in (10_000, 100_000, 1_000_000):
            pin_col = torch.empty(64 * n_nodes, dtype=torch.int32).pin_memory().numpy()
            pin_row = torch.empty(n_nodes + 1, dtype=torch.int64).pin_memory().numpy()
            best = None
            for _ in range(3):
                prm = P.PRM(pmap)
                t0 = time.perf_counter(); prm.grow_graph(pin_pts[:n_nodes], 0.1, 2.0, col_out=pin_col, row_ptr_out=pin_row); t1 = time.perf_counter()
                if best is None or t1 - t0 < best[0]:
                    best = (t1 - t0, [round(float(x), 3) for x in prm.phase_ms], int(len(prm.col)))
            resident = None
            for _ in range(3):      # the roadmap left on the device (for porrt_sssp_worlds_prm / porrt_edge_validity_csr_i8): no column copy
                prm = P.PRM(pmap)
                t0 = time.perf_counter(); prm.grow_graph(pin_pts[:n_nodes], 0.1, 2.0, fetch_col=False, row_ptr_out=pin_row); t1 = time.perf_counter()
                resident = t1 - t0 if resident is None else min(resident, t1 - t0)
            ex["prm_build"]["V%d" % n_nodes] = {"ms": 1e3 * best[0], "ms_roadmap_left_on_device": 1e3 * resident, "directed_edges": best[2],
                                                "candidate_edge_checks": int(best[1][7]),
                                                "phase_ms[radii,bin,radius,kd_rank,order,edges,csr]": best[1][:7]}
        # re-validating a whole roadmap (e.g. after the map changed): its adjacency goes through porrt_edge_validity_csr_i8,
        # 4 B per edge + 8 B per node in, 1 B per edge out; every edge of a PRM is valid, so every pixel is looked at
        try:
            n_nodes = 1_000_000
            prm = P.PRM(pmap)
            prm.grow_graph(pin_pts[:n_nodes], 0.1, 2.0, col_out=pin_col, row_ptr_out=pin_row)
            n_e = int(pin_row[n_nodes])
            pin_v8 = torch.empty(n_e, dtype=torch.int8).pin_memory().numpy()
            tree = P.KdTree(ctx, pin_pts[:n_nodes], cell_size=r)
            best = None
            for _ in range(3):
                t0 = time.perf_counter(); pmap.transition_validator_adjacency(pin_row[:n_nodes + 1], pin_col[:n_e], vid_out=pin_v8); t1 = time.perf_counter()
                best = t1 - t0 if best is None else min(best, t1 - t0)
            ex["roadmap_revalidation_e2e"] = {"nodes": n_nodes, "directed_edges": n_e, "ms": 1e3 * best, "edges_per_s": n_e / best,
                                              "edge_world_checks_per_s": n_e * N_WORLDS / best, "all_valid": bool((pin_v8 >= 0).all()),
                                              "h2d_bytes": 4 * n_e + 8 * (n_nodes + 1), "d2h_bytes": n_e,
                                              "call": "porrt_edge_validity_csr_i8 (adjacency in, validity ids out)"}
            del tree
        except Exception as e:
            ex["roadmap_revalidation_e2e"] = {"error": repr(e)}
        # plan_qmdp at PRM scale (SURVEY 8(d): SSSP per world on the roadmap the builder just left on the device): 1e6 nodes x 64
        # worlds, 4 final nodes per world; nothing but the final lists goes in, the 512 MB table stays on the device
        try:
            n_nodes = 1_000_000
            prm = P.PRM(pmap)
            prm.grow_graph(pin_pts[:n_nodes], 0.1, 2.0, col_out=pin_col, row_ptr_out=pin_row)
            n_e = int(pin_row[n_nodes])
            rng = np.random.default_rng(9)
            finals = [rng.choice(n_nodes, 4, replace=False).tolist() for _ in range(N_WORLDS)]
            best = None
            for _ in range(2):
                t0 = time.perf_counter(); _, rounds = P.dijkstra_worlds_resident_prm(pmap, n_nodes, finals, want_dist=False); t1 = time.perf_counter()
                ph = ctx.last_phase_ms()[:2]
                if best is None or t1 - t0 < best[0]:
                    best = (t1 - t0, ph, rounds)
            pairs = float(best[1][1])
            ex["qmdp_prm_scale"] = {"nodes": n_nodes, "directed_edges": n_e, "worlds": N_WORLDS, "finals_per_world": 4,
                                    "ms": 1e3 * best[0], "device_ms": best[1][0], "rounds": int(best[2]),
                                    "parent_world_pairs": pairs, "full_sweep_pairs": float(n_e) * N_WORLDS,
                                    "equivalent_full_sweeps": pairs / (float(n_e) * N_WORLDS),
                                    "gather_bytes": pairs * 32.0, "gather_gbs": pairs * 32.0 / (best[1][0] * 1e-3) / 1e9 if best[1][0] > 0 else None,
                                    "call": "porrt_sssp_worlds_prm (frontier relaxation over the [node][world] table in global memory, "
                                            "sssp_frontier.cu); gather_bytes = one 32-byte sector of the value table per (parent, world) pair",
                                    "cpu_note": "the reference runs one heap dijkstra per world: 64 x (1e6 nodes, 5.3e7 edges) single-threaded"}
        except Exception as e:
            import traceback
            ex["qmdp_prm_scale"] = {"error": repr(e) + " | " + traceback.format_exc()[-300:]}
        omap = O.GridMap(pmap.occ, pmap.zones, [-1.0, -1.0], [1.0, 1.0], O.DOOR, 0.3)
        for n_nodes in (10_000, 100_000):
            oprm = O.PRM(omap, [-1.0, -1.0], [1.0, 1.0], seed=0)
            oprm.init(pts[0])
            ex["prm_build"]["V%d" % n_nodes]["cpu_ms_1thread"] = 1e3 * oprm.add_samples(pts[1:n_nodes], 0.1, 2.0)
    except Exception as e:  # side numbers must never take the headline down
        import traceback
        ex["error"] = repr(e) + " | " + traceback.format_exc()[-400:]
    try:
        ex["refiner"] = refiner_measurement(ctx, pmap)
    except Exception as e:
        import traceback
        ex["refiner"] = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
    try:
        ex["mmprm_z6"] = mmprm_measurement(ctx)
    except Exception as e:
        import traceback
        ex["mmprm_z6"] = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
    try:
        ex["belief_c3"] = belief_measurement(ctx)
    except Exception as e:
        import traceback
        ex["belief_c3"] = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
    try:
        ex["belief_c4"] = belief_measurement(ctx, Z=12, visibility=0.2, max_step=0.05, search_radius=5.0, check="sweeps")
    except Exception as e:
        import traceback
        ex["belief_c4"] = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
    return ex


def multi_gpu_measurements(ctx, pmap, rank, world, dev):
    """N > 1 only, called by EVERY rank (collective): the other two BASELINE metrics at N GPUs.
    NN queries: vertex set replicated, 1e6 queries per rank (weak scaling, no data-path collective), device ms = max over ranks.
    PRM build: ONE roadmap of 1e6 samples built by all ranks together (strong scaling): sharded radius + edge batches, NCCL
    all-gather of the valid pairs, CSR assembled on every rank (csrc/comm.cu, graph.cu)."""
    import torch
    import torch.distributed as dist
    import po_rrt_b200 as P
    from po_rrt_b200 import shard, synth
    out = {}

    def rmax(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    V = Q = 1_000_000
    pts, qs = synth.points(V, seed=3), synth.points(Q, seed=4 + rank)
    r = 2.0 * (np.log(V) / V) ** 0.5
    tree = P.KdTree(ctx, pts, cell_size=r)
    pin_ids = torch.empty(64 * Q, dtype=torch.int32).pin_memory().numpy()
    pin_k = torch.empty((Q, 16), dtype=torch.int32).pin_memory().numpy()
    pin_d = torch.empty((Q, 16), dtype=torch.float64).pin_memory().numpy()
    tree.nearest_neighbors(qs[:1000], r)
    res = {}
    for name, call, n_ph in (("radius", lambda: tree.nearest_neighbors(qs, r, cap=64 * Q, ids_out=pin_ids), 2),
                             ("nearest", lambda: tree.nearest_neighbor(qs), 1),
                             ("knn16", lambda: tree.knn(qs, 16, ids_out=pin_k, dist_out=pin_d), 1)):
        best = None
        for _ in range(3):
            dist.barrier()
            t0 = time.perf_counter(); call(); t1 = time.perf_counter()
            dms, wall = rmax(sum(ctx.last_phase_ms()[:n_ph])), rmax(t1 - t0)
            if best is None or dms < best[0]:
                best = (dms, wall)
        res[name] = {"queries_per_rank": Q, "device_ms_max": best[0], "queries_per_s_device": Q * world / (best[0] * 1e-3),
                     "queries_per_s_e2e": Q * world / best[1]}
    out["nn"] = res

    # replicas: every rank builds its own roadmap (its own sample stream) at the same time -- how independent planning problems
    # / seeds scale (weak); ms = max over ranks for one roadmap each
    pin_col = torch.empty(64 * V, dtype=torch.int32).pin_memory().numpy()
    pin_row = torch.empty(V + 1, dtype=torch.int64).pin_memory().numpy()
    my_pts = torch.from_numpy(synth.points(V, seed=30 + rank)).pin_memory().numpy()
    pts = torch.from_numpy(pts).pin_memory().numpy()
    best = None
    for _ in range(3):
        dist.barrier()
        prm = P.PRM(pmap)
        t0 = time.perf_counter(); prm.grow_graph(my_pts, 0.1, 2.0, col_out=pin_col, row_ptr_out=pin_row); t1 = time.perf_counter()
        wall = rmax(t1 - t0)
        if best is None or wall < best:
            best = wall
    out["prm_build_replicas"] = {"V": V, "roadmaps": world, "ms_max_over_ranks": 1e3 * best, "roadmaps_per_s": world / best,
                                 "scaling": "weak"}

    shard.init_comm(ctx)
    best = None
    for _ in range(3):
        dist.barrier()
        prm = P.PRM(pmap)
        t0 = time.perf_counter(); prm.grow_graph(pts, 0.1, 2.0, col_out=pin_col, fetch_col=(rank == 0), row_ptr_out=pin_row); t1 = time.perf_counter()
        wall = rmax(t1 - t0)
        if best is None or wall < best[0]:
            best = (wall, [round(float(x), 3) for x in prm.phase_ms[:7]], ctx.last_phase_ms()[:1], int(prm.row_ptr[-1]))
    resident = None
    for _ in range(3):
        dist.barrier()
        prm = P.PRM(pmap)
        t0 = time.perf_counter(); prm.grow_graph(pts, 0.1, 2.0, fetch_col=False, row_ptr_out=pin_row); t1 = time.perf_counter()
        wall = rmax(t1 - t0)
        resident = wall if resident is None else min(resident, wall)
    out["prm_build_sharded"] = {"V": V, "ms_max_over_ranks": 1e3 * best[0], "ms_roadmap_left_on_device": 1e3 * resident,
                                "directed_edges": best[3], "exchange_ms": best[2],
                                "phase_ms_rank0[radii,bin,radius,kd_rank,order,edges,csr]": best[1], "scaling": "strong",
                                "note": "one roadmap built by all ranks; bins, kd ranks and the CSR assembly are replicated, "
                                        "radius + order + edge batches are sharded; the CSR ends device-resident on every rank, "
                                        "rank 0 alone copies the column array to the host"}
    # belief-space planning at the config-4 shape: the columns of every belief level are sharded over the ranks and all-gathered
    # before the next level reads them (graph.cu / colsolve.cu); every rank ends with the whole table
    try:
        prob = belief_problem(12, 0.2, 0.05, 5.0)
        dist.barrier()
        plan, best, _ = belief_run(ctx, prob)
        wall, dev_ms = rmax(best[0]), rmax(best[2][0])
        solo = P.Context(dev.index)
        try:
            ref_plan, ref_best, _ = belief_run(solo, prob, reps=2)
            same = bool(np.array_equal(ref_plan.dist, plan.dist))
        finally:
            solo.close()
        tsame = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(tsame, op=dist.ReduceOp.MIN)
        out["belief_c4_sharded"] = {"nodes": int(plan.dist.shape[0]), "beliefs": int(plan.dist.shape[1]), "ms_max_over_ranks": 1e3 * wall,
                                    "backups_device_ms_max": dev_ms, "single_gpu_ms_rank0": 1e3 * ref_best[0],
                                    "single_gpu_backups_device_ms": ref_best[2][0],
                                    "phase_ms_rank0[tables,upload+types,backups,result]": [round(x, 3) for x in best[1]],
                                    "bit_exact_vs_single_gpu_all_ranks": bool(tsame.item() == 1.0), "scaling": "strong"}
    except Exception as e:
        import traceback
        out["belief_c4_sharded"] = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
    ctx.comm_destroy()
    return out


def refiner_measurement(ctx, pmap, n_pieces=64, n_states=30, n_iterations=1000):
    """PTOPolicyRefiner::partial_shortcut (SURVEY 8(f) rank 1) on the c5 map: n_pieces jagged path pieces (random walks through
    free space), n_iterations trials each; the device runs the trials of all pieces in shared speculative waves, the oracle runs
    them one by one like the reference.  States and commit counts must be identical."""
    from oracle import pyoracle as O
    rng = np.random.default_rng(12)
    omap = O.GridMap(pmap.occ, pmap.zones, [-1.0, -1.0], [1.0, 1.0], O.DOOR, 0.3)
    pieces = []
    while len(pieces) < n_pieces:
        starts = rng.uniform(-0.9, 0.9, (4000, 1, 2))
        walks = np.clip(starts + np.cumsum(rng.uniform(-0.01, 0.01, (4000, n_states, 2)), 1), -0.99, 0.99)
        a, b = walks[:, :-1].reshape(-1, 2), walks[:, 1:].reshape(-1, 2)
        ok = (pmap.transition_validator(np.ascontiguousarray(a), np.ascontiguousarray(b)) >= 0).reshape(4000, n_states - 1).all(1)
        ok &= (pmap.state_validity(np.ascontiguousarray(walks[:, 0])) >= 0)
        pieces += [w for w in walks[ok]][: n_pieces - len(pieces)]
    rows = np.ones((n_pieces, pmap.n_validities), np.uint8)
    pmap.partial_shortcut_batch(pieces, rows, n_iterations)   # warm-up at full size: pinned / device staging is allocated here
    t0 = time.perf_counter(); got, commits, waves = pmap.partial_shortcut_batch(pieces, rows, n_iterations); t_gpu = time.perf_counter() - t0
    t0 = time.perf_counter()
    want = [omap.refiner_partial_shortcut(p, rows[k], n_iterations) for k, p in enumerate(pieces)]
    t_cpu = time.perf_counter() - t0
    exact = all(np.array_equal(got[k], want[k][0]) and commits[k] == want[k][1] for k in range(n_pieces))
    return {"pieces": n_pieces, "states_per_piece": n_states, "trials_per_piece": n_iterations, "device_round_trips": int(waves),
            "commits": int(commits.sum()), "gpu_ms": 1e3 * t_gpu, "cpu_oracle_ms_1thread": 1e3 * t_cpu, "bit_exact": bool(exact)}


def belief_problem(Z, visibility, max_step, search_radius, n_min=5000):
    """the PTO roadmap of a BASELINE config-3 / config-4 shaped problem on a stand-in shelf map, grown by the oracle (sequential
    growth is out of scope, SURVEY 8)"""
    from po_rrt_b200 import synth
    from oracle import pyoracle as O
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    low, up = [-1.0, -1.0], [1.0, 1.0]
    omap = O.GridMap(occ, zones, low, up, O.SHELF, visibility)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    pto = O.PTO(omap, low, up, seed=0)
    t0 = time.perf_counter(); rc = pto.grow_graph((0.0, -0.9), O.SquareGoal(goals, 0.05), max_step, search_radius, n_min, 100000); t_grow = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError("roadmap growth failed (rc %d)" % rc)
    return {"occ": occ, "zones": zones, "low": low, "up": up, "visibility": visibility, "pto": pto, "Z": Z, "grow_ms": 1e3 * t_grow}


def belief_run(ctx, prob, reps=3, copy=None):
    """plan_belief_space on the device: reachable beliefs + visibility + implicit belief graph + value backups + policy;
    best of `reps` wall times, the phases of the best run and the column solver's device counters.  copy=None: what the planner
    needs -- the policy and its expected cost; the V x B table stays on the device and is fetched afterwards for the checks."""
    import po_rrt_b200 as P
    pmap = P.MapShelfDomain(ctx, prob["occ"], prob["low"], prob["up"])
    pmap.add_zones(prob["zones"], prob["visibility"])
    pto, Z = prob["pto"], prob["Z"]
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    fm = P.words_from_bits(fin_bits)
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, [1.0 / Z] * Z, fin_ids, fm, copy=copy)
        t = time.perf_counter() - t0
        if best is None or t < best[0]:
            best = (t, [float(x) for x in plan.phase_ms], list(ctx.last_phase_ms()[:2]))
    if plan.dist is None:
        t0 = time.perf_counter(); plan.fetch_table(); best = best + (1e3 * (time.perf_counter() - t0),)
    return plan, best, (xy, nvid, rp, col, ev, fin_ids, fm, pmap)


def belief_measurement(ctx, Z=8, n_min=5000, visibility=0.5, max_step=0.1, search_radius=2.0, check="oracle"):
    """BASELINE config 3 (8 goal zones, B = 255 beliefs; main.rs:757-799) / config 4 (12 zones, B = 4095; main.rs:386-411) shapes on a
    stand-in shelf map: belief-space planning = implicit belief graph + value backups on the device (rows C2-C4).  check = "oracle":
    against the oracle's materialised belief graph + conditional_dijkstra, bit for bit (config 4 is intractable there, main.rs:385);
    check = "sweeps": against the library's second, independent schedule (order-free sweeps over the table in global memory)."""
    import po_rrt_b200 as P
    prob = belief_problem(Z, visibility, max_step, search_radius, n_min)
    plan, best, (xy, nvid, rp, col, ev, fin_ids, fm, pmap) = belief_run(ctx, prob)
    V, E, B = len(nvid), len(col), len(plan.beliefs)
    out = {"zones": Z, "nodes": V, "directed_edges": E, "beliefs": B, "belief_nodes": V * B, "rounds_max": int(plan.sweeps),
           "gpu_ms_total": 1e3 * best[0],
           "gpu_phase_ms[tables,upload+types,backups,result]": [round(x, 3) for x in best[1]],
           "call": "plan_belief_space: porrt_reachable_belief_states + porrt_visibility + porrt_belief_vi + porrt_extract_policy -> "
                   "the policy and its expected cost; the V*B table stays on the device (the policy walk fetches the value columns it "
                   "visits) and comes over on demand through porrt_belief_result",
           "table_fetch_ms": round(best[3], 3) if len(best) > 3 else None,
           "roadmap_growth_cpu_ms": round(prob["grow_ms"], 1)}
    dev_ms, offers = best[2]
    if dev_ms and dev_ms > 0:
        out["backups_device"] = {"ms": dev_ms, "edge_records": int(offers), "l2_bytes": int(offers) * 12,
                                 "l2_gbs": offers * 12 / (dev_ms * 1e-3) / 1e9,
                                 "full_sweep_records": E * B, "equivalent_full_sweeps": offers / float(E * B),
                                 "note": "on-chip column solver (colsolve.cu): a record = one 12-byte (parent, validity id, cost) entry of "
                                         "the transposed adjacency read from L2 when a node's value improved; the value table never "
                                         "leaves shared memory between the first and the last round of a column"}
    if check == "oracle":
        pto = prob["pto"]
        b0 = [1.0 / Z] * Z
        t0 = time.perf_counter(); pto.build_belief_graph(b0); t_build = time.perf_counter() - t0
        t0 = time.perf_counter(); want = pto.compute_expected_costs_to_goals(); t_dp = time.perf_counter() - t0
        t0 = time.perf_counter(); opol = pto.extract_policy(); t_pol = time.perf_counter() - t0
        out["cpu_oracle_ms[build_belief_graph,conditional_dijkstra,extract_policy]"] = [round(1e3 * t_build, 1), round(1e3 * t_dp, 1), round(1e3 * t_pol, 2)]
        out["bit_exact"] = bool(np.array_equal(plan.dist.reshape(-1), want) and
                                np.array_equal(plan.policy_node.astype(np.int64) * B + plan.policy_belief, opol.original))
        # the run's last step in the reference (main.rs:442): refine_solution(PartialShortCut(1500))
        P.refine_policy_shortcut(ctx, plan, 1500)
        t0 = time.perf_counter(); ref = P.refine_policy_shortcut(ctx, plan, 1500); t_ref = time.perf_counter() - t0
        t0 = time.perf_counter(); oref = pto.refine_policy_shortcut(1500); t_oref = time.perf_counter() - t0
        out["refine_shortcut_1500"] = {"gpu_ms": 1e3 * t_ref, "cpu_oracle_ms_1thread": 1e3 * t_oref, "pieces_nodes": int(len(ref["node"])),
                                       "commits": int(ref["commits"]), "expected_cost_before": float(plan.expected_cost),
                                       "expected_cost_after": float(ref["expected_cost"]),
                                       "bit_exact": bool(ref["xy"].tobytes() == oref.xy.tobytes() and ref["expected_cost"] == oref.expected_costs)}
        # the other strategy (main.rs:221,270): refine_solution(Reparent(0.3)) -- every candidate transition of every tree in one device batch
        P.refine_policy_reparent(ctx, plan, 0.3)
        t0 = time.perf_counter(); rep = P.refine_policy_reparent(ctx, plan, 0.3); t_rep = time.perf_counter() - t0
        t0 = time.perf_counter(); orep = pto.refine_policy_reparent(0.3); t_orep = time.perf_counter() - t0
        out["refine_reparent_0.3"] = {"gpu_ms": 1e3 * t_rep, "cpu_oracle_ms_1thread": 1e3 * t_orep, "tree_nodes": int(rep["tree_nodes"]),
                                      "transitions_checked": int(rep["transitions"]), "policy_nodes_after": int(len(rep["node"])),
                                      "bit_exact": bool(rep["xy"].tobytes() == orep.xy.tobytes() and np.array_equal(rep["parent"], orep.parent) and
                                                        rep["expected_cost"] == orep.expected_costs)}
    else:
        keep = plan.dist.copy()
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 1)
        try:
            t0 = time.perf_counter()
            other = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, [1.0 / Z] * Z, fin_ids, fm, copy=False)
            same_policy = bool(np.array_equal(other.policy_node, plan.policy_node) and np.array_equal(other.policy_belief, plan.policy_belief) and
                               other.expected_cost == plan.expected_cost)
            out["global_sweeps_ms_total"] = 1e3 * (time.perf_counter() - t0)
            out["global_sweeps_phase_ms"] = [round(float(x), 3) for x in other.phase_ms]
            out["global_sweeps"] = int(other.sweeps)
        finally:
            ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
        out["bit_exact_vs_global_sweeps"] = bool(np.array_equal(other.dist, keep)) and same_policy
    return out

_REAL_STDOUT = None


def mmprm_measurement(ctx, Z=6, n_iter=2500):
    """multi-modal PRM (SURVEY 8(f) rank 3; map_shelves_tamp_prm.rs test shape :539-552: 6 shelves, plan(.., 0.1, 2.0, 2500)): the oracle
    runs the reference algorithm (and so decides the RNG schedule), the product rebuilds all mode PRMs + belief graph + expected
    costs on the GPU from the schedule"""
    import po_rrt_b200 as P
    from po_rrt_b200 import synth
    from oracle import pyoracle as O
    occ, zones = synth.shelf_map(200, n_zones=Z)
    low, up = [-1.0, -1.0], [1.0, 1.0]
    omap = O.GridMap(occ, zones, low, up, O.SHELF, 0.5)
    smap = P.MapShelfDomain(ctx, occ, low, up)
    smap.add_zones(zones, 0.5)
    tamp = O.TampPRM(omap, low, up)
    opol = tamp.plan((0.0, -0.9), [1.0 / Z] * Z, 0.1, 2.0, n_iter)
    sch = tamp.schedule()
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        dist, graph, pol, phase = P.mmprm_plan(smap, sch)
        t = time.perf_counter() - t0
        if best is None or t < best[0]:
            best = (t, [round(float(x), 3) for x in phase[:3]], [round(float(x), 3) for x in ctx.last_phase_ms()[:7]])
    exact = bool(np.array_equal(dist, sch["expected_costs"]) and np.array_equal(pol[0].astype(np.int64), opol.original))
    return {"zones": Z, "modes": int(len(sch["mode_belief_id"])), "prm_nodes_total": int(len(sch["samples"])),
            "belief_graph_edges": int(len(graph.col)), "sweeps": int(graph.sweeps), "gpu_ms_total": 1e3 * best[0],
            "gpu_phase_ms[prm builds,graph assembly,value backups]": best[1],
            "prm_phase_ms[radii,bin,radius,kd_rank,order,edges,csr]": best[2],
            "cpu_oracle_ms[grow_mm_prm,build_belief_graph,conditional_dijkstra,extract_policy]": [round(1e3 * float(x), 1) for x in tamp.seconds],
            "bit_exact": exact}


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was diverted to stderr"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def host_threads():
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm must still use the box's cores
    return max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import po_rrt_b200 as P
    from po_rrt_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: po_rrt_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = P.Context(local_rank)
    # host locality: this process's pinned buffers and copy-issuing thread sit on the NUMA node next to its GPU
    # (N ranks on a two-socket box otherwise push their H2D / D2H through the socket interconnect); undone before the CPU baseline
    affinity0 = os.sched_getaffinity(0)
    numa_node = ctx.bind_host_thread() if world > 1 else -1
    occ, zones, a, b = make_inputs(args, rank)
    pmap = P.Map(ctx, occ, [-1.0, -1.0], [1.0, 1.0])
    pmap.add_zones(zones, 0.3)
    assert pmap.n_worlds() == N_WORLDS
    E = args.edges

    # ---- device-resident arm
    stream = torch.cuda.Stream(device=dev)  # a real (non-default) stream: kernels and the timing events share it
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    d_a, d_b = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)
    d_vid = torch.empty(E, dtype=torch.int32, device=dev)
    d_mask = torch.empty(E, dtype=torch.int64, device=dev)
    lib, h = ctx.lib, ctx.h

    def step_dev():
        ctx.check(lib.porrt_edge_validity_dev(h, d_a.data_ptr(), d_b.data_ptr(), E, d_vid.data_ptr(), d_mask.data_ptr()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    for _ in range(args.warmup):
        step_dev()
    barrier()
    launches0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        step_dev()
    ev1.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = ctx.launch_count() - launches0
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = E * world * N_WORLDS * args.steps / (ms_max * 1e-3)

    # algorithmic bytes of one launch (SURVEY 8(d)): 32 B endpoints + 8 B mask + 4 B id + 1 B per line pixel
    ppm = args.map_size / 2.0
    ai = torch.floor((args.map_size - 1) - (d_a[:, 1] + 1.0) * ppm); aj = torch.floor((d_a[:, 0] + 1.0) * ppm)
    bi = torch.floor((args.map_size - 1) - (d_b[:, 1] + 1.0) * ppm); bj = torch.floor((d_b[:, 0] + 1.0) * ppm)
    n_px = float((torch.maximum((ai - bi).abs(), (aj - bj).abs()) + 1).sum().item())
    del ai, aj, bi, bj
    alg_bytes = 44.0 * E + n_px
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    kernel_s = ms / args.steps * 1e-3
    achieved = alg_bytes / kernel_s / 1e9
    traffic, pipes = None, None  # dram bytes / pipe utilisation of one launch, from the committed ncu capture of this command
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "edge_traffic.json")))
        if tr["edges_per_launch"] == E and args.map_size == 8192:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            pipes = tr.get("pipes")
    except Exception:
        pass
    # the L2-resident gather rate (SURVEY 8(d): "an L2 peak the builder must measure"): random independent 32-byte sector reads
    # over a 64 MiB buffer, measured here and now on this GPU
    l2_peak = C.c_double()
    ctx.check(lib.porrt_measure_l2_gather(h, 64 << 20, C.byref(l2_peak)))
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "algorithmic_bytes_per_launch": alg_bytes, "mean_pixels_per_edge": n_px / E,
                "kernel": "edge_validity_v3_kernel<DOOR,false>",
                "hbm_streams": {"achieved": 44.0 * E / kernel_s / 1e9, "frac": 44.0 * E / kernel_s / 1e9 / peak,
                                "note": "the 32 B in + 12 B out per edge that actually cross HBM"},
                "l2": {"achieved": n_px / kernel_s / 1e9, "peak": l2_peak.value, "unit": "GB/s", "frac": n_px / kernel_s / 1e9 / l2_peak.value,
                       "note": "pixel bytes (1 B per line pixel) per second against the measured rate of random 32-byte sector reads "
                               "from a 64 MiB L2-resident buffer (porrt_measure_l2_gather)"},
                "bound_note": "algorithmic bytes / kernel time against the HBM peak (SURVEY 8(d)); measured DRAM traffic ~ the 44 B/edge "
                              "streams: the pixels are served by the class plane in shared memory and L2-resident bitmaps, the kernel "
                              "is bound by integer issue (profiles/: ncu pipe utilisation)",
                "ncu_pipes": pipes, "kernel_ms": ms / args.steps}

    # ---- end-to-end arms: HOST (pinned) buffers through the C ABI, H2D + kernel + D2H inside the timed region.
    # The headline `e2e` is the call the planners make -- transition_validator(&PTONode, &PTONode) -> Option<usize>
    # (pto_graph.rs:133-139, call sites pto.rs:105 / prm.rs:93) batched: the nodes' states are resident on the device like a
    # roadmap's vertices (uploaded once, outside the timed region), an edge is a pair of node ids in and one validity id out.
    # `e2e_variants` holds the other shapes of the same call, down to raw coordinates with per-world bitvecs out.
    ctx.set_stream(None)
    h_a, h_b = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    h_vid = torch.empty(E, dtype=torch.int32).pin_memory()
    h_mask = torch.empty(E, dtype=torch.int64).pin_memory()
    h_vid8 = torch.empty(E, dtype=torch.int8).pin_memory()
    h_fi = torch.arange(0, E, dtype=torch.int32).pin_memory()
    h_ti = torch.arange(E, 2 * E, dtype=torch.int32).pin_memory()
    want_vid = d_vid.cpu()
    want_mask = d_mask.cpu()
    if args.dump_outputs and rank == 0:      # nothing after the timed loop has written d_vid / d_mask: the last step's results
        dump_outputs(args.dump_outputs, want_vid.numpy(), want_mask.numpy())
    del d_a, d_b, d_vid, d_mask
    torch.cuda.empty_cache()
    tree = P.KdTree(ctx, np.concatenate([a, b]), cell_size=0.01)        # the vertex set: 2E node states, resident

    def run_e2e(call, check):
        call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            call()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        check()
        return E * world * N_WORLDS * e2e_steps / float(t.item())

    def chk32():
        assert torch.equal(h_vid, want_vid), "e2e result differs from the device-resident one"

    def chk8():
        assert torch.equal(h_vid8.to(torch.int32), want_vid), "e2e byte result differs from the device-resident one"

    def chk32m():
        chk32()
        assert torch.equal(h_mask, want_mask)

    e2e_steps = max(2, min(args.steps, 5))
    variants = {}
    specs = [("node_ids_in__validity_id_out", 8, 1, chk8,
              lambda: ctx.check(lib.porrt_edge_validity_indexed_i8(h, h_fi.data_ptr(), h_ti.data_ptr(), E, h_vid8.data_ptr()))),
             ("coordinates_in__id_and_world_mask_out", 32, 12, chk32m,
              lambda: ctx.check(lib.porrt_edge_validity(h, h_a.data_ptr(), h_b.data_ptr(), E, h_vid.data_ptr(), h_mask.data_ptr()))),
             ("coordinates_in__validity_id_out", 32, 1, chk8,
              lambda: ctx.check(lib.porrt_edge_validity_i8(h, h_a.data_ptr(), h_b.data_ptr(), E, h_vid8.data_ptr()))),
             ("node_ids_in__id_and_world_mask_out", 8, 12, chk32m,
              lambda: ctx.check(lib.porrt_edge_validity_indexed(h, h_fi.data_ptr(), h_ti.data_ptr(), E, h_vid.data_ptr(), h_mask.data_ptr())))]
    if args.no_extras:
        specs = specs[:2]
    for name, bi_, bo_, check, call in specs:
        h_vid.zero_(); h_vid8.zero_(); h_mask.zero_()
        v = run_e2e(call, check)
        variants[name] = {"value": v, "unit": UNIT, "edges_per_s": v / N_WORLDS, "h2d_bytes_per_step": bi_ * E, "d2h_bytes_per_step": bo_ * E}
    e2e_main = variants["node_ids_in__validity_id_out"]
    e2e_value = e2e_main["value"]

    # N > 1: how the end-to-end path scales on this host -- the same call by rank 0 ALONE (the others wait), against all ranks at once
    e2e_scaling = None
    if world > 1:
        solo = None
        dist.barrier()
        if rank == 0:
            specs[0][4]()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                specs[0][4]()
            torch.cuda.synchronize()
            solo = E * N_WORLDS * e2e_steps / (time.perf_counter() - t0)
        dist.barrier()
        if rank == 0:
            e2e_scaling = {"one_rank_alone": solo, "all_ranks_together": e2e_value, "efficiency": e2e_value / (world * solo),
                           "note": "same box, same call (node ids in, validity id out); the ranks share the host's PCIe root / memory"}
    del tree

    multi = None
    if world > 1 and not args.no_extras:
        try:
            multi = multi_gpu_measurements(ctx, pmap, rank, world, dev)
        except Exception as e:  # side numbers must never take the headline down (a failed rank leaves the others to NCCL's timeout)
            import traceback
            multi = {"error": repr(e) + " | " + traceback.format_exc()[-400:]}
        if rank == 0 and isinstance(multi, dict):
            multi["e2e_scaling"] = e2e_scaling

    # ---- batch-size sweep of the device-resident kernel (BASELINE config 5 names 1e6 - 1e8 edge checks)
    sizes = None
    if not args.no_extras:
        try:
            sizes = {}
            for n_e in (1_000_000, 100_000_000):
                sa, sb = synth.edges(n_e, seed=50 + rank)
                da, db = torch.from_numpy(sa).to(dev), torch.from_numpy(sb).to(dev)
                dv = torch.empty(n_e, dtype=torch.int32, device=dev)
                dm = torch.empty(n_e, dtype=torch.int64, device=dev)
                torch.cuda.set_stream(stream)
                ctx.set_stream(stream.cuda_stream)
                reps = 20 if n_e <= 1_000_000 else 3
                for _ in range(2):
                    ctx.check(lib.porrt_edge_validity_dev(h, da.data_ptr(), db.data_ptr(), n_e, dv.data_ptr(), dm.data_ptr()))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(reps):
                    ctx.check(lib.porrt_edge_validity_dev(h, da.data_ptr(), db.data_ptr(), n_e, dv.data_ptr(), dm.data_ptr()))
                e1.record(stream)
                torch.cuda.synchronize()
                t_ms = e0.elapsed_time(e1) / reps
                sizes["E%d" % n_e] = {"ms": t_ms, "edges_per_s": n_e / (t_ms * 1e-3), "value": n_e * N_WORLDS / (t_ms * 1e-3), "unit": UNIT}
                ctx.set_stream(None)
                del da, db, dv, dm, sa, sb
                torch.cuda.empty_cache()
        except Exception as e:
            sizes = {"error": repr(e)}

    line = None
    os.sched_setaffinity(0, affinity0)
    if rank == 0:
        base, oracle_vid, _ = cpu_baseline(args, occ, zones, a, b)
        n = len(oracle_vid)
        assert np.array_equal(want_vid.numpy()[:n].astype(np.int64), oracle_vid), "GPU result differs from the oracle"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": workload_config(args),
                "edges_per_s": value / N_WORLDS,
                "roofline": roofline, "cpu_baseline": base,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 8 * E, "d2h_bytes_per_step": 1 * E,
                        "steps": e2e_steps, "edges_per_s": e2e_value / N_WORLDS,
                        "call": "porrt_edge_validity_indexed_i8: transition_validator(&PTONode, &PTONode) -> Option<usize> batched over "
                                "pinned host buffers -- node-id pairs in, one validity id out; node states resident on the device "
                                "(uploaded once, outside the timed region, like a roadmap's vertices)"},
                "e2e_variants": variants,
                "gpu_launches": int(launches), "clocks": clocks, "parity_checked_edges": n}

    # ---- side measurements of the other BASELINE metrics (kNN queries/s, PRM build ms); not part of `value`
    if rank == 0 and not args.no_extras:
        line["extras"] = side_measurements(ctx, pmap, args)
        line["extras"]["edge_batch_sizes_device"] = sizes
        line["extras"]["host_numa_node_rank0"] = numa_node
        if multi is not None:
            line["extras"]["multi_gpu"] = multi
    if rank == 0:
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
