"""The value-column driver (graph.cu) at the edges of its two schedules: every colsolve_push_kernel<C, MODE> instantiation with a full
and a partly filled last CTA, both sides of every shared-memory band of the column solver, both worklist overflow paths (the column
solver's COLSOLVE_QCAP queue, the frontier relaxation's push list) and degenerate roadmaps.  World columns against the oracle's
dijkstra over PTOGraphWorldView (pto_graph.rs:245-303), belief columns against the oracle's materialised belief graph
(pto.rs:185-275), bit for bit; every case once on the schedule the driver picks and once on the frontier relaxation
(OPT_FORCE_GLOBAL_SWEEPS)."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

COLSOLVE_SMEM_MAX = 227 * 1024   # colsolve.cuh
COLSOLVE_QCAP = 1024
FRONTIER_LAUNCHES_PER_LEVEL = 32   # sf_relax: two kernels per round, the host looks back every 16 rounds


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def colsolve_schedule(V, n_columns, sm_count, E=0, n_validities=1):
    """The host rule of colsolve_fits and colsolve_level (colsolve.cu:256-287) for one level of n_columns columns ->
    (on_chip, C, columns of the last CTA); (False, None, None) when the driver takes the frontier relaxation."""
    fits = 0 < V <= 65535 and E < 2 ** 32 and n_validities <= 256 and V * 9 + 280 + COLSOLVE_QCAP * 2 <= COLSOLVE_SMEM_MAX
    if not fits:
        return False, None, None
    cap = (COLSOLVE_SMEM_MAX - 280 - COLSOLVE_QCAP * 2 - V) // (V * 8)
    cmax = 6 if cap >= 6 else 4 if cap >= 4 else 2 if cap >= 2 else 1
    waves = -(-n_columns // (cmax * sm_count))
    want = -(-n_columns // (waves * sm_count))
    C = min(1 if want <= 1 else 2 if want <= 2 else 4 if want <= 4 else 6, cmax)
    return True, C, n_columns - (-(-n_columns // C) - 1) * C


def _csr(V, src, dst):
    order = np.lexsort((dst, src))
    row_ptr = np.concatenate([[0], np.cumsum(np.bincount(src, minlength=V))]).astype(np.int64)
    return row_ptr, np.ascontiguousarray(dst[order], np.int32)


def _pairs(xy, radius):
    """every pair of points at most `radius` apart, once"""
    p = cKDTree(xy).query_pairs(radius, output_type="ndarray")
    return p[:, 0], p[:, 1]


def _roadmap(xy, radius):
    """every pair of points at most `radius` apart, both directions, as CSR"""
    a, b = _pairs(xy, radius)
    return _csr(len(xy), np.concatenate([a, b]), np.concatenate([b, a]))


def _radius(V, degree):
    """the radius that gives `degree` neighbours on average to V uniform points in [-1, 1]^2"""
    return math.sqrt(4.0 * degree / (math.pi * V))


def _oracle_graph(xy, row_ptr, col, nvid, bits):
    og = O.PTOGraph(validities=bits)
    for k in range(len(xy)):
        og.add_node(xy[k], int(nvid[k]))
    src = np.repeat(np.arange(len(xy)), np.diff(row_ptr))
    for u, v in zip(src.tolist(), col.tolist()):
        og.add_edge(u, v, 0)
    return og


def _world_oracle(xy, row_ptr, col, nvid, bits, finals):
    og = _oracle_graph(xy, row_ptr, col, nvid, bits)
    return np.stack([og.dijkstra(f, world=w) if len(f) else np.full(len(xy), np.inf) for w, f in enumerate(finals)])


def _plain_oracle(xy, row_ptr, col, finals):
    og = _oracle_graph(xy, row_ptr, col, np.zeros(len(xy), np.int32), np.ones((1, 1), np.uint8))
    return og.dijkstra(finals) if len(finals) else np.full(len(xy), np.inf)


def _launches(ctx, force, call):
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, force)
    try:
        n0 = ctx.launch_count()
        out = call()
        return out, ctx.launch_count() - n0
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)


def _check_schedule(launches, on_chip, levels=1):
    """an on-chip level is one launch of the column solver; a frontier level is at least FRONTIER_LAUNCHES_PER_LEVEL launches"""
    if on_chip:
        assert launches < FRONTIER_LAUNCHES_PER_LEVEL * levels, launches
    else:
        assert launches >= FRONTIER_LAUNCHES_PER_LEVEL * levels, launches


def _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, expect):
    """porrt_sssp_worlds on both schedules == want; `expect` = the (on_chip, C, nc) the host rule must give.  bits None: the
    plain-graph call (n_worlds = 0, one column, finals = finals[0])."""
    V, W = len(xy), len(finals)
    n_val = 1 if bits is None else len(bits)
    assert colsolve_schedule(V, W, sm_count, int(row_ptr[-1]), n_val) == expect
    for force in (0, 1):
        if bits is None:
            got, launches = _launches(ctx, force, lambda: P.dijkstra_worlds(ctx, row_ptr, col, xy, None, None, finals[0])[0][None])
        else:
            words = P.words_from_bits(bits)
            got, launches = _launches(ctx, force, lambda: P.dijkstra_worlds(ctx, row_ptr, col, xy, nvid, words, finals)[0])
        np.testing.assert_array_equal(got, want, err_msg="force_global_sweeps=%d" % force)
        _check_schedule(launches, expect[0] and not force)


def _finals(rng, V, nvid, bits, W, k=3):
    """k random finals per world and one that is invalid in the world (where there is one)"""
    out = []
    for w in range(W):
        f = set(rng.choice(V, k, replace=False).tolist())
        bad = np.nonzero(bits[nvid, w] == 0)[0]
        if len(bad):
            f.add(int(rng.choice(bad)))
        out.append(sorted(f))
    return out


def _world_problem(V, W, n_ids, seed, degree=12.0, p_valid=0.75):
    """V random points joined within a radius, a synthetic validity table of n_ids ids x W worlds (one id holds in no world)"""
    xy = synth.points(V, seed=seed)
    row_ptr, col = _roadmap(xy, _radius(V, degree))
    rng = np.random.default_rng(seed + 1000)
    bits = (rng.random((n_ids, W)) < p_valid).astype(np.uint8)
    bits[n_ids - 1] = 0
    nvid = rng.integers(0, n_ids, V).astype(np.int32)
    return xy, row_ptr, col, nvid, bits, _finals(rng, V, nvid, bits, W)


# ---------------------------------------------------------------------------------------------- 1: every <C, WORLD>
@pytest.fixture(scope="module")
def worlds_3000():
    """V = 3000 (up to 6 columns per CTA fit), 888 worlds; the cases take the first W of them (ceil(W / 64) mask words)"""
    xy, row_ptr, col, nvid, bits, finals = _world_problem(3000, 888, 6, seed=31)
    finals[100] = []                                      # a world without finals: its row stays +inf
    return xy, row_ptr, col, nvid, bits, finals, _world_oracle(xy, row_ptr, col, nvid, bits, finals)


@pytest.mark.parametrize("W,C,nc", [(1, 1, 1), (150, 2, 2), (151, 2, 1), (300, 4, 4), (299, 4, 3), (888, 6, 6), (601, 6, 1),
                                    (887, 6, 5)])
def test_world_columns_per_cta(ctx, sm_count, worlds_3000, W, C, nc):
    """colsolve_push_kernel<C, COLSOLVE_WORLD> for C = 1, 2, 4, 6, with a full and a partly filled last CTA (padding columns)"""
    xy, row_ptr, col, nvid, bits, finals, want = worlds_3000
    if sm_count != 148 and colsolve_schedule(len(xy), W, sm_count)[1:] != (C, nc):
        pytest.skip("the column counts are chosen for 148 SMs")
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits[:, :W], finals[:W], want[:W], (True, C, nc))
    assert np.isfinite(want[:W]).any()
    if W > 100:
        assert np.isinf(want[100]).all()


# ---------------------------------------------------------------------------------------------- 2: through porrt_sssp_worlds_prm
@pytest.mark.parametrize("n_zones,C", [(8, 2), (9, 4)])
def test_world_columns_per_cta_on_resident_prm(ctx, sm_count, n_zones, C):
    """plan_qmdp's caller on a PRM of 3000 nodes over door maps of 8 / 9 zones (256 / 512 worlds)"""
    occ, zones = synth.door_map(size=1024, n_zones=n_zones)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    W = pmap.n_worlds()
    assert W == 2 ** n_zones
    xy = synth.points(3000, seed=40 + n_zones)
    prm = P.PRM(pmap)
    prm.init(xy[:1])
    prm.grow_graph(xy[1:], 0.1, 2.0)
    V = len(xy)
    rng = np.random.default_rng(n_zones)
    finals = [sorted(rng.choice(V, 3, replace=False).tolist()) for _ in range(W)]
    finals[W - 1] = []
    # the oracle: node validity id = state validity, an obstacle -> an extra id that holds in no world (as the product does)
    nvid = omap.state_validity(xy)
    wv = omap.world_validities()
    nvid = np.where(nvid >= 0, nvid, len(wv)).astype(np.int32)
    bits = np.vstack([wv, np.zeros((1, W), np.uint8)])
    want = _world_oracle(xy, prm.row_ptr, prm.col, nvid, bits, finals)
    on_chip, c, nc = colsolve_schedule(V, W, sm_count, int(prm.row_ptr[-1]), len(bits))
    assert on_chip and (c == C or sm_count != 148), (c, nc)
    for force in (0, 1):
        (got, _), launches = _launches(ctx, force, lambda: P.dijkstra_worlds_resident_prm(pmap, V, finals))
        np.testing.assert_array_equal(got, want, err_msg="force_global_sweeps=%d" % force)
        _check_schedule(launches, not force)
    assert np.isfinite(want).any() and np.isinf(want[W - 1]).all()
    assert len({want[w].tobytes() for w in range(W - 1)}) > 1


# ---------------------------------------------------------------------------------------------- 3: shared-memory bands
@pytest.mark.parametrize("V,W,expect", [(4696, 600, (True, 6, 6)), (4697, 600, (True, 4, 4)),
                                        (6973, 300, (True, 4, 4)), (6974, 300, (True, 2, 2)),
                                        (13536, 150, (True, 2, 2)), (13537, 150, (True, 1, 1)),
                                        (25568, 3, (True, 1, 1)), (25569, 3, (False, None, None))])
def test_world_columns_at_shared_memory_bands(ctx, sm_count, V, W, expect):
    """the largest V of each columns-per-CTA band and the one after it: the dynamic shared memory colsolve_level asks for and the
    kernel's carve-up agree at the top of the band; 25568 is the last on-chip size"""
    if sm_count != 148 and colsolve_schedule(V, W, sm_count) != expect:
        pytest.skip("the column counts are chosen for 148 SMs")
    xy, row_ptr, col, nvid, bits, finals = _world_problem(V, W, 5, seed=V)
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, expect)
    assert np.isfinite(want).any()


@pytest.mark.parametrize("V,on_chip", [(25568, True), (25569, False)])
def test_plain_graph_at_the_on_chip_limit(ctx, sm_count, V, on_chip):
    """the plain-graph call (n_worlds = 0: one column, every node valid) on both sides of colsolve_fits"""
    xy = synth.points(V, seed=V + 1)
    row_ptr, col = _roadmap(xy, _radius(V, 8.0))
    finals = sorted(np.random.default_rng(V).choice(V, 4, replace=False).tolist())
    want = _plain_oracle(xy, row_ptr, col, finals)[None]
    _check_worlds(ctx, sm_count, xy, row_ptr, col, None, None, [finals], want, (True, 1, 1) if on_chip else (False, None, None))
    assert np.isfinite(want).sum() > V // 2


# ---------------------------------------------------------------------------------------------- belief columns
def _hand_built_pto(omap, n_nodes, radius, goal_states, goal_masks, seed):
    """a roadmap over `omap` assembled by hand in the oracle's PTO (graph + reachability): random valid states + the goal states
    (n_nodes + len(goal_states) nodes), bi-edges between the pairs within `radius` whose transition the oracle validates; finals =
    the goal nodes"""
    rng = np.random.default_rng(seed)
    pts = np.zeros((0, 2))
    while len(pts) < n_nodes:
        c = rng.uniform(-0.95, 0.95, (2 * n_nodes, 2))
        pts = np.vstack([pts, c[omap.state_validity(c) >= 0]])[:n_nodes]
    goals = []
    for g in goal_states:                                  # the nearest valid state left of / around the goal position
        cand = np.array([[g[0] - dx, g[1] + dy] for dx in (0.0, 0.03, 0.06, 0.09, -0.03) for dy in (0.0, 0.03, -0.03)])
        ok = np.nonzero(omap.state_validity(cand) >= 0)[0]
        assert len(ok), g
        goals.append(cand[ok[0]])
    pts = np.vstack([pts, goals])
    vids = omap.state_validity(pts)
    assert (vids >= 0).all()
    pto = O.PTO(omap, util.LOW, util.UP)
    ones = [1] * omap.n_worlds
    for p, v in zip(pts, vids):
        pto.graph.add_node(p, int(v))
    pto.reach.set_root(ones)
    for _ in range(len(pts) - 1):
        pto.reach.add_node(ones)
    ii, jj = _pairs(pts, radius)
    ev = omap.edge_validity(pts[ii], pts[jj])
    for a, b, v in zip(ii[ev >= 0], jj[ev >= 0], ev[ev >= 0]):
        pto.graph.add_bi_edge(int(a), int(b), int(v))
    for k, m in enumerate(goal_masks):
        pto.reach.add_final_node(n_nodes + k, list(m))
    return pto


def _shelf(ctx, n_zones, visibility):
    occ, zones = synth.shelf_map(200, n_zones=n_zones)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, visibility)
    zp = omap.zone_positions()
    goal_states = [(float(zp[z][0]) - 0.06, float(zp[z][1])) for z in range(n_zones)]
    goal_masks = [[1 if k == z else 0 for k in range(n_zones)] for z in range(n_zones)]
    return omap, pmap, goal_states, goal_masks


def _belief_oracle(pto, b0):
    pto.build_belief_graph(b0)
    want = pto.compute_expected_costs_to_goals()
    typ = pto.belief_graph.export()[0]
    return want, typ


def _check_beliefs(ctx, sm_count, pmap, pto, b0, want, typ, on_chip):
    """porrt_belief_vi on both schedules: the whole V x B table and the node types == the oracle's"""
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    beliefs = pto.beliefs()
    V, B = len(xy), len(beliefs)
    levels = np.unique((beliefs > 0).sum(1), return_counts=True)[1]
    for n in levels:
        assert colsolve_schedule(V, int(n), sm_count, len(col), pmap.n_validities)[0] == on_chip
    for force in (0, 1):
        plan, launches = _launches(ctx, force, lambda: P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids,
                                                                           P.words_from_bits(fin_bits)))
        np.testing.assert_array_equal(plan.beliefs, beliefs)
        np.testing.assert_array_equal(plan.dist.reshape(-1), want, err_msg="force_global_sweeps=%d" % force)
        np.testing.assert_array_equal(plan.type.reshape(-1).astype(np.int32), typ, err_msg="force_global_sweeps=%d" % force)
        assert plan.expected_cost == want[0]
        _check_schedule(launches, on_chip and not force, levels=len(levels))
    return V, B


@pytest.mark.parametrize("V,on_chip", [(25568, True), (25569, False)])
def test_belief_columns_at_the_on_chip_limit(ctx, sm_count, V, on_chip):
    """porrt_belief_vi on a 3-zone shelf map (B = 7) with a roadmap of exactly 25568 (last on-chip size, C = 1) and 25569 nodes"""
    Z = 3
    omap, pmap, goal_states, goal_masks = _shelf(ctx, Z, 0.3)
    pto = _hand_built_pto(omap, V - Z, _radius(V, 14.0), goal_states, goal_masks, seed=V)
    b0 = [1.0 / Z] * Z
    want, typ = _belief_oracle(pto, b0)
    n, B = _check_beliefs(ctx, sm_count, pmap, pto, b0, want, typ, on_chip)
    assert (n, B) == (V, 7)
    assert colsolve_schedule(V, 3, sm_count, 0, pmap.n_validities) == ((True, 1, 1) if on_chip else (False, None, None))
    assert np.isfinite(want[0]) and (typ == O.OBSERVATION).any()


# ---------------------------------------------------------------------------------------------- 5: column-solver queue overflow
def test_world_columns_queue_overflow(ctx, sm_count):
    """more than COLSOLVE_QCAP sources in one column: the first round's dirty nodes do not fit the CTA's queue, the rest stay dirty"""
    V, W = 5000, 8
    xy, row_ptr, col, nvid, bits, _ = _world_problem(V, W, 6, seed=55)
    rng = np.random.default_rng(56)
    finals = [sorted(rng.choice(V, 1500, replace=False).tolist()) for _ in range(W)]
    assert min(len(f) for f in finals) > COLSOLVE_QCAP
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, (True, 1, 1))
    assert ((want > 0) & np.isfinite(want)).sum() > W * 1000


def test_belief_columns_queue_overflow(ctx, sm_count):
    """a shelf roadmap with a high visibility: a column of a later level starts with more than COLSOLVE_QCAP finite Observation values"""
    Z = 3
    omap, pmap, goal_states, goal_masks = _shelf(ctx, Z, 1.5)
    pto = _hand_built_pto(omap, 5000 - Z, _radius(5000, 12.0), goal_states, goal_masks, seed=57)
    b0 = [1.0 / Z] * Z
    want, typ = _belief_oracle(pto, b0)
    B = len(pto.beliefs())
    sources = ((typ == O.OBSERVATION) & np.isfinite(want)).reshape(-1, B).sum(0)
    assert sources.max() > COLSOLVE_QCAP, sources
    _check_beliefs(ctx, sm_count, pmap, pto, b0, want, typ, True)


# ---------------------------------------------------------------------------------------------- 6: frontier push-list overflow
def test_world_columns_push_list_overflow(ctx, sm_count):
    """V = 30000 takes the frontier relaxation; 75 % of the nodes are finals in every one of 200 worlds, so the first round has more
    (node, world) pairs than the push list holds and sf_classify_kernel defers the rest"""
    V, W = 30000, 200
    xy, row_ptr, col, nvid, bits, _ = _world_problem(V, W, 5, seed=66)
    rng = np.random.default_rng(67)
    finals = [np.sort(rng.choice(V, 3 * V // 4, replace=False)) for _ in range(W)]
    pair_cap = min(V * W, max(4 << 20, 4 * V))            # sf_state_layout
    assert sum(len(f) for f in finals) > pair_cap
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, (False, None, None))
    assert ((want > 0) & np.isfinite(want)).any()


# ---------------------------------------------------------------------------------------------- 7: degenerate roadmaps
def _degenerate(name):
    """-> xy, row_ptr, col, nvid, bits, finals of a small world problem"""
    rng = np.random.default_rng(sum(map(ord, name)))
    W = 3
    if name == "one_node":
        xy, row_ptr, col = np.zeros((1, 2)), np.zeros(2, np.int64), np.zeros(0, np.int32)
        return xy, row_ptr, col, np.zeros(1, np.int32), np.ones((1, 2), np.uint8), [[0], []]
    if name == "no_edges":
        xy = synth.points(50, seed=5)
        row_ptr, col = np.zeros(51, np.int64), np.zeros(0, np.int32)
    elif name == "one_point":                             # zero-cost edges, a zero-size bounding box, mean edge length 0
        xy = np.full((40, 2), 0.25)
        row_ptr, col = _roadmap(xy, 0.1)
    elif name == "vertical_line":
        xy = np.stack([np.full(300, -0.3), rng.uniform(-1.0, 1.0, 300)], 1)
        row_ptr, col = _roadmap(xy, 0.02)
    elif name == "self_loops_and_duplicates":
        xy = synth.points(400, seed=8)
        a, b = _pairs(xy, 0.15)
        dup = rng.choice(len(a), len(a) // 3, replace=False)
        loops = np.arange(0, 400, 3)
        src = np.concatenate([a, b, a[dup], b[dup], loops, loops])
        dst = np.concatenate([b, a, b[dup], a[dup], loops, loops])
        row_ptr, col = _csr(400, src, dst)
    elif name in ("repeated_finals", "every_node_final"):
        xy = synth.points(400, seed=9)
        row_ptr, col = _roadmap(xy, 0.15)
    V = len(xy)
    bits = (rng.random((4, W)) < 0.7).astype(np.uint8)
    nvid = rng.integers(0, 4, V).astype(np.int32)
    finals = [sorted(rng.choice(V, 3, replace=False).tolist()) for _ in range(W)]
    if name == "repeated_finals":
        finals = [f + f[:2] for f in finals]
    if name == "every_node_final":
        finals[1] = list(range(V))
    return xy, row_ptr, col, nvid, bits, finals


@pytest.mark.parametrize("name", ["one_node", "no_edges", "one_point", "vertical_line", "self_loops_and_duplicates",
                                  "repeated_finals", "every_node_final"])
def test_world_columns_degenerate(ctx, sm_count, name):
    xy, row_ptr, col, nvid, bits, finals = _degenerate(name)
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, (True, 1, 1))
    if name == "one_point":
        assert set(np.unique(want)) <= {0.0, np.inf}


def test_plain_graph_degenerate(ctx, sm_count):
    """one node, final and not final; no edges at all"""
    xy = np.zeros((1, 2))
    for finals in ([0], []):
        want = _plain_oracle(xy, np.zeros(2, np.int64), np.zeros(0, np.int32), finals)[None]
        assert want[0, 0] == (0.0 if finals else np.inf)
        _check_worlds(ctx, sm_count, xy, np.zeros(2, np.int64), np.zeros(0, np.int32), None, None, [finals], want, (True, 1, 1))
    xy = synth.points(50, seed=6)
    _check_worlds(ctx, sm_count, xy, np.zeros(51, np.int64), np.zeros(0, np.int32), None, None, [[7, 9]],
                  _plain_oracle(xy, np.zeros(51, np.int64), np.zeros(0, np.int32), [7, 9])[None], (True, 1, 1))


@pytest.mark.parametrize("n_validities,on_chip", [(256, True), (257, False)])
def test_world_columns_validity_id_255(ctx, sm_count, n_validities, on_chip):
    """nodes of validity id 255 (the top bit of the column solver's 4-word mask) with 256 ids, on chip, and with 257 ids, which
    only the frontier relaxation takes; 70 worlds: two words of the validity table"""
    V, W = 600, 70
    xy = synth.points(V, seed=n_validities)
    row_ptr, col = _roadmap(xy, _radius(V, 8.0))
    rng = np.random.default_rng(n_validities)
    bits = (rng.random((n_validities, W)) < 0.6).astype(np.uint8)
    ids = [0, 64, 254, 255] + ([256] if n_validities > 256 else [])
    nvid = rng.choice(ids, V).astype(np.int32)
    nvid[: V // 3] = 255
    finals = _finals(rng, V, nvid, bits, W)
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    _check_worlds(ctx, sm_count, xy, row_ptr, col, nvid, bits, finals, want, (True, 1, 1) if on_chip else (False, None, None))
    assert bits[255].any() and not bits[255].all() and np.isfinite(want[:, nvid == 255]).any()


# ---------------------------------------------------------------------------------------------- a second device
_TWO_DEVICES = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import po_rrt_b200 as P
a = np.load(sys.argv[2])
finals = np.split(a["fin"], a["fptr"][1:-1])
ctxs = [P.Context(0), P.Context(1)]
out = []
for c in ctxs:
    n0 = c.launch_count()
    d = P.dijkstra_worlds(c, a["row_ptr"], a["col"], a["xy"], a["nvid"], a["words"], finals)[0]
    out.append((d, c.launch_count() - n0))
np.savez(sys.argv[3], dist=np.stack([d for d, _ in out]), launches=np.array([n for _, n in out]))
for c in ctxs:
    c.close()
"""


def test_world_columns_on_a_second_device(ctx, sm_count, tmp_path):
    """the column solver's opt-in to more than 48 KB of dynamic shared memory holds for the current device only: a process that
    solves on device 0 and then on device 1 (V = 7000, C = 1: about 65 KB) must get the same table from both.  A fresh process,
    so that nothing has opted in on either device before."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    V, W = 7000, 4
    xy, row_ptr, col, nvid, bits, finals = _world_problem(V, W, 5, seed=77)
    assert colsolve_schedule(V, W, sm_count, int(row_ptr[-1]), len(bits)) == (True, 1, 1)
    assert V * 8 + 256 + (V + 3) // 4 * 4 + COLSOLVE_QCAP * 2 + 16 > 48 * 1024
    fptr = np.concatenate([[0], np.cumsum([len(f) for f in finals])]).astype(np.int64)
    np.savez(tmp_path / "in.npz", xy=xy, row_ptr=row_ptr, col=col, nvid=nvid, words=P.words_from_bits(bits), fptr=fptr,
             fin=np.concatenate(finals).astype(np.int32))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _TWO_DEVICES, root, str(tmp_path / "in.npz"), str(tmp_path / "out.npz")], cwd=root,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = np.load(tmp_path / "out.npz")
    want = _world_oracle(xy, row_ptr, col, nvid, bits, finals)
    for dev in range(2):
        np.testing.assert_array_equal(res["dist"][dev], want, err_msg="device %d" % dev)
        _check_schedule(int(res["launches"][dev]), True)
