"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.
Integer / index results must be bit-exact; f64 values are compared for exact equality unless stated."""
import math
import os

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu
INF = float("inf")


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------------------------- maps
def _check_edges(omap, pmap, a, b):
    want = omap.edge_validity(a, b)
    got, masks = pmap.transition_validator(a, b, want_masks=True)
    assert got.dtype == np.int32
    np.testing.assert_array_equal(got.astype(np.int64), want)
    wv = pmap.world_validities_words()
    exp_masks = np.where((want >= 0)[:, None], wv[np.clip(want, 0, None)], 0)
    np.testing.assert_array_equal(masks, exp_masks)
    got8 = pmap.transition_validator(a, b, compact=True)          # one signed byte per edge, same codes
    assert got8.dtype == np.int8
    np.testing.assert_array_equal(got8.astype(np.int64), want)
    return want


def test_door_map_info_and_validities(ctx):
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    assert (pmap.n_zones, pmap.n_worlds(), pmap.n_validities) == (omap.n_zones, omap.n_worlds, omap.n_validities) == (3, 8, 4)
    np.testing.assert_array_equal(pmap.world_validities(), omap.world_validities())
    np.testing.assert_array_equal(pmap.zone_positions(), omap.zone_positions())


def test_door_edges_random(ctx):
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(200_000, seed=2, max_len=0.1)
    want = _check_edges(omap, pmap, a, b)
    # the batch exercises every outcome
    assert (want == -1).any() and (want == omap.n_validities - 1).any() and ((want >= 0) & (want < 3)).any()


def test_door_edges_long_and_degenerate(ctx):
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(50_000, seed=7, max_len=2.5)      # up to the whole map: many 128-pixel rounds
    _check_edges(omap, pmap, a, b)
    p = synth.points(5_000, seed=8)
    _check_edges(omap, pmap, p, p)                        # zero-length edges (dx_oct == 0)
    q = p + np.array([1.0 / 256, 0.0])                    # one-pixel steps (dx_oct == 1)
    _check_edges(omap, pmap, p, np.clip(q, -1, 1 - 2.0 ** -20))


def test_door_edges_direction_matters(ctx):
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(100_000, seed=9, max_len=0.3)
    fwd = _check_edges(omap, pmap, a, b)
    bwd = _check_edges(omap, pmap, b, a)
    assert (fwd != bwd).any()  # a->b and b->a visit different pixels (SURVEY A5)


def test_door_edges_panics(ctx):
    """adjacent zones (multi-zone assert), gray pixels without zone id (unwrap), out-of-bounds endpoints"""
    size = 256
    occ = np.full((size, size), 255, np.uint8)
    zones = np.full((size, size), 255, np.uint8)
    occ[100:140, 60:70] = 128; zones[100:140, 60:70] = 0
    occ[100:140, 70:80] = 128; zones[100:140, 70:80] = 1     # touches zone 0
    occ[100:140, 84:90] = 0                                   # obstacle right after
    occ[30:40, 30:200] = 90                                   # gray without zone id
    occ[200:210, :] = 0
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    rng = np.random.default_rng(4)
    a = rng.uniform(-1.2, 1.2, (150_000, 2))                  # some endpoints outside the map
    b = a + rng.uniform(-0.4, 0.4, (150_000, 2))
    want = _check_edges(omap, pmap, a, b)
    for code in (O.PANIC_OOB, O.PANIC_ZONE_UNWRAP, O.PANIC_MULTI_ZONE, O.NONE):
        assert (want == code).any(), code
    sv = omap.state_validity(a)
    np.testing.assert_array_equal(pmap.state_validity(a).astype(np.int64), sv)
    assert (sv == O.PANIC_OOB).any() and (sv == O.PANIC_ZONE_UNWRAP).any()


def test_edge_large_map_path(ctx):
    """maps whose class plane does not fit in shared memory (> ~14000^2 px) take map.cu's kernel (class bytes in global
    memory); forced here on small maps, it must give the same bits"""
    ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 1)
    try:
        occ, zones = util.small_door_map(512, 3)
        omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
        a, b = synth.edges(120_000, seed=31, max_len=0.4)
        _check_edges(omap, pmap, a, b)
        a, b = synth.edges(20_000, seed=32, max_len=2.5)        # edges across the whole map (> 32 strips)
        _check_edges(omap, pmap, a, b)
        rng = np.random.default_rng(33)
        a = rng.uniform(-1.1, 1.1, (40_000, 2)); b = a + rng.uniform(-0.3, 0.3, (40_000, 2))
        _check_edges(omap, pmap, a, b)                          # some end points outside the map
        occ, zones = synth.shelf_map(400, n_rects=20, n_zones=5, seed=6)
        omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.6)
        a, b = synth.edges(60_000, seed=34, max_len=0.5)
        _check_edges(omap, pmap, a, b)
    finally:
        ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)


def test_edge_large_map_path_real(ctx):
    """a 15008^2 map: the class plane (220 KiB + guards) no longer leaves room for the warps' queues -> large-map kernel"""
    size = 15008
    occ, zones = synth.door_map(size=size, n_rects=2048, n_zones=3, seed=17)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(300_000, seed=35, max_len=0.05)
    want = _check_edges(omap, pmap, a, b)
    assert (want == -1).any() and (want >= 0).any()
    occ, zones = util.small_door_map(256, 2)
    util.make_pair(ctx, occ, zones, P.DOOR, 0.3)                # release the big grids' successor state


def test_edges_odd_map_sizes(ctx):
    """maps whose sides are not multiples of the 16-pixel blocks, and a non-square one"""
    rng = np.random.default_rng(40)
    for (H, W) in ((200, 200), (333, 517), (1000, 250)):
        occ = np.full((H, W), 255, np.uint8)
        for _ in range(60):
            h, w = rng.integers(3, max(4, H // 6)), rng.integers(3, max(4, W // 6))
            i, j = rng.integers(0, H - h), rng.integers(0, W - w)
            occ[i:i + h, j:j + w] = 0
        zones = np.full((H, W), 255, np.uint8)
        occ[H // 2:H // 2 + 9, W // 3:W // 3 + 7] = 128; zones[H // 2:H // 2 + 9, W // 3:W // 3 + 7] = 0
        occ[H - 12:H - 3, W - 11:W - 2] = 128; zones[H - 12:H - 3, W - 11:W - 2] = 1   # zone touching the last (partial) blocks
        omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
        a, b = synth.edges(80_000, seed=41, max_len=0.6)
        want = _check_edges(omap, pmap, a, b)
        assert (want == -1).any() and (want >= 0).any()
        _check_edges(omap, pmap, b, a)


def test_door_without_zones(ctx):
    occ, _ = util.small_door_map(256, 1)
    occ[occ == 128] = 255
    omap, pmap = util.make_pair(ctx, occ, None, P.DOOR)
    assert pmap.n_worlds() == 1 and pmap.n_validities == 1
    a, b = synth.edges(50_000, seed=3, max_len=0.2)
    _check_edges(omap, pmap, a, b)
    np.testing.assert_array_equal(pmap.state_validity(a).astype(np.int64), omap.state_validity(a))


def test_shelf_edges_states_visibility(ctx):
    occ, zones = synth.shelf_map(400, n_rects=20, n_zones=5, seed=6)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.6)
    assert pmap.n_worlds() == omap.n_worlds == 5 and pmap.n_validities == 1
    np.testing.assert_array_equal(pmap.world_validities(), omap.world_validities())
    a, b = synth.edges(150_000, seed=12, max_len=0.5)
    want = _check_edges(omap, pmap, a, b)
    assert (want == 0).any() and (want == -1).any()
    np.testing.assert_array_equal(pmap.state_validity(a).astype(np.int64), omap.state_validity(a))
    pts = synth.points(20_000, seed=13)
    wm, wp = omap.visible_zones(pts)
    gm, gs = pmap.visible_zones(pts)
    np.testing.assert_array_equal(gm, wm)
    np.testing.assert_array_equal(gs.astype(np.int64), wp)
    assert (wm != 0).any()


def test_door_visibility(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.5)
    pts = synth.points(30_000, seed=14)
    wm, wp = omap.visible_zones(pts)
    gm, gs = pmap.visible_zones(pts)
    np.testing.assert_array_equal(gm, wm)
    np.testing.assert_array_equal(gs.astype(np.int64), wp)
    assert len(np.unique(wm)) >= 3


def test_edges_host_pipeline_multi_chunk(ctx):
    """> 1 Mi edges: exercises the chunked H2D | kernel | D2H pipeline and pageable staging"""
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(3_500_000, seed=21, max_len=0.05)
    _check_edges(omap, pmap, a, b)


@pytest.mark.parametrize("n", [2_150_001, 4_194_312 + 8, 2_150_000])
def test_edges_host_pipeline_odd_chunk_sizes(ctx, n):
    """chunk sizes that are not multiples of 4 edges: every array of a device slot must still be 16-byte aligned (the kernels
    read endpoints as 16-byte vectors); pageable and pinned buffers, with and without masks, coordinates and node ids"""
    import torch
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    a, b = synth.edges(n, seed=22, max_len=0.03)
    want = omap.edge_validity(a, b)
    wv = pmap.world_validities_words()
    exp_masks = np.where((want >= 0)[:, None], wv[np.clip(want, 0, None)], 0)
    got, masks = pmap.transition_validator(a, b, want_masks=True)                      # pageable, masks
    np.testing.assert_array_equal(got.astype(np.int64), want)
    np.testing.assert_array_equal(masks, exp_masks)
    np.testing.assert_array_equal(pmap.transition_validator(a, b).astype(np.int64), want)   # pageable, no masks
    pa, pb = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    pv = torch.empty(n, dtype=torch.int32).pin_memory()
    pm = torch.empty((n, 1), dtype=torch.int64).pin_memory()
    c = ctx
    c.check(c.lib.porrt_edge_validity(c.h, pa.data_ptr(), pb.data_ptr(), n, pv.data_ptr(), pm.data_ptr()))      # pinned, masks
    np.testing.assert_array_equal(pv.numpy().astype(np.int64), want)
    np.testing.assert_array_equal(pm.numpy().view(np.uint64), exp_masks)
    pv.zero_()
    c.check(c.lib.porrt_edge_validity(c.h, pa.data_ptr(), pb.data_ptr(), n, pv.data_ptr(), None))               # pinned, no masks
    np.testing.assert_array_equal(pv.numpy().astype(np.int64), want)
    p8 = torch.empty(n, dtype=torch.int8).pin_memory()
    c.check(c.lib.porrt_edge_validity_i8(c.h, pa.data_ptr(), pb.data_ptr(), n, p8.data_ptr()))                  # pinned, bytes
    np.testing.assert_array_equal(p8.numpy().astype(np.int64), want)
    # the same edges as node pairs and as an adjacency over the resident vertex set
    tree = P.KdTree(ctx, np.concatenate([a, b]), cell_size=0.02)
    fi, ti = np.arange(n, dtype=np.int32), np.arange(n, 2 * n, dtype=np.int32)
    got, masks = pmap.transition_validator_nodes(fi, ti, want_masks=True)
    np.testing.assert_array_equal(got.astype(np.int64), want)
    np.testing.assert_array_equal(masks, exp_masks)
    np.testing.assert_array_equal(pmap.transition_validator_nodes(fi, ti, compact=True).astype(np.int64), want)
    del tree


def test_reachable_belief_states(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.5)
    for b0 in ([0.25] * 4, [0.1, 0.1, 0.1, 0.7], [0.5, 0.5, 0.0, 0.0]):
        np.testing.assert_array_equal(pmap.reachable_belief_states(b0), omap.reachable_belief_states(b0))
    assert len(pmap.reachable_belief_states([0.25] * 4)) == 9      # map_io.rs:711-712
    occ, zones = synth.shelf_map(200, n_zones=4)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    np.testing.assert_array_equal(pmap.reachable_belief_states([0.25] * 4), omap.reachable_belief_states([0.25] * 4))


# ---------------------------------------------------------------------------------------------- nearest neighbours
NODES = [[3.0, 6.0], [17.0, 15.0], [13.0, 15.0], [6.0, 12.0], [9.0, 1.0], [2.0, 7.0], [10.0, 19.0]]
CENTERS = [[17.0, 15.0], [9.1, 1.0], [2.0, 8.0], [15.0, 13.0], [3.0, 5.0], [13.0, 7.0]]


def test_kdtree_golden_through_gpu(ctx):  # nearest_neighbor.rs:237-311
    tree = P.KdTree(ctx, NODES)
    for c in CENTERS:
        d = sorted(((math.sqrt((n[0] - c[0]) ** 2 + (n[1] - c[1]) ** 2), i) for i, n in enumerate(NODES)))
        ids, dist, _ = tree.nearest_neighbor([c])
        assert ids[0] == d[0][1] and dist[0] == d[0][0]
        for radius in range(1, 10):
            offs, hits = tree.nearest_neighbors([c], float(radius))
            assert list(hits) == sorted(i for dd, i in d if dd <= radius)
    # filtered sequences (:267-311): validator = reach bit
    def filt(q, excluded):
        reach = np.ones(len(NODES), np.uint64)
        reach[list(excluded)] = 0
        return int(tree.nearest_neighbor([q], reach, [0])[0][0])
    seq = [(0, []), (5, [0]), (3, [0, 5]), (4, [0, 5, 3]), (2, [0, 5, 3, 4]), (6, [0, 5, 3, 4, 2]), (1, [0, 5, 3, 4, 2, 6])]
    for expect, excl in seq:
        assert filt([3.1, 6.0], excl) == expect
    for expect, excl in [(2, []), (1, [2]), (6, [2, 1]), (3, [2, 1, 6])]:
        assert filt([13.0, 15.1], excl) == expect
    assert filt([3.1, 6.0], range(7)) == -1


def _oracle_tree(pts):
    t = O.KdTree(pts[0], 0)
    t.add_batch(pts[1:], 1)
    return t


def test_radius_query_vs_oracle(ctx):
    pts = synth.points(50_000, seed=3)
    q = synth.points(4_000, seed=4)
    otree = _oracle_tree(pts)
    tree = P.KdTree(ctx, pts, cell_size=0.02)
    rng = np.random.default_rng(5)
    radius = rng.uniform(0.0, 0.05, len(q))
    radius[:10] = 0.0
    q[:5] = pts[:5]                                           # exact duplicates at radius 0
    offs, ids = tree.nearest_neighbors(q, radius)
    ooffs, oids, tot = otree.radius_batch(q, radius, cap=len(ids) + 10)
    assert tot == len(ids)
    np.testing.assert_array_equal(offs, ooffs)
    for k in range(len(q)):
        got = ids[offs[k]:offs[k + 1]]
        assert (np.diff(got) > 0).all()
        np.testing.assert_array_equal(got, np.sort(oids[ooffs[k]:ooffs[k + 1]]))
    assert list(ids[offs[0]:offs[1]]) == [0]
    # kd pre-order restored by rank
    rank = tree.preorder_rank()
    for k in range(0, len(q), 37):
        got = ids[offs[k]:offs[k + 1]]
        np.testing.assert_array_equal(got[np.argsort(rank[got], kind="stable")], oids[ooffs[k]:ooffs[k + 1]])


@pytest.mark.parametrize("huge", [False, True])
def test_radius_query_large_segments(ctx, huge):
    """> 256 hits per query: block-level sorting network (257..4096 entries); with `huge`, one query beyond that sends the call
    to the global radix sort instead"""
    pts = synth.points(20_000, seed=33)
    q = synth.points(300, seed=34)
    otree = _oracle_tree(pts)
    tree = P.KdTree(ctx, pts, cell_size=0.05)
    radius = np.where(np.arange(300) % 3 == 0, 0.3, 0.02)
    if huge:
        radius[7] = 0.9
    offs, ids = tree.nearest_neighbors(q, radius)
    rank = tree.preorder_rank()
    assert (np.diff(offs) > 256).any() and (np.diff(offs) < 64).any() and (np.diff(offs).max() > 4096) == huge
    for k in range(300):
        got = ids[offs[k]:offs[k + 1]]
        want = otree.nearest_neighbors(q[k], radius[k])
        np.testing.assert_array_equal(got, np.sort(want))
        np.testing.assert_array_equal(got[np.argsort(rank[got], kind="stable")], want)


def test_kd_preorder_rank_device(ctx):
    """level-synchronous device construction == sequential insertion (incl. duplicate points and collinear runs)"""
    rng = np.random.default_rng(8)
    pts = rng.uniform(-1, 1, (30_000, 2))
    pts[100:200] = pts[0:100]                      # exact duplicates go right, in insertion order
    pts[300:400, 0] = 0.25                         # equal x
    pts[500:600] = np.round(pts[500:600] * 4) / 4  # lattice points: many ties on both axes
    tree = P.KdTree(ctx, pts)
    rank = tree.preorder_rank()
    otree = _oracle_tree(pts)
    order = otree.nearest_neighbors([0.0, 0.0], 10.0)          # everything, in kd pre-order
    np.testing.assert_array_equal(np.argsort(rank), order)
    chain = np.arange(2000, dtype=np.float64)[:, None] * np.array([[1e-3, 1e-3]]) - 1.0   # sorted input: depth == n
    np.testing.assert_array_equal(P.KdTree(ctx, chain).preorder_rank(), np.arange(2000))


def test_kd_preorder_rank_two_phase_start(ctx):
    """single trees of >= 8 * 65536 points are built top tree first, then everybody else from where a read-only walk leaves
    them (graph.cu: kd_walk_kernel); the order must still be the one of sequential insertion (nearest_neighbor.rs:29-46)"""
    rng = np.random.default_rng(18)
    n = 600_000
    pts = rng.uniform(-1, 1, (n, 2))
    pts[70_000:70_500] = pts[0:500]                       # duplicates of top-tree points among the later ones
    pts[200_000:200_400] = pts[100_000:100_400]           # duplicates among the later points
    pts[300_000:301_000, 0] = pts[5, 0]                   # a run with a top-tree node's x
    pts[400_000:400_800] = np.round(pts[400_000:400_800] * 8) / 8
    rank = P.KdTree(ctx, pts).preorder_rank()
    order = _oracle_tree(pts).nearest_neighbors([0.0, 0.0], 10.0)
    np.testing.assert_array_equal(np.argsort(rank), order)


def test_radius_threshold_boundary(ctx):
    """inclusive `<=` on the sqrt-ed distance: hits at exactly r, misses one ulp below"""
    pts = np.array([[0.0, 0.0], [3.0, 4.0], [1.0, 1.0], [-0.3, 0.4]])
    tree = P.KdTree(ctx, pts)
    q = np.zeros((6, 2))
    r = np.array([5.0, np.nextafter(5.0, 0), math.sqrt(2.0), np.nextafter(math.sqrt(2.0), 0), 0.5, np.nextafter(0.5, 0)])
    offs, ids = tree.nearest_neighbors(q, r)
    otree = _oracle_tree(pts)
    for k in range(6):
        assert sorted(otree.nearest_neighbors(q[k], r[k])) == list(ids[offs[k]:offs[k + 1]])
    assert list(ids[offs[0]:offs[1]]) == [0, 1, 2, 3] and list(ids[offs[1]:offs[2]]) == [0, 2, 3]


def test_prefix_and_filtered_radius(ctx):
    pts = synth.points(20_000, seed=31)
    tree = P.KdTree(ctx, pts, cell_size=0.03)
    k = np.arange(1, 20_000, 7)
    offs, ids = tree.nearest_neighbors(pts[k], 0.04, prefix_limit=k)
    d = None
    for n, kk in enumerate(k[:200]):
        got = ids[offs[n]:offs[n + 1]]
        dd = np.sqrt(((pts[:kk] - pts[kk]) ** 2).sum(1))
        np.testing.assert_array_equal(got, np.nonzero(dd <= 0.04)[0])
    rng = np.random.default_rng(2)
    reach = rng.integers(0, 2 ** 63, len(pts), dtype=np.uint64)
    world = rng.integers(0, 63, 300).astype(np.uint32)
    offs, ids = tree.nearest_neighbors(pts[:300], 0.05, reach_mask=reach, world=world)
    for n in range(300):
        dd = np.sqrt(((pts - pts[n]) ** 2).sum(1))
        ok = ((reach >> np.uint64(world[n])) & np.uint64(1)).astype(bool)
        np.testing.assert_array_equal(ids[offs[n]:offs[n + 1]], np.nonzero((dd <= 0.05) & ok)[0])


def test_nearest_vs_oracle(ctx):
    pts = synth.points(30_000, seed=41)
    q = np.vstack([synth.points(5_000, seed=42), synth.points(200, seed=43, low=-1.5, up=1.5)])
    otree = _oracle_tree(pts)
    tree = P.KdTree(ctx, pts)
    ids, dist, ties = tree.nearest_neighbor(q)
    want = otree.nearest_batch(q)
    assert (ties == 1).all()
    np.testing.assert_array_equal(ids.astype(np.int64), want)
    np.testing.assert_array_equal(dist, np.sqrt(((pts[want] - q) ** 2).sum(1)))
    # filtered: random reachability bits, world per query (pto.rs:74-77)
    rng = np.random.default_rng(44)
    reach = rng.integers(0, 2 ** 63, len(pts), dtype=np.uint64)
    world = rng.integers(0, 63, len(q)).astype(np.uint32)
    ids, _, ties = tree.nearest_neighbor(q, reach, world)
    want = otree.nearest_batch(q, reach, world)
    np.testing.assert_array_equal(ids[ties == 1].astype(np.int64), want[ties == 1])
    assert (ties == 1).all()


def test_knn_vs_bruteforce(ctx):
    pts = synth.points(8_000, seed=51)
    q = synth.points(500, seed=52)
    tree = P.KdTree(ctx, pts)
    for k in (1, 5, 16, 32):
        ids, dist = tree.knn(q, k)
        d2 = ((pts[None, :, :] - q[:, None, :]) ** 2).sum(2)
        order = np.lexsort((np.broadcast_to(np.arange(len(pts)), d2.shape), d2), axis=1)[:, :k]
        np.testing.assert_array_equal(ids, order)
        np.testing.assert_array_equal(dist, np.sqrt(np.take_along_axis(d2, order, 1)))
    ids, dist = P.KdTree(ctx, pts[:3]).knn(q[:4], 5)   # fewer vertices than k: padded
    assert (ids[:, 3:] == -1).all() and np.isinf(dist[:, 3:]).all()


# ---------------------------------------------------------------------------------------------- PRM
def _prm_compare(ctx, occ, zones, kind, n_iter, max_step, search_radius, start=(0.0, 0.0)):
    omap, pmap = util.make_pair(ctx, occ, zones, kind, 0.3)
    oprm = O.PRM(omap, util.LOW, util.UP, seed=0)
    oprm.init(start)
    oprm.grow_graph(max_step, search_radius, n_iter)
    samples = O.Pcg64(0).sample_states(util.LOW, util.UP, n_iter)   # the ContinuousSampler stream the oracle consumed
    prm = P.PRM(pmap)
    prm.init(start)
    prm.grow_graph(samples, max_step, search_radius)
    xy, _, rp, col, _ = oprm.graph.export(0)
    np.testing.assert_array_equal(prm.states, xy)
    np.testing.assert_array_equal(prm.row_ptr, rp)
    np.testing.assert_array_equal(prm.col, col)                      # children in the reference's insertion order
    _, _, rpp, colp, _ = oprm.graph.export(1)
    np.testing.assert_array_equal(prm.row_ptr, rpp)
    np.testing.assert_array_equal(prm.col, colp)                     # parents(k) == children(k) as sequences
    return prm, oprm


def test_nn_tiles_equal_thread_per_query(ctx):
    """nn_tile.cu (TMA-staged tiles) against nn.cu's thread-per-query kernels on the same batches: mixed radii (some wider
    than a cell -> index-list fallback), prefix limits, reachability filters, NaN / far-away queries, clustered vertices
    (tiles that exceed the staging buffer), k = 1 / 5 / 16 / 32"""
    rng = np.random.default_rng(77)
    pts = np.vstack([synth.points(60_000, seed=71), 0.02 * rng.standard_normal((30_000, 2)) + [0.3, -0.2]])   # dense cluster
    tree = P.KdTree(ctx, pts, cell_size=0.02)
    q = np.vstack([synth.points(12_000, seed=72), 0.02 * rng.standard_normal((4_000, 2)) + [0.3, -0.2],
                   synth.points(500, seed=73, low=-1.6, up=1.6)])
    q[7] = [np.nan, 0.1]
    radius = rng.uniform(0.0, 0.03, len(q)); radius[::50] = 0.08; radius[3] = -1.0; radius[11] = np.nan
    prefix = rng.integers(0, len(pts) + 1, len(q)).astype(np.uint32)
    reach = rng.integers(0, 2 ** 63, len(pts), dtype=np.uint64)
    world = rng.integers(0, 63, len(q)).astype(np.uint32)

    def run():
        out = {}
        out["r"] = tree.nearest_neighbors(q, radius)
        out["rp"] = tree.nearest_neighbors(q, radius, prefix_limit=prefix)
        out["rf"] = tree.nearest_neighbors(q, radius, reach_mask=reach, world=world)
        out["nn"] = tree.nearest_neighbor(q)
        out["nnf"] = tree.nearest_neighbor(q, reach_mask=reach, world=world)
        for k in (5, 16, 32):
            out["k%d" % k] = tree.knn(q, k)
        return out

    got = run()
    ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 1)
    try:
        want = run()
    finally:
        ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 0)
    for key in want:
        for a, b in zip(got[key], want[key]):
            np.testing.assert_array_equal(a, b, err_msg=key)
    assert len(got["r"][1]) > 100_000


def test_prm_build_door(ctx):
    occ, zones = util.small_door_map(512, 3)
    prm, _ = _prm_compare(ctx, occ, zones, P.DOOR, 6000, 0.1, 2.0)
    assert len(prm.col) > 20_000


def test_prm_build_shelf_reference_params(ctx):  # prm.rs:136-155: grow_graph(0.1, 5.0, 1500)
    occ, zones = synth.shelf_map(200, n_zones=2)
    _prm_compare(ctx, occ, zones, P.SHELF, 1500, 0.1, 5.0)


def test_prm_build_wide_rows(ctx):
    """a wide connection radius: neighbour lists of ~170 and late lists beyond 256 entries (block-level segment sort)"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    prm, _ = _prm_compare(ctx, occ, zones, P.SHELF, 6000, 0.4, 8.0)
    assert np.diff(prm.row_ptr).max() > 600


def test_prm_build_large_result_in_row_blocks(ctx):
    """>= 2^18 nodes: the one-pass thread- / warp-per-query radius kernels, kd ranks by pointer jumping and, with a caller-owned
    column buffer, the result copy in row blocks that overlaps the CSR assembly -- against the oracle's sequential add_sample
    (280 k nodes, 1.2e7 directed edges) and against the fetch-afterwards path"""
    n_iter = 280_000
    occ, zones = util.small_door_map(1024, 3)
    prm, oprm = _prm_compare(ctx, occ, zones, P.DOOR, n_iter, 0.1, 2.0)      # columns fetched after the build
    samples = O.Pcg64(0).sample_states(util.LOW, util.UP, n_iter)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    col_out = np.full(len(prm.col) + 1000, -7, np.int32)
    row_out = np.zeros(n_iter + 2, np.int64)
    prm2 = P.PRM(pmap)
    prm2.init((0.0, 0.0))
    prm2.grow_graph(samples, 0.1, 2.0, col_out=col_out, row_ptr_out=row_out)  # columns leave in row blocks during the build
    np.testing.assert_array_equal(prm2.row_ptr, prm.row_ptr)
    np.testing.assert_array_equal(prm2.col, prm.col)
    assert (col_out[len(prm.col):] == -7).all()                               # nothing written past the last edge
    small = np.empty(1000, np.int32)                                          # a buffer that is too small: size query + fetch
    prm3 = P.PRM(pmap)
    prm3.init((0.0, 0.0))
    with pytest.raises(P.PorrtError):
        prm3.grow_graph(samples, 0.1, 2.0, col_out=small)


def test_prm_plan_path(ctx):
    occ, zones = synth.shelf_map(200, n_zones=2)
    prm, oprm = _prm_compare(ctx, occ, zones, P.SHELF, 2500, 0.1, 5.0)
    # PRM::plan_path (prm.rs:111-122): nearest start/goal vertex, dijkstra towards the goal
    tree = P.KdTree(ctx, prm.states)
    ids, _, _ = tree.nearest_neighbor([[0.0, 0.0], [-0.7, 0.8]])
    dist, sweeps = P.dijkstra_worlds(ctx, prm.row_ptr, prm.col, prm.states, None, None, [int(ids[1])])
    want = oprm.graph.dijkstra([int(ids[1])])
    np.testing.assert_array_equal(dist, want)
    assert np.isfinite(dist[ids[0]])


# ---------------------------------------------------------------------------------------------- SSSP
def test_dijkstra_golden_through_gpu(ctx):  # pto_graph.rs:625-678
    def run(g, finals, **kw):
        xy, nvid, rp, col, ev = g.export(0)
        d, _ = P.dijkstra_worlds(ctx, rp, col, xy, None, None, finals)
        return list(d)
    from test_oracle_golden import minimal_graph, grid_graph, oriented_grid_graph, diamond_graph_2_worlds
    assert run(minimal_graph(), [1]) == [1.0, 0.0]
    assert run(grid_graph(), [8]) == [4.0, 3.0, 2.0, 3.0, 2.0, 1.0, 2.0, 1.0, 0.0]
    assert run(grid_graph(), [7, 5]) == [3.0, 2.0, 1.0, 2.0, 1.0, 0.0, 1.0, 0.0, 1.0]
    assert run(grid_graph(), []) == [INF] * 9
    assert run(oriented_grid_graph(), [3]) == [2.0, 1.0, INF, 0.0]
    g = diamond_graph_2_worlds()
    xy, nvid, rp, col, ev = g.export(0)
    d, _ = P.dijkstra_worlds(ctx, rp, col, xy, nvid, P.words_from_bits([[1, 0], [0, 1], [1, 1]]), [[3], [3]])
    s2 = math.sqrt(2.0)
    assert d.tolist() == [[s2 + s2, INF, s2, 0.0], [s2 + s2, s2, INF, 0.0]]


def _grow_pto(omap, start, goals, max_step, search_radius, n_min, n_max=100000):
    goal = O.SquareGoal(goals, 0.05)
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    rc = pto.grow_graph(start, goal, max_step, search_radius, n_min, n_max)
    assert rc == 0, rc
    return pto


def test_qmdp_costs_shelf_config2(ctx):
    """BASELINE config 2 shape: PTO growth (sequential, CPU side) on a 2-shelf map, then plan_qmdp on the GPU"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[0][0]) - 0.06, float(zp[0][1])), [1, 0]), ((float(zp[1][0]) - 0.06, float(zp[1][1])), [0, 1])]
    pto = _grow_pto(omap, (-0.8, -0.8), goals, 0.05, 5.0, 2000)
    want = pto.plan_qmdp()
    xy, nvid, rp, col, ev = pto.graph.export(0)
    finals = [pto.reach.get_final_nodes_for_world(w) for w in range(2)]
    got, sweeps = P.dijkstra_worlds(ctx, rp, col, xy, nvid, pmap.world_validities_words(), finals)
    np.testing.assert_array_equal(got, want)   # bit-exact f64
    assert np.isfinite(want).any()
    # the extracted QMDP policy (qmdp_policy_extractor.rs:176-199: react_qmdp(&[-0.8, -0.8], &vec![0.5, 0.5], 0.2)): start node by
    # the device 1-NN, walk over the device-computed cost table; common path and per-world paths as in the reference
    tree = P.KdTree(ctx, xy)
    for start, belief, horizon in (((-0.8, -0.8), [0.5, 0.5], 0.2), ((-0.8, -0.8), [0.9, 0.1], 1.0), ((0.2, 0.1), [0.3, 0.7], 0.5)):
        ids, _, ties = tree.nearest_neighbor([start])
        assert ties[0] == 1 and ids[0] == pto.kdtree.nearest_neighbor(start)
        paths, n_common = P.react_qmdp(ctx, rp, col, xy, got, int(ids[0]), belief, horizon)
        want_paths = pto.react_qmdp(start, belief, horizon)
        for w in range(2):
            np.testing.assert_array_equal(xy[paths[w]], want_paths[w])
        assert n_common >= 1 and len(paths[0]) > n_common


def test_qmdp_costs_door(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    pto = _grow_pto(omap, (-0.8, -0.8), [((0.8, 0.8), [1, 1, 1, 1])], 0.05, 5.0, 3000)
    want = pto.plan_qmdp()
    xy, nvid, rp, col, ev = pto.graph.export(0)
    finals = [pto.reach.get_final_nodes_for_world(w) for w in range(4)]
    got, _ = P.dijkstra_worlds(ctx, rp, col, xy, nvid, pmap.world_validities_words(), finals)
    np.testing.assert_array_equal(got, want)
    assert not np.array_equal(want[0], want[3])


# ---------------------------------------------------------------------------------------------- belief space
def _belief_compare(ctx, omap, pmap, pto, b0):
    pto.build_belief_graph(b0)
    want = pto.compute_expected_costs_to_goals()
    typ, bid, rp_b, col_b = pto.belief_graph.export()
    opol = pto.extract_policy()
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits))
    B = len(plan.beliefs)
    np.testing.assert_array_equal(plan.beliefs, pto.beliefs())
    np.testing.assert_array_equal(plan.dist.reshape(-1), want)                 # bit-exact expected costs
    np.testing.assert_array_equal(plan.type.reshape(-1).astype(np.int32), typ)  # Unknown / Action / Observation
    assert plan.expected_cost == opol.expected_costs
    np.testing.assert_array_equal(plan.policy_node.astype(np.int64) * B + plan.policy_belief, opol.original)
    np.testing.assert_array_equal(plan.policy_parent.astype(np.int64), opol.parent)
    np.testing.assert_array_equal(np.nonzero(plan.policy_leaf)[0], opol.leafs)
    return plan, want, typ


def test_belief_planning_door(ctx):
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    pto = _grow_pto(omap, (-0.8, -0.8), [((0.8, 0.8), [1, 1, 1, 1])], 0.05, 5.0, 3000)
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [0.1, 0.1, 0.1, 0.7])
    assert (typ == O.OBSERVATION).any() and (typ == O.ACTION).any() and np.isfinite(want[0])
    assert plan.policy_leaf.sum() >= 2


def test_belief_planning_shelf_config2(ctx):
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[0][0]) - 0.06, float(zp[0][1])), [1, 0]), ((float(zp[1][0]) - 0.06, float(zp[1][1])), [0, 1])]
    pto = _grow_pto(omap, (-0.8, -0.8), goals, 0.05, 5.0, 2000)
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [0.2, 0.8])
    assert np.isfinite(want[0])


def test_belief_planning_shelf_8_goals_config3(ctx):
    """BASELINE config 3 shape (8 goal zones, B = 255 reachable beliefs) on a stand-in map, at the reference's literal
    n_iter_min = 5000 (main.rs:104, grow_graph(start (0,-1)-like, 0.1, 2.0, 5000, 100000), main.rs:757-799)"""
    Z = 8
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    pto = _grow_pto(omap, (0.0, -0.9), goals, 0.1, 2.0, 5000)
    assert pto.n_it() >= 5000
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [1.0 / Z] * Z)
    assert len(plan.beliefs) == 255 and np.isfinite(want[0]) and plan.policy_leaf.sum() == Z
    # QMDP on the same roadmap: 8 world-view dijkstras at once
    xy, nvid, rp, col, ev = pto.graph.export(0)
    finals = [pto.reach.get_final_nodes_for_world(w) for w in range(Z)]
    got, _ = P.dijkstra_worlds(ctx, rp, col, xy, nvid, pmap.world_validities_words(), finals)
    np.testing.assert_array_equal(got, pto.plan_qmdp())
    # the same two problems through the sweeps over global memory (the path of roadmaps too large for colsolve.cu)
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 1)
    try:
        fin_ids, fin_bits = pto.reach.finals()
        plan2 = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, [1.0 / Z] * Z, fin_ids, P.words_from_bits(fin_bits))
        got2, _ = P.dijkstra_worlds(ctx, rp, col, xy, nvid, pmap.world_validities_words(), finals)
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    np.testing.assert_array_equal(plan2.dist, plan.dist)
    np.testing.assert_array_equal(got2, got)


def test_belief_planning_12_goals_config4_full_size(ctx):
    """BASELINE config 4 shape at FULL size (12 goal zones, B = 4095 beliefs, grow_graph(.., 0.05, 5.0, 5000, ..), main.rs:386-411) on a
    stand-in map.  The reference's materialised belief graph is 'typically intractable' here (main.rs:385) and so is the oracle's, so
    the 1.9e7-entry result is checked through what can be verified independently:
      * the 12 fully informed beliefs have no observation edges, their columns are plain shortest paths: bit-equal to the oracle's
        `dijkstra` towards that world's final nodes;
      * the table is a fixed point (a second run gives the same bits) and informing never hurts: the root's expected cost under the
        uniform belief is at least the probability-weighted cost of the informed columns;
      * the policy ends in 12 leaves, one per world."""
    Z = 12
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.2)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    pto = _grow_pto(omap, (0.0, -0.9), goals, 0.05, 5.0, 5000)
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    b0 = [1.0 / Z] * Z
    plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits))
    assert plan.beliefs.shape == (4095, Z) and plan.dist.shape == (len(xy), 4095)
    informed = {int(np.argmax(b)): k for k, b in enumerate(plan.beliefs) if b.max() == 1.0}
    assert sorted(informed) == list(range(Z))
    for z, b in informed.items():
        want = pto.graph.dijkstra(pto.reach.get_final_nodes_for_world(z))
        np.testing.assert_array_equal(plan.dist[:, b], want, err_msg="world %d" % z)
        assert (plan.type[:, b] != P.NODE_OBSERVATION).all()
    again = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits))
    np.testing.assert_array_equal(again.dist, plan.dist)
    # the two independent schedules -- on-chip column solver level by level (colsolve.cu) and order-free sweeps over the table in
    # global memory (graph.cu) -- must give every one of the 1.9e7 entries bit for bit
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 1)
    try:
        sweeps = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits))
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    np.testing.assert_array_equal(sweeps.dist, plan.dist)
    np.testing.assert_array_equal(sweeps.type, plan.type)
    root = plan.dist[0, 0]
    assert np.isfinite(root) and root >= sum(plan.dist[0, informed[z]] for z in range(Z)) / Z - 1e-12
    assert plan.expected_cost == root and int(plan.policy_leaf.sum()) == Z
    leaf_worlds = sorted(int(np.argmax(plan.beliefs[b])) for b in plan.policy_belief[plan.policy_leaf != 0])
    assert leaf_worlds == list(range(Z))


def _hand_built_roadmap(omap, n_nodes, radius, goal_states, goal_masks, seed):
    """a small roadmap over `omap` assembled by hand in the oracle's PTO (graph + reachability): random valid states + the goal
    states, bi-edges between all pairs within `radius` whose transition the oracle validates; finals = the goal nodes"""
    rng = np.random.default_rng(seed)
    pts = []
    while len(pts) < n_nodes:
        c = rng.uniform(-0.95, 0.95, (4 * n_nodes, 2))
        pts += [p for p, v in zip(c, omap.state_validity(c)) if v >= 0][: n_nodes - len(pts)]
    for g in goal_states:                                  # the nearest valid state left of / around the goal position
        cand = np.array([[g[0] - dx, g[1] + dy] for dx in (0.0, 0.03, 0.06, 0.09, -0.03) for dy in (0.0, 0.03, -0.03)])
        ok = np.nonzero(omap.state_validity(cand) >= 0)[0]
        assert len(ok), g
        pts.append(cand[ok[0]])
    pts = np.array(pts)
    vids = omap.state_validity(pts)
    assert (vids >= 0).all()
    pto = O.PTO(omap, util.LOW, util.UP)
    ones = [1] * omap.n_worlds
    for p, v in zip(pts, vids):
        pto.graph.add_node([float(p[0]), float(p[1])], int(v))
    pto.reach.set_root(ones)
    for _ in range(len(pts) - 1):
        pto.reach.add_node(ones)
    d = np.linalg.norm(pts[:, None, :] - pts[None, :, :], axis=2)
    ii, jj = np.nonzero(np.triu(d <= radius, 1))
    ev = omap.edge_validity(pts[ii], pts[jj])
    for a, b, v in zip(ii, jj, ev):
        if v >= 0:
            pto.graph.add_bi_edge(int(a), int(b), int(v))
    for k, m in enumerate(goal_masks):
        pto.reach.add_final_node(n_nodes + k, list(m))
    return pto


def test_belief_planning_12_goals_full_table_vs_oracle(ctx):
    """BASELINE config 4's belief space (12 goal zones, B = 4095 reachable beliefs) on a roadmap small enough for the oracle's
    MATERIALISED belief graph (pto.rs:185-259): every one of the V x 4095 expected costs, every node type and the whole policy
    must equal the reference algorithm's"""
    Z = 12
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.3)
    zp = omap.zone_positions()
    goal_states = [(float(zp[z][0]) - 0.08, float(zp[z][1])) for z in range(Z)]
    goal_masks = [[1 if k == z else 0 for k in range(Z)] for z in range(Z)]
    pto = _hand_built_roadmap(omap, 280, 0.3, goal_states, goal_masks, seed=77)
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [1.0 / Z] * Z)
    assert plan.beliefs.shape == (4095, Z) and plan.dist.shape == (292, 4095)
    assert np.isfinite(want[0]) and int(plan.policy_leaf.sum()) == Z
    assert (typ == O.OBSERVATION).sum() > 1000


def test_seven_door_zones_two_mask_words(ctx):
    """7 door zones = 128 worlds: world masks are two u64 words wide (mask_words = 2) in the edge kernel's outputs, the world
    validity table, the per-world SSSP (plan_qmdp) and the reachability filter of the nearest-neighbour search"""
    occ, zones = synth.door_map(size=1024, n_rects=1500, n_zones=7, seed=23)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    assert (pmap.n_zones, pmap.n_worlds(), pmap.n_validities, pmap.mask_words) == (7, 128, 8, 2)
    np.testing.assert_array_equal(pmap.world_validities(), omap.world_validities())
    a, b = synth.edges(400_000, seed=24, max_len=0.15)
    want = _check_edges(omap, pmap, a, b)                      # ids + [n, 2]-word masks
    assert all((want == z).any() for z in range(7)) and (want == 7).any() and (want == -1).any()
    ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 1)
    try:
        _check_edges(omap, pmap, a[:100_000], b[:100_000])
    finally:
        ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)
    # node ids + masks through the indexed entry point
    tree = P.KdTree(ctx, np.concatenate([a[:50_000], b[:50_000]]), cell_size=0.02)
    fi, ti = np.arange(50_000, dtype=np.int32), np.arange(50_000, 100_000, dtype=np.int32)
    got, masks = pmap.transition_validator_nodes(fi, ti, want_masks=True)
    wv = pmap.world_validities_words()
    np.testing.assert_array_equal(got.astype(np.int64), want[:50_000])
    np.testing.assert_array_equal(masks, np.where((want[:50_000] >= 0)[:, None], wv[np.clip(want[:50_000], 0, None)], 0))
    # plan_qmdp over 128 world views of a PTO roadmap (goal valid in every world)
    pto = _grow_pto(omap, (-0.8, -0.8), [((0.8, 0.8), [1] * 128)], 0.05, 5.0, 2500)
    want_costs = pto.plan_qmdp()
    xy, nvid, rp, col, ev = pto.graph.export(0)
    finals = [pto.reach.get_final_nodes_for_world(w) for w in range(128)]
    got_costs, _ = P.dijkstra_worlds(ctx, rp, col, xy, nvid, wv, finals)
    np.testing.assert_array_equal(got_costs, want_costs)
    assert len({want_costs[w].tobytes() for w in range(128)}) > 1      # the worlds really differ
    # filtered 1-NN / radius search with 128-bit reachability masks (pto.rs:74-77), worlds on both sides of bit 64
    reach = pto.reach.all(len(xy))                                     # [V, 128] bits
    rw = P.words_from_bits(reach)
    assert rw.shape == (len(xy), 2)
    rng = np.random.default_rng(25)
    q = rng.uniform(-1, 1, (4000, 2))
    world = rng.integers(0, 128, 4000).astype(np.uint32)
    tree = P.KdTree(ctx, xy, cell_size=0.05)
    ids, dist, ties = tree.nearest_neighbor(q, reach_mask=rw, world=world)
    d = np.linalg.norm(xy[None, :, :] - q[:, None, :], axis=2)
    d_f = np.where(reach[:, world].T != 0, d, np.inf)
    best = d_f.min(1)
    for k in range(len(q)):
        if np.isfinite(best[k]):
            assert ids[k] >= 0 and reach[ids[k], world[k]] and abs(dist[k] - best[k]) <= 1e-12, k
        else:
            assert ids[k] == -1
    offs, rid = tree.nearest_neighbors(q, 0.12, reach_mask=rw, world=world)
    for k in range(0, len(q), 7):
        exp = np.nonzero((d[k] <= 0.12 - 1e-12) & (reach[:, world[k]] != 0))[0]
        got_k = rid[offs[k]:offs[k + 1]]
        assert set(exp) <= set(got_k) and all(reach[j, world[k]] for j in got_k) and (d[k, got_k] <= 0.12 + 1e-12).all()
    # the belief space of 7 doors: hash() (common.rs:352-355) wraps from 20 worlds on, reachable_belief_states silently merges
    # colliding beliefs (map_io.rs:515-546) and conditional_dijkstra then panics on the mangled successor table; the product
    # must follow the reference into the same panic, not compute something else
    small = _grow_pto(omap, (0.6, 0.6), [((0.8, 0.8), [1] * 128)], 0.05, 5.0, 200)        # 184 nodes
    small.build_belief_graph([1.0 / 128] * 128)
    assert len(small.beliefs()) == 1441                                # 3^7 = 2187 without the collisions
    with pytest.raises(RuntimeError):
        small.compute_expected_costs_to_goals()
    xy, nvid, rp, col, ev = small.graph.export(0)
    fin_ids, fin_bits = small.reach.finals()
    np.testing.assert_array_equal(pmap.reachable_belief_states([1.0 / 128] * 128), small.beliefs())
    with pytest.raises(P.PorrtError) as ei:
        P.plan_belief_space(pmap, rp, col, ev, xy, nvid, [1.0 / 128] * 128, fin_ids, P.words_from_bits(fin_bits))
    assert ei.value.code == 5


def test_c5_full_shape_every_edge(ctx):
    """BASELINE config 5 at full shape: the synthetic 8192^2 map, 6 door zones = 64 worlds, 2^24 edges from each of two seeds,
    EVERY edge against the oracle (OpenMP over edges), through coordinates, node ids (int32 and byte results) and the adjacency
    entry point; states and visibility on the same map"""
    import os
    occ, zones = synth.door_map(size=8192, n_zones=6, seed=1)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    assert pmap.n_worlds() == 64 and pmap.mask_words == 1
    threads = max(1, len(os.sched_getaffinity(0)))
    wv = pmap.world_validities_words()
    E = 1 << 24
    for seed in (2, 3):
        a, b = synth.edges(E, seed=seed)
        want, _ = omap.edge_validity_timed(a, b, threads)
        got, masks = pmap.transition_validator(a, b, want_masks=True)
        np.testing.assert_array_equal(got, want.astype(np.int32))
        np.testing.assert_array_equal(masks[:, 0], np.where(want >= 0, wv[np.clip(want, 0, None), 0], 0))
        del masks
        if seed == 2:
            assert all((want == z).any() for z in range(6)) and (want == 6).any() and (want == -1).any()
            tree = P.KdTree(ctx, np.concatenate([a, b]), cell_size=0.01)
            fi, ti = np.arange(E, dtype=np.int32), np.arange(E, 2 * E, dtype=np.int32)
            np.testing.assert_array_equal(pmap.transition_validator_nodes(fi, ti), want.astype(np.int32))
            np.testing.assert_array_equal(pmap.transition_validator_nodes(fi, ti, compact=True), want.astype(np.int8))
            # the same batch as an adjacency: row r (a "new node" b_r = vertex E + r) lists its one neighbour a_r
            rows = 1 << 20
            rp = np.zeros(2 * E + 1, np.int64)
            rp[E + 1:E + rows + 1] = np.arange(1, rows + 1)
            rp[E + rows + 1:] = rows
            np.testing.assert_array_equal(pmap.transition_validator_adjacency(rp, fi[:rows]), want[:rows].astype(np.int8))
            del tree
            pts = a[:2_000_000]
            np.testing.assert_array_equal(pmap.state_validity(pts).astype(np.int64), omap.state_validity(pts))
            wm, wp = omap.visible_zones(pts[:300_000])
            gm, gs = pmap.visible_zones(pts[:300_000])
            np.testing.assert_array_equal(gm, wm)
            np.testing.assert_array_equal(gs.astype(np.int64), wp)
            assert (wm != 0).any()
    occ, zones = util.small_door_map(256, 2)
    util.make_pair(ctx, occ, zones, P.DOOR, 0.3)                # drop the big map


def test_build_belief_graph_mock(ctx):
    """pto.rs:548-590 'mock graph growth' on a stand-in map: node 2 sees the door, belief jump only there"""
    size = 200
    occ = np.full((size, size), 255, np.uint8)
    zones = np.full((size, size), 255, np.uint8)
    occ[85:95, 150:160] = 128        # the door, around (0.55, 0.1)
    zones[85:95, 150:160] = 0
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.15)
    pto = O.PTO(omap, util.LOW, util.UP)
    pto.set_mock(2, [[0, 1], [1, 1]])
    for s, v in [([0.55, -0.8], 1), ([-0.42, -0.38], 1), ([0.54, 0.0], 1), ([0.54, 0.1], 0), ([-0.97, 0.65], 1), ([0.55, 0.9], 1)]:
        pto.graph.add_node(s, v)
    for a, b, v in [(0, 1, 1), (1, 2, 1), (2, 3, 0), (3, 5, 0), (1, 4, 1), (4, 5, 1)]:
        pto.graph.add_bi_edge(a, b, v)
    pto.reach.set_root([1, 1])
    for _ in range(5):
        pto.reach.add_node([1, 1])
    pto.reach.add_final_node(5, [1, 1])
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [0.5, 0.5])
    typ_o, bid, rp_b, col_b = pto.belief_graph.export()
    assert list(col_b[rp_b[6]:rp_b[7]]) == [7, 8]       # observation transitions (pto.rs:579)
    assert plan.type[2, 0] == P.NODE_OBSERVATION


# ---------------------------------------------------------------------------------------------- policy refinement
def _path_through_free_space(omap, rng, n_states, step):
    """a jagged polyline of valid states (what a policy path piece looks like before refinement)"""
    for _ in range(1000):
        p = rng.uniform(-0.9, 0.9, 2)
        if omap.state_validity(p[None])[0] >= 0:
            break
    pts = [p]
    while len(pts) < n_states:
        q = np.clip(pts[-1] + rng.uniform(-step, step, 2), -0.95, 0.95)
        if omap.state_validity(q[None])[0] >= 0 and omap.edge_validity(pts[-1][None], q[None])[0] >= 0:
            pts.append(q)
    return np.array(pts)


def test_refiner_is_transition_valid(ctx):
    """pto_policy_refiner.rs:395-423, batched, incl. the order in which the reference's panics would fire"""
    occ, zones = util.small_door_map(512, 3)
    occ[40:44, 40:120] = 77                                    # gray without zone id: unwrap panic
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    rng = np.random.default_rng(5)
    a = rng.uniform(-1.1, 1.1, (60_000, 2))
    b = a + rng.uniform(-0.08, 0.08, (60_000, 2))
    for compat in ([1, 1, 1, 1], [0, 1, 0, 1], [1, 0, 0, 0]):
        want = omap.refiner_transition_valid(a, b, compat)
        valid, status = pmap.is_transition_valid(a, b, compat)
        np.testing.assert_array_equal(valid.astype(np.int64), (want == 1).astype(np.int64))
        np.testing.assert_array_equal(status.astype(np.int64), np.where(want < 0, want, 0))
    assert (want == 1).any() and (want == 0).any() and (want == O.PANIC_OOB).any() and (want == O.PANIC_ZONE_UNWRAP).any()


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_refiner_partial_shortcut(ctx, kind):
    """pto_policy_refiner.rs:158-206 on stand-in maps: the speculative waves must reproduce the sequential trial-by-trial
    result bit for bit (states and number of commits), with far fewer device round trips than trials"""
    rng = np.random.default_rng(9)
    if kind == "door":
        occ, zones = util.planning_door_map(200)
        omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.5)
        compats = ([1, 1, 1], [0, 1, 1], [1, 0, 1])        # validities: zone 0, zone 1, free
    else:
        occ, zones = synth.shelf_map(200, n_rects=10, n_zones=4, seed=5)
        omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
        compats = ([1],)
    total_commits = waves_sum = trials_sum = 0
    for n_states, n_it in ((3, 50), (12, 400), (40, 1500), (90, 600)):
        path = _path_through_free_space(omap, rng, n_states, 0.08)
        for compat in compats:
            want_states, want_commits = omap.refiner_partial_shortcut(path, compat, n_it)
            assert want_commits >= 0
            got_states, commits, waves = pmap.partial_shortcut(path, compat, n_it)
            np.testing.assert_array_equal(got_states, want_states)      # bit-exact f64
            assert commits == want_commits
            assert 1 <= waves <= n_it
            total_commits += commits
            waves_sum += waves; trials_sum += n_it
    assert total_commits > 20
    assert waves_sum * 3 < trials_sum, (waves_sum, trials_sum)            # speculation pays: > 3 trials per device round trip
    # all pieces of a policy in shared waves (refine_solution's loop): same results, round trips of the slowest piece only
    pieces = [_path_through_free_space(omap, rng, n, 0.08) for n in (25, 2, 60, 9, 33, 3, 48)]
    rows = [compats[k % len(compats)] for k in range(len(pieces))]
    got, commits, waves = pmap.partial_shortcut_batch(pieces, rows, 500)
    single_waves = []
    for k, piece in enumerate(pieces):
        want_states, want_commits = omap.refiner_partial_shortcut(piece, rows[k], 500)
        np.testing.assert_array_equal(got[k], want_states)
        assert commits[k] == max(want_commits, 0)
        single_waves.append(pmap.partial_shortcut(piece, rows[k], 500)[2])
    assert waves == max(single_waves) and waves < sum(single_waves)
    # fewer than 3 states: nothing to do (pto_policy_refiner.rs:163-165)
    st, c, w = pmap.partial_shortcut(path[:2], compats[0], 100)
    np.testing.assert_array_equal(st, path[:2])
    assert (c, w) == (0, 0)


# ---------------------------------------------------------------------------------------------- multi-GPU (SURVEY 8(e))
def test_sharded_paths_multi_gpu():
    """scripts/multi_gpu_check.py under torchrun on min(2, visible GPUs) ranks: sharded PRM build / plan_qmdp / gathered edge
    masks are bit-identical to the single-GPU results and to the oracle (with one GPU only the world-1 plumbing runs)"""
    import os
    import socket
    import subprocess
    import sys
    import torch
    n = min(2, torch.cuda.device_count())
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "scripts", "multi_gpu_check.py")]
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "multi_gpu_check: ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ---------------------------------------------------------------------------------------------- explicit belief graphs
class _RecordingBeliefGraph:
    """stands in for O.BeliefGraph while the reference's hand-built test graphs are constructed: keeps the oracle graph and
    the (state, belief_id, type) / edge lists the product needs as arrays"""

    def __init__(self, beliefs):
        self.o = _ORACLE_BG(beliefs)
        self.beliefs = np.asarray(beliefs, np.float64)
        self.nodes, self.children = [], []

    def add_node(self, s, belief_id, node_type):
        self.nodes.append((tuple(s), belief_id, node_type))
        self.children.append([])
        return self.o.add_node(s, belief_id, node_type)

    def add_edge(self, a, b):
        self.children[a].append(b)
        self.o.add_edge(a, b)

    def product(self, ctx):
        rp = np.zeros(len(self.nodes) + 1, np.int64)
        for k, c in enumerate(self.children):
            rp[k + 1] = rp[k] + len(c)
        col = np.array([v for c in self.children for v in c], np.int32)
        xy = np.array([n[0] for n in self.nodes], np.float64)
        return P.BeliefGraph(ctx, rp, col, xy, [n[2] for n in self.nodes], [n[1] for n in self.nodes], self.beliefs)


_ORACLE_BG = O.BeliefGraph


def _check_policy(g, pg, d):
    opol = g.o.extract_policy(d)
    node, parent, leaf, cost = pg.extract_policy(d)
    np.testing.assert_array_equal(node.astype(np.int64), opol.original)
    np.testing.assert_array_equal(parent.astype(np.int64), opol.parent)
    np.testing.assert_array_equal(np.nonzero(leaf)[0], opol.leafs)
    assert cost == opol.expected_costs
    return opol


@pytest.mark.parametrize("which", [1, 2])
def test_conditional_dijkstra_golden_through_gpu(ctx, which, monkeypatch):  # belief_graph.rs:500-567
    import test_oracle_golden as golden
    monkeypatch.setattr(O, "BeliefGraph", _RecordingBeliefGraph)
    bs = [[0.4, 0.6], [1.0, 0.0], [0.0, 1.0]]
    g = golden.create_graph_1(bs) if which == 1 else golden.create_graph_2(bs)
    finals = [3, 10, 16] if which == 1 else [8, 17, 27]
    pg = g.product(ctx)
    d = pg.conditional_dijkstra(finals)
    np.testing.assert_array_equal(d, g.o.conditional_dijkstra(finals))        # bit-exact f64
    if which == 1:
        assert d[4] == bs[0][0] * d[5] + bs[0][1] * d[11]                      # belief_graph.rs:528
        assert d[0] < d[1] and d[4] < d[0] and d[16] < d[15]
    else:
        assert int(np.argmax(d)) == 10 and d.max() == 8.0                      # :557-560
    opol = _check_policy(g, pg, d)
    assert len(opol.leafs) == 2


def test_conditional_dijkstra_random_graphs(ctx):
    """random Action / Observation graphs (zero-length observation edges, unreachable parts, several finals) against the
    oracle's label-correcting heap version: identical bits, identical policy"""
    rng = np.random.default_rng(7)
    for trial in range(6):
        nb, nw = 6, 4
        beliefs = rng.uniform(0.05, 1.0, (nb, nw))
        beliefs[1:, :] *= rng.integers(0, 2, (nb - 1, nw)) | np.eye(nw, dtype=np.int64)[rng.integers(0, nw, nb - 1)]
        beliefs /= beliefs.sum(1, keepdims=True)
        n_base = 300 + 50 * trial
        pts = rng.uniform(-1, 1, (n_base, 2))
        g = _RecordingBeliefGraph(beliefs)
        ids = {}
        for b in range(nb):
            for k in range(n_base):
                ids[(k, b)] = g.add_node(pts[k], b, O.ACTION)
        # observation nodes: node (k, 0) observes into two other beliefs with overlapping support
        obs = set(rng.choice(n_base, n_base // 10, replace=False).tolist()) - {0}
        for k in obs:
            kids = [b for b in rng.choice(np.arange(1, nb), 2, replace=False)
                    if (np.where(beliefs[b] > 0, beliefs[0], 0.0)).sum() > 0]
            if not kids:
                continue
            g.nodes[ids[(k, 0)]] = (g.nodes[ids[(k, 0)]][0], 0, O.OBSERVATION)
            g.o = None
            for b in kids:
                g.children[ids[(k, 0)]].append(ids[(k, b)])
        # action edges between near base nodes, inside every belief, skipping observation nodes as sources
        d2 = ((pts[:, None, :] - pts[None, :, :]) ** 2).sum(-1)
        near = [np.nonzero((d2[k] < 0.03) & (np.arange(n_base) != k))[0] for k in range(n_base)]
        for b in range(nb):
            for k in range(n_base):
                if g.nodes[ids[(k, b)]][2] == O.OBSERVATION:
                    continue
                for j in near[k]:
                    g.children[ids[(k, b)]].append(ids[(int(j), b)])
        # rebuild the oracle graph with the final types / edges (types were changed after add_node above)
        og = _ORACLE_BG(beliefs)
        for s, b, t in g.nodes:
            og.add_node(s, b, t)
        for a, ch in enumerate(g.children):
            for c in ch:
                og.add_edge(a, c)
        g.o = og
        finals = [ids[(int(k), b)] for b in range(1, nb) for k in rng.choice(n_base, 2, replace=False)]
        pg = g.product(ctx)
        d = pg.conditional_dijkstra(finals)
        np.testing.assert_array_equal(d, og.conditional_dijkstra(finals))
        assert np.isfinite(d).sum() > n_base
        if np.isfinite(d[0]):
            _check_policy(g, pg, d)


def test_conditional_dijkstra_panics(ctx):
    """belief_graph.rs:130 / :140: an evaluated Observation node with p == 0 towards a child, an Unknown-typed parent of a
    reached node; neither fires when the offending node is never evaluated"""
    beliefs = [[0.5, 0.5], [1.0, 0.0], [0.0, 1.0]]
    xy = [[0, 0], [1, 0], [2, 0], [3, 0]]

    def run(types, bids, edges, finals):
        rp = np.zeros(5, np.int64)
        for a, _ in edges:
            rp[a + 1:] += 1
        col = [b for a, b in sorted(edges, key=lambda e: e[0])]
        return P.BeliefGraph(ctx, rp, col, xy, types, bids, beliefs).conditional_dijkstra(finals)

    A_, O_, U_ = P.NODE_ACTION, P.NODE_OBSERVATION, P.NODE_UNKNOWN
    # node 1 (belief 1) "observes" into belief 2: p = 0 -> panic once its child 2 is reached
    with pytest.raises(P.PorrtError) as e:
        run([A_, O_, A_, A_], [0, 1, 2, 2], [(0, 1), (1, 2), (2, 3)], [3])
    assert e.value.code == 5
    d = run([A_, O_, A_, A_], [0, 1, 2, 2], [(0, 1), (1, 2), (2, 3)], [])      # nothing reached: no evaluation, no panic
    assert np.isinf(d).all()
    with pytest.raises(P.PorrtError) as e:
        run([A_, U_, A_, A_], [0, 0, 0, 0], [(0, 1), (1, 2), (2, 3)], [3])
    assert e.value.code == 5
    d = run([A_, A_, A_, U_], [0, 0, 0, 0], [(0, 1), (1, 2), (2, 3)], [2])      # the Unknown node has no reached child
    np.testing.assert_array_equal(d, [2.0, 1.0, 0.0, np.inf])


# ---------------------------------------------------------------------------------------------- multi-modal PRM (SURVEY 8(f) rank 3)
@pytest.mark.parametrize("n_zones,start,n_iter", [(2, (-0.9, 0.0), 2500), (4, (0.0, -0.9), 1200)])
def test_mmprm_plan_vs_oracle(ctx, n_zones, start, n_iter):
    """MapShelfDomainTampPRM::plan (map_shelves_tamp_prm.rs:308-326; its tests :506-552 use plan(start, uniform belief, 0.1, 2.0,
    2500)): the oracle runs the reference algorithm and records the RNG-decided schedule; the product rebuilds every mode's PRM,
    the belief graph and the expected costs from that schedule on the GPU -- identical graph, bit-identical costs, same policy"""
    occ, zones = synth.shelf_map(200, n_zones=n_zones)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    tamp = O.TampPRM(omap, util.LOW, util.UP)
    opol = tamp.plan(start, [1.0 / n_zones] * n_zones, 0.1, 2.0, n_iter)
    sch = tamp.schedule()
    assert len(sch["mode_belief_id"]) >= n_zones + 1 and len(sch["tr_pairs"]) > 0
    dist, graph, (node, parent, leaf, cost), phase = P.mmprm_plan(pmap, sch)
    typ, bid, rp, col = tamp.belief_graph.export()
    np.testing.assert_array_equal(graph.row_ptr, rp)                       # every mode's PRM adjacency + observation edges
    np.testing.assert_array_equal(graph.col.astype(np.int64), col)
    np.testing.assert_array_equal(graph.node_type.astype(np.int32), typ)
    np.testing.assert_array_equal(graph.belief_id, bid)
    np.testing.assert_array_equal(dist, sch["expected_costs"])             # bit-exact f64
    assert np.isfinite(dist[0])
    np.testing.assert_array_equal(node.astype(np.int64), opol.original)
    np.testing.assert_array_equal(parent.astype(np.int64), opol.parent)
    np.testing.assert_array_equal(np.nonzero(leaf)[0], opol.leafs)
    assert cost == opol.expected_costs and len(opol.leafs) == n_zones


def test_edges_between_nodes_by_id(ctx):
    """porrt_edge_validity_indexed == porrt_edge_validity on the nodes' states (ids, masks, panic codes), pageable and pinned
    buffers, several pipeline chunks"""
    import torch
    occ, zones = util.small_door_map(512, 3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    pts = synth.points(50_000, seed=21)
    pts[:200] = np.random.default_rng(1).uniform(-1.2, 1.2, (200, 2))        # some nodes outside the map: panic codes
    tree = P.KdTree(ctx, pts)
    rng = np.random.default_rng(5)
    n = 1_300_000
    fi = rng.integers(0, len(pts), n).astype(np.int32)
    ti = (fi + rng.integers(1, 40, n)).astype(np.int32) % len(pts)            # short and long edges
    ti[:100_000] = np.argsort(pts[:, 0])[rng.integers(0, len(pts) - 1, 100_000)].astype(np.int32)
    want_vid, want_mask = pmap.transition_validator(pts[fi], pts[ti], want_masks=True)
    got_vid, got_mask = pmap.transition_validator_nodes(fi, ti, want_masks=True)
    np.testing.assert_array_equal(got_vid, want_vid)
    np.testing.assert_array_equal(got_mask, want_mask)
    np.testing.assert_array_equal(got_vid[:20000].astype(np.int64), omap.edge_validity(pts[fi[:20000]], pts[ti[:20000]]))
    pf, pt = torch.from_numpy(fi).pin_memory().numpy(), torch.from_numpy(ti).pin_memory().numpy()
    pv = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    got2 = pmap.transition_validator_nodes(pf, pt, vid_out=pv)
    np.testing.assert_array_equal(got2, want_vid)
    assert (want_vid >= 0).any() and (want_vid == -1).any() and (want_vid < -1).any()
    with pytest.raises(P.PorrtError):
        pmap.transition_validator_nodes(np.array([0, len(pts)], np.int32), np.array([1, 2], np.int32))


# ---------------------------------------------------------------------------------------------- empty / degenerate inputs
def test_empty_and_degenerate_inputs(ctx):
    """batches of zero, single vertices, k larger than the vertex set, graphs without edges or goals: every entry point answers
    (or refuses with an error code) instead of faulting"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    e0 = np.zeros((0, 2))
    assert len(pmap.transition_validator(e0, e0)) == 0
    assert len(pmap.state_validity(e0)) == 0
    vz, st = pmap.visible_zones(e0)
    assert len(vz) == 0 and len(st) == 0
    # one vertex
    tree = P.KdTree(ctx, np.array([[0.25, -0.5]]))
    offs, ids = tree.nearest_neighbors(e0, 0.1)
    assert list(offs) == [0] and len(ids) == 0
    offs, ids = tree.nearest_neighbors([[0.25, -0.5], [0.9, 0.9]], [0.0, 0.05])
    assert list(offs) == [0, 1, 1] and list(ids) == [0]                       # radius 0 finds the exact duplicate only
    nid, nd, ties = tree.nearest_neighbor([[0.0, 0.0], [5.0, 5.0]])
    assert list(nid) == [0, 0]
    kid, kd = tree.knn([[0.0, 0.0]], 4)                                        # k > V: the missing entries are marked
    assert kid[0, 0] == 0 and (kid[0, 1:] < 0).all() and np.isinf(kd[0, 1:]).all()
    assert len(pmap.transition_validator_nodes(np.zeros(0, np.int32), np.zeros(0, np.int32))) == 0
    # PRM with one and two samples
    for n in (1, 2):
        prm = P.PRM(pmap)
        prm.grow_graph(np.array([[0.0, 0.0], [0.01, 0.0]])[:n], 0.1, 2.0)
        oprm = O.PRM(omap, util.LOW, util.UP, seed=0)
        oprm.add_samples(np.array([[0.0, 0.0], [0.01, 0.0]])[:n], 0.1, 2.0)
        _, _, rp, col, _ = oprm.graph.export(0)
        np.testing.assert_array_equal(prm.row_ptr, rp)
        np.testing.assert_array_equal(prm.col, col)
    # value backups: a graph without edges, no goals, a goal only
    xy = np.array([[0.0, 0.0], [0.1, 0.0], [0.2, 0.0]])
    rp, col = np.zeros(4, np.int64), np.zeros(0, np.int32)
    d, _ = P.dijkstra_worlds(ctx, rp, col, xy, None, None, [1])
    np.testing.assert_array_equal(d, [np.inf, 0.0, np.inf])
    d, _ = P.dijkstra_worlds(ctx, rp, col, xy, None, None, [])
    assert np.isinf(d).all()
    g = P.BeliefGraph(ctx, rp, col, xy, [P.NODE_ACTION] * 3, [0, 0, 0], [[1.0, 0.0]])
    np.testing.assert_array_equal(g.conditional_dijkstra([2]), [np.inf, np.inf, 0.0])
    assert np.isinf(g.conditional_dijkstra([])).all()
    node, parent, leaf, cost = g.extract_policy(g.conditional_dijkstra([0]))   # the root is a goal: a policy of one node
    assert list(node) == [0] and list(parent) == [-1] and cost == 0.0


# ---------------------------------------------------------------------------------------------- BASELINE config 1: RRT* (sequential caller)
def test_rrt_star_through_per_query_wrappers(ctx):
    """rrt.rs:269-304 shape (RRT* on a MapShelfDomain, plan(start, goal, 0.1, 2.0, 2500, 10000)): the planner is sequential and
    stays on the host; run over the oracle and over the product's per-query calls it must grow the same tree"""
    import rrt_mirror as R
    occ, zones = synth.shelf_map(200, n_zones=2)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    start = [0.0, -0.8]
    zp = omap.zone_positions()
    gx = next(float(zp[0][0]) - dx for dx in (0.06, 0.1, 0.15, 0.2, 0.3) if omap.state_validity([[float(zp[0][0]) - dx, float(zp[0][1])]])[0] >= 0)
    goal = O.SquareGoal([((gx, float(zp[0][1])), [1])], 0.05)
    samples = O.Pcg64(0).sample_states(util.LOW, util.UP, 2500)
    want = R.grow_tree(R.OracleBackend(omap, start), samples, start, goal, 0.1, 2.0, 900, 2500)
    got = R.grow_tree(R.ProductBackend(pmap, start), samples, start, goal, 0.1, 2.0, 900, 2500)
    np.testing.assert_array_equal(got[0], want[0])      # states (steered samples)
    np.testing.assert_array_equal(got[1], want[1])      # parents after choose-parent and rewiring
    np.testing.assert_array_equal(got[2], want[2])      # dist_from_root, bit-exact
    assert got[3] == want[3] and len(want[3]) > 0 and len(want[0]) > 600


def test_pto_growth_through_per_query_wrappers(ctx):
    """PTO::grow_graph (pto.rs:55-139; configs 2-4 grow their roadmap with it) is sequential and stays on the host.  The oracle's
    restatement runs twice: on its own functions, and with every per-query answer -- 1-NN filtered by the reachability bit of the
    sampled world, radius search in kd order, state validity ids, the candidate edges' validity ids -- coming from the C ABI.
    Door map: validity ids differ per zone, so reachability (and with it the filter) really depends on them."""
    import rrt_mirror as R
    occ, zones = util.planning_door_map(200)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    goal = O.SquareGoal([((0.8, 0.8), [1, 1, 1, 1])], 0.05)
    ref = O.PTO(omap, util.LOW, util.UP, seed=0)
    assert ref.grow_graph((-0.8, -0.8), goal, 0.05, 5.0, 700, 100000) == 0
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    pto.set_hooks(R.ProductPTOBackend(pmap))
    assert pto.grow_graph((-0.8, -0.8), goal, 0.05, 5.0, 700, 100000) == 0
    assert pto.n_it() == ref.n_it()
    for which in (0, 1):
        for a, b in zip(pto.graph.export(which), ref.graph.export(which)):
            np.testing.assert_array_equal(a, b)              # states, node validity ids, adjacency in insertion order, edge ids
    fa, fb = pto.reach.finals(), ref.reach.finals()
    assert list(fa[0]) == list(fb[0]) and np.array_equal(np.asarray(fa[1]), np.asarray(fb[1]))
    assert len(np.unique(ref.graph.export(0)[1])) > 1        # several validity ids occur among the nodes


def test_malformed_graphs_are_refused(ctx):
    """edge targets / validity ids outside their range must come back as PORRT_ERR_INVALID_ARG, not reach a kernel"""
    occ, zones = synth.shelf_map(200, n_zones=2)
    _, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    xy = np.array([[0.0, 0.0], [0.1, 0.0], [0.2, 0.0]])
    rp = np.array([0, 1, 2, 2], np.int64)
    for bad_col in ([1, 3], [-1, 2]):
        with pytest.raises(P.PorrtError) as e:
            P.dijkstra_worlds(ctx, rp, np.array(bad_col, np.int32), xy, None, None, [2])
        assert e.value.code == 1
        with pytest.raises(P.PorrtError) as e:
            P.BeliefGraph(ctx, rp, bad_col, xy, [P.NODE_ACTION] * 3, [0, 0, 0], [[1.0, 0.0]]).conditional_dijkstra([2])
        assert e.value.code == 1
    with pytest.raises(P.PorrtError) as e:      # row_ptr not monotone
        P.dijkstra_worlds(ctx, np.array([0, 2, 1, 2], np.int64), np.array([1, 2], np.int32), xy, None, None, [2])
    assert e.value.code == 1
    with pytest.raises(P.PorrtError) as e:      # edge validity id beyond the table
        P.plan_belief_space(pmap, rp, np.array([1, 2], np.int32), np.array([0, 7], np.int32), xy, np.zeros(3, np.int32), [0.5, 0.5], [2],
                            P.words_from_bits([[1, 1]]))
    assert e.value.code == 1


def test_vertices_append_equals_full_set(ctx):
    """KdTree::add (nearest_neighbor.rs:29-46): a vertex set grown by porrt_vertices_append -- one by one and in ragged batches --
    answers radius / 1-NN / k-NN queries and ranks its kd pre-order exactly like the same set uploaded at once, and like the
    oracle's incrementally built kd-tree."""
    rng = np.random.default_rng(21)
    pts = rng.uniform(-1, 1, (3000, 2))
    pts[100] = pts[7]                                     # an exact duplicate
    q = rng.uniform(-1, 1, (500, 2))
    whole = P.KdTree(ctx, pts, cell_size=0.05)
    want_offs, want_ids = whole.nearest_neighbors(q, 0.08)
    want_nn = whole.nearest_neighbor(q)
    want_knn = whole.knn(q, 5)
    want_rank = whole.preorder_rank()
    otree = O.KdTree(pts[0], 0)
    otree.add_batch(pts[1:], 1)
    grown = P.KdTree(ctx, pts[:1], cell_size=0.05)
    k = 1
    for step in (1, 1, 1, 5, 64, 1, 700, 1, 2225):       # sums to 2999
        grown.add(pts[k:k + step])
        k += step
        if step == 1:                                     # query between appends: the grid is rebuilt for the grown set each time
            offs, ids = grown.nearest_neighbors(q[:20], 0.3)
            ooffs, oids, _ = otree_prefix_radius(pts[:k], q[:20], 0.3)
            np.testing.assert_array_equal(offs, ooffs)
            np.testing.assert_array_equal(ids, oids)
    assert k == len(pts) and grown.n == len(pts)
    offs, ids = grown.nearest_neighbors(q, 0.08)
    np.testing.assert_array_equal(offs, want_offs)
    np.testing.assert_array_equal(ids, want_ids)
    for a, b in zip(grown.nearest_neighbor(q), want_nn):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(grown.knn(q, 5), want_knn):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(grown.preorder_rank(), want_rank)
    # the oracle's kd-tree gives the same sets (ids ascending after sorting its kd-ordered lists)
    ooffs, oids, _ = otree.radius_batch(q, 0.08, cap=len(ids) + 8)
    np.testing.assert_array_equal(offs, ooffs)
    for j in range(len(q)):
        np.testing.assert_array_equal(ids[offs[j]:offs[j + 1]], np.sort(oids[ooffs[j]:ooffs[j + 1]]))
    # node ids of appended vertices are usable by the indexed edge checks
    occ, zones = synth.door_map(size=256, n_zones=2, seed=3)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    t2 = P.KdTree(ctx, pts[:10])
    t2.add(pts[10:50])
    a, b = rng.integers(0, 50, 400).astype(np.int32), rng.integers(0, 50, 400).astype(np.int32)
    np.testing.assert_array_equal(pmap.transition_validator_nodes(a, b).astype(np.int64), omap.edge_validity(pts[a], pts[b]))


def otree_prefix_radius(pts, q, r):
    """brute-force radius sets (ids ascending) over the first len(pts) vertices, with the reference's predicate sqrt(d2) <= r"""
    offs, ids = [0], []
    for p in q:
        d = np.sqrt((pts[:, 0] - p[0]) * (pts[:, 0] - p[0]) + (pts[:, 1] - p[1]) * (pts[:, 1] - p[1]))
        hit = np.nonzero(d <= r)[0]
        ids += list(hit)
        offs.append(len(ids))
    return np.asarray(offs, np.int64), np.asarray(ids, np.int32), None


def test_c_abi_harness(tmp_path):
    """the C ABI called from plain C (tests/c_abi_harness.c, gcc -std=c99), not through ctypes"""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "c_abi_harness")
    libdir = os.path.join(root, "po_rrt_b200")
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Wextra", "-pedantic", "-I", os.path.join(root, "include"),
                    os.path.join(root, "tests", "c_abi_harness.c"), "-o", exe, "-L", libdir, "-lporrt_b200", "-lm",
                    "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "c_abi_harness: ok" in r.stdout, r.stdout + r.stderr


def test_qmdp_on_resident_prm(ctx):
    """porrt_sssp_worlds_prm: world-view shortest paths on the roadmap porrt_prm_build left on the device, through both value-backup
    paths (on-chip column solver; frontier relaxation over global memory), against the oracle's dijkstra over PTOGraphWorldView on
    the same graph (pto_graph.rs:245-303)."""
    occ, zones = synth.door_map(size=512, n_rects=600, n_zones=3, seed=11)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    xy = synth.points(2500, seed=8)
    prm = P.PRM(pmap)
    prm.init(xy[:1])
    prm.grow_graph(xy[1:], 0.1, 2.0)
    V, W = len(xy), 8
    rng = np.random.default_rng(4)
    finals = [sorted(rng.choice(V, 3, replace=False).tolist()) for _ in range(W)]
    finals[5] = []                                                   # a world without final node: its row stays +inf
    got, rounds = P.dijkstra_worlds_resident_prm(pmap, V, finals)
    ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 1)
    try:
        got2, rounds2 = P.dijkstra_worlds_resident_prm(pmap, V, finals)
    finally:
        ctx.set_option(P.OPT_FORCE_GLOBAL_SWEEPS, 0)
    np.testing.assert_array_equal(got2, got)
    assert rounds > 0 and rounds2 > 0
    # the oracle: same graph, node validity id = state validity (obstacle -> an extra validity that holds in no world)
    nvid = omap.state_validity(xy).astype(np.int64)
    wv = omap.world_validities()
    none = len(wv)
    og = O.PTOGraph(validities=[list(map(int, m)) for m in wv] + [[0] * W])
    for k in range(V):
        og.add_node(xy[k], int(nvid[k]) if nvid[k] >= 0 else none)
    for u in range(V):
        for e in range(prm.row_ptr[u], prm.row_ptr[u + 1]):
            og.add_edge(u, int(prm.col[e]), 0)
    for w in range(W):
        want = og.dijkstra(finals[w], world=w) if finals[w] else np.full(V, np.inf)
        np.testing.assert_array_equal(got[w], want, err_msg="world %d" % w)
    assert np.isfinite(got).any() and np.isinf(got[5]).all()


def _py_conditional_dijkstra(row_ptr, col, xs, node_type, belief_id, beliefs, finals):
    """conditional_dijkstra's fixed point (belief_graph.rs:89-182) in plain Python floats, any state dimension: chaotic iteration from
    +inf with the reference's operand order per backup (norm2 summed in dimension order from 0.0, Observation sums in stored child
    order from 0.0) -- monotone, so it ends at the same bits as the heap version"""
    import math
    V = len(xs)
    dist = [math.inf] * V
    for f in finals:
        dist[f] = 0.0

    def norm2(a, b):
        d2 = 0.0
        for xa, xb in zip(a, b):
            dx = xb - xa
            d2 += dx * dx
        return math.sqrt(d2)

    def tp(pb, cb):
        s = 0.0
        for p, q in zip(beliefs[cb], beliefs[pb]):
            s = s + (q if p > 0.0 else 0.0)
        return s
    xs = [list(map(float, x)) for x in xs]
    cost = [[norm2(xs[u], xs[v]) for v in col[row_ptr[u]:row_ptr[u + 1]]] for u in range(V)]
    changed = True
    while changed:
        changed = False
        for u in range(V):
            kids = col[row_ptr[u]:row_ptr[u + 1]]
            if len(kids) == 0:
                continue
            if node_type[u] == O.ACTION:
                alt = min(c + dist[v] for c, v in zip(cost[u], kids))
            else:
                alt = 0.0
                for c, v in zip(cost[u], kids):
                    alt += tp(belief_id[u], belief_id[v]) * (c + dist[v])
            if alt < dist[u]:
                dist[u] = alt
                changed = True
    return np.array(dist)


@pytest.mark.parametrize("dim", [3, 7, 9])
def test_conditional_dijkstra_nd(ctx, dim):
    """BeliefGraph<N> for the other state dimensions the reference's planner is instantiated with (pto_c.rs:236-240):
    porrt_conditional_dijkstra_nd / porrt_extract_policy_graph_nd against the fixed point in plain Python floats (bit for bit), and
    -- with the extra coordinates held at zero -- against the two-dimensional entry points"""
    rng = np.random.default_rng(100 + dim)
    nb, nw, n_base = 4, 3, 120
    beliefs = np.array([[0.5, 0.3, 0.2], [0.625, 0.375, 0.0], [0.0, 0.0, 1.0], [0.0, 1.0, 0.0]])
    for flat in (False, True):
        pts = rng.uniform(-1, 1, (n_base, dim))
        if flat:
            pts[:, 2:] = 0.0
        xs, btype, bid = [], [], []
        for k in range(n_base):
            for b in range(nb):
                xs.append(pts[k]); btype.append(O.ACTION); bid.append(b)
        idx = lambda k, b: k * nb + b
        children = [[] for _ in range(n_base * nb)]
        obs = set(rng.choice(np.arange(1, n_base), n_base // 8, replace=False).tolist())
        for k in obs:                                   # belief 0 splits into {worlds 0, 1} and {world 2}
            btype[idx(k, 0)] = O.OBSERVATION
            children[idx(k, 0)] = [idx(k, 1), idx(k, 2)]
        d2 = ((pts[:, None, :] - pts[None, :, :]) ** 2).sum(-1)
        thr = np.sort(d2, axis=1)[:, 7].max()
        for k in range(n_base):
            near = np.nonzero((d2[k] <= thr) & (np.arange(n_base) != k))[0][:12]
            for b in range(nb):
                if btype[idx(k, b)] == O.ACTION:
                    children[idx(k, b)] = [idx(int(j), b) for j in near]
        row_ptr = np.zeros(len(children) + 1, np.int64)
        row_ptr[1:] = np.cumsum([len(c) for c in children])
        col = np.array([c for ch in children for c in ch], np.int32)
        finals = [idx(int(k), b) for b in (1, 2, 3) for k in rng.choice(n_base, 2, replace=False)]
        xs = np.array(xs)
        g = P.BeliefGraph(ctx, row_ptr, col, xs, btype, bid, beliefs, dim=dim)
        got = g.conditional_dijkstra(finals)
        want = _py_conditional_dijkstra(row_ptr.tolist(), col.tolist(), xs, btype, bid, beliefs.tolist(), finals)
        np.testing.assert_array_equal(got, want)
        assert np.isfinite(got[0]) and np.isfinite(got).sum() > n_base
        node, parent, leaf, cost = g.extract_policy(got)
        assert cost == got[0] and node[0] == 0 and parent[0] == -1 and leaf.sum() >= 1
        for k in range(1, len(node)):                   # every policy edge is an edge of the graph
            assert node[k] in col[row_ptr[node[parent[k]]]:row_ptr[node[parent[k]] + 1]]
        if flat:
            g2 = P.BeliefGraph(ctx, row_ptr, col, xs[:, :2].copy(), btype, bid, beliefs)
            d2d = g2.conditional_dijkstra(finals)
            np.testing.assert_array_equal(got, d2d)
            n2, p2, l2, c2 = g2.extract_policy(d2d)
            np.testing.assert_array_equal(node, n2); np.testing.assert_array_equal(parent, p2); np.testing.assert_array_equal(leaf, l2)
            assert cost == c2


@pytest.mark.parametrize("kind,Z,n_min", [("shelf", 4, 1500), ("door", 2, 2500)])
def test_refine_solution_partial_shortcut(ctx, kind, Z, n_min):
    """PTOPolicyRefiner::refine_solution(RefinmentStrategy::PartialShortCut(n)) (pto_policy_refiner.rs:85-133; main.rs:442 runs it with
    n = 1500 after every PTO plan): Policy::decompose, build_path_piece + partial_shortcut per piece, recompose and the policy's
    expected cost -- states bit for bit, same tree, same leaves, same expected cost as the oracle's restatement."""
    if kind == "shelf":
        occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
        omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
        zp = omap.zone_positions()
        goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
        pto = _grow_pto(omap, (0.0, -0.9), goals, 0.1, 2.0, n_min)
        b0 = [1.0 / Z] * Z
    else:
        occ, zones = util.planning_door_map(200)
        omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
        pto = _grow_pto(omap, (-0.8, -0.8), [((0.8, 0.8), [1, 1, 1, 1])], 0.05, 5.0, n_min)
        b0 = [0.1, 0.1, 0.1, 0.7]
    plan, _, _ = _belief_compare(ctx, omap, pmap, pto, b0)
    B = len(plan.beliefs)
    for n_it in (0, 300, 1500):
        want = pto.refine_policy_shortcut(n_it)
        got = P.refine_policy_shortcut(ctx, plan, n_it)
        assert got["xy"].tobytes() == want.xy.tobytes(), n_it                       # refined states, bit for bit
        np.testing.assert_array_equal(got["node"].astype(np.int64) * B + got["belief"], want.original)
        np.testing.assert_array_equal(got["belief"], want.belief_id)
        np.testing.assert_array_equal(got["parent"], want.parent)
        np.testing.assert_array_equal(np.nonzero(got["is_leaf"])[0], want.leafs)
        assert got["expected_cost"] == want.expected_costs, n_it
        assert int(got["is_leaf"].sum()) == int(plan.policy_leaf.sum())   # the reference's own check: pto_policy_refiner.rs:448 (leafs preserved)
    assert got["commits"] > 0 and got["expected_cost"] <= plan.expected_cost + 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("kind,Z,n_min", [("shelf", 4, 1500), ("shelf", 3, 2500), ("door", 2, 2500)])
def test_refine_solution_reparent(ctx, kind, Z, n_min):
    """PTOPolicyRefiner::refine_solution(RefinmentStrategy::Reparent(radius)) (pto_policy_refiner.rs:85-133,208-322; main.rs:221,270
    run Reparent(0.3)): build_tree + reparent(radius / 2) per piece, recompose -- all candidate transitions in one device batch, the
    label-correcting loop on the host; the recomposed policy equals the oracle's restatement node for node, cost bit for bit."""
    if kind == "shelf":
        occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
        omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
        zp = omap.zone_positions()
        goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
        pto = _grow_pto(omap, (0.0, -0.9), goals, 0.1, 2.0, n_min)
        b0 = [1.0 / Z] * Z
    else:
        occ, zones = util.planning_door_map(200)
        omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
        pto = _grow_pto(omap, (-0.8, -0.8), [((0.8, 0.8), [1, 1, 1, 1])], 0.05, 5.0, n_min)
        b0 = [0.1, 0.1, 0.1, 0.7]
    plan, _, _ = _belief_compare(ctx, omap, pmap, pto, b0)
    B = len(plan.beliefs)
    improved = False
    for radius in (0.0, 0.05, 0.15, 0.3):
        want = pto.refine_policy_reparent(radius)
        got = P.refine_policy_reparent(ctx, plan, radius)
        assert got["xy"].tobytes() == want.xy.tobytes(), radius
        np.testing.assert_array_equal(got["node"].astype(np.int64) * B + got["belief"], want.original)
        np.testing.assert_array_equal(got["belief"], want.belief_id)
        np.testing.assert_array_equal(got["parent"], want.parent)
        np.testing.assert_array_equal(np.nonzero(got["is_leaf"])[0], want.leafs)
        assert got["expected_cost"] == want.expected_costs, radius
        assert int(got["is_leaf"].sum()) == int(plan.policy_leaf.sum())   # the reference's own check: pto_policy_refiner.rs:477,507 (leafs preserved)
        assert got["tree_nodes"] >= len(plan.policy_node) and got["transitions"] >= got["tree_nodes"]   # every node is its own neighbour
        improved |= got["expected_cost"] != plan.expected_cost
    assert improved   # at least one radius changes the policy


def test_value_backups_on_a_roadmap_beyond_shared_memory(ctx):
    """27 k roadmap nodes: a value column no longer fits in shared memory, so belief-space planning and plan_qmdp run through the
    frontier relaxation over global memory (sssp_frontier.cu) WITHOUT any option being set -- against the oracle, bit for bit."""
    Z = 3
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=Z, seed=5)
    omap, pmap = util.make_pair(ctx, occ, zones, P.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(Z)]) for z in range(Z)]
    pto = _grow_pto(omap, (0.0, -0.9), goals, 0.05, 5.0, 29000)
    assert pto.graph.n_nodes() > 26000
    plan, want, typ = _belief_compare(ctx, omap, pmap, pto, [0.5, 0.3, 0.2])
    assert len(plan.beliefs) == 7 and np.isfinite(want[0])
    xy, nvid, rp, col, ev = pto.graph.export(0)
    finals = [pto.reach.get_final_nodes_for_world(w) for w in range(Z)]
    got, rounds = P.dijkstra_worlds(ctx, rp, col, xy, nvid, pmap.world_validities_words(), finals)
    np.testing.assert_array_equal(got, pto.plan_qmdp())
    assert rounds > 0
