"""Radius, 1-NN and k-NN queries against an exact brute force, on every kernel path and at every capacity edge.

Three paths answer a nearest-neighbour batch: the TMA-staged tiles of nn_tile.cu (batches of >= 2048 queries), nn.cu's warp per
query (k-NN queries the tiles leave over, up to 65536 of them) and nn.cu's thread per query (everything else, and every query
under OPT_FORCE_THREAD_PER_QUERY_NN).  Every case here runs once at a tile-sized batch and once under the option, and both runs
are compared with a numpy brute force in f64 with the reference's operation order (common.rs:203-213): dx = qx - vx,
dy = qy - vy, d2 = dx*dx + dy*dy (separate ufuncs: no FMA), a radius hit is sqrt(d2) <= r.

Which path a query took is read from the library's PORRT_DEBUG line "nn tiles: M queries, F left to the thread-per-query
kernels": each capacity case asserts F on both sides of its limit, so a case cannot pass on the wrong side of it.  The
populations are built on the host with a restatement of the cell grid (nn_vertices_set_dev, cell_coord) and counted there
before the device sees them."""
import math
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- the limits under test, restated
NT_W = 8                 # nn_tile.cu:22   cells per tile along x
NT_CAP_KNN = 768         # nn_tile.cu:25   staged vertices per k-NN tile
NR_CAP = 704             # nn_tile.cu:160  staged vertices per radius tile
NR_CCAP = 176            # nn_tile.cu:161  merged candidates of a query cell's 3 x 3 cells
NR_LCAP = 80             # nn_tile.cu:162  hits per query kept by the tile
NT_BINS = 32             # nn_tile.cu:476  d2 histogram bins of the k-NN tile
NT_SLACK = 16            # nn_tile.cu:477  candidates beyond k the k-NN tile keeps
HIST_SAT = 255           # nn_tile.cu:551  a histogram bin saturates at 255
TILE_MIN_BATCH = 2048    # nn_tile.cu:648  nn_tile_usable
STAGE_PER_QUERY = 64     # nn_tile.cu:688  staging buffer: m * 64 + 4096 hits
STAGE_EXTRA = 4096
RADIUS_WIDE_CELLS = 64   # nn.cu:386       prefix-restricted queries over more cells get a warp each ...
WIDE_MIN_BATCH = 1024    # nn.cu:555       ... in batches of at least 1024
RADIUS_STAGE_CAP = 96    # nn.cu:403       hits per query kept in the one-pass slot
ONE_PASS_MAX = 8 << 20   # nn.cu:587       leftover queries answered in one pass
SEG_REG_CAP = 256        # nn.cu:726       segment sort in registers ...
SEG_MID_CAP = 4096       # nn.cu:727       ... in shared memory, then the global radix sort
WARP_KNN_MAX = 65536     # nn.cu:1112      leftover k-NN queries that get a warp each
DBL_MAX = np.finfo(np.float64).max


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture
def probe(monkeypatch, capfd):
    """-> read(): the (M, F) pairs of the tile calls since the last read"""
    monkeypatch.setenv("PORRT_DEBUG", "1")
    capfd.readouterr()

    def read():
        err = capfd.readouterr().err
        return [(int(a), int(b)) for a, b in re.findall(r"nn tiles: (\d+) queries, (\d+) left to the thread-per-query kernels", err)]
    return read


# ---------------------------------------------------------------------------------------------- brute force
def _d2(q, v):
    dx = np.subtract(q[:, None, 0], v[None, :, 0])
    dy = np.subtract(q[:, None, 1], v[None, :, 1])
    return np.add(np.multiply(dx, dx), np.multiply(dy, dy))


def _chunks(m, n):
    step = max(1, min(m, 4_000_000 // max(n, 1)))
    for a in range(0, m, step):
        yield a, min(m, a + step)


def _passes(n, a, b, prefix, reach, world):
    ok = np.ones((b - a, n), bool)
    ids = np.arange(n)
    if prefix is not None:
        ok &= ids[None, :] < np.asarray(prefix, np.int64)[a:b, None]
    if reach is not None:
        reach = np.asarray(reach, np.uint64).reshape(n, -1)
        w = np.asarray(world, np.int64)[a:b]
        word = w // 64
        inside = word < reach.shape[1]
        bits = (reach[:, np.minimum(word, reach.shape[1] - 1)].T >> (w % 64).astype(np.uint64)[:, None]) & np.uint64(1)
        ok &= (bits == 1) & inside[:, None]
    return ok


def bf_radius(v, q, r, prefix=None, reach=None, world=None):
    v, q = np.asarray(v, np.float64), np.asarray(q, np.float64)
    r = np.broadcast_to(np.asarray(r, np.float64), (len(q),))
    counts, ids = np.zeros(len(q), np.int64), []
    with np.errstate(all="ignore"):
        for a, b in _chunks(len(q), len(v)):
            hit = (np.sqrt(_d2(q[a:b], v)) <= r[a:b, None]) & _passes(len(v), a, b, prefix, reach, world)
            counts[a:b] = hit.sum(1)
            ids.append(np.nonzero(hit)[1].astype(np.int32))
    return np.concatenate([[0], np.cumsum(counts)]), np.concatenate(ids) if ids else np.zeros(0, np.int32)


def bf_nearest(v, q, reach=None, world=None):
    """-> (id, dist, ties): smallest (d2, id), its sqrt, the number of vertices at exactly that d2; -1 / inf / 0 if none"""
    v, q = np.asarray(v, np.float64), np.asarray(q, np.float64)
    ids, dist, ties = np.full(len(q), -1, np.int32), np.full(len(q), np.inf), np.zeros(len(q), np.int32)
    with np.errstate(all="ignore"):
        for a, b in _chunks(len(q), len(v)):
            d2 = _d2(q[a:b], v)
            ok = ~np.isnan(d2) & _passes(len(v), a, b, None, reach, world)
            d2 = np.where(ok, d2, np.nan)
            any_ = ok.any(1)
            best = np.full(b - a, np.inf)
            best[any_] = np.nanmin(d2[any_], 1)
            at = ok & (d2 == best[:, None])
            ids[a:b] = np.where(any_, np.argmax(at, 1), -1)
            dist[a:b] = np.where(any_, np.sqrt(best), np.inf)
            ties[a:b] = np.where(any_, at.sum(1), 0)
    return ids, dist, ties


def bf_knn(v, q, k):
    """-> (ids [m, k], dist [m, k]): the first k of lexsort((id, d2)), NaN distances left out, padded with -1 / inf"""
    v, q = np.asarray(v, np.float64), np.asarray(q, np.float64)
    ids, dist = np.full((len(q), k), -1, np.int32), np.full((len(q), k), np.inf)
    kk = min(k, len(v))
    with np.errstate(all="ignore"):
        for a, b in _chunks(len(q), len(v)):
            d2 = _d2(q[a:b], v)
            order = np.lexsort((np.broadcast_to(np.arange(len(v)), d2.shape), np.where(np.isnan(d2), np.inf, d2)), axis=1)[:, :kk]
            dk = np.take_along_axis(d2, order, 1)
            ok = ~np.isnan(dk)
            ids[a:b, :kk] = np.where(ok, order, -1)
            dist[a:b, :kk] = np.where(ok, np.sqrt(dk), np.inf)
    return ids, dist


def check_radius(tree, v, q, r, **kw):
    woffs, wids = bf_radius(v, q, r, kw.get("prefix_limit"), kw.get("reach_mask"), kw.get("world"))
    offs, ids = tree.nearest_neighbors(q, r, cap=max(len(wids), 1), **kw)   # (one call: no retry on ERR_CAPACITY)
    np.testing.assert_array_equal(offs, woffs)
    np.testing.assert_array_equal(ids, wids)
    return woffs, wids


def check_nearest(tree, v, q, reach=None, world=None):
    got = tree.nearest_neighbor(q, reach, world)
    want = bf_nearest(v, q, reach, world)
    for g, w, name in zip(got, want, ("id", "dist", "ties")):
        np.testing.assert_array_equal(g, w, err_msg=name)
    return want


def check_knn(tree, v, q, k):
    ids, dist = tree.knn(q, k)
    wids, wdist = bf_knn(v, q, k)
    np.testing.assert_array_equal(ids, wids)
    np.testing.assert_array_equal(dist, wdist)


def both_paths(ctx, probe, check):
    """check() at the batch size given (the tiles where usable), then under OPT_FORCE_THREAD_PER_QUERY_NN.
    -> the (M, F) lines of the first run"""
    probe()
    check()
    lines = probe()
    ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 1)
    try:
        check()
    finally:
        ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 0)
    assert probe() == [], "the forced run must not touch the tiles"
    return lines


# ---------------------------------------------------------------------------------------------- host restatement of the grid
def cell_coord(v, org, cell, n_cells):
    """nn_dev.cuh cell_coord: floor((v - org) * inv_cell), NaN and negatives to 0, clamped to n_cells - 1"""
    with np.errstate(all="ignore"):
        c = np.floor(np.multiply(np.subtract(v, org), 1.0 / cell))
    c = np.where(c > 0.0, c, 0.0)
    return np.minimum(c, n_cells - 1).astype(np.int64)


def grid_of(xy, cell):
    """the grid nn_vertices_set_dev builds for an explicit cell size -> (org, (cells_x, cells_y))"""
    lo, hi = xy.min(0), xy.max(0)
    cx, cy = (int(np.floor((hi[d] - lo[d]) / cell)) + 1 for d in (0, 1))
    assert cx * cy <= 1 << 24
    return lo, (cx, cy)


def cell_counts(xy, cell):
    org, (cx, cy) = grid_of(xy, cell)
    ix, iy = cell_coord(xy[:, 0], org[0], cell, cx), cell_coord(xy[:, 1], org[1], cell, cy)
    return np.bincount(iy * cx + ix, minlength=cx * cy).reshape(cy, cx)


def populate(counts, rng, cell=1.0, disk=None):
    """vertices in cell interiors: counts[cy, cx] per cell (within `disk` of the cell's centre if given, else uniform in
    [0.05, 0.95] of the cell), ids shuffled, plus two pins at (0, 0) and ((W - 1/2) cell, (H - 1/2) cell) that fix the bounding
    box and with it the grid.  The counts are checked with the host restatement."""
    counts = np.asarray(counts)
    H, W = counts.shape
    pts = []
    for (cy, cx), n in np.ndenumerate(counts):
        if not n:
            continue
        if disk is None:
            u = rng.uniform(0.05, 0.95, (n, 2))
        else:
            a, rr = rng.uniform(0, 2 * np.pi, n), disk * np.sqrt(rng.uniform(0, 1, n))
            u = 0.5 + np.stack([rr * np.cos(a), rr * np.sin(a)], 1)
        pts.append((np.array([cx, cy]) + u) * cell)
    body = np.vstack(pts) if pts else np.zeros((0, 2))
    body = body[rng.permutation(len(body))]
    xy = np.vstack([[[0.0, 0.0], [(W - 0.5) * cell, (H - 0.5) * cell]], body])
    want = counts.copy()
    want[0, 0] += 1
    want[H - 1, W - 1] += 1
    np.testing.assert_array_equal(cell_counts(xy, cell), want)
    return xy


def queries_in(cx, cy, n, rng, cell=1.0, spread=0.15):
    return (np.array([cx, cy]) + 0.5 + rng.uniform(-spread, spread, (n, 2))) * cell


# ---------------------------------------------------------------------------------------------- 1. threshold arithmetic
R0 = 1.3407807929942596e154   # sqrt_rn(DBL_MAX): the largest r whose square is finite


@pytest.mark.parametrize("r", [3 * 5e-324, 1e-8, 1.0, 1e150, np.nextafter(R0, 0), R0, np.nextafter(R0, np.inf), 1e200, DBL_MAX])
def test_radius_threshold_ulps(ctx, probe, r):
    """vertices at exactly r, one ulp below and one ulp above, along both axes and on a diagonal, from a query at the origin;
    radii whose square overflows, underflows or is subnormal.  Where r * r overflows, d2 of a vertex at r is +inf and
    sqrt(inf) <= r fails: the reference has no hit there."""
    ds = [x for x in (np.nextafter(r, 0), r, np.nextafter(r, np.inf)) if np.isfinite(x)]
    v = [[0.0, 0.0]] + [[d, 0.0] for d in ds] + [[0.0, d] for d in ds] + [[0.6 * d, 0.8 * d] for d in ds]
    v = np.array(v)
    tree = P.KdTree(ctx, v, cell_size=max(r, 1e-300))
    m = TILE_MIN_BATCH
    q = np.zeros((m, 2))
    rad = np.full(m, r)
    rad[1:8] = [np.inf, 0.0, -0.0, -1.0, np.nan, -np.inf, np.nextafter(0, 1)]
    q[8] = [np.nan, 0.0]
    q[9] = [0.0, np.nan]
    want = {}

    def check():
        want["r"] = check_radius(tree, v, q, rad)
    lines = both_paths(ctx, probe, check)
    assert lines == [(m, 0)], lines                 # every query, radius_threshold included, ran in the tiles
    offs, ids = want["r"]
    hits = set(ids[offs[0]:offs[1]])
    with np.errstate(all="ignore"):
        passes = [bool(np.sqrt(d * d) <= r) for d in ds]   # vertex 1 + j sits at ds[j] on the x axis
    assert [1 + j in hits for j in range(len(ds))] == passes and 0 in hits
    if 1e-8 <= r <= 1e150:
        assert passes == [True, True, False]        # both sides of the threshold reached
    elif r >= 1e200:
        assert not passes[1]                        # r * r overflows: no hit at exactly r
    if r > 1e-150:   # (below, d2 underflows to 0 while |dx| > r: the oracle's kd-tree prunes such vertices by coordinate)
        oracle = O.KdTree(v[0], 0)
        oracle.add_batch(v[1:], 1)
        for t in (0, 1, 2, 3, 5, 8):
            assert sorted(oracle.nearest_neighbors(q[t], float(rad[t]))) == list(ids[offs[t]:offs[t + 1]])


def test_radius_finite_r_with_overflowing_d2(ctx, probe):
    """r = 1e200, a vertex 1e160 away: d2 = 1e320 overflows to +inf and sqrt(inf) <= 1e200 is false, so it is no hit.  A
    threshold of +inf for a finite r let it through on every path."""
    v = np.array([[0.0, 0.0], [1e160, 0.0], [0.0, -1e160], [1e100, 1e100]])
    tree = P.KdTree(ctx, v, cell_size=1e200)
    q = np.zeros((TILE_MIN_BATCH, 2))

    def check():
        offs, ids = check_radius(tree, v, q, 1e200)
        assert list(ids[offs[0]:offs[1]]) == [0, 3]
    assert both_paths(ctx, probe, check) == [(TILE_MIN_BATCH, 0)]


# ---------------------------------------------------------------------------------------------- 2. grid geometry
def _all_queries(ctx, probe, tree, v, q, r, ks=(1, 8)):
    def check():
        check_radius(tree, v, q, r)
        check_nearest(tree, v, q)
        for k in ks:
            if k > 1:
                check_knn(tree, v, q, k)
    return both_paths(ctx, probe, check)


@pytest.mark.parametrize("cell", [0.1, 0.125])
def test_vertices_and_queries_on_cell_boundaries(ctx, probe, cell):
    """a lattice of vertices at multiples of a non-dyadic (0.1) and a dyadic (0.125) cell, queries on the lattice, on its
    midpoints and outside the bounding box on every side and corner; radius = one cell (exact hits along the axes, ties of
    four everywhere)"""
    rng = np.random.default_rng(1)
    g = np.arange(24) * cell
    v = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    span = g[-1]
    inner = v[rng.integers(0, len(v), 1200)]
    mids = inner + cell / 2
    out = []
    for sx in (-1, 0, 1):
        for sy in (-1, 0, 1):
            if sx or sy:
                out.append(np.array([span / 2 + sx * (span / 2 + 3 * cell), span / 2 + sy * (span / 2 + 3 * cell)]) + rng.uniform(-cell, cell, (40, 2)))
    q = np.vstack([inner, mids, *out, v[:8] + [[span + 10, 0]]])
    assert len(q) >= TILE_MIN_BATCH
    tree = P.KdTree(ctx, v, cell_size=cell)
    lines = _all_queries(ctx, probe, tree, v, q, cell)
    assert [m for m, _ in lines] == [len(q)] * 3


@pytest.mark.parametrize("cells_x", [1, 7, 8, 9, 15, 16, 17])
@pytest.mark.parametrize("cells_y", [1, 5])
def test_grid_widths(ctx, probe, cells_x, cells_y):
    """cells_x % 8 in {1, 7, 0} and partial last tiles; one-row and one-column grids"""
    rng = np.random.default_rng(cells_x * 10 + cells_y)
    counts = rng.integers(0, 6, (cells_y, cells_x))
    counts[0, 0] = counts[-1, -1] = 0
    v = populate(counts, rng)
    assert cell_counts(v, 1.0).shape == (cells_y, cells_x)
    q = np.vstack([rng.uniform(-0.5, [cells_x + 0.5, cells_y + 0.5], (TILE_MIN_BATCH, 2)), v[:50]])
    tree = P.KdTree(ctx, v, cell_size=1.0)
    _all_queries(ctx, probe, tree, v, q, rng.uniform(0, 1.2, len(q)), ks=(1, 3, 8))


@pytest.mark.parametrize("shape", ["one", "identical", "horizontal", "vertical"])
def test_degenerate_sets(ctx, probe, shape):
    rng = np.random.default_rng(3)
    if shape == "one":
        v = np.array([[0.25, -0.5]])
    elif shape == "identical":
        v = np.tile([[0.3, 0.7]], (500, 1))
    elif shape == "horizontal":
        v = np.stack([rng.uniform(-1, 1, 700), np.full(700, 0.2)], 1)
    else:
        v = np.stack([np.full(700, -0.4), rng.uniform(-1, 1, 700)], 1)
    q = np.vstack([rng.uniform(-1.5, 1.5, (TILE_MIN_BATCH, 2)), v[:20]])
    tree = P.KdTree(ctx, v, cell_size=0.05)
    _all_queries(ctx, probe, tree, v, q, 0.1, ks=(1, 2, 32))
    if shape == "identical":
        _, _, ties = tree.nearest_neighbor(q[:4])
        assert (ties == 500).all()


@pytest.mark.parametrize("offset", [1e6, 1e12])
@pytest.mark.parametrize("cell", [0.01, 2.0 ** -7])
def test_large_coordinate_offsets(ctx, probe, offset, cell):
    """a unit square at 1e6 and at 1e12: the cell of a vertex comes from floor((v - org) * inv_cell), the ring bound of the
    k-NN search from org + c * cell; queries on and next to cell boundaries"""
    rng = np.random.default_rng(int(math.log10(offset)))
    v = offset + rng.uniform(0, 1, (3000, 2))
    b = offset + np.floor(rng.uniform(0, 1, (600, 1)) / cell) * cell
    q = np.vstack([offset + rng.uniform(-0.1, 1.1, (1500, 2)),
                   np.hstack([b, offset + rng.uniform(0, 1, (600, 1))]),
                   np.hstack([np.nextafter(b, -np.inf), offset + rng.uniform(0, 1, (600, 1))])])
    tree = P.KdTree(ctx, v, cell_size=cell)
    _all_queries(ctx, probe, tree, v, q, cell * 0.9, ks=(1, 4, 16))


def test_ring_bound_at_a_rounded_cell_side(ctx, probe):
    """cell 0.1: x = 0.3 lies in cell 3 (0.3 * 10 rounds to 3) while the side of cell 3 computed as 3 * 0.1 is 0.30000000000000004.
    A query at 0.29999999999999993 (cell 2) has vertex B one ulp to its left and vertex A = 0.3 one ulp to its right, equally far;
    A has the lower id, so it is the nearest (2 ties).  A bound that trusts org + c * cell ends the ring search after the query's
    own cell with B; the relative 1e-9 shrink it once had does not help at a bound of 2 ulps.  k = 2 adds a vertex on the query.
    800 vertices at x in [0.65, 0.85] overfill the k-NN tile, so k = 2 goes to the warp kernel; 1-NN is certified by the tile,
    which sees all 3 x 3 cells; forced, the thread kernel answers both."""
    qx = np.nextafter(0.3, 0)
    assert cell_coord(0.3, 0.0, 0.1, 10) == 3 and cell_coord(qx, 0.0, 0.1, 10) == 2 and 3 * 0.1 > 0.3
    rng = np.random.default_rng(15)
    v = np.array([[0.3, 0.0], [np.nextafter(qx, 0), 0.0], [qx, 0.0], [0.0, 0.0], [0.95, 0.0]])
    v = np.vstack([v, np.stack([rng.uniform(0.65, 0.85, 800), np.zeros(800)], 1)])
    assert grid_of(v, 0.1)[1] == (10, 1)
    q = np.tile([[qx, 0.0]], (TILE_MIN_BATCH, 1))
    tree = P.KdTree(ctx, v[[0, 1, 3, 4]], cell_size=0.1)

    def check1():
        ids, _, ties = check_nearest(tree, v[[0, 1, 3, 4]], q)
        assert ids[0] == 0 and ties[0] == 2
    assert both_paths(ctx, probe, check1) == [(len(q), 0)]
    tree = P.KdTree(ctx, v, cell_size=0.1)

    def check2():
        check_knn(tree, v, q, 2)
        assert list(tree.knn(q[:1], 2)[0][0]) == [2, 0]
    assert both_paths(ctx, probe, check2) == [(len(q), len(q))]


_NONFINITE_SPAN = textwrap.dedent("""
    import numpy as np, po_rrt_b200 as P
    ctx = P.Context(0)
    for xy in ([[-1e308, 0.0], [1e308, 0.0]], [[0.0, -1e308], [0.0, 1e308]], [[-DBL, -DBL], [DBL, DBL]]):
        try:
            P.KdTree(ctx, np.array(xy))
        except P.PorrtError as e:
            assert e.code == 1, e
        else:
            raise SystemExit("accepted")
    tree = P.KdTree(ctx, np.array([[-1e308, 0.0]]))
    tree.add([[1e308, 0.0]])
    try:
        tree.nearest_neighbor([[0.0, 0.0]])
    except P.PorrtError as e:
        assert e.code == 1, e
    else:
        raise SystemExit("accepted after add")
    tree.set(np.array([[0.0, 0.0], [1.0, 1.0]]))
    assert tree.nearest_neighbor([[0.9, 0.9]])[0][0] == 1
    print("refused")
""").replace("DBL", repr(float(DBL_MAX)))


def test_bounding_box_span_overflow_is_refused():
    """corners near -DBL_MAX and +DBL_MAX: a span of +inf used to keep the cell-size loop going forever; now it is refused.
    Run in a child process so that a regression fails on the timeout instead of stalling the suite."""
    r = subprocess.run([sys.executable, "-c", _NONFINITE_SPAN], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "refused" in r.stdout, r.stdout + r.stderr


def test_nan_vertices_are_refused(ctx):
    """fmin / fmax skip NaN, so a NaN vertex passed the non-finite check and was binned into cell 0 where no query found it"""
    for bad in ([np.nan, 0.0], [0.0, np.nan], [np.inf, 0.0], [0.0, -np.inf]):
        v = np.array([[0.0, 0.0], bad, [1.0, 1.0]])
        with pytest.raises(P.PorrtError) as e:
            P.KdTree(ctx, v)
        assert e.value.code == 1
    tree = P.KdTree(ctx, np.random.default_rng(0).uniform(-1, 1, (5000, 2)))
    tree.add([[0.5, 0.5], [np.nan, np.nan]])
    with pytest.raises(P.PorrtError) as e:
        tree.nearest_neighbors(np.zeros((4, 2)), 0.1)
    assert e.value.code == 1
    v = np.array([[0.0, 0.0], [1.0, 1.0]])
    tree.set(v)
    check_nearest(tree, v, [[0.9, 0.8]])


# ---------------------------------------------------------------------------------------------- 3. capacity edges
def test_tile_batch_threshold(ctx, probe):
    rng = np.random.default_rng(4)
    v = rng.uniform(-1, 1, (5000, 2))
    tree = P.KdTree(ctx, v, cell_size=0.05)
    for m in (TILE_MIN_BATCH - 1, TILE_MIN_BATCH):
        q = rng.uniform(-1, 1, (m, 2))
        lines = _all_queries(ctx, probe, tree, v, q, 0.04, ks=(1, 5))
        assert [mm for mm, _ in lines] == ([m] * 3 if m >= TILE_MIN_BATCH else [])


def _staged_tile_counts(n_staged, query_cell_vertices, shape=(6, 16)):
    """query cell (1, 2) of tile 0 in row 2 (query columns 0..7, staged columns 0..8, rows 1..3): query_cell_vertices in the
    query cell, the rest of n_staged in columns 5..8 of rows 1..3, out of every query cell's reach"""
    counts = np.zeros(shape, np.int64)
    counts[2, 1] = query_cell_vertices
    fill = n_staged - query_cell_vertices
    counts[1:4, 5:9] = fill // 12
    counts[1:4, 5:9].flat[:fill % 12] += 1
    assert counts[1:4, 0:9].sum() == n_staged and counts[1:4, 0:3].sum() == query_cell_vertices
    return counts


@pytest.mark.parametrize("n_staged", [NR_CAP, NR_CAP + 1])
def test_radius_tile_staging_cap(ctx, probe, n_staged):
    rng = np.random.default_rng(n_staged)
    v = populate(_staged_tile_counts(n_staged, 20), rng)
    q = queries_in(1, 2, TILE_MIN_BATCH, rng)
    tree = P.KdTree(ctx, v, cell_size=1.0)
    assert bf_radius(v, q, 0.3)[0][-1] > TILE_MIN_BATCH
    lines = both_paths(ctx, probe, lambda: check_radius(tree, v, q, 0.3))
    assert lines == [(len(q), 0 if n_staged <= NR_CAP else len(q))]


@pytest.mark.parametrize("n_staged", [NT_CAP_KNN, NT_CAP_KNN + 1])
def test_knn_tile_staging_cap(ctx, probe, n_staged):
    """k > 1 needs the staged tile; k = 1 reads an unstaged one from global memory"""
    rng = np.random.default_rng(n_staged)
    v = populate(_staged_tile_counts(n_staged, 20), rng)
    q = queries_in(1, 2, TILE_MIN_BATCH, rng)
    tree = P.KdTree(ctx, v, cell_size=1.0)
    assert both_paths(ctx, probe, lambda: check_knn(tree, v, q, 4)) == [(len(q), 0 if n_staged <= NT_CAP_KNN else len(q))]
    assert both_paths(ctx, probe, lambda: check_nearest(tree, v, q)) == [(len(q), 0)]


@pytest.mark.parametrize("n_cand", [NR_CCAP, NR_CCAP + 1])
def test_radius_candidates_per_query_cell(ctx, probe, n_cand):
    rng = np.random.default_rng(n_cand)
    counts = np.zeros((6, 16), np.int64)
    counts[1:4, 0:3] = (n_cand - 20) // 8
    counts[1:4, 0:3].flat[[0, 1, 2, 3, 5, 6, 7, 8][:(n_cand - 20) % 8]] += 1
    counts[2, 1] = 20
    counts[2, 5] = 30                     # another query cell of the tile, with few candidates
    assert counts[1:4, 0:3].sum() == n_cand
    v = populate(counts, rng)
    q = np.vstack([queries_in(1, 2, TILE_MIN_BATCH, rng), queries_in(5, 2, 300, rng)])
    tree = P.KdTree(ctx, v, cell_size=1.0)
    lines = both_paths(ctx, probe, lambda: check_radius(tree, v, q, 0.3))
    assert lines == [(len(q), 0 if n_cand <= NR_CCAP else TILE_MIN_BATCH)]


@pytest.mark.parametrize("n_hits", [NR_LCAP, NR_LCAP + 1, RADIUS_STAGE_CAP, RADIUS_STAGE_CAP + 1])
def test_hits_per_query(ctx, probe, n_hits):
    """every query sees exactly n_hits: the tile keeps NR_LCAP of them, the thread-per-query slot RADIUS_STAGE_CAP (beyond it a
    second walk writes the list to its place)"""
    rng = np.random.default_rng(n_hits)
    counts = np.zeros((6, 16), np.int64)
    counts[2, 1] = n_hits
    counts[2, 3] = 7
    v = populate(counts, rng, disk=0.1)
    q = queries_in(1, 2, TILE_MIN_BATCH, rng, spread=0.03)
    offs, _ = bf_radius(v, q, 0.2)
    assert (np.diff(offs) == n_hits).all()
    # as many queries without hits, in an empty cell: the m * 64 + 4096 staging buffer then holds every list
    q = np.vstack([q, queries_in(10, 4, TILE_MIN_BATCH, rng)])
    assert len(q) * STAGE_PER_QUERY + STAGE_EXTRA >= TILE_MIN_BATCH * n_hits
    tree = P.KdTree(ctx, v, cell_size=1.0)
    lines = both_paths(ctx, probe, lambda: check_radius(tree, v, q, 0.2))
    assert lines == [(len(q), 0 if n_hits <= NR_LCAP else TILE_MIN_BATCH)]


@pytest.mark.parametrize("n_hits", [STAGE_PER_QUERY, 72])
def test_radius_staging_buffer_full(ctx, probe, n_hits):
    """4096 queries with n_hits each: at 64 the m * 64 + 4096 staging buffer holds them all; at 72 the warps that reserve
    after it is full (32 queries x 72 hits each) send their queries on, and the total comes from the scan"""
    rng = np.random.default_rng(n_hits)
    counts = np.zeros((12, 24), np.int64)
    cells = [(1 + 3 * a, 1 + 3 * b) for a in range(8) for b in range(4)]
    for cx, cy in cells:
        counts[cy, cx] = n_hits
    v = populate(counts, rng, disk=0.1)
    q = np.vstack([queries_in(cx, cy, 128, rng, spread=0.03) for cx, cy in cells])
    m = len(q)
    tree = P.KdTree(ctx, v, cell_size=1.0)
    assert (np.diff(bf_radius(v, q, 0.2)[0]) == n_hits).all()
    lines = both_paths(ctx, probe, lambda: check_radius(tree, v, q, 0.2))
    cap = m * STAGE_PER_QUERY + STAGE_EXTRA
    fit = min(m // 32, cap // (32 * n_hits))
    assert lines == [(m, m - 32 * fit)]
    assert (lines[0][1] == 0) == (n_hits == STAGE_PER_QUERY)


@pytest.mark.parametrize("m", [WIDE_MIN_BATCH - 1, WIDE_MIN_BATCH])
@pytest.mark.parametrize("r", [5.6, 5.8])
def test_prefix_queries_over_many_cells(ctx, probe, m, r):
    """prefix-restricted queries whose cell cover is 12 x 5 = 60 (<= 64) or 13 x 5 = 65 cells, in batches below and at the
    size that gives the wide ones a warp each"""
    rng = np.random.default_rng(int(r * 10) + m)
    counts = rng.integers(3, 12, (5, 20))
    v = populate(counts, rng)
    q = np.stack([rng.integers(6, 13, m) + 0.25, rng.uniform(0.1, 4.9, m)], 1)
    rr = r * 1.000000001 + 1e-300
    cover = (cell_coord(q[:, 0] + rr, 0.0, 1.0, 20) - cell_coord(q[:, 0] - rr, 0.0, 1.0, 20) + 1) * 5
    assert (cover == (60 if r == 5.6 else 65)).all() and ((cover > RADIUS_WIDE_CELLS) == (r == 5.8)).all()
    prefix = rng.integers(0, len(v) + 1, m).astype(np.uint32)
    prefix[:4] = [0, 1, len(v), len(v) + 10]
    tree = P.KdTree(ctx, v, cell_size=1.0)
    both_paths(ctx, probe, lambda: check_radius(tree, v, q, r, prefix_limit=prefix))


@pytest.mark.parametrize("n_hits", [SEG_REG_CAP, SEG_REG_CAP + 1, SEG_MID_CAP, SEG_MID_CAP + 1])
def test_radius_list_sort_segments(ctx, probe, n_hits):
    """lists the thread-per-query kernels fill in cell order and sort by id: in registers up to 256 entries, in shared memory up
    to 4096, by the global radix sort beyond"""
    rng = np.random.default_rng(n_hits)
    a, rr = rng.uniform(0, 2 * np.pi, n_hits), 2.0 * np.sqrt(rng.uniform(0, 1, n_hits))
    v = np.vstack([[[-3.0, -3.0], [3.0, 3.0]], np.stack([rr * np.cos(a), rr * np.sin(a)], 1)])
    v = v[np.r_[0, 1, 2 + rng.permutation(n_hits)]]
    q = rng.uniform(-0.01, 0.01, (TILE_MIN_BATCH, 2))
    tree = P.KdTree(ctx, v, cell_size=0.5)
    assert (np.diff(bf_radius(v, q, 2.05)[0]) == n_hits).all()
    lines = both_paths(ctx, probe, lambda: check_radius(tree, v, q, 2.05))
    assert lines == [(len(q), len(q))]


@pytest.mark.parametrize("n_dup", [NT_SLACK + 8, NT_SLACK + 9, HIST_SAT, HIST_SAT + 1, 300])
def test_knn_candidate_list_and_histogram(ctx, probe, n_dup):
    """k = 8 with n_dup exact duplicates as the nearest vertices: the tile keeps k + 16 candidates (the k-th place then falls
    inside the tie group), one more sends the query on; a histogram bin saturates at 255 (and must not wrap)"""
    k = 8
    rng = np.random.default_rng(n_dup)
    counts = np.zeros((6, 16), np.int64)
    counts[2, 3] = 10
    v = populate(counts, rng)
    dup = np.tile([[1.7, 2.5]], (n_dup, 1))
    v = np.vstack([v[:2], dup, v[2:]])
    v = v[np.r_[0, 1, 2 + rng.permutation(len(v) - 2)]]
    q = np.tile([[1.5, 2.5]], (TILE_MIN_BATCH, 1))
    tree = P.KdTree(ctx, v, cell_size=1.0)
    lines = both_paths(ctx, probe, lambda: check_knn(tree, v, q, k))
    assert lines == [(len(q), 0 if n_dup <= k + NT_SLACK else len(q))]
    d, dd = np.sqrt(_d2(q[:1], v))[0], np.sqrt(_d2(q[:1], dup[:1]))[0, 0]
    assert (d == dd).sum() == n_dup and (d < dd).sum() == 0


@pytest.mark.parametrize("m", [WARP_KNN_MAX, WARP_KNN_MAX + 1])
def test_knn_leftover_warp_limit(ctx, probe, m):
    """queries far outside the box cannot be certified by the tiles: all m come back, a warp each up to 65536, else a thread"""
    rng = np.random.default_rng(m)
    v = populate(rng.integers(0, 4, (10, 10)), rng)
    q = np.stack([np.full(m, -100.0) + rng.uniform(-1, 1, m), rng.uniform(3, 7, m)], 1)
    q[::97, 1] = np.round(q[::97, 1])
    tree = P.KdTree(ctx, v, cell_size=1.0)

    def check():
        check_nearest(tree, v, q)
        check_knn(tree, v, q, 3)
    assert both_paths(ctx, probe, check) == [(m, m), (m, m)]


def test_k_range(ctx, probe):
    """k across the KMAX = 1 / 8 / 32 instantiations of all three k-NN kernels; k = 0 and k = 33 are refused"""
    rng = np.random.default_rng(9)
    v = np.vstack([rng.uniform(-1, 1, (6000, 2)), 0.01 * rng.standard_normal((1500, 2)) + [0.4, 0.4]])
    q = np.vstack([rng.uniform(-1.2, 1.2, (3000, 2)), 0.01 * rng.standard_normal((500, 2)) + [0.4, 0.4]])
    tree = P.KdTree(ctx, v, cell_size=0.03)
    for k in (1, 2, 7, 8, 9, 16, 31, 32):
        lines = both_paths(ctx, probe, lambda: check_knn(tree, v, q, k))
        assert len(lines) == 1 and 0 < lines[0][1] < len(q)
    for k in (0, 33):
        with pytest.raises(P.PorrtError):
            tree.knn(q[:10], k)


def test_one_pass_limit(ctx):
    """8 << 20 leftover queries are answered in one pass, one more in a count pass and a fill pass: the same lists as the same
    queries in chunks, and as the brute force on a sample"""
    rng = np.random.default_rng(10)
    v = rng.uniform(-1, 1, (20_000, 2))
    tree = P.KdTree(ctx, v, cell_size=0.02)
    q = rng.uniform(-1, 1, (ONE_PASS_MAX + 1, 2))
    ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 1)
    try:
        big = tree.nearest_neighbors(q, 0.01, cap=4 * len(q))
        edge = tree.nearest_neighbors(q[:ONE_PASS_MAX], 0.01, cap=4 * len(q))
        parts = [tree.nearest_neighbors(q[a:a + (1 << 21)], 0.01) for a in range(0, len(q), 1 << 21)]
    finally:
        ctx.set_option(P.OPT_FORCE_THREAD_PER_QUERY_NN, 0)
    offs, ids = big
    np.testing.assert_array_equal(edge[0], offs[:ONE_PASS_MAX + 1])
    np.testing.assert_array_equal(edge[1], ids[:offs[ONE_PASS_MAX]])
    np.testing.assert_array_equal(np.concatenate([p[1] for p in parts]), ids)
    np.testing.assert_array_equal(np.diff(offs), np.concatenate([np.diff(p[0]) for p in parts]))
    sample = np.r_[np.arange(0, len(q), 4099), len(q) - 1]
    woffs, wids = bf_radius(v, q[sample], 0.01)
    for j, t in enumerate(sample):
        np.testing.assert_array_equal(ids[offs[t]:offs[t + 1]], wids[woffs[j]:woffs[j + 1]])


# ---------------------------------------------------------------------------------------------- 4. ties
TIE = np.array([[3, 4], [-3, 4], [3, -4], [-3, -4], [4, 3], [-4, 3], [4, -3], [-4, -3], [5, 0], [-5, 0], [0, 5], [0, -5]], np.float64)


@pytest.mark.parametrize("cell,expect_left", [(8.0, 0), (1.0, TILE_MIN_BATCH)])
def test_equidistant_sets(ctx, probe, cell, expect_left):
    """twelve vertices at distance exactly 5 of the query, some duplicated: 40 copies of one (two per lane for eight lanes of
    the warp kernel) and 1-3 of the others, with decoys in their cells.  cell = 8: the tile certifies them (thread kernel of
    nn_tile.cu); cell = 1: they lie three to five rings out and the warp kernel answers; forced: the thread kernel of nn.cu.
    Reach filters mask part of the tie group, the lowest id included."""
    rng = np.random.default_rng(int(cell))
    c = np.array([20.0, 20.0])
    pts = [c + t for t in TIE for _ in range(1 + (hash(tuple(t)) % 3))]
    pts += [c + TIE[4]] * 40
    pts += list(c + TIE * 1.01 + rng.uniform(-0.3, 0.3, (12, 2)))                # decoys, a little farther out
    pts += list(rng.uniform(0, 40, (200, 2)) * [1, 1])
    pts = [p for p in pts if np.hypot(*(p - c)) >= 5.0]
    v = np.vstack([[[0.0, 0.0], [44.0, 44.0]], np.array(pts)[rng.permutation(len(pts))]])
    q = np.tile(c, (TILE_MIN_BATCH, 1))
    n_tie = int((np.sqrt(_d2(q[:1], v))[0] == 5.0).sum())
    assert n_tie >= 52
    tree = P.KdTree(ctx, v, cell_size=cell)
    reach = np.ones(len(v), np.uint64)
    tied = np.nonzero(np.sqrt(_d2(q[:1], v))[0] == 5.0)[0]
    reach[tied[::3]] = 0
    world = np.zeros(len(q), np.uint32)
    world[1::2] = 1                                   # world 1: nothing passes

    def check():
        ids, _, ties = check_nearest(tree, v, q)
        assert ties[0] == n_tie and ids[0] == tied[0]
        ids, _, ties = check_nearest(tree, v, q, reach, world)
        assert ties[0] == n_tie - len(tied[::3]) and ids[0] == tied[1] and ids[1] == -1 and ties[1] == 0
        for k in (5, 16, 32):
            check_knn(tree, v, q, k)
    lines = both_paths(ctx, probe, check)
    assert lines[:2] == [(len(q), expect_left), (len(q), len(q) // 2 if expect_left == 0 else len(q))]


# ---------------------------------------------------------------------------------------------- 5. filters
@pytest.mark.parametrize("words", [1, 2, 3])
def test_prefix_and_reach_filters(ctx, probe, words):
    rng = np.random.default_rng(words)
    v = rng.uniform(-1, 1, (4000, 2))
    m = TILE_MIN_BATCH + 100
    q = np.vstack([rng.uniform(-1, 1, (m - 200, 2)), v[:200]])
    reach = rng.integers(0, 2 ** 63, (len(v), words), dtype=np.uint64) | (rng.integers(0, 2, (len(v), words)).astype(np.uint64) << np.uint64(63))
    worlds = np.array([0, 63, 64, 127, 128, 64 * words - 1, 64 * words, 64 * words + 5], np.uint32)
    world = worlds[rng.integers(0, len(worlds), m)]
    prefix = rng.integers(0, len(v) + 1, m).astype(np.uint32)
    prefix[:5] = [0, 1, len(v), len(v) + 1, 0xffffffff]
    tree = P.KdTree(ctx, v, cell_size=0.04)

    def check():
        check_radius(tree, v, q, 0.035, prefix_limit=prefix)
        check_radius(tree, v, q, 0.035, reach_mask=reach, world=world)
        check_radius(tree, v, q, 0.035, prefix_limit=prefix, reach_mask=reach, world=world)
        check_nearest(tree, v, q, reach, world)
    both_paths(ctx, probe, check)
    oracle = O.KdTree(v[0], 0)
    oracle.add_batch(v[1:], 1)
    ok = world < 64                                    # the oracle's filtered nearest takes one mask word per vertex
    if words == 1:
        want = oracle.nearest_batch(q[ok], reach[:, 0], world[ok])
        np.testing.assert_array_equal(tree.nearest_neighbor(q[ok], reach, world[ok])[0], want)


# ---------------------------------------------------------------------------------------------- 6. appended sets
def test_appended_sets(ctx, probe):
    """set, query at tile size (merge scripts built), add (inside and beyond the old box), query again: the grid and the merge
    scripts are rebuilt for the whole set"""
    rng = np.random.default_rng(12)
    v = rng.uniform(-1, 1, (3000, 2))
    q = rng.uniform(-1.5, 1.5, (TILE_MIN_BATCH + 7, 2))
    tree = P.KdTree(ctx, v, cell_size=0.05)

    def check():
        check_radius(tree, v, q, 0.04)
        check_nearest(tree, v, q)
        check_knn(tree, v, q, 6)
    both_paths(ctx, probe, check)
    for extra in (rng.uniform(-1, 1, (500, 2)), rng.uniform(-1.5, 1.5, (1, 2)), rng.uniform(1, 1.5, (700, 2))):
        tree.add(extra)
        v = np.vstack([v, extra])
        both_paths(ctx, probe, check)
