"""The policy refiners (refine.cu) against the oracle at the trial loop's piece, chain and panic edges, and Reparent at its radius
boundaries on both candidate searches.

partial_shortcut runs its whole trial loop in shortcut_loop_kernel: one CTA per piece (at most 1024 states), shortcut states
written with a 128-thread stride, the `&&` chain decided 32 transitions at a time by a ballot ("the first non-1 wins; a panic
counts only if the chain reaches it"), compatibility rows indexed by piece while trials are indexed by the active-piece list, and
on a panic the host reports the lowest panicking piece and leaves every caller state untouched.  Each case here is compared with
the oracle bit for bit (states, commits, error codes), and the cases that claim a situation run through mirror_shortcut, a Python
restatement of the trial loop that records what each trial exercised: the case then asserts that its situation occurred.

Reparent finds each tree node's radius / 2 candidates with an all-pairs sweep in kd pre-order (trees of up to
PORRT_OPT_REPARENT_BRUTE_MAX_NODES nodes, 4096 by default) or with the kd search; both must give the oracle's KdTree hits in the
oracle's order (the order decides heap ties in the label-correcting loop).  Every reparent case runs on both searches, at radii
taken from the plan's own geometry: a belief-graph child exactly at the build_tree radius, and two consecutive path nodes exactly
at radius / 2, each also at the next double below."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util

pytestmark = pytest.mark.gpu

# ---- the limits under test, restated
SHORTCUT_MAX_STATES = 1024   # refine.cu  SHORTCUT_MAX_STATES
SHORTCUT_THREADS = 128       # refine.cu  SHORTCUT_THREADS: stride of the shortcut-state loops
CHAIN_CHUNK = 32             # refine.cu  one ballot decides 32 transitions of the chain
MAX_PAIRS = 1 << 26          # refine.cu  reparent candidate transitions of one call
ERR_INVALID_ARG, ERR_PANIC, ERR_UNSUPPORTED = 1, 5, 6
ALL_BRUTE, ALL_KD, DEFAULT = 1 << 40, 0, -1   # PORRT_OPT_REPARENT_BRUTE_MAX_NODES values
INF = float("inf")


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------------------------- mirror of partial_shortcut
class Coverage:
    """what the trials of a case exercised (counts per situation; panic codes reached / left unreached)"""

    def __init__(self):
        self.n = dict.fromkeys(("n_tr>=33", "n_tr>=129", "stop>=32", "commit n_tr>128", "reject n_tr>128", "unreached panic",
                                "unreached panic same chunk", "reached panic", "reached panic>=32"), 0)
        self.reached, self.unreached = set(), set()

    def record(self, n_tr, first, decision, res):
        self.n["n_tr>=33"] += n_tr >= 33
        self.n["n_tr>=129"] += n_tr >= 129
        self.n["stop>=32"] += decision != 1 and first >= CHAIN_CHUNK
        self.n["commit n_tr>128"] += decision == 1 and n_tr > SHORTCUT_THREADS
        self.n["reject n_tr>128"] += decision == 0 and n_tr > SHORTCUT_THREADS
        if decision == 0:
            later = np.flatnonzero(res[first + 1:] < -1) + first + 1
            if len(later):
                self.n["unreached panic"] += 1
                self.n["unreached panic same chunk"] += int(later[0]) // CHAIN_CHUNK == first // CHAIN_CHUNK
                self.unreached.update(int(c) for c in res[later])
        if decision < -1:
            self.n["reached panic"] += 1
            self.n["reached panic>=32"] += first >= CHAIN_CHUNK
            self.reached.add(decision)

    def need(self, *names):
        for k in names:
            assert self.n[k] > 0, "the case never exercised %r: %s" % (k, self.n)


def mirror_shortcut(omap, states, compat, n_iterations, seed, cov):
    """pto_policy_refiner.rs:158-206 restated: trials from DiscreteSampler(seed) (O.Pcg64(seed).gen_range_usize), every
    transition of a trial checked with the oracle's is_transition_valid, then the `&&` chain: the first non-1 decides.
    -> (states, commits) or (None, panic code)"""
    st = np.array(states, np.float64).reshape(-1, 2)
    L = len(st)
    if L <= 2:
        return st, 0
    rng = O.Pcg64(seed)
    commits = 0
    for _ in range(n_iterations):
        joint = rng.gen_range_usize(2)
        a = rng.gen_range_usize(L - 2)
        b = a + 2 + rng.gen_range_usize(L - a - 2)
        n_tr = b - a
        lam = np.arange(n_tr, dtype=np.float64) / float(n_tr)
        cut = st[a:b].copy()
        cut[:, joint] = st[a, joint] * (1.0 - lam) + st[b, joint] * lam          # a * (1 - lambda) + b * lambda, no FMA
        res = omap.refiner_transition_valid(cut, np.concatenate([cut[1:], st[b:b + 1]]), compat)
        stop = np.flatnonzero(res != 1)
        first = int(stop[0]) if len(stop) else n_tr
        decision = int(res[first]) if len(stop) else 1
        cov.record(n_tr, first, decision, res)
        if decision < -1:
            return None, decision
        if decision == 1:
            st[a:b] = cut
            commits += 1
    return st, commits


# ---------------------------------------------------------------------------------------------- maps and pieces
# Lanes: a path piece runs along y = y0 with a 1-px jitter and dips under "patches" drawn just above the lane.  A shortcut of the
# jittered coordinate y flattens the dip and crosses the patch: obstacle or excluded zone -> the chain stops there (0), gray
# without zone / two adjacent zones -> a panic, reached or not depending on what comes first.
DIP, RAMP, INSET, HALF = 0.06, 0.03, 0.012, 0.016
LANES = {                                    # y0: [(x1, x2, patch)]
    "free": (0.78, [(-0.5, -0.4, "obstacle"), (-0.15, -0.05, "zone0"), (0.2, 0.3, "obstacle"), (0.55, 0.65, "zone0")]),
    "unwrap": (0.5, [(-0.55, -0.47, "obstacle"), (-0.45, -0.35, "unwrap"), (0.1, 0.2, "zone0"), (0.5, 0.6, "unwrap")]),
    "multi": (0.22, [(-0.6, -0.5, "zone0"), (-0.1, -0.04, "obstacle"), (-0.03, 0.07, "multi"), (0.45, 0.55, "multi")]),
}
UNWRAP_SPOT = (-0.4, 0.5)                    # the middle of the lane "unwrap" patch at x in [-0.45, -0.35]


def _lane_y(name, x):
    y0, dips = LANES[name]
    y = np.full_like(x, y0)
    for x1, x2, _ in dips:
        down = np.clip((x - (x1 - RAMP)) / RAMP, 0, 1) * np.clip(((x2 + RAMP) - x) / RAMP, 0, 1)
        y = y - DIP * down
    return y


def lane_piece(name, L, x0=-0.92, x1=0.92, seed=0):
    x = np.linspace(x0, x1, L)
    y = _lane_y(name, x) + np.random.default_rng(seed + 1000 * L).uniform(-0.003, 0.003, L)
    return np.ascontiguousarray(np.stack([x, y], 1))


def _px(H, W, x, y):
    ppm = W / 2.0                                                      # map on [-1, 1]^2 (Map::to_pixel, map_io.rs:91)
    return int((H - 1) - (y + 1.0) * ppm), int((x + 1.0) * ppm)


def lanes_map(H, W, kind):
    """door (kind DOOR: zones 0, 1, 2; n_validities 4) or shelf (low obstacles 180 as patches) map with the lanes' patches"""
    occ = np.full((H, W), 255, np.uint8)
    zones = np.full((H, W), 255, np.uint8)

    def rect(xa, xb, ya, yb, v, z=255):
        i0, j0 = _px(H, W, xa, yb)
        i1, j1 = _px(H, W, xb, ya)
        occ[i0:i1 + 1, j0:j1 + 1] = v
        zones[i0:i1 + 1, j0:j1 + 1] = z
    for name, (y0, dips) in LANES.items():
        for x1, x2, patch in dips:
            xa, xb, ya, yb = x1 + INSET, x2 - INSET, y0 - HALF, y0 + HALF
            if kind == P.SHELF:
                rect(xa, xb, ya, yb, 0 if patch == "obstacle" else 180)
            elif patch == "obstacle":
                rect(xa, xb, ya, yb, 0)
            elif patch == "unwrap":
                rect(xa, xb, ya, yb, 77)
            elif patch == "multi":
                xm = 0.5 * (xa + xb)
                rect(xa, xm, ya, yb, 128, 1)
                rect(xm, xb, ya, yb, 128, 2)
            else:
                rect(xa, xb, ya, yb, 128, int(patch[-1]))
    if kind == P.SHELF:
        zones[:] = 255
        for z, (x, y) in enumerate([(-0.8, -0.8), (0.8, -0.8)]):
            i, j = _px(H, W, x, y)
            zones[i - 2:i + 2, j - 2:j + 2] = z
    rect(-0.8, -0.6, -0.8, -0.6, 0)                                    # an obstacle away from every lane
    return occ, zones


def border_piece(L, seed=0):
    """a vertical piece along the far border x = 1: every state at x = 1 - 2^-52 or 1 - 2^-51 is inside the map (x + 1 rounds
    below 2), but a shortcut of x between them can round to 1 - 2^-53, whose x + 1 rounds to 2.0: pixel column W, PANIC_OOB"""
    rng = np.random.default_rng(seed)
    x = np.where(rng.random(L) < 0.5, 1.0 - 2.0 ** -52, 1.0 - 2.0 ** -51)
    y = np.linspace(-0.9, -0.3, L)
    return np.ascontiguousarray(np.stack([x, y], 1))


@pytest.fixture(scope="module")
def door_maps():
    return lanes_map(512, 512, P.DOOR)


@pytest.fixture(scope="module")
def shelf_maps():
    return lanes_map(512, 512, P.SHELF)


def _pair(ctx, maps, kind):
    return util.make_pair(ctx, maps[0], maps[1], kind, 0.3)


DOOR_ROWS = ([1, 1, 1, 1], [0, 1, 1, 1], [1, 0, 0, 1])     # validities: zone 0, zone 1, zone 2, free
SHELF_ROWS = ([1],)


# ---------------------------------------------------------------------------------------------- device calls
def raw_batch(ctx, pieces, rows, n_iterations, seed, ptr=None):
    """porrt_partial_shortcut_batch on caller buffers -> (rc, message, states after, commits after); commits start at -7"""
    if ptr is None:
        ptr = np.zeros(len(pieces) + 1, np.int32)
        ptr[1:] = np.cumsum([len(p) for p in pieces])
    ptr = np.ascontiguousarray(ptr, np.int32)
    st = np.ascontiguousarray(np.concatenate([np.reshape(p, (-1, 2)) for p in pieces]) if len(pieces) else np.zeros((1, 2)), np.float64)
    rw = np.ascontiguousarray(np.asarray(rows, np.uint8))
    commits = np.full(len(ptr) - 1, -7, np.int32)
    waves = C.c_int32(-7)
    rc = ctx.lib.porrt_partial_shortcut_batch(ctx.h, P.api._p(st), P.api._p(ptr), len(ptr) - 1, P.api._p(rw), int(n_iterations),
                                              C.c_uint64(int(seed)), P.api._p(commits), C.byref(waves))
    msg = (ctx.lib.porrt_last_error(ctx.h) or b"").decode() if rc else ""
    return rc, msg, st, commits


def check_batch(ctx, omap, pieces, rows, n_iterations, seed=0, cov=None):
    """device batch == oracle per piece (states bit for bit, commits); a panic anywhere: PORRT_ERR_PANIC naming the lowest
    panicking piece's code, caller states untouched, commits zeroed.  cov: also run the mirror and require it to agree.
    -> the oracle's (states, rc) per piece"""
    want = [omap.refiner_partial_shortcut(p, rows[k], n_iterations, seed) for k, p in enumerate(pieces)]
    if cov is not None:
        for k, p in enumerate(pieces):
            m_st, m_rc = mirror_shortcut(omap, p, rows[k], n_iterations, seed, cov)
            assert m_rc == want[k][1], (k, m_rc, want[k][1])
            if m_rc >= 0:
                assert m_st.tobytes() == want[k][0].tobytes(), k
    before = np.concatenate([np.reshape(p, (-1, 2)) for p in pieces]).copy()
    rc, msg, st, commits = raw_batch(ctx, pieces, rows, n_iterations, seed)
    panics = [c for _, c in want if c < 0]
    if panics:
        assert rc == ERR_PANIC, (rc, msg)
        assert "(code %d)" % panics[0] in msg, (msg, panics)
        assert st.tobytes() == before.tobytes()                       # the caller's states stay untouched
        assert (commits == 0).all()
    else:
        assert rc == 0, msg
        off = 0
        for k, p in enumerate(pieces):
            n = len(p)
            assert st[off:off + n].tobytes() == want[k][0].tobytes(), (k, n)
            assert commits[k] == want[k][1], (k, commits[k], want[k][1])
            off += n
    return want


# ---------------------------------------------------------------------------------------------- partial_shortcut: piece lengths
LENGTHS = (3, 4, 33, 34, 129, 130, 1023, 1024)


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_piece_lengths_at_chunk_stride_and_capacity_edges(ctx, kind, door_maps, shelf_maps):
    """pieces of 3, 4, 33, 34, 129, 130, 1023 and 1024 states on lanes without panics: long trials (n_tr > 32, > 128) both commit
    and get rejected, and some chains stop at index >= 32"""
    omap, pmap = _pair(ctx, door_maps if kind == "door" else shelf_maps, P.DOOR if kind == "door" else P.SHELF)
    rows = DOOR_ROWS if kind == "door" else SHELF_ROWS
    cov = Coverage()
    for L in LENGTHS:
        piece = lane_piece("free", L, seed=L)
        assert (omap.state_validity(piece) >= 0).all()
        for row in rows:
            check_batch(ctx, omap, [piece], [row], 700, 0, cov)
            st, commits, waves = pmap.partial_shortcut(piece, row, 700)                 # the one-piece entry point
            want_st, want_c = omap.refiner_partial_shortcut(piece, row, 700)
            assert st.tobytes() == want_st.tobytes() and commits == want_c and waves == 1
    cov.need("n_tr>=33", "n_tr>=129", "stop>=32", "commit n_tr>128", "reject n_tr>128")


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_piece_limit_and_malformed_batches(ctx, kind, door_maps, shelf_maps):
    """1025 states: PORRT_ERR_UNSUPPORTED with states untouched and every out_commits entry zeroed; a decreasing piece_ptr is
    refused; n_iterations = 0 changes nothing; pieces of 0, 1 and 2 states between active ones are left as they are"""
    omap, pmap = _pair(ctx, door_maps if kind == "door" else shelf_maps, P.DOOR if kind == "door" else P.SHELF)
    row = [1] * omap.n_validities
    big, ok = lane_piece("free", SHORTCUT_MAX_STATES + 1), lane_piece("free", 40)
    pieces = [ok, big, ok]
    before = np.concatenate(pieces).copy()
    rc, msg, st, commits = raw_batch(ctx, pieces, [row] * 3, 50, 0)
    assert rc == ERR_UNSUPPORTED, (rc, msg)
    assert st.tobytes() == before.tobytes() and (commits == 0).all(), commits
    ptr = np.array([0, 40, 30, 80], np.int32)                         # decreasing
    rc, msg, st, commits = raw_batch(ctx, [ok, ok], [row] * 3, 50, 0, ptr=ptr)
    assert rc == ERR_INVALID_ARG, (rc, msg)
    assert st.tobytes() == np.concatenate([ok, ok]).tobytes()
    rc, msg, st, commits = raw_batch(ctx, pieces[:1] * 2, [row] * 2, 0, 0)
    assert rc == 0 and st.tobytes() == np.concatenate([ok, ok]).tobytes() and (commits == 0).all()
    mixed = [lane_piece("free", 34, seed=1), ok[:0], ok[:1], lane_piece("free", 130, seed=2), ok[:2], ok[:0], lane_piece("free", 33, seed=3)]
    want = check_batch(ctx, omap, mixed, [row] * len(mixed), 400, 0)
    assert [c for _, c in want] [1:3] == [0, 0] and want[3][1] > 0


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_batch_beyond_one_wave_with_a_row_per_piece(ctx, kind, door_maps, shelf_maps):
    """more than 148 active pieces (more CTAs than SMs), each with its own compatibility row, skipped short pieces interleaved so
    that a piece's CTA index and its piece index differ, 1500 trials"""
    omap, pmap = _pair(ctx, door_maps if kind == "door" else shelf_maps, P.DOOR if kind == "door" else P.SHELF)
    rng = np.random.default_rng(7)
    pieces, rows = [], []
    nv = omap.n_validities
    for k in range(200):
        if k % 5 == 2:
            pieces.append(lane_piece("free", int(rng.integers(0, 3)), seed=k))
        else:
            L = int(rng.integers(5, 90))
            x0 = float(rng.uniform(-0.92, 0.2))
            pieces.append(lane_piece("free", L, x0=x0, x1=min(0.92, x0 + 0.02 * L), seed=k))
        rows.append(np.r_[rng.integers(0, 2, nv - 1), 1] if nv > 1 else [int(k % 7 != 3)])
    want = check_batch(ctx, omap, pieces, rows, 1500, 0)
    active = [k for k, p in enumerate(pieces) if len(p) > 2]
    assert len(active) > 148 and active != list(range(len(active)))
    assert sum(c for _, c in want) > 100
    if nv > 1:   # the rows decide something: the same pieces under all-ones rows commit differently
        alt = [omap.refiner_partial_shortcut(p, [1] * nv, 1500)[1] for p in pieces]
        assert alt != [c for _, c in want]


# ---------------------------------------------------------------------------------------------- panics
def _shelf_border_pieces():
    return [border_piece(L, seed=L) for L in (34, 130, 300)]


def test_panics_reached_and_unreached_door(ctx, door_maps):
    """gray without zone (PANIC_ZONE_UNWRAP), two adjacent zones (PANIC_MULTI_ZONE) and shortcut states that round onto the far
    border (PANIC_OOB): some only behind the chain's first false (no panic, the oracle's states), some reached, one at chain index
    >= 32; every reached one is PORRT_ERR_PANIC with the oracle's code and the caller's states untouched"""
    omap, pmap = _pair(ctx, door_maps, P.DOOR)
    assert omap.state_validity([UNWRAP_SPOT])[0] == O.PANIC_ZONE_UNWRAP
    cov = Coverage()
    for name in ("unwrap", "multi"):
        for L in (34, 130, 400, 1024):
            for row in DOOR_ROWS:
                check_batch(ctx, omap, [lane_piece(name, L, seed=L)], [row], 600, 0, cov)
    for L in (34, 130, 300):
        check_batch(ctx, omap, [border_piece(L, seed=L)], [DOOR_ROWS[0]], 600, 0, cov)
    # the first transition's FROM state panics (zone unwrap) and its TO state is out of the map whichever coordinate the trial
    # interpolates (x beyond the right border, y below the bottom one; a y above the top saturates to row 0): the reference
    # checks `from` first
    first = np.array([UNWRAP_SPOT, [1.5, -1.5], [0.0, 0.0]])
    want = check_batch(ctx, omap, [first], [DOOR_ROWS[0]], 5, 0, cov)
    assert want[0][1] == O.PANIC_ZONE_UNWRAP
    cov.need("unreached panic", "unreached panic same chunk", "reached panic", "reached panic>=32")
    assert cov.reached >= {O.PANIC_ZONE_UNWRAP, O.PANIC_MULTI_ZONE, O.PANIC_OOB}, cov.reached
    assert cov.unreached >= {O.PANIC_ZONE_UNWRAP, O.PANIC_MULTI_ZONE}, cov.unreached


def test_panics_reached_and_unreached_shelf(ctx, shelf_maps):
    """the shelf domain: low obstacles stop chains (validity None), the far border panics (PANIC_OOB)"""
    omap, pmap = _pair(ctx, shelf_maps, P.SHELF)
    cov = Coverage()
    for piece in _shelf_border_pieces():
        check_batch(ctx, omap, [piece], [SHELF_ROWS[0]], 600, 0, cov)
    for L in (130, 1024):          # a lane through low obstacles that ends a few ulps inside the far border
        lane = lane_piece("free", L, x0=0.4, x1=1.0 - 2.0 ** -52, seed=L)
        check_batch(ctx, omap, [lane], [SHELF_ROWS[0]], 600, 0, cov)
    cov.need("reached panic", "reached panic>=32")
    assert cov.reached == {O.PANIC_OOB}


def test_batch_panics_name_the_lowest_piece(ctx, door_maps):
    """two pieces of one batch panic with different codes: the message names the lower-indexed piece's code, in either order,
    with clean pieces before, between and after them"""
    omap, pmap = _pair(ctx, door_maps, P.DOOR)
    row = DOOR_ROWS[0]
    clean = [lane_piece("free", L, seed=L) for L in (40, 90, 2)]
    unwrap = next(p for p in (lane_piece("unwrap", L, seed=L) for L in (130, 400, 1024)) if omap.refiner_partial_shortcut(p, row, 600)[1] == O.PANIC_ZONE_UNWRAP)
    multi = next(p for p in (lane_piece("multi", L, seed=L) for L in (130, 400, 1024)) if omap.refiner_partial_shortcut(p, row, 600)[1] == O.PANIC_MULTI_ZONE)
    for a, b, code in ((unwrap, multi, O.PANIC_ZONE_UNWRAP), (multi, unwrap, O.PANIC_MULTI_ZONE)):
        pieces = [clean[0], a, clean[1], clean[2], b, clean[0]]
        check_batch(ctx, omap, pieces, [row] * len(pieces), 600, 0)
        rc, msg, _, _ = raw_batch(ctx, pieces, [row] * len(pieces), 600, 0)
        assert rc == ERR_PANIC and "(code %d)" % code in msg, msg


# ---------------------------------------------------------------------------------------------- seeds and map shapes
SEEDS = (0, 1, (1 << 63) + 5, (1 << 64) - 1)


@pytest.mark.parametrize("seed", SEEDS)
def test_sampler_seeds_batch(ctx, seed, door_maps, shelf_maps):
    for maps, kind, rows in ((door_maps, P.DOOR, DOOR_ROWS), (shelf_maps, P.SHELF, SHELF_ROWS)):
        omap, pmap = _pair(ctx, maps, kind)
        pieces = [lane_piece("free", L, seed=L) for L in (3, 33, 2, 129, 500)]
        cov = Coverage()
        want = check_batch(ctx, omap, pieces, [rows[k % len(rows)] for k in range(len(pieces))], 800, seed, cov)
        if seed:   # a different trial list than seed 0
            assert [c for _, c in want] != [c for _, c in check_batch(ctx, omap, pieces, [rows[k % len(rows)] for k in range(len(pieces))], 800, 0)]


def test_long_transitions_on_a_4096_px_map_and_a_non_square_map(ctx):
    """sparse pieces on a 4096 x 4096 door map: every transition walks hundreds of pixels (several rounds of walk_warp's
    32-pixel steps); and a 301 x 237 map, sides no multiple of 16"""
    occ, zones = lanes_map(4096, 4096, P.DOOR)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    cov = Coverage()
    pieces = [lane_piece(name, L, seed=L) for name in ("free", "unwrap", "multi") for L in (8, 12, 33)]
    for k, p in enumerate(pieces):
        d = np.hypot(*np.diff(p, axis=0).T).max() * omap.ppm
        assert d > 100, d
        check_batch(ctx, omap, [p], [DOOR_ROWS[k % 3]], 300, 0, cov)
    assert cov.reached and cov.n["n_tr>=33"] == 0
    occ, zones = lanes_map(301, 237, P.DOOR)
    omap, pmap = util.make_pair(ctx, occ, zones, P.DOOR, 0.3)
    cov = Coverage()
    for name in ("free", "unwrap", "multi"):
        for L in (33, 130, 700):
            check_batch(ctx, omap, [lane_piece(name, L, seed=L)], [DOOR_ROWS[L % 3]], 500, 0, cov)
    cov.need("n_tr>=129", "commit n_tr>128", "reached panic")


# ---------------------------------------------------------------------------------------------- the refiners on a plan
def _door_pto(start=(-0.8, -0.8), max_step=0.05, n_min=1000, omap_=None, hooks=None):
    occ, zones = util.planning_door_map(200)
    omap = omap_ or O.GridMap(occ, zones, util.LOW, util.UP, O.DOOR, 0.3)
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    if hooks is not None:
        pto.set_hooks(hooks)
    assert pto.grow_graph(start, O.SquareGoal([((0.8, 0.8), [1, 1, 1, 1])], 0.05), max_step, 5.0, n_min, 100000) == 0
    pto.build_belief_graph([0.1, 0.1, 0.1, 0.7])
    pto.compute_expected_costs_to_goals()
    return pto, occ, zones, [0.1, 0.1, 0.1, 0.7]


def _shelf_pto():
    occ, zones = synth.shelf_map(200, n_rects=10, n_zones=4, seed=5)
    omap = O.GridMap(occ, zones, util.LOW, util.UP, O.SHELF, 0.5)
    zp = omap.zone_positions()
    goals = [((float(zp[z][0]) - 0.08, float(zp[z][1])), [1 if k == z else 0 for k in range(4)]) for z in range(4)]
    pto = O.PTO(omap, util.LOW, util.UP, seed=0)
    assert pto.grow_graph((0.0, -0.9), O.SquareGoal(goals, 0.05), 0.1, 2.0, 1500, 100000) == 0
    pto.build_belief_graph([0.25] * 4)
    pto.compute_expected_costs_to_goals()
    return pto, occ, zones, [0.25] * 4


@pytest.fixture(scope="module")
def plans():
    return {"door": _door_pto(), "shelf": _shelf_pto()}


def _device_plan(ctx, pto, occ, zones, b0):
    """upload the map and plan in belief space on the device (the refiners read the ctx's last plan); -> (pmap, plan, B)"""
    kind = pto.map.kind
    pmap = (P.Map if kind == O.DOOR else P.MapShelfDomain)(ctx, occ, util.LOW, util.UP)
    pmap.add_zones(zones, 0.3 if kind == O.DOOR else 0.5)
    xy, nvid, rp, col, ev = pto.graph.export(0)
    fin_ids, fin_bits = pto.reach.finals()
    plan = P.plan_belief_space(pmap, rp, col, ev, xy, nvid, b0, fin_ids, P.words_from_bits(fin_bits))
    opol = pto.extract_policy()
    B = len(plan.beliefs)
    np.testing.assert_array_equal(plan.policy_node.astype(np.int64) * B + plan.policy_belief, opol.original)
    return pmap, plan, B


def _same_policy(got, want, B, what):
    assert got["xy"].tobytes() == want.xy.tobytes(), what
    np.testing.assert_array_equal(got["node"].astype(np.int64) * B + got["belief"], want.original, err_msg=str(what))
    np.testing.assert_array_equal(got["parent"], want.parent, err_msg=str(what))
    np.testing.assert_array_equal(np.nonzero(got["is_leaf"])[0], want.leafs, err_msg=str(what))
    assert got["expected_cost"] == want.expected_costs, what


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_refine_policy_shortcut_sampler_seeds(ctx, plans, kind):
    pto, occ, zones, b0 = plans[kind]
    pmap, plan, B = _device_plan(ctx, pto, occ, zones, b0)
    costs = set()
    for seed in SEEDS:
        want = pto.refine_policy_shortcut(600, seed)
        got = P.refine_policy_shortcut(ctx, plan, 600, seed)
        _same_policy(got, want, B, seed)
        costs.add(want.expected_costs)
    assert len(costs) > 1     # the seed reaches the trials


def _reparent_both_searches(ctx, pto, plan, B, radius, force_large=False):
    """Reparent(radius) with every tree on the all-pairs sweep and with every tree on the kd search: both equal the oracle
    and each other (tree sizes and candidate counts included) -> the device result"""
    want = pto.refine_policy_reparent(radius)
    res = []
    try:
        if force_large:
            ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 1)
        for brute in (ALL_BRUTE, ALL_KD):
            ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, brute)
            got = P.refine_policy_reparent(ctx, plan, radius)
            _same_policy(got, want, B, (radius, brute))
            res.append(got)
    finally:
        ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, DEFAULT)
        ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)
    assert (res[0]["tree_nodes"], res[0]["transitions"]) == (res[1]["tree_nodes"], res[1]["transitions"]), radius
    return res[0]


def _norm2(a, b):                    # common.rs:203-213
    dx, dy = b[0] - a[0], b[1] - a[1]
    return math.sqrt(dx * dx + dy * dy)


@pytest.mark.parametrize("kind", ["door", "shelf"])
def test_reparent_radius_boundaries_on_both_searches(ctx, plans, kind):
    """build_tree's `d <= radius` with a belief-graph child exactly at the radius, and reparent's radius / 2 with two consecutive
    path nodes exactly at it (radius = 2 * their distance: the halving is exact), each also at the next double below; plus the
    default threshold at Reparent(0.3)"""
    pto, occ, zones, b0 = plans[kind]
    pmap, plan, B = _device_plan(ctx, pto, occ, zones, b0)
    xy = pto.graph.export(0)[0]
    _, _, rp, col = pto.belief_graph.export()
    pieces, _ = P.policy_decompose(plan.policy_parent)
    bg = plan.policy_node.astype(np.int64) * B + plan.policy_belief
    # ---- build_tree: a child of a path node, not on the piece, at exactly the radius
    tree_edge = 0
    tried = 0
    for piece in pieces:
        on_piece = set(int(bg[k]) for k in piece)
        for k in piece:
            s = xy[plan.policy_node[k]]
            for c in col[rp[bg[k]]:rp[bg[k] + 1]]:
                d = _norm2(s, xy[int(c) // B])
                if int(c) in on_piece or d == 0.0 or tried >= 6:
                    continue
                tried += 1
                at = _reparent_both_searches(ctx, pto, plan, B, d)
                below = _reparent_both_searches(ctx, pto, plan, B, np.nextafter(d, 0.0))
                tree_edge += at["tree_nodes"] > below["tree_nodes"]
    assert tried > 0 and tree_edge > 0, "no child at exactly the radius changed a tree"
    # ---- reparent: two consecutive path nodes at exactly radius / 2; pick pairs whose d^2 is above fl(r2 * r2), so only the
    # prefilter's margin keeps them (an exact d^2 <= r2^2 test would drop them)
    pairs = 0
    for piece in pieces:
        for u, v in zip(piece[:-1], piece[1:]):
            a, b = xy[plan.policy_node[u]], xy[plan.policy_node[v]]
            d = _norm2(a, b)
            dx, dy = b[0] - a[0], b[1] - a[1]
            if d == 0.0 or not d * d < dx * dx + dy * dy or pairs >= 3:
                continue
            pairs += 1
            at = _reparent_both_searches(ctx, pto, plan, B, 2.0 * d)
            below = _reparent_both_searches(ctx, pto, plan, B, np.nextafter(2.0 * d, 0.0))
            assert at["transitions"] > below["transitions"] or at["tree_nodes"] != below["tree_nodes"], d
    assert pairs > 0
    # ---- the default threshold
    want = pto.refine_policy_reparent(0.3)
    got = P.refine_policy_reparent(ctx, plan, 0.3)
    _same_policy(got, want, B, 0.3)
    assert _reparent_both_searches(ctx, pto, plan, B, 0.3)["transitions"] == got["transitions"]


def test_reparent_unbounded_radius_and_pair_limit(ctx, plans):
    """radius = inf on a small roadmap (every descendant in the tree, every pair a candidate) equals the oracle on both
    searches; on the full roadmap the pairs exceed 2^26 and the call is refused with PORRT_ERR_UNSUPPORTED"""
    pto, occ, zones, b0 = _door_pto(start=(0.3, -0.2), max_step=0.1, n_min=30)
    pmap, plan, B = _device_plan(ctx, pto, occ, zones, b0)
    got = _reparent_both_searches(ctx, pto, plan, B, INF)
    assert got["transitions"] > got["tree_nodes"]
    pto, occ, zones, b0 = plans["door"]
    pmap, plan, B = _device_plan(ctx, pto, occ, zones, b0)
    _, _, rp, col = pto.belief_graph.export()
    for brute in (ALL_BRUTE, ALL_KD):
        ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, brute)
        try:
            with pytest.raises(P.PorrtError) as e:
                P.refine_policy_reparent(ctx, plan, INF)
            assert e.value.code == ERR_UNSUPPORTED and "2^26" in str(e.value)
        finally:
            ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, DEFAULT)
    assert len(rp) - 1 > math.isqrt(MAX_PAIRS)      # a tree of every belief node would hold more than 2^26 pairs


class _CleanMapAnswers:
    """PTO.set_hooks backend: the growth's per-query answers from a map without the stripe (the oracle's own primitives)"""

    def __init__(self, omap):
        self.omap, self.tree, self.states = omap, None, []

    def add_vertex(self, q, node_id):
        if self.tree is None:
            self.tree = O.KdTree(q, 0)
        else:
            self.tree.add(q, node_id)
        self.states.append(q)

    def nearest_filtered(self, q, world, reach_words):
        ok = np.flatnonzero((reach_words[:, 0] >> np.uint64(world)) & np.uint64(1))
        if not len(ok):
            return 0
        st = np.asarray(self.states)
        dx, dy = st[ok, 0] - q[0], st[ok, 1] - q[1]
        return int(ok[int(np.argmin(np.sqrt(dx * dx + dy * dy)))])

    def radius(self, q, r):
        return [int(i) for i in self.tree.nearest_neighbors(q, r)]

    def state_validity(self, q):
        return int(self.omap.state_validity([q])[0])

    def edges(self, frm, to):
        return [int(v) for v in self.omap.edge_validity(frm, to)]


def test_reparent_panic_through_the_pair_batch(ctx):
    """a gray pixel without zone id that neither the growth nor any observation crosses, but a pair of a reparent tree does:
    the oracle panics (RuntimeError), the device refuses with PORRT_ERR_PANIC, on the default edge kernel and on the large-map
    kernel, with either candidate search"""
    clean, occ, zones, b0 = _door_pto(start=(-0.8, -0.8), max_step=0.05, n_min=300)
    xy = clean.graph.export(0)[0]
    opol = clean.extract_policy()
    B = len(clean.beliefs())
    node_px = {tuple(clean.map.to_pixel(s)) for s in xy}
    zp = clean.map.zone_positions()
    spot = None
    for k in range(1, len(opol.parent)):
        a, b = xy[int(opol.original[opol.parent[k]]) // B], xy[int(opol.original[k]) // B]
        far = min(_norm2(p, z) for p in (a, b) for z in zp) > 0.45
        if _norm2(a, b) == 0.0 or not far:
            continue
        line = O.bresenham(clean.map.to_pixel(a).astype(np.int64), clean.map.to_pixel(b).astype(np.int64))
        for i, j in line[1:-1]:
            if (i, j) not in node_px and occ[i, j] == 255:
                spot, radius = (int(i), int(j)), 2.0 * _norm2(a, b)
                break
        if spot:
            break
    assert spot is not None
    striped = occ.copy()
    striped[spot] = 77
    omap_s = O.GridMap(striped, zones, util.LOW, util.UP, O.DOOR, 0.3)
    pto, _, _, _ = _door_pto(start=(-0.8, -0.8), max_step=0.05, n_min=300, omap_=omap_s, hooks=_CleanMapAnswers(clean.map))
    for x, y in zip(pto.graph.export(0), clean.graph.export(0)):
        np.testing.assert_array_equal(x, y)                       # the growth never saw the stripe
    assert pto.extract_policy().original.tolist() == opol.original.tolist()
    with pytest.raises(RuntimeError):
        pto.refine_policy_reparent(radius)
    pmap, plan, B = _device_plan(ctx, pto, striped, zones, b0)
    for large in (0, 1):
        for brute in (ALL_BRUTE, ALL_KD):
            ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, large)
            ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, brute)
            try:
                with pytest.raises(P.PorrtError) as e:
                    P.refine_policy_reparent(ctx, plan, radius)
                assert e.value.code == ERR_PANIC and "(code %d)" % O.PANIC_ZONE_UNWRAP in str(e.value), str(e.value)
            finally:
                ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)
                ctx.set_option(P.OPT_REPARENT_BRUTE_MAX_NODES, DEFAULT)
    # the clean map: the same call goes through
    pmap, plan, B = _device_plan(ctx, clean, occ, zones, b0)
    _same_policy(P.refine_policy_reparent(ctx, plan, radius), clean.refine_policy_reparent(radius), B, radius)
