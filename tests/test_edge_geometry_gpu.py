"""Edge validity pixel by pixel: lines built so that ONE chosen pixel decides the answer exactly at a strip (16 px), item
(7 strips = 112 px) or block boundary, maps whose every block is mixed or special so that 32 long lanes fill a warp's queues,
and the device-resident entry points the benchmark times.  Every result is compared for exact equality with the oracle, on both
edge kernels (the class-plane kernel of edge3.cu and the large-map kernel of map.cu), in three edge orders and through every
input form (coordinates with masks, compact bytes, node ids, adjacency rows)."""
import os

import numpy as np
import pytest

from oracle import pyoracle as O
import po_rrt_b200 as P
from po_rrt_b200 import synth
import porrt_testutil as util


LOW, UP = util.LOW, util.UP
BS, G = 16, 7                                                   # pixels per strip / block side, strips per item
LENGTHS = (0, 1, 2, 15, 16, 17, 31, 32, 33, 111, 112, 113, 223, 224, 225)
KS = (0, 1, 15, 16, 17, 111, 112, 113, "dx-1", "dx", "random")


@pytest.fixture(scope="module")
def ctx():
    c = P.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------------------------- line geometry
def line_offsets(d, k):
    """offset of pixel k from the start of the line with deltas d = b - a ([n, 2] (di, dj)), closed form:
    k * U + floor(k * dy / dx) * V, U / V the unit steps along the major / minor axis (major = i when |di| >= |dj|)"""
    d = np.asarray(d, np.int64).reshape(-1, 2)
    k = np.broadcast_to(np.asarray(k, np.int64), (len(d),))
    ad, s = np.abs(d), np.sign(d)
    major_i = ad[:, 0] >= ad[:, 1]
    dx = np.where(major_i, ad[:, 0], ad[:, 1])
    dy = np.where(major_i, ad[:, 1], ad[:, 0])
    m = k * dy // np.maximum(dx, 1)
    di = np.where(major_i, k * s[:, 0], m * s[:, 0])
    dj = np.where(major_i, m * s[:, 1], k * s[:, 1])
    return np.stack([di, dj], 1)


def major_length(d):
    d = np.abs(np.asarray(d, np.int64).reshape(-1, 2))
    return d.max(1)


def minor_unit(d):
    """unit step along the minor axis (sign of the minor delta, + when it is 0)"""
    d = np.asarray(d, np.int64).reshape(-1, 2)
    major_i = np.abs(d[:, 0]) >= np.abs(d[:, 1])
    sv = np.where(np.where(major_i, d[:, 1], d[:, 0]) < 0, -1, 1)
    return np.stack([np.where(major_i, 0, sv), np.where(major_i, sv, 0)], 1)


def line_pixels(a, b):
    """every pixel of one line a -> b, [dx + 1, 2]"""
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    dx = int(major_length(b - a)[0])
    return a + line_offsets(np.repeat((b - a)[None], dx + 1, 0), np.arange(dx + 1))


def pixel_centres(H, W, ij, low=LOW, up=UP):
    """coordinates whose GridMap.to_pixel is ij: i = sat((H-1) - (y - low) * ppm), j = sat((x - low) * ppm) at pixel centres.
    Indices >= H / W give points outside the map (negative ones cannot be reached: the conversion saturates at 0)."""
    ij = np.asarray(ij, np.int64).reshape(-1, 2)
    assert (ij >= 0).all()
    ppm = W / (up[0] - low[0])
    return np.stack([low[0] + (ij[:, 1] + 0.5) / ppm, low[1] + (H - 1 - ij[:, 0] - 0.5) / ppm], 1)


def test_line_offsets_match_bresenham():
    """the closed form the designs below rely on equals the oracle's Bresenham in every octant, on axis-aligned lines, exact
    diagonals and zero-length lines (no GPU needed)"""
    rng = np.random.default_rng(1)
    lines = [rng.integers(-300, 300, (3000, 2)), rng.integers(-40, 40, (1000, 2))]
    for L in (0, 1, 2, 7, 16, 113, 250):
        for si in (-1, 1):
            for sj in (-1, 1):
                lines.append(np.array([[si * L, 0], [0, sj * L], [si * L, sj * L]]))             # axis-aligned, diagonals
        lines.append(np.array([[L, L - 1], [L - 1, L], [-L, 1 - L], [1 - L, -L]]))             # near-ties
    d = np.concatenate(lines)
    starts = rng.integers(-50, 400, (len(d), 2))
    octants = set()
    for (ai, aj), (di, dj) in zip(starts, d):
        want = O.bresenham((int(ai), int(aj)), (int(ai + di), int(aj + dj)))
        got = line_pixels((ai, aj), (ai + di, aj + dj))
        np.testing.assert_array_equal(got, want, err_msg=str(((ai, aj), (di, dj))))
        octants.add((abs(di) >= abs(dj), di < 0, dj < 0))
    assert len(octants) == 8


# ---------------------------------------------------------------------------------------------- designs
class Case:
    """one map and the pixel endpoints of its lines; `dec` = k of the pixel built to decide the line (-1: none), `hit` = the
    decisive pixel is on the line (False: near miss, the pixel one step beside it along the minor axis)"""

    def __init__(self, name, kind, occ, zones, visibility=0.3):
        self.name, self.kind, self.occ, self.zones, self.visibility = name, kind, occ, zones, visibility
        self.H, self.W = occ.shape
        self.a, self.b, self.dec, self.hit = [], [], [], []

    def add(self, a, b, dec=-1, hit=True):
        self.a.append(np.asarray(a, np.int64).reshape(-1, 2))
        self.b.append(np.asarray(b, np.int64).reshape(-1, 2))
        n = len(self.a[-1])
        self.dec.append(np.broadcast_to(np.asarray(dec, np.int64), (n,)).copy())
        self.hit.append(np.broadcast_to(np.asarray(hit, bool), (n,)).copy())

    def done(self):
        self.a, self.b = np.concatenate(self.a), np.concatenate(self.b)
        self.dec, self.hit = np.concatenate(self.dec), np.concatenate(self.hit)
        self.xa, self.xb = pixel_centres(self.H, self.W, self.a), pixel_centres(self.H, self.W, self.b)
        return self


def _k_of(spec, dx, rng):
    if spec == "dx-1":
        k = dx - 1
    elif spec == "dx":
        k = dx
    elif spec == "random":
        k = int(rng.integers(0, dx + 1))
    else:
        k = spec
    return int(min(max(k, 0), dx))


def _shapes(rng, part=0, n_parts=1, long_lines=0, max_long=700):
    """line shapes (deltas, decisive k, start residue (ai % 16, aj % 16)) over all 8 octants, |di| == |dj| ties, axis-aligned and
    zero-length lines, every length of LENGTHS and every k of KS; the start residues run through all 256 values"""
    out = []
    combos = [(dx, spec, octant) for dx in LENGTHS for spec in KS for octant in range(8)]
    mine = np.random.default_rng(7).permutation(len(combos)) % n_parts == part     # a fixed split over the maps of one design
    for (dx, spec, octant), take in zip(combos, mine):
        if not take:
            continue
        major_i, su, sv = octant & 1, 1 - 2 * ((octant >> 1) & 1), 1 - 2 * ((octant >> 2) & 1)
        kind = int(rng.integers(0, 4))                         # axis-aligned, |di| == |dj| tie, or any slope in between
        dy = 0 if kind == 0 or dx <= 1 else (dx if kind == 1 else int(rng.integers(1, dx)))
        d = (su * dx, sv * dy) if major_i else (sv * dy, su * dx)
        out.append((d, _k_of(spec, dx, rng)))
    for _ in range(long_lines):
        dx = int(rng.integers(300, max_long))
        dy = int(rng.integers(0, dx + 1))
        su, sv = rng.choice([-1, 1], 2)
        d = (su * dx, sv * dy) if rng.integers(2) else (sv * dy, su * dx)
        out.append((d, int(rng.integers(0, dx + 1))))
    res = [(t % 16, (t // 16) % 16) for t in range(len(out))]
    order = rng.permutation(len(out))                          # residues are not tied to one length or k
    return [(out[i][0], out[i][1], res[r]) for r, i in enumerate(order)]


def _place(rng, H, W, d, res):
    """a start a with a % 16 == res such that a and a + d are in the map, or None"""
    a = []
    for ax, size in ((0, H), (1, W)):
        lo, hi = max(0, -d[ax]), size - 1 - max(0, d[ax])
        first = lo + ((res[ax] - lo) % BS)
        if first > hi:
            return None
        a.append(first + BS * int(rng.integers(0, (hi - first) // BS + 1)))
    return np.array(a, np.int64)


def _near_miss(rng, H, W, a, b):
    """the line shifted by one pixel along its minor axis (either side that stays in the map), or None"""
    v = minor_unit(b - a)[0]
    for s in rng.permutation([-1, 1]):
        a2, b2 = a + s * v, b + s * v
        if (a2 >= 0).all() and (b2 >= 0).all() and a2[0] < H and b2[0] < H and a2[1] < W and b2[1] < W:
            return a2, b2
    return None


def _door_obstacles(name, H, W, seed, part, n_parts):
    """DOOR map, free but for the isolated obstacle pixels the lines are built around, a few all-blocking blocks and lines that
    start in them, and lines that leave or enter the map"""
    rng = np.random.default_rng(seed)
    occ = np.full((H, W), 255, np.uint8)
    zones = np.full((H, W), 255, np.uint8)
    occ[H - 2, 1] = 128; zones[H - 2, 1] = 0                   # one zone, far from everything
    c = Case(name, P.DOOR, occ, zones)
    for d, k, res in _shapes(rng, part, n_parts, long_lines=32):
        a = _place(rng, H, W, d, res)
        if a is None:
            continue
        b = a + d
        p = a + line_offsets(d, k)[0]
        occ[p[0], p[1]] = 0
        c.add(a, b, k, True)
        nm = _near_miss(rng, H, W, a, b)
        if nm is not None:
            c.add(nm[0], nm[1], k, False)
    # all-blocking blocks (class "blocked"): lines that start in them are decided before any strip is looked at
    for _ in range(6):
        bi, bj = int(rng.integers(2, H // BS - 2)), int(rng.integers(2, W // BS - 2))
        occ[bi * BS:(bi + 1) * BS, bj * BS:(bj + 1) * BS] = 0
        for _ in range(12):
            a = np.array([bi * BS + rng.integers(0, BS), bj * BS + rng.integers(0, BS)])
            b = np.clip(a + rng.integers(-150, 150, 2), 0, [H - 1, W - 1])
            c.add(a, b, 0, True)
            c.add(b, a)
    # end outside the map (i >= H or j >= W): an obstacle before the line leaves decides (Obstacle), else PANIC_OOB; start
    # outside: PANIC_OOB whatever lies on the line in the map
    for t in range(160):
        out_i = t % 2 == 0
        L = int(rng.choice([3, 17, 40, 113, 230]))
        if out_i:
            a = np.array([H - 1 - rng.integers(0, L), rng.integers(0, W)])
            b = np.array([H + rng.integers(0, 20), a[1] + rng.integers(-L, L + 1)])
        else:
            a = np.array([rng.integers(0, H), W - 1 - rng.integers(0, L)])
            b = np.array([a[0] + rng.integers(-L, L + 1), W + rng.integers(0, 20)])
        b = np.maximum(b, 0)
        px = line_pixels(a, b)
        inside = (px[:, 0] < H) & (px[:, 1] < W)
        k_exit = int(np.argmin(inside))                          # first pixel outside
        if t % 4 < 2:
            k = int(rng.integers(0, k_exit))
            occ[px[k, 0], px[k, 1]] = 0
            c.add(a, b, k, True)
            a2 = a + rng.choice([-1, 1]) * minor_unit(b - a)[0]  # near miss: shifted along the minor axis, end still outside
            if (a2 >= 0).all() and (b + (a2 - a) >= 0).all() and a2[0] < H and a2[1] < W:
                c.add(a2, b + (a2 - a), k, False)
        else:
            c.add(b, a)                                          # start outside, back into the map: PANIC_OOB
            p = px[int(rng.integers(0, k_exit))]
            occ[p[0], p[1]] = 0
    return c.done()


def _door_gray(name, H, W, seed, part, n_parts):
    """DOOR map with zones 0..3: per line a single zone pixel, two zones (also on adjacent pixels across a strip boundary), an
    obstacle and a zone pixel in either order, gray without a zone id (PANIC_ZONE_UNWRAP) before or after an obstacle"""
    rng = np.random.default_rng(seed)
    occ = np.full((H, W), 255, np.uint8)
    zones = np.full((H, W), 255, np.uint8)
    Z = 4
    for z in range(Z):                                         # every zone id has pixels, far from the lines' region
        occ[H - 1, 2 * z] = 128; zones[H - 1, 2 * z] = z
    c = Case(name, P.DOOR, occ, zones)

    def put(p, what):
        if what == "obst":
            occ[p[0], p[1]] = 0; zones[p[0], p[1]] = 255
        elif what == "unwrap":
            occ[p[0], p[1]] = 90; zones[p[0], p[1]] = 255
        else:
            occ[p[0], p[1]] = 128; zones[p[0], p[1]] = what

    t = 0
    for d, k, res in _shapes(rng, part, n_parts, long_lines=24):
        a = _place(rng, H, W, d, res)
        if a is None or a[0] >= H - 2:
            continue
        b = a + d
        dx = int(major_length(d)[0])
        px = a + line_offsets(np.repeat(np.asarray(d)[None], dx + 1, 0), np.arange(dx + 1))
        if (px[:, 0] >= H - 2).any():
            continue
        t += 1
        v = t % 8
        z1 = int(rng.integers(0, Z)); z2 = (z1 + 1 + int(rng.integers(0, Z - 1))) % Z
        if v == 0 or dx == 0:
            put(px[k], z1)                                       # one zone pixel: validity z1
        elif v == 1:
            # two zones on adjacent pixels, the second one first in its strip (major coordinate crosses a block edge)
            major = 0 if abs(d[0]) >= abs(d[1]) else 1
            cross = np.nonzero(px[1:, major] // BS != px[:-1, major] // BS)[0]
            k1 = int(rng.choice(cross)) if len(cross) else max(0, k - 1)
            put(px[k1], z1); put(px[k1 + 1], z2)
            k = k1 + 1
        else:
            k1, k2 = sorted(rng.choice(dx + 1, 2, replace=False)) if dx >= 1 else (0, 0)
            k1, k2 = int(k1), int(k2)
            if v == 2:
                put(px[k1], "obst"); put(px[k2], z1)             # obstacle first
            elif v == 3:
                put(px[k1], z1); put(px[k2], "obst")             # zone first
            elif v == 4:
                put(px[k], "unwrap")                             # gray without zone id
            elif v == 5:
                put(px[k1], "unwrap"); put(px[k2], "obst")       # the panic comes first
            elif v == 6:
                put(px[k1], "obst"); put(px[k2], "unwrap")       # the obstacle comes first
            else:
                put(px[k1], z1); put(px[k2], z1)                 # the same zone twice: validity z1
            k = k1
        c.add(a, b, k, True)
        nm = _near_miss(rng, H, W, a, b)
        if nm is not None and nm[0][0] < H - 2 and nm[1][0] < H - 2:
            c.add(nm[0], nm[1], k, False)
    return c.done()


def _shelf(name, H, W, seed, part, n_parts):
    """SHELF map: a low (127..254) or a high (< 127) obstacle decides each line"""
    rng = np.random.default_rng(seed)
    occ = np.full((H, W), 255, np.uint8)
    zones = np.full((H, W), 255, np.uint8)
    for z in range(3):
        zones[H - 1, 3 * z] = z
    c = Case(name, P.SHELF, occ, zones, visibility=0.6)
    lows, highs = (127, 128, 200, 253, 254), (0, 1, 64, 126)
    for t, (d, k, res) in enumerate(_shapes(rng, part, n_parts, long_lines=32)):
        a = _place(rng, H, W, d, res)
        if a is None:
            continue
        p = a + line_offsets(d, k)[0]
        occ[p[0], p[1]] = rng.choice(lows) if t % 2 else rng.choice(highs)
        c.add(a, a + d, k, True)
        nm = _near_miss(rng, H, W, a, a + d)
        if nm is not None:
            c.add(nm[0], nm[1], k, False)
    return c.done()


def _last_pixel(c, occ, rng, a, b, share=0.04, zones=None):
    """a few per cent of the lines get one blocking pixel (or, with zones, a zone pixel) as their last pixel"""
    for t in range(len(a)):
        if rng.random() < share:
            occ[b[t][0], b[t][1]] = 0
            c.add(a[t], b[t], int(major_length(b[t] - a[t])[0]), True)
        elif zones is not None and rng.random() < share:
            occ[b[t][0], b[t][1]] = 128; zones[b[t][0], b[t][1]] = 1
            c.add(a[t], b[t], int(major_length(b[t] - a[t])[0]), True)
        else:
            c.add(a[t], b[t])


def _stripes(name, H, W, seed, vertical=False, gray=False):
    """blocking (or, with `gray`, zone) pixels on every odd row, long free lines on the even rows in both directions: every
    block is mixed (special), every strip of every lane is queued and the queues drain several times per warp batch"""
    rng = np.random.default_rng(seed)
    Hl, Wl = (W, H) if vertical else (H, W)                      # built along rows, transposed for columns
    occ = np.full((Hl, Wl), 255, np.uint8)
    zones = np.full((Hl, Wl), 255, np.uint8)
    if gray:
        rows = np.arange(1, Hl, 2)
        occ[1::2, :] = 128
        zones[1::2, :] = ((rows // 2) % 4)[:, None]
    else:
        occ[1::2, :] = 0
        occ[1, 0] = 128; zones[1, 0] = 0                        # the one zone the map needs, on a blocking row
    if vertical:
        occ, zones = occ.T.copy(), zones.T.copy()
    c = Case(name, P.DOOR, occ, zones)
    r = np.arange(0, Hl - 1, 2)
    j0 = rng.integers(0, 64, len(r))
    j1 = Wl - 1 - rng.integers(0, 64, len(r))
    a = np.stack([r, np.where(r % 4 == 0, j0, j1)], 1)
    b = np.stack([r, np.where(r % 4 == 0, j1, j0)], 1)
    if vertical:
        a, b = a[:, ::-1].copy(), b[:, ::-1].copy()
    _last_pixel(c, occ, rng, a, b, zones=zones if gray else None)
    return c.done()


def _checker(name, H, W, seed):
    """pixels with (i + j) odd block: every block is mixed; anti-diagonal (and diagonal) lines through the free pixels"""
    rng = np.random.default_rng(seed)
    ii, jj = np.indices((H, W))
    occ = np.where((ii + jj) % 2 == 1, 0, 255).astype(np.uint8)
    zones = np.full((H, W), 255, np.uint8)
    zones[0, 0] = 0; occ[0, 0] = 128
    c = Case(name, P.DOOR, occ, zones)
    n = 1200
    L = rng.integers(900, min(H, W) - 1, n)
    i0 = np.array([rng.integers(l, H) for l in L])              # anti-diagonal a = (i0, j0) -> (i0 - L, j0 + L)
    j0 = np.array([rng.integers(0, W - l) for l in L])
    j0 += (i0 + j0) % 2 * np.where(j0 + 1 < W - L, 1, -1)       # start on a free pixel
    a = np.stack([i0, j0], 1)
    b = a + np.stack([-L, L], 1)
    diag = np.arange(n) % 3 == 2                                 # every third one on the main diagonal
    b[diag] = a[diag] - np.stack([L[diag], L[diag]], 1)
    ok = (b >= 0).all(1) & (b[:, 0] < H) & (b[:, 1] < W)
    a, b = a[ok], b[ok]
    back = rng.random(len(a)) < 0.5                              # both directions
    a[back], b[back] = b[back].copy(), a[back].copy()
    _last_pixel(c, occ, rng, a, b)
    return c.done()


BOUNDARY_CASES = {
    "door_obst_1000_a": lambda: _door_obstacles("door_obst_1000_a", 1000, 1000, 101, 0, 4),
    "door_obst_777x1200_b": lambda: _door_obstacles("door_obst_777x1200_b", 777, 1200, 102, 1, 4),
    "door_obst_1000_c": lambda: _door_obstacles("door_obst_1000_c", 1000, 1000, 103, 2, 4),
    "door_obst_777x1200_d": lambda: _door_obstacles("door_obst_777x1200_d", 777, 1200, 104, 3, 4),
    "door_gray_1000_a": lambda: _door_gray("door_gray_1000_a", 1000, 1000, 111, 0, 2),
    "door_gray_777x1200_b": lambda: _door_gray("door_gray_777x1200_b", 777, 1200, 112, 1, 2),
    "shelf_1000_a": lambda: _shelf("shelf_1000_a", 1000, 1000, 121, 0, 2),
    "shelf_777x1200_b": lambda: _shelf("shelf_777x1200_b", 777, 1200, 122, 1, 2),
}
QUEUE_CASES = {
    "stripes_rows_2100": lambda: _stripes("stripes_rows_2100", 2100, 2100, 131),
    "stripes_cols_2050x2200": lambda: _stripes("stripes_cols_2050x2200", 2050, 2200, 132, vertical=True),
    "checker_2100": lambda: _checker("checker_2100", 2100, 2100, 133),
    "gray_stripes_2100x2048": lambda: _stripes("gray_stripes_2100x2048", 2100, 2048, 134, gray=True),
}


def design_stats(c):
    """what the design exercises, from the generator alone: the share of lines whose decisive pixel is the first or last pixel of
    a strip (major coordinate at a block edge) or of an item (7 strips from the edge's first strip), and the share of lines with
    both ends in the map that cross a mixed or special block and no all-blocking one (their strips go through the queues)"""
    blocking = (c.occ != 255) if c.kind == P.SHELF else (c.occ == 0)
    gray = (c.occ != 0) & (c.occ != 255) if c.kind == P.DOOR else np.zeros_like(blocking)
    hb, wb = -(-c.H // BS), -(-c.W // BS)
    pad = lambda x: np.pad(x, ((0, hb * BS - c.H), (0, wb * BS - c.W))).reshape(hb, BS, wb, BS).sum((1, 3))
    n_in = pad(np.ones_like(blocking, np.int64))
    n_bl, n_gr = pad(blocking.astype(np.int64)), pad(gray.astype(np.int64))
    cls = np.where(n_gr > 0, 3, np.where(n_bl == 0, 0, np.where(n_bl == n_in, 2, 1)))
    strip = item = queued = inside = 0
    for a, b, k in zip(c.a, c.b, c.dec):
        px = line_pixels(a, b)
        major = 0 if abs(b[0] - a[0]) >= abs(b[1] - a[1]) else 1
        if k >= 0 and len(px) > 1:
            cm, c0, step = px[k, major], px[0, major], np.sign(b[major] - a[major])
            first, last = (cm % BS == 0, cm % BS == BS - 1) if step > 0 else (cm % BS == BS - 1, cm % BS == 0)
            s = abs(cm // BS - c0 // BS)
            strip += bool(first or last)
            item += bool((first and s % G == 0 and s > 0) or (last and s % G == G - 1))
        if (px[[0, -1], 0] < c.H).all() and (px[[0, -1], 1] < c.W).all():
            inside += 1
            k_cls = cls[px[:, 0] // BS, px[:, 1] // BS]
            queued += bool(((k_cls == 1) | (k_cls == 3)).any() and not (k_cls == 2).any())
    n = len(c.a)
    return {"lines": n, "at_strip_boundary": strip / n, "at_item_boundary": item / n, "through_queues": queued / max(inside, 1)}


# ---------------------------------------------------------------------------------------------- running a case
def _orders(c, seed=0):
    n = len(c.a)
    length = major_length(c.b - c.a)
    return {"generated": np.arange(n), "by_length": np.argsort(length, kind="stable"),
            "shuffled": np.random.default_rng(seed).permutation(n)}


def _run_forms(ctx, pmap, xa, xb, want, wv):
    """every input form against the oracle's ids `want`; masks = world_validities_words()[id] (0 for negative ids)"""
    n = len(xa)
    exp_masks = np.where((want >= 0)[:, None], wv[np.clip(want, 0, None)], 0)
    got, masks = pmap.transition_validator(xa, xb, want_masks=True)
    bad = np.nonzero(got.astype(np.int64) != want)[0]
    assert len(bad) == 0, "coordinates: %d mismatches, first %s: got %d want %d" % (len(bad), bad[0], got[bad[0]], want[bad[0]])
    np.testing.assert_array_equal(masks, exp_masks)
    np.testing.assert_array_equal(pmap.transition_validator(xa, xb, compact=True).astype(np.int64), want)
    tree = P.KdTree(ctx, np.concatenate([xa, xb]))
    fi, ti = np.arange(n, dtype=np.int32), np.arange(n, 2 * n, dtype=np.int32)
    got, masks = pmap.transition_validator_nodes(fi, ti, want_masks=True)
    np.testing.assert_array_equal(got.astype(np.int64), want)
    np.testing.assert_array_equal(masks, exp_masks)
    rp = np.zeros(2 * n + 1, np.int64)                            # row n + r (node b_r) lists its one neighbour a_r
    rp[n + 1:] = np.arange(1, n + 1)
    np.testing.assert_array_equal(pmap.transition_validator_adjacency(rp, fi).astype(np.int64), want)
    del tree


def _check_case(ctx, c):
    omap, pmap = util.make_pair(ctx, c.occ, c.zones, c.kind, c.visibility)
    sample = np.random.default_rng(0).choice(len(c.a), min(len(c.a), 64), replace=False)
    for t in sample:                                             # the coordinates give back the intended pixels
        np.testing.assert_array_equal(omap.to_pixel(c.xa[t]), c.a[t])
        np.testing.assert_array_equal(omap.to_pixel(c.xb[t]), c.b[t])
    want = omap.edge_validity(c.xa, c.xb)
    wv = pmap.world_validities_words()
    for large in (0, 1):
        ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, large)
        try:
            for name, perm in _orders(c).items():
                try:
                    _run_forms(ctx, pmap, c.xa[perm], c.xb[perm], want[perm], wv)
                except AssertionError as e:
                    raise AssertionError("%s, %s kernel, %s order: %s" % (c.name, "large-map" if large else "class-plane", name, e))
        finally:
            ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)
    return omap, want


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BOUNDARY_CASES))
def test_one_pixel_decides(ctx, name):
    c = BOUNDARY_CASES[name]()
    omap, want = _check_case(ctx, c)
    decided = c.dec >= 0
    hits, misses = decided & c.hit, decided & ~c.hit
    if c.kind == P.SHELF or name.startswith("door_obst"):
        # the design really exercises both outcomes: hits are blocked, near misses mostly free (or leave the map)
        assert (want[hits] < 0).mean() >= 0.95, (want[hits] < 0).mean()
        free = want[misses] == omap.n_validities - 1
        if name.startswith("door_obst"):
            free |= want[misses] == O.PANIC_OOB
        assert free.mean() >= 0.90, free.mean()
    if name.startswith("door_obst"):
        assert (want == O.PANIC_OOB).any() and (want == -1).any() and (want == omap.n_validities - 1).any()
    if name.startswith("door_gray"):
        for code in (O.PANIC_ZONE_UNWRAP, O.PANIC_MULTI_ZONE, -1, 0, 1, 2, 3, omap.n_validities - 1):
            assert (want == code).any(), code
    st = design_stats(c)
    assert st["at_strip_boundary"] > 0.05 and st["at_item_boundary"] > 0.005, st


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(QUEUE_CASES))
def test_full_warp_queues(ctx, name):
    c = QUEUE_CASES[name]()
    omap, want = _check_case(ctx, c)
    free = want == omap.n_validities - 1
    assert free.mean() > 0.85 and (want == -1).any(), free.mean()
    assert design_stats(c)["through_queues"] > 0.99


# ---------------------------------------------------------------------------------------------- device-resident entry points
_BENCH = {}


def _bench_map(ctx):
    """the benchmark's map (6 door zones, 64 worlds) uploaded to ctx; the oracle's twin is built once per module"""
    if "occ" not in _BENCH:
        _BENCH["occ"], _BENCH["zones"] = synth.door_map(size=8192, n_zones=6, seed=1)
        _BENCH["omap"] = O.GridMap(_BENCH["occ"], _BENCH["zones"], LOW, UP, O.DOOR, 0.3)
    pmap = P.Map(ctx, _BENCH["occ"], LOW, UP)
    pmap.add_zones(_BENCH["zones"], 0.3)
    return _BENCH["omap"], pmap


def _edges_dev(ctx, stream, a, b, want_masks, sentinel=-7):
    """porrt_edge_validity_dev on `stream`, inputs and outputs as torch device tensors -> (ids, masks or None) on the host"""
    import torch
    n = len(a)
    da, db = torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda()
    dv = torch.full((max(n, 1),), sentinel, dtype=torch.int32, device="cuda")
    dm = torch.full((max(n, 1),), sentinel, dtype=torch.int64, device="cuda") if want_masks else None
    for t in (da, db, dv) + ((dm,) if want_masks else ()):
        assert t.data_ptr() % 16 == 0
    stream.wait_stream(torch.cuda.current_stream())
    ctx.check(ctx.lib.porrt_edge_validity_dev(ctx.h, da.data_ptr(), db.data_ptr(), n, dv.data_ptr(),
                                              dm.data_ptr() if want_masks else None))
    stream.synchronize()
    return dv.cpu().numpy(), (dm.cpu().numpy().view(np.uint64) if want_masks else None)


def _on_stream(ctx, fn):
    import torch
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    try:
        return fn(stream)
    finally:
        ctx.set_stream(None)


@pytest.mark.gpu
def test_edge_validity_dev_benchmark_call(ctx):
    """the benchmark's inputs as one launch of 2^24 edges on a non-default stream, with and without masks, on both kernels"""
    omap, pmap = _bench_map(ctx)
    a, b = synth.edges(1 << 24, seed=2)
    want, _ = omap.edge_validity_timed(a, b, max(1, len(os.sched_getaffinity(0))))
    assert all((want == z).any() for z in range(6)) and (want == 6).any() and (want == -1).any()
    wv = pmap.world_validities_words()
    exp_masks = np.where(want >= 0, wv[np.clip(want, 0, None), 0], 0)
    for large in (0, 1):
        ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, large)
        try:
            got, masks = _on_stream(ctx, lambda s: _edges_dev(ctx, s, a, b, True))
            np.testing.assert_array_equal(got, want.astype(np.int32))
            np.testing.assert_array_equal(masks, exp_masks)
            del masks
            got, _ = _on_stream(ctx, lambda s: _edges_dev(ctx, s, a, b, False))
            np.testing.assert_array_equal(got, want.astype(np.int32))
        finally:
            ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)


@pytest.mark.gpu
def test_edge_validity_dev_launch_shapes(ctx):
    """batch sizes at the launch-shape boundaries: the 4-warp minimum per CTA, one CTA per SM, the cap of 32 warps per CTA and
    the first edges of the persistent loop's second round"""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    omap, pmap = _bench_map(ctx)
    wv = pmap.world_validities_words()
    for n in (0, 1, 31, 32, 33, 128 * sm - 1, 128 * sm + 1, 1024 * sm - 1, 1024 * sm + 1):
        a, b = synth.edges(max(n, 1), seed=50 + n % 97, max_len=0.2)
        a, b = a[:n], b[:n]
        want = omap.edge_validity(a, b)
        for large in (0, 1):
            ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, large)
            try:
                for masks_on in (True, False):
                    got, masks = _on_stream(ctx, lambda s: _edges_dev(ctx, s, a, b, masks_on))
                    if n == 0:
                        assert got[0] == -7 and (masks is None or masks[0] == np.uint64(2 ** 64 - 7))   # nothing written
                        continue
                    np.testing.assert_array_equal(got[:n], want.astype(np.int32), err_msg="n=%d large=%d" % (n, large))
                    if masks_on:
                        np.testing.assert_array_equal(masks[:n], np.where(want >= 0, wv[np.clip(want, 0, None), 0], 0))
            finally:
                ctx.set_option(P.OPT_FORCE_LARGE_MAP_PATH, 0)


@pytest.mark.gpu
def test_state_validity_and_visibility_dev(ctx):
    import torch
    omap, pmap = _bench_map(ctx)
    a, _ = synth.edges(1 << 21, seed=2)
    pts = np.ascontiguousarray(a)
    vis = np.ascontiguousarray(pts[:300_000])

    def run(stream):
        dp, dq = torch.from_numpy(pts).cuda(), torch.from_numpy(vis).cuda()
        dv = torch.empty(len(pts), dtype=torch.int32, device="cuda")
        dm = torch.empty(len(vis), dtype=torch.int64, device="cuda")
        ds = torch.empty(len(vis), dtype=torch.int32, device="cuda")
        stream.wait_stream(torch.cuda.current_stream())
        ctx.check(ctx.lib.porrt_state_validity_dev(ctx.h, dp.data_ptr(), len(pts), dv.data_ptr()))
        ctx.check(ctx.lib.porrt_visibility_dev(ctx.h, dq.data_ptr(), len(vis), dm.data_ptr(), ds.data_ptr()))
        stream.synchronize()
        return dv.cpu().numpy(), dm.cpu().numpy().view(np.uint64), ds.cpu().numpy()

    sv, mask, status = _on_stream(ctx, run)
    np.testing.assert_array_equal(sv.astype(np.int64), omap.state_validity(pts))
    wm, wp = omap.visible_zones(vis)
    np.testing.assert_array_equal(mask, wm)
    np.testing.assert_array_equal(status.astype(np.int64), wp)
    assert (wm != 0).any() and (sv == omap.n_validities - 1).any() and (sv == -1).any()


@pytest.mark.gpu
def test_vertices_set_dev_with_bounding_box(ctx):
    """the vertex set uploaded from device memory with an explicit bounding box (the points' own and a larger one) answers
    indexed edge validity, radius and 1-NN queries as the same set uploaded from the host, and as the oracle"""
    import torch
    omap, pmap = _bench_map(ctx)
    a, b = synth.edges(100_000, seed=61, max_len=0.1)
    pts = np.ascontiguousarray(np.concatenate([a, b]))
    n = len(a)
    fi, ti = np.arange(n, dtype=np.int32), np.arange(n, 2 * n, dtype=np.int32)
    want = omap.edge_validity(a, b)
    rng = np.random.default_rng(62)
    q = rng.uniform(-1.05, 1.05, (5000, 2))
    q[:50] = pts[rng.integers(0, len(pts), 50)]                   # queries on vertices: distance 0
    radius = 0.01
    otree = O.KdTree(pts[0], 0)
    otree.add_batch(pts[1:], 1)
    ooffs, oids, _ = otree.radius_batch(q, radius, cap=1 << 22)
    onn = otree.nearest_batch(q)

    def queries():
        tree = P.KdTree(ctx)
        tree.n = len(pts)
        offs, ids = tree.nearest_neighbors(q, radius)
        nid, ndist, ties = tree.nearest_neighbor(q)
        return pmap.transition_validator_nodes(fi, ti), offs, ids, nid, ndist, ties

    host_tree = P.KdTree(ctx, pts)
    host = queries()
    np.testing.assert_array_equal(host[0].astype(np.int64), want)
    np.testing.assert_array_equal(host[1], ooffs)
    for k in range(0, len(q), 7):
        np.testing.assert_array_equal(host[2][host[1][k]:host[1][k + 1]], np.sort(oids[ooffs[k]:ooffs[k + 1]]))
    one = host[5] == 1
    assert one.mean() > 0.99
    np.testing.assert_array_equal(host[3][one], onn[one])
    d = np.linalg.norm(pts[onn] - q, axis=1)
    np.testing.assert_allclose(host[4], d, rtol=0, atol=1e-15)
    lo, hi = pts.min(0), pts.max(0)
    dp = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    for blo, bhi in ((lo, hi), (lo - 0.37, hi + 0.5)):
        blo, bhi = np.ascontiguousarray(blo, np.float64), np.ascontiguousarray(bhi, np.float64)
        ctx.check(ctx.lib.porrt_vertices_set_dev(ctx.h, dp.data_ptr(), len(pts), 0.0, blo.ctypes.data, bhi.ctypes.data))
        got = queries()
        for g, h in zip(got, host):
            np.testing.assert_array_equal(g, h)
    del host_tree
