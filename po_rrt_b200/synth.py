"""Synthetic inputs of the named shapes (SURVEY.md 8(d)): occupancy grids with door zones / shelves, edge batches,
vertex and query sets.  numpy's PCG64 is used here (generator choice does not matter for inputs; seeds are stated)."""
import numpy as np


def door_map(size=8192, n_rects=4096, side_lo=16, side_hi=112, n_zones=6, seed=1, zone_w=32, zone_h=256):
    """Free grid (255) with axis-aligned obstacle rectangles (0) covering ~25 %, and n_zones door rectangles of gray 128 in the
    occupancy grid / zone id in the zone grid, at least 1024*size/8192 px apart so no edge of <= 410 px crosses two zones."""
    rng = np.random.default_rng(seed)
    occ = np.full((size, size), 255, np.uint8)
    s = size / 8192.0
    lo, hi = max(1, int(side_lo * s)), max(2, int(side_hi * s))  # same count, scaled sides: coverage stays ~25 %
    for _ in range(n_rects):
        h, w = rng.integers(lo, hi + 1, 2)
        i, j = rng.integers(0, size - h), rng.integers(0, size - w)
        occ[i:i + h, j:j + w] = 0
    zones = np.full((size, size), 255, np.uint8)
    zw, zh = max(2, int(zone_w * s)), max(4, int(zone_h * s))
    cols = 3
    rows = (n_zones + cols - 1) // cols
    for z in range(n_zones):
        # two rows of three (the c5 layout); more zones: as many rows as needed, still >= size/8 apart
        ci = int((0.25 + 0.5 * (z // cols)) * size) if rows <= 2 else int((z // cols + 0.25) / rows * size)
        cj = int((0.2 + 0.3 * (z % cols)) * size)
        occ[ci:ci + zh, cj:cj + zw] = 128
        zones[ci:ci + zh, cj:cj + zw] = z
    return occ, zones


def shelf_map(size=200, n_rects=12, n_zones=2, seed=5):
    """MapShelfDomain stand-in: high obstacles (0), low obstacles (180: observable through), shelves = zones."""
    rng = np.random.default_rng(seed)
    occ = np.full((size, size), 255, np.uint8)
    occ[0, :] = occ[-1, :] = 0
    occ[:, 0] = occ[:, -1] = 0
    for k in range(n_rects):
        h, w = rng.integers(size // 25, size // 8, 2)
        i, j = rng.integers(size // 10, size - h - size // 10), rng.integers(size // 10, size - w - size // 10)
        occ[i:i + h, j:j + w] = 0 if k % 3 else 180
    zones = np.full((size, size), 255, np.uint8)
    for z in range(n_zones):
        i = int((0.15 + 0.7 * (z + 0.5) / n_zones) * size)
        j = int(0.88 * size)
        occ[i - 3:i + 3, j - 3:j + 3] = 255
        zones[i - 2:i + 2, j - 2:j + 2] = z
    return occ, zones


def pixel_centres(size):
    """(x, y) of every pixel centre of a size x size map on [-1, 1]^2; row 0 is the top (largest y), as Map::to_pixel reads it"""
    c = (np.arange(size) + 0.5) / size * 2.0 - 1.0
    return np.meshgrid(c, c[::-1])


def rrt_map(size=1024, n_rects=4096, seed=7, clear=((-0.8, -0.8), (0.8, 0.8)), clear_r=0.06):
    """Single-world stand-in for the RRT* config's map (BASELINE config 1): free grid with obstacle rectangles (0) on [-1, 1]^2, no
    zones, and a free disc of radius clear_r around each point of `clear` (the start and the goal)."""
    occ, _ = door_map(size=size, n_rects=n_rects, n_zones=0, seed=seed)
    x, y = pixel_centres(size)
    for px, py in clear:
        occ[(x - px) ** 2 + (y - py) ** 2 <= clear_r ** 2] = 255
    return occ


def edges(n, seed=2, max_len=0.1, low=-1.0, up=1.0):
    """a uniform in [low,up)^2; b = a + l*(cos t, sin t), l ~ U[0,max_len], clamped into [low, up - 2^-20]"""
    rng = np.random.default_rng(seed)
    a = rng.uniform(low, up, (n, 2))
    l = rng.uniform(0.0, max_len, n)
    t = rng.uniform(0.0, 2 * np.pi, n)
    b = a + np.stack([l * np.cos(t), l * np.sin(t)], 1)
    b = np.clip(b, low, up - 2.0 ** -20)
    a = np.clip(a, low, up - 2.0 ** -20)
    return np.ascontiguousarray(a), np.ascontiguousarray(b)


def points(n, seed=3, low=-1.0, up=1.0):
    return np.ascontiguousarray(np.random.default_rng(seed).uniform(low, up, (n, 2)))
