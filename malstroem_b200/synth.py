"""Deterministic synthetic DEMs (the benchmark / test input of SURVEY.md §8(d)).

`fractal_dem` is an integer-arithmetic fBm: OCTAVES octaves of hashed-lattice value noise with a
fixed-point smoothstep interpolation, summed in int64 and quantised to whole millimetres; the float32
elevation is `float32(mm) * float32(0.001)` (one rounding).  Every cell depends only on
(seed, row, col), so row-bands can be generated independently on each GPU, and because no floating
point is involved before the last multiply the numpy version here and the CUDA kernel
(csrc/synth.cu, `ms_synth_fractal_dev`) produce bit-identical rasters.

This module is numpy-only on purpose: it is input generation, not part of the hot path.
"""
import numpy as np

OCTAVES = 10
TOP_SHIFT = 10            # coarsest lattice spacing = 2**TOP_SHIFT cells
RELIEF_MM = 200000        # 0 .. 200 m
HURST_Q16 = 40342         # 2**-0.7 in Q16: amplitude ratio between octaves


def _amplitudes():
    """Per-octave amplitude in Q16 so that the amplitudes sum to 1.0 (65536)."""
    a = [1 << 16]
    for _ in range(1, OCTAVES):
        a.append((a[-1] * HURST_Q16) >> 16)
    tot = sum(a)
    return [(x << 16) // tot for x in a]


AMPL_Q16 = _amplitudes()


def _hash(ix, iy, o, seed):
    """32-bit integer hash of lattice point (uint32 arithmetic, wraps)."""
    h = (ix.astype(np.uint32) * np.uint32(0x9E3779B1)) ^ (iy.astype(np.uint32) * np.uint32(0x85EBCA77))
    h = h ^ np.uint32((seed * 0xC2B2AE3D + o * 0x27D4EB2F) & 0xFFFFFFFF)
    h ^= h >> np.uint32(15)
    h *= np.uint32(0x2C1B3C6D)
    h ^= h >> np.uint32(12)
    h *= np.uint32(0x297A2D39)
    h ^= h >> np.uint32(15)
    return (h >> np.uint32(16)).astype(np.int64)        # 0 .. 65535


def fractal_mm(rows, cols, seed=1, row0=0, col0=0):
    """Elevation in integer millimetres for the window [row0,row0+rows) x [col0,col0+cols)."""
    y = (np.arange(rows, dtype=np.int64) + row0)[:, None]
    x = (np.arange(cols, dtype=np.int64) + col0)[None, :]
    total = np.zeros((rows, cols), np.int64)
    with np.errstate(over='ignore'):
        for o in range(OCTAVES):
            sh = TOP_SHIFT - o
            if sh > 0:
                ix, iy = x >> sh, y >> sh
                tx = ((x & ((1 << sh) - 1)) << 16) >> sh
                ty = ((y & ((1 << sh) - 1)) << 16) >> sh
            else:
                ix, iy = x, y
                tx = np.zeros_like(x)
                ty = np.zeros_like(y)
            sx = (((tx * tx) >> 16) * ((3 << 16) - 2 * tx)) >> 16
            sy = (((ty * ty) >> 16) * ((3 << 16) - 2 * ty)) >> 16
            h00 = _hash(ix, iy, o, seed)
            h10 = _hash(ix + 1, iy, o, seed)
            h01 = _hash(ix, iy + 1, o, seed)
            h11 = _hash(ix + 1, iy + 1, o, seed)
            top = h00 + (((h10 - h00) * sx) >> 16)
            bot = h01 + (((h11 - h01) * sx) >> 16)
            v = top + (((bot - top) * sy) >> 16)            # 0 .. 65535
            total += v * AMPL_Q16[o]                        # Q32 of [0,1)
    return (total * RELIEF_MM) >> 32


def fractal_dem(rows, cols, seed=1, row0=0, col0=0):
    """float32 DEM, elevations 0..200 m on a 1 mm grid of values."""
    return fractal_mm(rows, cols, seed, row0, col0).astype(np.float32) * np.float32(0.001)


def pathological_dem(rows, cols, seed=1):
    """Stepped plateaus (large exact flats), concentric nested craters that straddle the k*rows/8
    band edges, and a raster-wide flat — the C5 stress input of SURVEY.md §8(d)."""
    y = np.arange(rows, dtype=np.int64)[:, None]
    x = np.arange(cols, dtype=np.int64)[None, :]
    base = fractal_mm(rows, cols, seed)
    mm = (base // 5000) * 5000                               # 5 m steps -> big exact flats
    # nested craters centred on band edges: rings of alternating rim / moat
    for k in range(1, 8):
        cy, cx = (k * rows) // 8, ((2 * k + 1) * cols) // 16
        rad = max(8, min(rows, cols) // 24)
        d = np.maximum(np.abs(y - cy), np.abs(x - cx))       # square rings: exact ties everywhere
        ring = d * 8 // rad
        inside = d < rad
        level = np.where(ring % 2 == 0, 20000 + 3000 * ring, 60000 - 2000 * ring)
        mm = np.where(inside, level, mm)
    mm[rows // 3: rows // 3 + max(2, rows // 16), :] = 100000  # raster-wide flat strip
    return mm.astype(np.float32) * np.float32(0.001)


def pathological_spiral_dem(rows, cols, seed=3):
    """BASELINE config 5 in small: stepped plateaus (large exact flats), concentric nested craters (depressions inside
    depressions, 6 levels) centred on rows k*rows/4 so that they straddle band edges, a spiral channel at one exact
    elevation (the longest geodesic one can fold into a square: stresses the no-flats wave and makes the capped fast
    path fail over to the generic one), and a flat running the whole width of the raster.  Integer millimetres ->
    float32, like fractal_dem."""
    y, x = np.mgrid[0:rows, 0:cols].astype(np.int64)
    mm = 60000 + 25 * (x + 2 * y)                         # a gentle plane, 25 mm per cell
    mm += (fractal_mm(rows, cols, seed=seed) - 100000) // 40
    mm = (mm // 2000) * 2000 + np.minimum(mm % 2000, 300)  # plateaus: 300 mm of slope, then an exact flat
    # nested craters
    for k in (1, 2, 3):
        cy, cx = k * rows // 4, (k * 2 - 1) * cols // 6
        r = np.sqrt((y - cy) ** 2 + (x - cx) ** 2)
        rad = min(rows, cols) // 7
        inside = r < rad
        ring = (r / max(rad / 12.0, 1.0)).astype(np.int64)           # 12 rings
        depth = np.where(ring % 2 == 0, 6000 + 700 * (11 - ring), 2500 + 300 * (11 - ring))   # moats and rims alternate
        mm = np.where(inside, mm[cy, cx] - depth, mm)
    # a flat across the whole raster
    band = (y >= rows * 5 // 8) & (y < rows * 5 // 8 + 6)
    mm = np.where(band, 30000, mm)
    # spiral channel, one cell wide, pitch 3, at one exact elevation; its outer end opens to the raster border
    s0 = min(rows, cols) // 3
    cy, cx = rows // 8 + s0 // 2, cols - s0 // 2 - 4
    lo = mm.min() - 5000
    yy, xx, step, d = cy, cx, 1, 0
    path = [(yy, xx)]
    moves = ((0, 1), (1, 0), (0, -1), (-1, 0))
    while step * 3 < s0:
        for _ in range(2):
            dy, dx = moves[d % 4]
            for _ in range(step * 3):
                yy += dy
                xx += dx
                path.append((yy, xx))
            d += 1
        step += 1
    py = np.clip(np.array([q[0] for q in path]), 1, rows - 2)
    px = np.clip(np.array([q[1] for q in path]), 1, cols - 2)
    mm[py, px] = lo
    # the outer end drains off the right border
    mm[py[-1], px[-1]:] = lo - 1000
    return (mm.astype(np.float32) * np.float32(0.001)).astype(np.float32)


def serpentine_path(rows, cols, pitch):
    """Cells (rows, cols index arrays, in flow order) of a one-cell channel that runs down column 1, along row rows-2,
    up column 1 + pitch, along row 1, ... every `pitch` columns, and then along its last row to the right border."""
    if pitch < 2 or rows < 5 or cols < pitch + 6:
        raise ValueError("serpentine: needs pitch >= 2, rows >= 5 and cols >= pitch + 6")
    xs = list(range(1, cols - 5, pitch))
    pr, pc = [], []
    down = np.arange(1, rows - 1)
    for k, x in enumerate(xs):
        seg = down if k % 2 == 0 else down[::-1]
        pr.append(seg)
        pc.append(np.full(seg.size, x))
        end = seg[-1]
        stop = xs[k + 1] if k + 1 < len(xs) else cols
        run = np.arange(x + 1, stop)
        pr.append(np.full(run.size, end))
        pc.append(run)
    return np.concatenate(pr), np.concatenate(pc)


def serpentine_dem(rows, cols, pitch=4, pit=False):
    """Walls of 100 and a serpentine channel (serpentine_path) whose bed falls by one step per cell to the right
    border: the whole raster drains down one path that crosses every row-band edge once per column of the channel
    (about cols / pitch times), with a flow accumulation that reaches nearly rows * cols there.  With `pit`, the third-last channel cell is a
    one-cell pit two steps below the channel cell after it: the only bluespot, whose watershed is nearly the whole
    raster.  The bed is an integer times a power of two, exact in float32 and below 64."""
    pr, pc = serpentine_path(rows, cols, pitch)
    n = pr.size
    scale = np.float32(2.0 ** -max(0, int(n).bit_length() - 6))
    bed = (n - np.arange(n)).astype(np.float32) * scale
    if pit:
        bed[n - 3] = bed[n - 1] - scale
    dem = np.full((rows, cols), 100.0, np.float32)
    dem[pr, pc] = bed
    return dem


def mask_dem(mask):
    """0 on the cells of `mask`, 10 elsewhere and on the raster border: every 8-connected component of the mask away
    from the border is one bluespot of depth 10, and the filled raster is one flat at 10."""
    dem = np.where(mask, np.float32(0.0), np.float32(10.0)).astype(np.float32)
    dem[0, :] = dem[-1, :] = dem[:, 0] = dem[:, -1] = 10.0
    return dem


def comb_mask(rows, cols):
    """Teeth in every third column from row 1 to row rows-2, joined in pairs by row rows-2 alone: two pieces of one
    component in every band but the last, which has at least two rows in any row-band split."""
    m = np.zeros((rows, cols), bool)
    teeth = list(range(3, cols - 1, 3))
    for x in teeth:
        m[1:rows - 1, x] = True
    for a, b in zip(teeth[0::2], teeth[1::2]):
        m[rows - 2, a:b + 1] = True
    return m


def speckle_mask(rows, cols, density=0.39, seed=1):
    """Independent cells at `density`: just below the 8-connected site-percolation threshold (0.407), many components,
    some hundreds of rows tall with long, thin branches."""
    return np.random.default_rng(seed).random((rows, cols)) < density


def pit_lattice_dem(rows, cols, seed=1):
    """Level ground at 10 with a one-cell pit on every cell of odd row and odd column away from the border.  No two
    pits touch, even diagonally, so each is a bluespot of its own: 1024 in a 64 x 64 tile, more than the 256-slot
    per-tile tables of the label-table pass hold.  Pit floors are 1 .. 9, seeded."""
    dem = np.full((rows, cols), 10.0, np.float32)
    pits = dem[1:rows - 1:2, 1:cols - 1:2]
    pits[...] = np.random.default_rng(seed).integers(1, 10, pits.shape).astype(np.float32)
    return dem


def pit_chain_dem(rows, cols, period=64):
    """Walls of 100 and one channel down column cols // 2: a pit in the middle of every `period` rows, a rim of two
    cells on every multiple of `period` rows, the rims falling by one per period away from the outlet at row 0 (so
    every pit spills over the rim below it into the next pit, away from the outlet, and the chain drains out over the
    60 of row 1).  With row bands of `period` rows each pit lies in its own band and spills across a band edge."""
    c = cols // 2
    r = np.arange(rows)
    mid = (r // period) * period + period // 2
    z = 10.0 + 0.25 * np.abs(r - mid)
    edge = (r % period == 0) | (r % period == period - 1)
    k = (r + 1) // period                              # the rim on rows k*period - 1, k*period
    z = np.where(edge & (r >= period - 1), 50.0 - k, z)
    dem = np.full((rows, cols), 100.0, np.float32)
    dem[1:rows - 1, c] = z[1:rows - 1]
    dem[1, c] = 60.0
    dem[0, c] = 5.0
    return dem


def sea_bowl_dem(rows, cols):
    """A bowl below sea level inside a rim of 30, drained by one channel at exactly 0 through the rim to the left
    edge of the raster: the whole interior is one lake whose fill level is 0.0, spanning every row band.  Zero has no
    binade, so the integer form of the no-flats solver refuses the raster and the float64 solver runs, on one GPU
    and across bands (a coastal DEM with the sea at 0 does the same)."""
    y, x = np.mgrid[0:rows, 0:cols].astype(np.float64)
    bowl = ((y - rows / 2) / rows) ** 2 + ((x - cols / 2) / cols) ** 2
    dem = (-20.0 + 39.0 * bowl).astype(np.float32)          # at most -0.5: no interior cell rounds to 0
    dem = (np.round(dem * 1000) / 1000).astype(np.float32)
    dem[:, :3] = dem[:, -3:] = 30.0
    dem[:3, :] = dem[-3:, :] = 30.0
    dem[rows // 3, :40] = 0.0                               # the outlet channel through the rim
    return dem
