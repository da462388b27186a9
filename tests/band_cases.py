"""Shared by the row-band tests: the CPU oracle on the whole raster, the comparison of a run with it, and what a
raster makes the band-edge logic do (computed in numpy from the oracle's results, so that a test can assert that its
input reaches the stress it is for)."""
import functools

import numpy as np
import scipy.ndimage
import torch

from malstroem_b200 import bands, synth
from oracle import port

DR = np.array((-1, -1, 0, 1, 1, 1, 0, -1))
DC = np.array((0, 1, 1, 1, 0, -1, -1, -1))
RASTERS = ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds")


def oracle_all(dem):
    filled = port.fill_terrain(dem)
    short, diag = port.minimum_safe_short_and_diag(dem)
    fnf = port.fill_terrain_no_flats(dem, short, diag)
    fd = port.terrain_flowdirection(fnf)
    acc = port.accumulated_flow(fd, fast=True)
    depths = filled - dem
    lab, n = port.connected_components(depths)
    ws = lab.copy()
    port.watersheds_from_labels(fd, ws, 0)
    return dict(filled=filled, depths=depths, fnf=fnf, flowdir=fd, accum=acc, labels=lab, wsheds=ws, n=n,
                stats=port.label_stats(depths, lab, n), count=port.label_count(ws),
                ppmin=port.label_min_index(fnf, lab, n), ppmax=port.label_max_index(acc, lab, n))


def check_tables(t, nlabels, want):
    """t: numpy tables of one run (at least nlabels + 1 entries each) against the oracle's."""
    assert nlabels == want["n"]
    m = want["n"] + 1
    for k in ("min", "max", "count"):
        assert np.array_equal(t["st_" + k][:m], want["stats"][k]), k
    np.testing.assert_allclose(t["st_sum"][:m], want["stats"]["sum"], rtol=1e-6, atol=1e-300)
    c = len(want["count"])
    assert np.array_equal(t["ws_count"][:c], want["count"]) and not t["ws_count"][c:m].any()
    for key in ("ppmin", "ppmax"):
        for f in ("row", "col", "value"):
            assert np.array_equal(t[key + "_" + f][:m], want[key][f]), key + "_" + f


def check(pipes, want):
    """Every raster of a banded run, and the tables of every rank, against the oracle's."""
    for name in RASTERS:
        got = torch.cat([p.out[name] for p in pipes]).cpu().numpy()
        assert np.array_equal(got, want[name]), name
    for p in pipes:                                   # every rank holds the same, complete tables
        check_tables({k: v.cpu().numpy() for k, v in p.tables.items()}, p.nlabels, want)


def band_of_row(rows, nbands):
    out = np.empty(rows, np.int64)
    for g, (r0, r1) in enumerate(bands.band_rows(rows, nbands)):
        out[r0:r1] = g
    return out


def d8_steps(fd):
    """(source flat index, target flat index) of every D8 step that stays on the raster."""
    rows, cols = fd.shape
    r, c = np.nonzero(fd <= 7)
    d = fd[r, c].astype(np.int64)
    tr, tc = r + DR[d], c + DC[d]
    ok = (tr >= 0) & (tr < rows) & (tc >= 0) & (tc < cols)
    return r[ok] * cols + c[ok], tr[ok] * cols + tc[ok]


def band_crossings(fd, nbands):
    """The D8 steps that cross a band edge: (source, target) flat indices."""
    rows, cols = fd.shape
    band = band_of_row(rows, nbands)
    s, t = d8_steps(fd)
    x = band[s // cols] != band[t // cols]
    return s[x], t[x]


def max_band_inflow(fd, accum, nbands):
    """The largest flow that enters one cell from the neighbouring band (the sum over the cells of that band that
    drain into it): the inflow the accumulation's band-entry cells carry into their band."""
    s, t = band_crossings(fd, nbands)
    inflow = np.zeros(fd.size, np.float64)
    np.add.at(inflow, t, accum.ravel()[s])
    return inflow.max() if s.size else 0.0


def band_presence(lab, nbands):
    """[label, band]: whether the label has cells in the band."""
    band = band_of_row(lab.shape[0], nbands)
    seen = np.zeros((lab.max() + 1, nbands), bool)
    r, c = np.nonzero(lab)
    seen[lab[r, c], band[r]] = True
    return seen


def labels_spanning_all_bands(lab, nbands):
    """Labels with cells in every band."""
    return np.nonzero(band_presence(lab, nbands).all(1))[0]


def split_in_first_band(lab, nbands):
    """Labels with two or more 8-connected pieces inside band 0 that also have cells in every band: the band-0 pieces
    are one component only through the other bands."""
    r1 = bands.band_rows(lab.shape[0], nbands)[0][1]
    out = []
    for L in labels_spanning_all_bands(lab, nbands):
        _, k = scipy.ndimage.label(lab[:r1] == L, structure=np.ones((3, 3)))
        if k >= 2:
            out.append(int(L))
    return out


def cross_band_ties(want, nbands):
    """Per table (st_min, st_max over depths; ppmin over fnf, ppmax over accum): the number of labels whose extreme
    value is held by cells in two or more bands, so that the min / max all-reduce meets equal values and the arg
    index has to be the smallest global one."""
    lab = want["labels"]
    band = band_of_row(lab.shape[0], nbands)
    r, c = np.nonzero(lab)
    L = lab[r, c]
    out = {}
    for key, raster, ext in (("st_min", want["depths"], want["stats"]["min"]),
                             ("st_max", want["depths"], want["stats"]["max"]),
                             ("ppmin", want["fnf"], want["ppmin"]["value"]),
                             ("ppmax", want["accum"], want["ppmax"]["value"])):
        at = raster[r, c] == ext[L]
        seen = np.zeros((lab.max() + 1, nbands), bool)
        seen[L[at], band[r[at]]] = True
        out[key] = int((seen.sum(1) >= 2).sum())
    return out


def labels_per_tile(lab, tile=64):
    """The number of distinct nonzero labels in each tile x tile tile (flat, row-major over the tiles)."""
    rows, cols = lab.shape
    tiles_x = -(-cols // tile)
    r, c = np.nonzero(lab)
    top = int(lab.max()) + 1
    key = ((r // tile) * tiles_x + c // tile) * top + lab[r, c]
    return np.bincount(np.unique(key) // top, minlength=tiles_x * -(-rows // tile))


def chain_spills_on_edges(dem, depths, nbands):
    """Pits (cells lower than all eight neighbours, inside a bluespot) whose spill along their column - the lower of
    the two crests met walking up and down the column from the pit - lies on one of the two rows of a band edge."""
    rows, cols = dem.shape
    edges = set()
    for r0, _ in bands.band_rows(rows, nbands)[1:]:
        edges.update((r0 - 1, r0))
    pad = np.pad(dem, 1, constant_values=np.inf)
    pit = depths > 0
    for dr in (-1, 0, 1):
        for dc in (-1, 0, 1):
            if dr or dc:
                pit &= dem < pad[1 + dr:1 + dr + rows, 1 + dc:1 + dc + cols]
    n = 0
    for r, c in zip(*np.nonzero(pit)):
        col = dem[:, c]
        up = down = r
        while up > 0 and col[up - 1] >= col[up]:
            up -= 1
        while down < rows - 1 and col[down + 1] >= col[down]:
            down += 1
        n += int((up if col[up] < col[down] else down) in edges)
    return n


# ------------------------------------------------------------------------------------ the stress rasters
def noise(rows, cols, seed):
    return np.random.default_rng(seed).random((rows, cols), dtype=np.float32) * np.float32(100.0)


def _interior(mask):
    m = mask.copy()
    m[0, :] = m[-1, :] = m[:, 0] = m[:, -1] = False
    return m


# name -> (builder, band counts); 960 rows split into 2, 3, 5 and 8 bands, 500 rows into 3 and 8 (450 - 512 rows make
# 8 bands of 64 rows)
CASES = {
    "noise": (lambda: noise(1024, 515, 2), (2, 3, 8)),
    "levels": (lambda: np.random.default_rng(1).integers(0, 3, (500, 257)).astype(np.float32), (3, 8)),
    "terraces": (lambda: ((synth.fractal_mm(960, 515, seed=4) // 20000) * 20000).astype(np.float32)
                 * np.float32(0.001), (3, 8)),
    "pit_chain": (lambda: synth.pit_chain_dem(500, 67), (8,)),
    "serpentine": (lambda: synth.serpentine_dem(1024, 512, 4), (4, 8)),
    "serpentine_pit": (lambda: synth.serpentine_dem(1024, 512, 4, pit=True), (3, 8)),
    "comb": (lambda: synth.mask_dem(synth.comb_mask(960, 515)), (2, 5, 8)),
    "speckle": (lambda: synth.mask_dem(synth.speckle_mask(960, 515)), (2, 5, 8)),
    "pit_lattice": (lambda: synth.pit_lattice_dem(320, 258), (2, 3)),
}
CASE_BANDS = [(name, nb) for name, (_, nbs) in CASES.items() for nb in nbs]


@functools.lru_cache(maxsize=None)
def case(name):
    """The raster of a case and the oracle's results on it (built once per process)."""
    dem = CASES[name][0]()
    return dem, oracle_all(dem)


def assert_reach(name, nb):
    """What the case is for, asserted on its input and the oracle's results."""
    dem, want = case(name)
    lab = want["labels"]
    if name == "noise":
        # bluespots cut by band edges (17 / 48 / 166 at 2 / 3 / 8 bands)
        assert (band_presence(lab, nb).sum(1) >= 2).sum() >= 15 * (nb - 1)
    elif name == "levels":
        # a bluespot whose lowest no-flats value is held in two bands: the arg-min goes to the smallest global index
        assert cross_band_ties(want, nb)["ppmin"] >= 1
    elif name == "terraces":
        assert sum(cross_band_ties(want, nb).values()) >= 1
    elif name == "pit_chain":
        # one pit per band, each spilling into the next across a band edge: the boundary graph is a path of nb nodes
        assert chain_spills_on_edges(dem, want["depths"], nb) == nb
    elif name == "serpentine":
        s, _ = band_crossings(want["flowdir"], nb)
        assert s.size >= 300                                         # 381 at 4 bands, 889 at 8
        assert max_band_inflow(want["flowdir"], want["accum"], nb) >= 1 << 16      # the high half of the wide inflow
    elif name == "serpentine_pit":
        assert want["n"] == 1 and want["count"][1] > 0.9 * dem.size
        assert 1 in labels_spanning_all_bands(want["wsheds"], nb)
    elif name in ("comb", "speckle"):
        m = _interior(dem == 0)
        assert np.array_equal(want["depths"] != 0, m)
        assert np.array_equal(lab, scipy.ndimage.label(m, structure=np.ones((3, 3)))[0])
        if name == "comb":
            assert split_in_first_band(lab, nb)
        else:
            assert (band_presence(lab, nb).sum(1) >= 2).sum() >= 15 * (nb - 1)     # 17 / 87 / 179
    elif name == "pit_lattice":
        # more bluespots (and watersheds) in a 64 x 64 tile than the per-tile tables of the label-table pass hold
        # (1024 in a full tile)
        assert labels_per_tile(lab).max() > 256 and labels_per_tile(want["wsheds"]).max() > 256
