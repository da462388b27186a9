"""The pipeline's bluespot labels and watersheds (csrc/labels.cu: roots numbered from per-row-segment root masks;
csrc/flow.cu: k_ws_tile writing the watershed raster directly, forest_resolve_ids for the paths that leave their
tile) bit for bit against the CPU oracle and against the generic in-place watersheds_from_labels (the ptr form), on
rasters built so that paths cross dozens of tiles, components span many tiles and are hooked across tile edges, and
roots sit in partial 64-cell row segments and in last columns."""
import numpy as np
import pytest

from malstroem_b200 import synth
from malstroem_b200.algorithms import flow
from malstroem_b200.pipeline import RasterPipeline
from oracle import port

pytestmark = pytest.mark.gpu
FT = 64


def tiles_touched(rows, cols, cells):
    r, c = np.divmod(cells, cols)
    return np.unique((r // FT) * (-(-cols // FT)) + c // FT).size


def run_and_check(dem, bluespot_filter=None):
    p = RasterPipeline(*dem.shape)
    h = p.run_host(dem, bluespot_filter=bluespot_filter)
    lab, ws, fd = h["labels"].numpy(), h["wsheds"].numpy(), h["flowdir"].numpy()
    assert np.array_equal(fd, port.terrain_flowdirection(port.fill_terrain_no_flats(
        dem, *port.minimum_safe_short_and_diag(dem))))
    if bluespot_filter is None:
        want_lab, n = port.connected_components(port.fill_terrain(dem) - dem)
        assert p.nlabels == n
        assert np.array_equal(lab, want_lab)
    else:
        n = p.nlabels
        assert 0 < n < p.stats["bluespots_raw"], "the filter should keep some bluespots and drop others"
        assert lab.max() == n and np.array_equal(np.unique(lab), np.arange(n + 1))
    want_ws = lab.copy()
    port.watersheds_from_labels(fd, want_ws, 0)
    assert np.array_equal(ws, want_ws)
    generic = lab.copy()
    flow.watersheds_from_labels(fd, generic, unassigned=0)
    assert np.array_equal(ws, generic)
    return p, lab, ws


@pytest.mark.parametrize("shape,pitch", [((300, 700), 4), ((700, 300), 5), ((200, 63), 4), ((130, 64), 3),
                                         ((129, 65), 4), ((257, 129), 6)])
@pytest.mark.parametrize("pit", [False, True])
def test_serpentine(shape, pitch, pit):
    dem = synth.serpentine_dem(*shape, pitch=pitch, pit=pit)
    p, lab, ws = run_and_check(dem)
    if pit:
        assert p.nlabels == 1
        # the one bluespot's watershed: at 300 x 700 and 700 x 300 every one of the 55 tiles drains into it
        cells = np.flatnonzero(ws.ravel() == 1)
        assert tiles_touched(*shape, cells) >= 2


@pytest.mark.parametrize("shape", [(300, 63), (300, 64), (300, 65), (260, 129), (513, 700)])
@pytest.mark.parametrize("kind", ["comb", "speckle"])
def test_masks(shape, kind):
    mask = synth.comb_mask(*shape) if kind == "comb" else synth.speckle_mask(*shape, seed=shape[1])
    p, lab, ws = run_and_check(synth.mask_dem(mask))
    assert p.nlabels > 1
    flat = lab.ravel()
    # the largest component spans several tiles, so roots were hooked across tile edges
    big = np.argmax(np.bincount(flat)[1:]) + 1
    assert tiles_touched(*shape, np.flatnonzero(flat == big)) >= 2
    if kind == "comb":
        return
    # roots (first cells) in the last column of a 64-cell segment or of the raster, and in a partial last segment
    first_col = np.unique(flat, return_index=True)[1][1:] % shape[1]
    assert ((first_col % FT == FT - 1) | (first_col == shape[1] - 2)).any()
    if shape[1] % FT > 1:          # (a partial segment of one column holds only the border)
        assert (first_col >= shape[1] // FT * FT).any()


@pytest.mark.parametrize("shape", [(400, 129), (257, 513)])
def test_filtered(shape):
    dem = synth.fractal_dem(*shape, seed=shape[1])
    run_and_check(dem, bluespot_filter="maxdepth > 0.05")


# ------------------------------------------------------------ watersheds_from_labels over interior no-direction cells
DR = np.array((-1, -1, 0, 1, 1, 1, 0, -1))
DC = np.array((0, 1, 1, 1, 0, -1, -1, -1))


def nodir_flowdir(rows, cols, seed):
    """D8 codes of a tilted random terrain (the noise is smaller than the tilt, so every path runs to the border across
    many tiles), then about 2 % of the interior cells set to 8 (no direction).  Only codes from terrain_flowdirection
    and 8: turning a code into 8 cannot close a cycle."""
    rng = np.random.default_rng(seed)
    r, c = np.mgrid[0:rows, 0:cols]
    sr, sc = rng.choice([-1.0, 1.0], 2)
    fd = port.terrain_flowdirection(sr * r + sc * 0.7 * c + rng.random((rows, cols)) * 0.5)
    stop = rng.random((rows, cols)) < 0.02
    stop[0, :] = stop[-1, :] = stop[:, 0] = stop[:, -1] = False
    fd[stop] = 8
    return fd


def path_ends(fd, labelled):
    """(end of every cell's path, first labelled cell or end on it) as flat indices, by pointer doubling in numpy."""
    rows, cols = fd.shape
    i = np.arange(fd.size)
    r, c = np.divmod(i, cols)
    d = fd.ravel().astype(np.int64)
    tr, tc = r + DR[np.minimum(d, 7)], c + DC[np.minimum(d, 7)]
    nxt = np.where((d <= 7) & (tr >= 0) & (tr < rows) & (tc >= 0) & (tc < cols), tr * cols + tc, i)
    end, stop = nxt, np.where(labelled.ravel(), i, nxt)
    for _ in range(int(fd.size).bit_length() + 1):
        end, stop = end[end], stop[stop]
    return end, stop


WS_DTYPES = [(np.int32, 0), (np.int32, 7), (np.int32, -1), (np.int64, 0), (np.int64, 7), (np.int64, -1),
             (np.uint32, 0), (np.uint32, 7), (np.int16, 0), (np.int16, 7), (np.int16, -1)]


@pytest.mark.parametrize("dt,unassigned", WS_DTYPES, ids=["%s-%d" % (np.dtype(d).name, u) for d, u in WS_DTYPES])
def test_watersheds_interior_nodir(dt, unassigned):
    """The general path of the public watersheds_from_labels (the label-free pointer forest and the border test of
    k_ws_assign): a cell whose path dies at an interior no-direction cell keeps its value, even when the path passes
    a labelled cell first.  Sparse labels (0.8 % of the cells; 0 is a label when `unassigned` is -1), values up to the
    dtype's range."""
    rows, cols = 333, 270
    k = WS_DTYPES.index((dt, unassigned))
    rng = np.random.default_rng(40 + k)
    fd = nodir_flowdir(rows, cols, k)
    hi = {np.int16: 30000, np.int32: 2 ** 31 - 1, np.uint32: 2 ** 32 - 1, np.int64: 2 ** 40}[dt]
    lab = np.full((rows, cols), unassigned, dt)
    on = rng.random((rows, cols)) < 0.008
    vals = rng.integers(0 if unassigned == -1 else 1, hi, on.sum(), dtype=np.int64)
    vals[vals == unassigned] += 1
    if unassigned == -1:
        vals[::10] = 0                       # 0 is a label like any other
    lab[on] = vals.astype(dt)
    labelled = lab != unassigned
    assert labelled.mean() < 0.01 and (unassigned != -1 or (lab == 0).any())
    # the reach: unlabelled cells whose path crosses a tile edge and then dies at an interior code-8 cell, and ones
    # whose path meets a labelled cell before it dies there
    end, stop = path_ends(fd, labelled)
    er, ec = np.divmod(end, cols)
    dies = (fd.ravel()[end] == 8) & (er > 0) & (ec > 0) & (er < rows - 1) & (ec < cols - 1) & ~labelled.ravel()
    start_tile = np.arange(fd.size) // cols // FT * 100 + np.arange(fd.size) % cols // FT
    assert (dies & (start_tile != er // FT * 100 + ec // FT)).sum() >= 10
    assert (dies & labelled.ravel()[stop]).sum() >= 10
    got, want = lab.copy(), lab.copy()
    assert flow.watersheds_from_labels(fd, got, unassigned=unassigned) is None
    port.watersheds_from_labels(fd, want, unassigned)
    assert got.dtype == dt and np.array_equal(got, want)
    assert (want != lab).sum() > 100 and (want.ravel()[dies] == unassigned).all()
