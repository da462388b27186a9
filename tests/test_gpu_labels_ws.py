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
