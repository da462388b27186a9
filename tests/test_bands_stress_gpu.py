"""Row bands on rasters built to make each stage's band-edge logic work hard (tests/band_cases.py): white noise (many
frozen fill components, a large boundary graph), exact ties across band edges, a chain of pits that spill into each
other across every band edge, a serpentine channel that carries half the raster across the band edges, and bluespot
masks whose components are joined only through other bands.  Each banded run, and the one-GPU run of the same raster,
must equal the CPU oracle bit for bit (label_stats 'sum' within 1e-6); each case also asserts that it reached the
stress it is for.  Short last bands and thin rasters come last."""
import numpy as np
import pytest
import torch

import band_cases as bc
from malstroem_b200 import bands, synth
from malstroem_b200.pipeline import TABLES, RasterPipeline

pytestmark = pytest.mark.gpu


def one_gpu(dem, want):
    p = RasterPipeline(*dem.shape)
    p.host_fnf = True
    h = p.run_host(dem)
    for name in bc.RASTERS:
        assert np.array_equal(h[name].numpy(), want[name]), name
    bc.check_tables({k: h[k].numpy() for k, _ in TABLES}, p.nlabels, want)


def banded(dem, want, nb):
    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb)
    try:
        bc.check(pipes, want)
        return dict(pipes[0].stats)
    finally:
        for p in pipes:
            p.close()


@pytest.mark.parametrize("name", list(bc.CASES))
def test_one_gpu_equals_oracle(name):
    dem, want = bc.case(name)
    one_gpu(dem, want)


@pytest.mark.parametrize("name,nb", bc.CASE_BANDS)
def test_bands_equal_oracle(name, nb):
    dem, want = bc.case(name)
    bc.assert_reach(name, nb)
    st = banded(dem, want, nb)
    if name == "noise":
        # many frozen fill components, a large boundary graph and many boundary roots of the labels: half of what a
        # B200 run saw (fill_frozen 191 / 389 / 1384, fill_graph_edges 810 / 1621 / 5824, cc_boundary_roots
        # 118 / 260 / 939 at 2 / 3 / 8 bands)
        floor = {2: (95, 405, 59), 3: (194, 810, 130), 8: (692, 2912, 469)}[nb]
        got = (st["fill_frozen"], st["fill_graph_edges"], st["cc_boundary_roots"])
        assert all(g >= f for g, f in zip(got, floor)), (got, floor)
    elif name == "pit_chain":
        # one frozen component per band; the lake down the column needs a no-flats exchange per band edge
        assert st["fill_frozen"] >= nb and st["noflat_exchanges"] >= nb - 1, st


@pytest.mark.parametrize("rows", [130, 131, 191])
@pytest.mark.parametrize("cols", [5, 67, 129, 515, 516])
def test_short_last_band_and_thin(rows, cols):
    """Last bands of 2, 3 and 63 rows (every cell of a 2-row band is an edge cell); widths that are not a multiple of 4
    (byte loads of the flow directions) and one that is."""
    for dem in (bc.noise(rows, cols, rows + cols), synth.fractal_dem(rows, cols, seed=rows * 7 + cols)):
        want = bc.oracle_all(dem)
        one_gpu(dem, want)
        banded(dem, want, 3)
