"""The stress rasters of tests/test_bands_stress_gpu.py (malstroem_b200.synth builders and the inline white noise,
integer levels and terraces) against the CPU oracle: each one has the property its banded case is meant to exercise at
the band counts it runs with.  Without this a builder could drift into a raster that no longer reaches that stress and
the GPU case would keep passing."""
import numpy as np
import pytest

import band_cases as bc
from malstroem_b200 import bands, synth


@pytest.mark.parametrize("name,nb", bc.CASE_BANDS)
def test_case_reaches_its_stress(name, nb):
    bc.assert_reach(name, nb)


def test_serpentine_path_is_one_channel():
    rows, cols, pitch = 130, 300, 4
    pr, pc = synth.serpentine_path(rows, cols, pitch)
    step = np.abs(np.diff(pr)) + np.abs(np.diff(pc))
    assert (step == 1).all() and len(set(zip(pr.tolist(), pc.tolist()))) == pr.size
    assert pc[-1] == cols - 1 and pr.min() == 1 and pr.max() == rows - 2
    dem = synth.serpentine_dem(rows, cols, pitch)
    assert (np.diff(dem[pr, pc]) < 0).all() and dem[pr, pc].max() < 64.0
    want = bc.oracle_all(dem)
    assert want["n"] == 0 and bc.band_crossings(want["flowdir"], 3)[0].size >= 250


@pytest.mark.parametrize("rows,last", [(130, 2), (131, 3), (191, 63)])
def test_short_last_band(rows, last):
    r = bands.band_rows(rows, 3)
    assert r[-1][1] - r[-1][0] == last
