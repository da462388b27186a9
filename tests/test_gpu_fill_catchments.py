"""The plain fill's catchment numbering (csrc/fill.cu: k_descent_tile numbers the local minima in tile order with a
decoupled look-back over the per-tile counts, forest_resolve_ids finishes the paths that leave their tile): the
number of catchments against a numpy count of the local minima, and long descents across many tiles and row bands
against the CPU oracle."""
import numpy as np
import pytest
import torch

from malstroem_b200 import bands
from malstroem_b200.algorithms import fill
from malstroem_b200.pipeline import RasterPipeline
from oracle import port

pytestmark = pytest.mark.gpu


def local_minima(dem):
    """Interior cells below all 8 neighbours in the strict order (z, flat index) of the descent."""
    rows, cols = dem.shape
    idx = np.arange(rows * cols).reshape(rows, cols)
    zc, ic = dem[1:-1, 1:-1], idx[1:-1, 1:-1]
    low = np.ones(zc.shape, bool)
    for dr in (-1, 0, 1):
        for dc in (-1, 0, 1):
            if dr or dc:
                zn = dem[1 + dr:rows - 1 + dr, 1 + dc:cols - 1 + dc]
                jn = idx[1 + dr:rows - 1 + dr, 1 + dc:cols - 1 + dc]
                low &= (zn > zc) | ((zn == zc) & (jn > ic))
    return int(low.sum())


def pipeline_run(dem):
    p = RasterPipeline(*dem.shape)
    p.host_fnf = True                 # also bring the no-flats surface back (an intermediate otherwise)
    h = p.run_host(dem)
    return p, h


def noise(rows, cols, seed):
    return np.random.default_rng(seed).random((rows, cols), dtype=np.float32) * np.float32(100.0)


def tilted_plane(rows, cols, seed):
    """Falls towards column 0 by 1 per cell, with noise of up to 1.5: most paths run across dozens of tiles to the
    left border, and the noise leaves some pits on the way."""
    c = np.arange(cols, dtype=np.float32)[None, :]
    rng = np.random.default_rng(seed)
    return (c + rng.random((rows, cols), dtype=np.float32) * np.float32(1.5)).astype(np.float32)


@pytest.mark.parametrize("shape,seed", [((2048, 2048), 1), ((3, 5000), 2), ((5000, 3), 3), ((65, 4099), 4),
                                        ((64, 64), 5), ((40, 50), 6)])
def test_catchment_count(shape, seed):
    dem = noise(*shape, seed)
    p, h = pipeline_run(dem)
    assert p.stats["catchments"] == 1 + local_minima(dem)
    assert np.array_equal(h["filled"].numpy(), port.fill_terrain(dem))


def test_long_descent_single():
    dem = tilted_plane(300, 4160, 7)
    f, d = fill.fill_terrain_and_depths(dem)
    want = port.fill_terrain(dem)
    assert np.array_equal(f, want)
    assert np.array_equal(d, want - dem)
    p, h = pipeline_run(dem)
    assert p.stats["catchments"] == 1 + local_minima(dem)
    assert p.stats["fill_jump_rounds"] > 1
    assert np.array_equal(h["filled"].numpy(), want)


def test_long_descent_bands():
    dem = tilted_plane(384, 4160, 8)
    _, h = pipeline_run(dem)
    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), 3)
    try:
        for name in ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds"):
            got = torch.cat([q.out[name] for q in pipes]).cpu().numpy()
            assert np.array_equal(got, h[name].numpy()), name
    finally:
        for q in pipes:
            q.close()
