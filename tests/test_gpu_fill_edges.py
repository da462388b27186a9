"""The plain fill's catchment edge list (csrc/fill.cu: k_tile_edges, Boruvka on the list) against the CPU oracle, bit
for bit, on inputs that stress it: exact flats (many equal edge weights), white noise (the most catchments and pairs
per tile: the per-tile table overflows), one large depression, nested craters, a chain of pits that merge one per
round, thin and odd shapes, and an edge list that outgrows the size chosen from the previous call."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from malstroem_b200 import _lib, synth
from malstroem_b200.algorithms import fill
from oracle import port

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check(dem):
    dem = np.ascontiguousarray(dem, np.float32)
    want = port.fill_terrain(dem)
    rows, cols = dem.shape
    if min(rows, cols) > 3:
        f, d = fill.fill_terrain_and_depths(dem)
    else:       # the numpy mirror follows the reference and rejects 3 rows / columns; the C ABI takes them
        f, d = np.empty_like(dem), np.empty_like(dem)
        with _lib.lock:
            _lib.check(_lib.lib().ms_fill_terrain(_lib.ptr(dem), _lib.ptr(f), _lib.ptr(d), rows, cols), "fill")
    assert np.array_equal(f, want)
    assert np.array_equal(d, want - dem)


def noise(rows, cols, seed):
    return np.random.default_rng(seed).random((rows, cols), dtype=np.float32) * np.float32(100.0)


def test_flats_and_plateaus():
    check(np.zeros((200, 300), np.float32))
    mm = synth.fractal_mm(300, 260, seed=4)
    check(((mm // 20000) * 20000).astype(np.float32) * np.float32(0.001))        # 20 m terraces
    rng = np.random.default_rng(1)
    check(rng.integers(0, 3, (257, 129)).astype(np.float32))                     # three levels, ties everywhere


def test_white_noise():
    check(noise(512, 640, 2))
    check(noise(130, 4099, 3))


def test_one_large_depression():
    y, x = np.mgrid[0:300, 0:400]
    bowl = 50.0 - 40.0 * np.exp(-(((y - 150) / 90.0) ** 2 + ((x - 200) / 120.0) ** 2))
    dem = bowl.astype(np.float32)
    dem[0, :] = dem[-1, :] = dem[:, 0] = dem[:, -1] = 100.0
    dem[0, 17] = 60.0                        # the one outlet
    check(dem)


def test_nested_craters():
    check(synth.pathological_dem(384, 448, 1))
    check(synth.pathological_spiral_dem(256, 320))


def test_chain_of_pits():
    # pits along a row, each spilling into the next over a slightly lower rim: one merge per pit down the chain
    cols = 1030
    dem = np.full((7, cols), 100.0, np.float32)
    k = np.arange(1, cols - 1)
    dem[3, 1:-1] = np.where(k % 2 == 1, 10.0, 50.0 - 0.01 * k)
    dem[3, 0] = 1.0
    check(dem)
    check(np.ascontiguousarray(dem.T))


@pytest.mark.parametrize("shape", [(3, 500), (500, 3), (3, 3), (67, 1000), (130, 4099), (129, 193), (64, 64),
                                   (65, 65), (1000, 67)])
def test_shapes(shape):
    rows, cols = shape
    check(synth.fractal_dem(rows, cols, seed=rows * 7 + cols))
    check(noise(rows, cols, rows + cols))


def test_edge_list_rerun():
    # a fresh process: a smooth DEM sizes the arena, white noise of the same size then has ~10x as many catchment
    # pairs, so its edge list overflows the first size and the tile pass runs again with the counted size
    code = textwrap.dedent("""
        import ctypes, sys
        import numpy as np
        sys.path.insert(0, %r)
        from malstroem_b200 import _lib, synth
        from malstroem_b200.algorithms import fill
        from oracle import port
        S = 1536
        smooth = synth.fractal_dem(S, S, seed=5)
        noisy = np.random.default_rng(6).random((S, S), dtype=np.float32) * np.float32(100.0)
        for _ in range(2):
            f, d = fill.fill_terrain_and_depths(smooth)
        assert np.array_equal(f, port.fill_terrain(smooth))
        L = _lib.lib()
        L.ms_profile(1)
        f, d = fill.fill_terrain_and_depths(noisy)
        buf = ctypes.create_string_buffer(1 << 16)
        L.ms_profile_report(buf, len(buf))
        L.ms_profile(0)
        want = port.fill_terrain(noisy)
        assert np.array_equal(f, want) and np.array_equal(d, want - noisy)
        n = sum(int(l.rsplit(" ", 3)[1]) for l in buf.value.decode().splitlines() if l.startswith("k_tile_edges"))
        print("tile passes", n)
    """ % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "tile passes 2" in r.stdout, r.stdout
