"""Row-band decomposition (SURVEY.md §8(e)) on one GPU, bands as threads of one process: every raster and table of
the banded run must equal the CPU oracle's result on the WHOLE raster bit for bit (label_stats 'sum' within 1e-6),
for several band counts, including bands whose lakes, flow paths and bluespots straddle the band edges."""
import numpy as np
import pytest
import torch

from band_cases import check, oracle_all
from malstroem_b200 import bands, synth
from oracle import port

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape,nbands,seed", [((320, 256), 2, 11), ((448, 200), 3, 12), ((512, 384), 4, 13),
                                               ((200, 330), 2, 14), ((640, 129), 5, 15)])
def test_bands_equal_oracle(shape, nbands, seed):
    dem = synth.fractal_dem(shape[0], shape[1], seed=seed)
    want = oracle_all(dem)
    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nbands)
    try:
        check(pipes, want)
    finally:
        for p in pipes:
            p.close()


def test_bands_lake_across_every_edge():
    """One basin spanning all bands (a bowl with a rim and a single outlet), plus a flat plateau: the spill graph,
    the no-flats wave, the accumulation forest and one bluespot all cross every band edge."""
    rows, cols = 384, 192
    y, x = np.mgrid[0:rows, 0:cols].astype(np.float64)
    bowl = ((y - rows / 2) / rows) ** 2 + ((x - cols / 2) / cols) ** 2
    dem = (50.0 + 40.0 * bowl).astype(np.float32)
    dem[:, :3] = dem[:, -3:] = 80.0
    dem[:3, :] = dem[-3:, :] = 80.0
    dem[rows // 3, :40] = 55.0                      # the outlet channel through the rim
    dem[200:260, 100:150] = np.float32(52.0)        # a plateau inside the lake area (exact flat)
    dem = (np.round(dem * 1000) / 1000).astype(np.float32)
    want = oracle_all(dem)
    for nb in (2, 3, 6):
        pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb)
        try:
            check(pipes, want)
        finally:
            for p in pipes:
                p.close()


def test_pathological_single_and_banded():
    """BASELINE config 5 in small (synth.pathological_spiral_dem): exact plateaus (79 % of the cells are lake / flat),
    nested craters on the band edges, a raster-wide flat and a spiral channel with a 9500-step geodesic, on one GPU
    and in bands."""
    from malstroem_b200.pipeline import RasterPipeline
    dem = synth.pathological_spiral_dem(768, 512)
    want = oracle_all(dem)
    p = RasterPipeline(768, 512)
    p.host_fnf = True                 # also bring the no-flats surface back (an intermediate otherwise)
    h = p.run_host(dem)
    for name in ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds"):
        assert np.array_equal(h[name].numpy(), want[name]), name
    assert p.nlabels == want["n"]
    for nb in (2, 3):
        pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb)
        try:
            check(pipes, want)
        finally:
            for q in pipes:
                q.close()


def test_pathological_plateaus_banded():
    """synth.pathological_dem: 5 m plateaus, square-ring craters on the k*rows/8 band edges, a raster-wide flat."""
    dem = synth.pathological_dem(512, 384)
    want = oracle_all(dem)
    for nb in (2, 8):
        pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb)
        try:
            check(pipes, want)
        finally:
            for q in pipes:
                q.close()


def test_pathological_float64_form_falls_back():
    """With the integer tile form switched off (MS_NF_INT=0, read once per process, hence the subprocess) the capped
    float64 form cannot carry the spiral's wave past the cap: the verification stencil must reject it and the
    generic solve must deliver the reference's bits."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import numpy as np\n"
        "from malstroem_b200 import synth\n"
        "from malstroem_b200.pipeline import RasterPipeline\n"
        "from oracle import port\n"
        "dem = synth.pathological_spiral_dem(768, 512)\n"
        "p = RasterPipeline(768, 512)\n"
        "p.host_fnf = True\n"
        "h = p.run_host(dem)\n"
        "short, diag = port.minimum_safe_short_and_diag(dem)\n"
        "assert np.array_equal(h['fnf'].numpy(), port.fill_terrain_no_flats(dem, short, diag))\n"
        "assert p.stats['noflat_reverify'] >= 1, p.stats\n"
        "print('fallback ok', p.stats)\n")
    env = dict(os.environ, MS_NF_INT="0", PYTHONPATH=root)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "fallback ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("shape,nbands,seed", [((512, 384), 4, 21), ((448, 300), 3, 22)])
def test_band_network_and_rain_equal_oracle(shape, nbands, seed):
    """SURVEY.md 8(f1,f2) across bands: downstream bluespots and rain events of the banded run == the oracle's
    pourpoint_network / rain_events on the whole raster (both pour-point variants), on every rank."""
    from malstroem_b200 import network
    dem = synth.fractal_dem(shape[0], shape[1], seed=seed)
    want = oracle_all(dem)
    mm = [10.0, 30.0, 100.0]
    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nbands,
                               after=lambda p: (p.network(0.16, mm), p.network(0.16, mm, use_accum_pourpoints=True)))
    try:
        area = np.zeros(want["n"] + 1)
        area[:len(want["count"])] = want["count"]
        area *= 0.16
        for k, key in enumerate(("ppmin", "ppmax")):
            cells = list(zip(want[key]["row"].tolist(), want[key]["col"].tolist()))
            nodes = port.pourpoint_network(want["flowdir"], want["labels"], cells, 0)
            parent = np.array([-1 if d["downstream_id"] is None else d["downstream_id"] for d in nodes])
            for p in pipes:
                got = p.after_result[k]
                assert np.array_equal(got["parent"].cpu().numpy(), parent), key
                ref = port.rain_events(parent, area, p.tables["st_sum"].cpu().numpy() * 0.16, mm, network.SUM_MODE)
                for q in ("rainv", "spillv", "v", "pctv"):
                    assert np.array_equal(got[q].cpu().numpy(), ref[q], equal_nan=True), (key, q)
    finally:
        for p in pipes:
            p.close()


@pytest.mark.parametrize("eps", [(1e-3, 1.5e-3), (0.01, 0.015)])
def test_band_seed_repair(eps):
    """fill_terrain_no_flats takes short / diag as arguments (fill.py:174); with steps of the size of the DEM's own
    height differences a lake rises above "seed" cells next to it (236 / 2604 of them here) and the seed assumption has
    to be repaired: the stencil rejects, the cells are banned, the solve is repeated.  One GPU does that in
    fill_no_flats_dev_impl, the bands in BandPipeline._noflats: both must give the reference's bits."""
    from malstroem_b200.algorithms import fill
    dem = synth.fractal_dem(320, 256, seed=5)
    want = port.fill_terrain_no_flats(dem, eps[0], eps[1])
    assert np.array_equal(fill.fill_terrain_no_flats(dem, eps[0], eps[1]), want)
    for nb in (2, 5):
        pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb, eps=eps)
        try:
            got = torch.cat([p.out["fnf"] for p in pipes]).cpu().numpy()
            assert np.array_equal(got, want)
            assert max(p.stats.get("noflat_repairs", 0) for p in pipes) >= 1, pipes[0].stats
            fd = torch.cat([p.out["flowdir"] for p in pipes]).cpu().numpy()
            assert np.array_equal(fd, port.terrain_flowdirection(want))
        finally:
            for p in pipes:
                p.close()
