"""Bluespot water levels and water-depth rasters on the GPU (csrc/flood.cu): levels and wet counts against the numpy
oracle (oracle/flood.py), rasters bit for bit against numpy from the levels the GPU returned, on the golden 188 x 250
DEM, a device-resident 1024^2 fractal run, a bluespot of over 3 M cells and a raster of bowls from 1 to ~10^5 cells
(all three segment-size paths in one call), integer cases that must be exact, and run-to-run determinism."""
import numpy as np
import pytest

from malstroem_b200 import flood
from malstroem_b200.algorithms import fill, label
from oracle import flood as oflood
from oracle import port

pytestmark = pytest.mark.gpu


def _levels_close(got, want, exact=False):
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    if exact:
        assert np.array_equal(got[m], want[m])
    else:
        assert (np.abs(got[m] - want[m]) <= 1e-12 * np.maximum(1.0, np.abs(want[m]))).all()


def _wet_from_levels(dem, lab, level):
    z = dem.astype(np.float64).ravel()
    l = lab.ravel()
    out = np.zeros(level.shape, np.int64)
    for e in range(level.shape[0]):
        with np.errstate(invalid="ignore"):
            w = (l > 0) & (z < level[e][l])
        out[e] = np.bincount(l[w], minlength=level.shape[1])
    return out


def _check(dem, filled, lab, v, ca, st_sum, exact=False):
    got = flood.water_levels(dem, filled, lab, v, ca, st_sum)
    want = oflood.water_levels(dem, filled, lab, v, ca, st_sum)
    _levels_close(got["level"], want["level"], exact)
    if exact:
        assert np.array_equal(got["wet"], want["wet"])
    else:
        same = got["level"] == want["level"]
        assert np.array_equal(got["wet"][same], want["wet"][same])
        full = want["wet"] == np.bincount(lab.ravel(), minlength=v.shape[-1])[None, :]
        assert np.array_equal(got["wet"][~full], _wet_from_levels(dem, lab, got["level"])[~full])
    for e in range(got["level"].shape[0]):
        d = flood.water_depth(dem, filled, lab, got["level"][e])
        assert d.dtype == np.float32
        assert np.array_equal(d, oflood.water_depth(dem, filled, lab, got["level"][e]))
    return got


def _network_volumes(dem, filled, lab, n, ca, mm):
    short, diag = port.minimum_safe_short_and_diag(dem)
    fnf = port.fill_terrain_no_flats(dem, short, diag)
    fd = port.terrain_flowdirection(fnf)
    mi = port.label_min_index(fnf, lab, n)
    cells = list(zip(mi["row"].tolist(), mi["col"].tolist()))
    parent = np.array([-1 if d["downstream_id"] is None else d["downstream_id"]
                       for d in port.pourpoint_network(fd, lab, cells, 0)])
    ws = lab.copy()
    port.watersheds_from_labels(fd, ws, 0)
    area = port.label_count(ws).astype(np.float64) * ca
    area = np.pad(area, (0, n + 1 - area.size))
    st_sum = port.label_stats(filled - dem, lab, n)["sum"]
    return port.rain_events(parent, area, st_sum * ca, mm, 1)["v"], st_sum


def test_golden_dtm188(dtm188):
    dem = dtm188["dtm"]
    filled = port.fill_terrain(dem)
    lab, n = port.connected_components(filled - dem)
    v, st_sum = _network_volumes(dem, filled, lab, n, 0.16, [10.0, 30.0, 100.0])
    got = _check(dem, filled, lab, v, 0.16, st_sum)
    assert (got["wet"] > 0).any()
    # st_sum computed by the library when not given
    again = flood.water_levels(dem, filled, lab, v, 0.16)
    assert np.array_equal(again["level"], got["level"], equal_nan=True)


def test_pipeline_fractal_1024():
    import torch
    from malstroem_b200.pipeline import RasterPipeline, synth_fractal
    size, ca, mm = 1024, 0.16, [10.0, 30.0, 100.0]
    pipe = RasterPipeline(size, size)
    pipe.run(synth_fractal(size, size, seed=2))
    net = pipe.network(cell_area=ca, events_mm=mm)
    fl = pipe.flood(net, ca)
    rasters = [pipe.water_depth(fl["level"][e]).cpu().numpy() for e in range(len(mm))]
    torch.cuda.synchronize()
    dem, filled = pipe.dem.cpu().numpy(), pipe.out["filled"].cpu().numpy()
    lab, depths = pipe.out["labels"].cpu().numpy(), pipe.out["depths"].cpu().numpy()
    n = pipe.nlabels
    st_sum, v = pipe.table("st_sum").cpu().numpy(), net["v"].cpu().numpy()
    level, wet = fl["level"].cpu().numpy(), fl["wet"].cpu().numpy()
    want = oflood.water_levels(dem, filled, lab, v, ca, st_sum)
    _levels_close(level, want["level"])
    same = level == want["level"]
    assert np.array_equal(wet[same], want["wet"][same]) and same.mean() > 0.9
    cap = st_sum * ca
    count = np.bincount(lab.ravel(), minlength=n + 1)
    L = np.zeros(n + 1)
    L[lab.ravel()] = filled.ravel()
    l = lab.ravel()
    for e in range(len(mm)):
        d = rasters[e]
        assert np.array_equal(d, oflood.water_depth(dem, filled, lab, level[e]))
        full = v[e] == cap
        full[0] = False
        assert np.array_equal(full[1:], (level[e] == L)[1:])
        on_full = full[l].reshape(lab.shape)
        assert np.array_equal(d[on_full], depths[on_full])
        assert (d[lab == 0] == 0).all() and (d <= depths).all()
        vol = np.bincount(l, weights=d.ravel().astype(np.float64), minlength=n + 1) * ca
        ok = ~np.isnan(v[e])
        ok[0] = False
        tol = 1e-6 * v[e][ok] + 4 * np.finfo(np.float64).eps * np.abs(L[ok]) * count[ok] * ca
        assert (np.abs(vol[ok] - v[e][ok]) <= tol).all()
    lv = np.where(np.isnan(level), -np.inf, level)
    assert (lv[1:] >= lv[:-1]).all()
    # determinism: the same call again, bit for bit
    fl2 = pipe.flood(net, ca)
    assert torch.equal(fl2["wet"], fl["wet"])
    assert np.array_equal(fl2["level"].cpu().numpy().view(np.int64), level.view(np.int64))
    assert np.array_equal(pipe.water_depth(fl2["level"][2]).cpu().numpy().view(np.int32), rasters[2].view(np.int32))


def _bowls(radii, plateau=1000):
    """Conical integer pits of the given radii on a flat plateau, packed in shelves: pit r holds the cells with
    floor(dist) < r (1 cell for r = 1, ~pi r^2 for large r)."""
    cols = 2 * max(radii) + 3 + 2 * sum(2 * r + 3 for r in radii[:4])
    shelves, x, y, h = [], 1, 1, 0
    for r in sorted(radii, reverse=True):
        w = 2 * r + 3
        if x + w > cols - 1:
            x, y, h = 1, y + h, 0
        shelves.append((y + r + 1, x + r + 1, r))
        x += w
        h = max(h, w)
    rows = y + h + 1
    dem = np.full((rows, cols), plateau, np.float32)
    rr, cc = np.mgrid[0:rows, 0:cols]
    for (cy, cx, r) in shelves:
        sl = (slice(cy - r, cy + r + 1), slice(cx - r, cx + r + 1))
        dist = np.floor(np.hypot(rr[sl] - cy, cc[sl] - cx))
        dem[sl] = np.where(dist < r, plateau - (r - dist), dem[sl])
    return dem


def _device_bluespots(dem):
    filled = fill.fill_terrain(dem)
    lab, n = label.connected_components(filled - dem)
    st_sum = label.label_stats(filled - dem, lab, n)["sum"]
    return filled, lab, n, st_sum


def test_many_bowls_all_paths_exact_and_deterministic():
    radii = [1] * 6 + [2, 3, 4, 5, 7, 9, 10, 12, 13, 15, 20, 30, 40, 50, 51, 52, 60, 80, 100, 128, 150, 178]
    dem = _bowls(radii)
    filled, lab, n, st_sum = _device_bluespots(dem)
    count = np.bincount(lab.ravel(), minlength=n + 1)
    assert n == len(radii) and count[1:].min() == 1 and count.max() > 9e4
    assert ((count > 512) & (count <= 8192)).any() and (count > 8192).sum() >= 5
    rng = np.random.default_rng(7)
    cap = st_sum.copy()
    v = np.floor(rng.random((17, n + 1)) * cap)
    v[0] = 0.0
    v[1] = cap
    v[2, ::3] = np.nan
    got = _check(dem, filled, lab, v, 1.0, st_sum, exact=True)
    for ne in (1, 3):
        part = flood.water_levels(dem, filled, lab, v[:ne], 1.0, st_sum)
        assert np.array_equal(part["level"], got["level"][:ne], equal_nan=True)
        assert np.array_equal(part["wet"], got["wet"][:ne])
    again = flood.water_levels(dem, filled, lab, v, 1.0, st_sum)
    assert np.array_equal(again["level"].view(np.int64), got["level"].view(np.int64))
    assert np.array_equal(again["wet"], got["wet"])
    d1 = flood.water_depth(dem, filled, lab, got["level"][5])
    d2 = flood.water_depth(dem, filled, lab, again["level"][5].copy())
    assert np.array_equal(d1.view(np.int32), d2.view(np.int32))


def test_one_large_bluespot():
    s = 2048
    rr, cc = np.mgrid[0:s, 0:s]
    dem = np.floor(((rr - 1023.5) ** 2 + (cc - 1023.5) ** 2) / 2000).astype(np.float32)
    filled, lab, n, st_sum = _device_bluespots(dem)
    count = np.bincount(lab.ravel(), minlength=n + 1)
    assert count[1:].max() >= 1 << 20
    rng = np.random.default_rng(3)
    v = np.floor(rng.random((3, n + 1)) * st_sum)
    _check(dem, filled, lab, v, 1.0, st_sum, exact=True)


def test_exact_cases():
    # a flat-bottomed bowl (z = 5 on a 10 x 10 floor, walls at 10), a single-cell pit, and background
    dem = np.full((16, 20), 10, np.float32)
    dem[3:13, 3:13] = 5
    dem[7, 16] = 8
    filled, lab, n, st_sum = _device_bluespots(dem)
    assert n == 2 and st_sum.tolist() == [0.0, 500.0, 2.0]
    v = np.array([[np.nan, 0.0, 0.0],            # v = 0: level at the floor, nothing wet
                  [np.nan, 100.0, 1.0],          # a level of 6 over the whole floor
                  [np.nan, 250.0, 2.0],          # v = cap of the pit
                  [np.nan, 500.0, np.nan],       # v = cap of the bowl; NaN volume
                  [5.0, 499.0, 1.5]])
    got = _check(dem, filled, lab, v, 1.0, st_sum, exact=True)
    assert got["level"][:, 1].tolist() == [5.0, 6.0, 7.5, 10.0, 9.99]
    assert got["wet"][:, 1].tolist() == [0, 100, 100, 100, 100]
    assert got["level"][:, 2].tolist()[:3] == [8.0, 9.0, 10.0] and np.isnan(got["level"][3, 2])
    assert got["wet"][:, 2].tolist() == [0, 1, 1, 0, 1]
    assert np.isnan(got["level"][:, 0]).all() and (got["wet"][:, 0] == 0).all()
    d = flood.water_depth(dem, filled, lab, got["level"][3])
    assert np.array_equal(d, np.where(lab == 1, filled - dem, 0).astype(np.float32))


def test_volumes_on_breakpoints():
    # a stepped trench z = 1, 2, 2, 3, 5 inside walls at 10: S = 1, 3, 5, 8, 13, j z_(j) - S_j = 0, 1, 1, 4, 12
    dem = np.full((7, 11), 10, np.float32)
    dem[3, 3:8] = [3, 1, 5, 2, 2]
    filled, lab, n, st_sum = _device_bluespots(dem)
    assert n == 1 and st_sum.tolist() == [0.0, 37.0]
    v = np.array([[np.nan, t] for t in (0.0, 1.0, 4.0, 12.0, 36.0)])
    got = _check(dem, filled, lab, v, 1.0, st_sum, exact=True)
    # on a breakpoint the level is the next value up and the cells at that value stay dry (z < h is strict)
    assert got["level"][:, 1].tolist() == [1.0, 2.0, 3.0, 5.0, 49.0 / 5.0]
    assert got["wet"][:, 1].tolist() == [0, 1, 3, 4, 5]


def test_errors():
    dem = np.full((8, 8), 10, np.float32)
    dem[2:6, 2:6] = 4
    filled = np.where(dem < 10, 7, 10).astype(np.float32)
    lab = (dem < 10).astype(np.int32)
    flood.water_levels(dem, filled, lab, [np.nan, 3.0], 1.0, [0.0, 48.0])
    bad = filled.copy()
    bad[2, 2] = 8
    with pytest.raises(ValueError, match="not uniform"):
        flood.water_levels(dem, bad, lab, [np.nan, 3.0], 1.0, [0.0, 48.0])
    with pytest.raises(IndexError):
        flood.water_levels(dem, filled, lab * 2, [np.nan, 3.0], 1.0, [0.0, 48.0])
    with pytest.raises(IndexError):
        flood.water_depth(dem, filled, lab * 2, [np.nan, 7.0])
    with pytest.raises(ValueError, match="negative"):
        flood.water_levels(dem, filled, lab, [np.nan, -1.0], 1.0, [0.0, 48.0])
