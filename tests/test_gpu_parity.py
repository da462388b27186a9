"""Parity of the CUDA path (through the C ABI, via the numpy mirrors of malstroem.algorithms) against the
reference's golden rasters, the stored outputs of the reference itself, and the CPU oracle on seeded
inputs.  Bit-exact for every raster, label and index; label_stats 'sum' within 1e-6 relative (north_star).
Mirrors /root/reference/tests/test_raster_{fill,flowdir,label}.py."""
import numpy as np
import pytest

from malstroem_b200 import synth
from malstroem_b200.algorithms import fill, flow, label
from oracle import port

pytestmark = pytest.mark.gpu
SUM_RTOL = 1e-6


def eq(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def check_stats(st, ref):
    assert len(st) == len(ref["min"])
    for k in ("min", "max", "count"):
        assert np.array_equal(st[k], ref[k]), k
    np.testing.assert_allclose(st["sum"], ref["sum"], rtol=SUM_RTOL, atol=1e-300)


def check_index(a, ref):
    assert len(a) == len(ref["value"])
    for k in ("value", "row", "col"):
        assert np.array_equal(a[k], ref[k]), k


# ---------------------------------------------------------------- golden rasters of the reference
def test_fill_golden(dtm188):
    assert eq(fill.fill_terrain(dtm188["dtm"]), dtm188["filled"])
    f, d = fill.fill_terrain_and_depths(dtm188["dtm"])
    assert eq(f, dtm188["filled"]) and eq(d, dtm188["depths"])


def test_fill_no_flats_golden(dtm188):
    short, diag = fill.minimum_safe_short_and_diag(dtm188["dtm"])
    assert short == dtm188["short"] and diag == dtm188["diag"]
    assert eq(fill.fill_terrain_no_flats(dtm188["dtm"], short, diag), dtm188["filled_no_flats"])


def test_negative_dem_values():
    dtm = np.full((10, 10), -9999, np.float32)
    dtm[4:6, 4:6] = 0
    short, diag = fill.minimum_safe_short_and_diag(dtm)
    filled = fill.fill_terrain_no_flats(dtm, short, diag)
    assert filled[1, 1] != -9999
    assert eq(filled, port.fill_terrain_no_flats(dtm, short, diag))


def test_flowdir_golden(dtm188):
    assert eq(flow.terrain_flowdirection(dtm188["filled_no_flats"]), dtm188["flowdir_noflats"])


def test_accum_golden(dtm188):
    acc = flow.accumulated_flow(dtm188["flowdir_noflats"])
    assert acc.min() >= 1 and acc.max() == 11158 and acc.sum() == 3578615
    assert eq(acc, dtm188["accum"])


@pytest.mark.parametrize("dt", [np.int32, np.int64, np.uint32, np.int16])
def test_watersheds_golden(dtm188, dt):
    ws = dtm188["labelled"].astype(dt)
    assert flow.watersheds_from_labels(dtm188["flowdir_noflats"], ws, unassigned=0) is None
    assert ws.dtype == dt and np.array_equal(ws, dtm188["wsheds"]) and ws.sum() == 2337891


def test_connected_components_golden(dtm188):
    lab, n = label.connected_components(dtm188["filled_no_flats"] - dtm188["filled"])
    assert lab.dtype == np.int32 and n == 525 and (lab == 0).sum() == 40029 and lab.sum() == 1561377
    assert eq(lab, dtm188["cc_diff_labels"])
    lab, n = label.connected_components(dtm188["depths"])
    assert n == dtm188["raw_nlabels"] and eq(lab, dtm188["raw_labels"])
    lab2, n2 = label.connected_components(dtm188["depths"] != 0)          # bool input (bluespots.py:170)
    assert n2 == n and eq(lab2, lab)


def test_label_tables_golden(dtm188):
    st = label.label_stats(dtm188["depths"], dtm188["labelled"])
    check_stats(st, {k: dtm188["lab_stats_" + k] for k in ("min", "max", "sum", "count")})
    mi = label.label_min_index(dtm188["filled_no_flats"], dtm188["labelled"])
    assert np.array_equal(mi["row"], dtm188["pp_cell_row"]) and np.array_equal(mi["col"], dtm188["pp_cell_col"])
    check_index(mi, {k: dtm188["lab_minidx_" + k] for k in ("value", "row", "col")})
    ma = label.label_max_index(dtm188["accum"], dtm188["labelled"])
    check_index(ma, {k: dtm188["lab_maxidx_" + k] for k in ("value", "row", "col")})
    assert np.array_equal(label.label_count(dtm188["wsheds"]), dtm188["lab_wshed_count"])


# ------------------------------------------------- stored outputs of the reference on small rasters
def _check_case(o):
    dem = o["dem"]
    f, dep = fill.fill_terrain_and_depths(dem)
    assert eq(f, o["filled_py"]) and eq(dep, o["depths"])
    short, diag = fill.minimum_safe_short_and_diag(dem)
    assert short == o["short"] and diag == o["diag"]
    fnf = fill.fill_terrain_no_flats(dem, short, diag)
    assert eq(fnf, o["fnf_py"])
    assert eq(flow.terrain_flowdirection(fnf, True), o["flowdir"])
    assert eq(flow.terrain_flowdirection(fnf, False), o["flowdir_noedge"])
    assert eq(flow.accumulated_flow(o["flowdir"]), o["accum"])
    lab, n = label.connected_components(dep)
    assert n == o["nlabels"] and eq(lab, o["labels"])
    ws = lab.copy()
    flow.watersheds_from_labels(o["flowdir"], ws, 0)
    assert eq(ws, o["wsheds"])
    assert np.array_equal(label.label_count(ws), o["wshed_count"])
    check_stats(label.label_stats(dep, lab), {k: o["stats_" + k] for k in ("min", "max", "sum", "count")})
    check_index(label.label_min_index(fnf, lab, n), {k: o["minidx_" + k] for k in ("value", "row", "col")})
    if "maxidx_value" in o:
        check_index(label.label_max_index(o["accum"], lab, n), {k: o["maxidx_" + k] for k in ("value", "row", "col")})


def test_small_cases(small_cases):
    cases, flows = small_cases
    for i, o in enumerate(cases):
        if min(o["dem"].shape) < 4:
            continue
        try:
            _check_case(o)
        except AssertionError as e:
            raise AssertionError("small case %d %s: %s" % (i, o["dem"].shape, e))
    for f in flows:                                   # NODIR cells, inward / undirected border cells
        ws = f["labels"].copy()
        flow.watersheds_from_labels(f["flowdir"], ws, 0)
        assert eq(ws, f["wsheds"])
        assert eq(flow.accumulated_flow(f["flowdir"]), port.accumulated_flow(f["flowdir"]))


def test_fractal256(fractal256):
    o = dict(fractal256)
    o["filled_py"], o["fnf_py"] = o["filled_cy"], o["fnf_cy"]
    _check_case(o)


# --------------------------------------------------------------- seeded inputs against the oracle
def _dems():
    rng = np.random.default_rng(7)
    yield "fractal_700x900", synth.fractal_dem(700, 900, seed=2)
    yield "fractal_1024", synth.fractal_dem(1024, 1024, seed=3)
    yield "levels_300x257", rng.integers(0, 12, (300, 257)).astype(np.float32)
    yield "noise_200x333", (rng.random((200, 333)) * 50).astype(np.float32)
    yield "pathological_512", synth.pathological_dem(512, 512, seed=1)
    yield "tiny_values", (synth.fractal_dem(150, 150, seed=4) * np.float32(1e-30)).astype(np.float32)
    yield "strip_4x500", synth.fractal_dem(4, 500, seed=5)
    yield "strip_500x4", synth.fractal_dem(500, 4, seed=5)
    yield "odd_65x129", synth.fractal_dem(65, 129, seed=6)


@pytest.mark.parametrize("name,dem", list(_dems()), ids=[n for n, _ in _dems()])
def test_whole_path_vs_oracle(name, dem):
    f, dep = fill.fill_terrain_and_depths(dem)
    assert eq(f, port.fill_terrain(dem))
    assert eq(dep, f - dem)
    short, diag = fill.minimum_safe_short_and_diag(dem)
    assert (short, diag) == port.minimum_safe_short_and_diag(dem)
    fnf = fill.fill_terrain_no_flats(dem, short, diag)
    assert eq(fnf, port.fill_terrain_no_flats(dem, short, diag))
    fd = flow.terrain_flowdirection(fnf)
    assert eq(fd, port.terrain_flowdirection(fnf))
    assert eq(flow.accumulated_flow(fd), port.accumulated_flow(fd, fast=True))
    lab, n = label.connected_components(dep)
    olab, on = port.connected_components(dep)
    assert n == on and eq(lab, olab)
    ws = lab.copy()
    flow.watersheds_from_labels(fd, ws, 0)
    ows = lab.copy()
    port.watersheds_from_labels(fd, ows, 0)
    assert eq(ws, ows)
    assert np.array_equal(label.label_count(ws), port.label_count(ws))
    check_stats(label.label_stats(dep, lab), port.label_stats(dep, lab))
    check_index(label.label_min_index(fnf, lab, n), port.label_min_index(fnf, lab, n))
    acc = port.accumulated_flow(fd, fast=True)
    check_index(label.label_max_index(acc, lab, n), port.label_max_index(acc, lab, n))


def test_no_flats_other_epsilons():
    dem = synth.fractal_dem(120, 160, seed=8)
    for short, diag in ((0, 0), (0.25, 0.4), (1e-3, 1.5e-3), (3.0, 4.5)):
        assert eq(fill.fill_terrain_no_flats(dem, short, diag), port.fill_terrain_no_flats(dem, short, diag)), (short, diag)


def test_label_functions_edge_cases():
    rng = np.random.default_rng(11)
    lab = rng.integers(0, 40, (77, 131)).astype(np.int32)
    data = rng.standard_normal((77, 131))
    data[rng.random((77, 131)) < 0.2] = 0.5          # ties: first cell in raster order must win
    data[3, 4] = -0.0
    # a label whose only values are +inf has no arg-min, one whose only values are -inf no arg-max (strict comparison
    # against the +inf / -inf start value); elsewhere the infinities are extremes
    data[lab == 5] = np.inf
    data[lab == 6] = -np.inf
    data[7, 8], data[9, 10] = np.inf, -np.inf
    for nl in (None, 39, 60):                         # tables longer than the labels present
        check_index(label.label_min_index(data, lab, nl), port.label_min_index(data, lab, nl))
        check_index(label.label_max_index(data, lab, nl), port.label_max_index(data, lab, nl))
        check_stats(label.label_stats(data, lab, nl), port.label_stats(data, lab, nl))
        check_stats(label.label_stats(data.astype(np.float32), lab, nl), port.label_stats(data.astype(np.float32), lab, nl))
    with pytest.raises(IndexError):
        label.label_stats(data, lab, 10)              # labels beyond the table (pure-Python reference: IndexError)
    keep = [bool(v) for v in rng.integers(0, 2, 40)]
    keep[0] = True
    keep2 = list(keep)
    assert eq(label.keep_labels(lab, keep), port.keep_labels(lab, keep2))
    assert keep[0] is False                           # label.py:94 mutates the caller's list
    assert np.array_equal(label.label_count(lab), np.bincount(lab.ravel()))
    with pytest.raises(ValueError):
        label.label_count(lab - 1)
    # foreground rule of scipy.ndimage.label: NaN and denormals count, -0.0 does not
    d = np.zeros((9, 9), np.float32)
    d[1, 1] = np.nan; d[1, 2] = 1e-45; d[5, 5] = -0.0; d[7, 7] = -3
    l, n = label.connected_components(d)
    ol, on = port.connected_components(d)
    assert n == on == 2 and eq(l, ol)


def test_error_behaviour():
    with pytest.raises(ValueError):
        fill.fill_terrain(np.zeros((8, 8), np.float64))           # Buffer dtype mismatch
    with pytest.raises(ValueError):
        fill.fill_terrain(np.zeros((3, 8), np.float32))           # processing area is zero
    with pytest.raises(ValueError):
        flow.terrain_flowdirection(np.zeros((8, 8), np.float32))
    with pytest.raises(ValueError):
        flow.accumulated_flow(np.zeros((8, 8), np.int32))


def test_synth_device_matches_numpy():
    import torch
    from malstroem_b200.pipeline import synth_fractal
    d = synth_fractal(300, 517, seed=3, row0=1000, col0=77).cpu().numpy()
    assert eq(d, synth.fractal_dem(300, 517, seed=3, row0=1000, col0=77))


def test_pipeline_matches_functions():
    import torch
    from malstroem_b200.pipeline import RasterPipeline
    dem = synth.fractal_dem(600, 800, seed=9)
    p = RasterPipeline(600, 800)
    p.host_fnf = True                 # also bring the no-flats surface back (an intermediate otherwise)
    h = p.run_host(dem)
    f, dep = fill.fill_terrain_and_depths(dem)
    assert eq(h["filled"].numpy(), f) and eq(h["depths"].numpy(), dep)
    short, diag = fill.minimum_safe_short_and_diag(dem)
    assert (p.short, p.diag) == (short, diag)
    fnf = port.fill_terrain_no_flats(dem, short, diag)
    assert eq(h["fnf"].numpy(), fnf)
    fd = port.terrain_flowdirection(fnf)
    assert eq(h["flowdir"].numpy(), fd)
    acc = port.accumulated_flow(fd, fast=True)
    assert eq(h["accum"].numpy(), acc)
    lab, n = port.connected_components(dep)
    assert p.nlabels == n and eq(h["labels"].numpy(), lab)
    ws = lab.copy(); port.watersheds_from_labels(fd, ws, 0)
    assert eq(h["wsheds"].numpy(), ws)
    m = n + 1
    st = port.label_stats(dep, lab)
    assert np.array_equal(h["st_min"].numpy()[:m], st["min"]) and np.array_equal(h["st_count"].numpy()[:m], st["count"])
    assert np.array_equal(h["st_max"].numpy()[:m], st["max"])
    np.testing.assert_allclose(h["st_sum"].numpy()[:m], st["sum"], rtol=SUM_RTOL)
    assert np.array_equal(h["ws_count"].numpy()[:m], port.label_count(ws))
    mi = port.label_min_index(fnf, lab, n)
    assert np.array_equal(h["ppmin_row"].numpy()[:m], mi["row"]) and np.array_equal(h["ppmin_col"].numpy()[:m], mi["col"])
    assert np.array_equal(h["ppmin_value"].numpy()[:m], mi["value"])
    ma = port.label_max_index(acc, lab, n)
    assert np.array_equal(h["ppmax_row"].numpy()[:m], ma["row"]) and np.array_equal(h["ppmax_col"].numpy()[:m], ma["col"])
    assert np.array_equal(h["ppmax_value"].numpy()[:m], ma["value"])


# ---------------------------------------------------------------- sizes beyond the CPU oracle: certificates
def test_certificates_4096():
    """SURVEY.md A.5: at sizes where the CPU oracle is impractical the results are certified by size-independent
    properties (tools/big_check.py): fixed point from above (fill), the library's verification stencil (no-flats),
    acc == 1 + sum of inflows with terminal sums == N, ws == label or ws(downstream).  The same tool certifies
    32768 x 32768 (BASELINE config 3) in profiles/."""
    import importlib.util
    import os
    import torch
    from malstroem_b200.pipeline import RasterPipeline, synth_fractal
    spec = importlib.util.spec_from_file_location(
        "big_check", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "big_check.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    p = RasterPipeline(4096, 3072)
    synth_fractal(4096, 3072, seed=7, out=p.dem)
    p.run()
    torch.cuda.synchronize()
    bad_fill, bad_acc, bad_ws, root_sum = mod.certify(p, CH=1024)
    assert (bad_fill, bad_acc, bad_ws) == (0, 0, 0) and root_sum == 4096 * 3072
    assert p.stats["noflat_reverify"] == 0
