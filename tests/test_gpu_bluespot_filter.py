"""The bluespot filter in the device-resident pipeline (csrc/bfilter.cu, ms_pipeline_filtered_host_dev) and across row
bands: keep decisions and rank tables against the CLI's filter lambda, the filtered rasters and tables against the
reference's own sequence run by the oracle (CC -> stats -> filter -> keep_labels -> CC -> watersheds -> tables), the
network and water levels on the filtered bluespots, edge filters, and the bands against the single-GPU run."""
import ctypes

import numpy as np
import pytest
import torch

from malstroem_b200 import _lib, bands, bluespot_filter as bf, network as mnetwork, synth
from malstroem_b200.pipeline import RasterPipeline
from oracle import flood as oflood
from oracle import port
from test_bands_flood_gpu import EDGE_PITS, _pits
from test_bluespot_filter_cpu import FILTERS, reference_decisions, stats_cases
from toolchain import parse_filter

pytestmark = pytest.mark.gpu
CLI = "area > 20.5 and maxdepth > 0.5 or volume > 2.5"
CA188 = 16 * 15 / 0.94
CA = 0.16
MIXED = "0.02 < maxdepth < 2 and not area < 0.5 or volume * 2 > 0.5"
TABLES = ("st_min", "st_max", "st_sum", "st_count", "ws_count", "ppmin_value", "ppmin_row", "ppmin_col",
          "ppmax_value", "ppmax_row", "ppmax_col")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _rank_table(keep):
    keep = np.asarray(keep, bool).copy()
    keep[0] = False
    return (np.cumsum(keep) * keep).astype(np.int32)


def _snapshot(p):
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy().copy() for k, v in p.out.items()}
    out.update({k: p.table(k).cpu().numpy().copy() for k in p.tables})
    out["n"] = p.nlabels
    return out


def _same(a, b, exact_sum=False):
    assert a["n"] == b["n"]
    for k in a:
        if k == "n":
            continue
        if k == "st_sum" and not exact_sum:
            np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=1e-300)
        else:
            assert np.array_equal(a[k], b[k]), k


# ---------------------------------------------------------------------------------------------- the kernels
@pytest.mark.parametrize("text", FILTERS)
def test_kernel_decisions_and_rank_table(text):
    for ca in (1.0, 0.5, CA188):
        count, vmax, vsum = stats_cases(ca, seed=len(text) + 7)
        count[0], vmax[0], vsum[0] = 5, 9.0, 9.0               # label 0 is never kept, whatever its stats
        want = _rank_table(reference_decisions(text, count, vmax, vsum, ca))
        n = count.size - 1
        dev = {k: torch.from_numpy(v).cuda() for k, v in (("c", count), ("m", vmax), ("s", vsum))}
        lut = torch.full((n + 1,), -7, dtype=torch.int32, device="cuda")
        filt = bf.compile_filter(text).struct(ca)
        nk = ctypes.c_int64(-1)
        _lib.check(_lib.lib().ms_bluespot_filter_dev(ctypes.byref(filt), n, dev["m"].data_ptr(), dev["s"].data_ptr(),
                                                     dev["c"].data_ptr(), lut.data_ptr(), ctypes.byref(nk), _stream()))
        assert np.array_equal(lut.cpu().numpy(), want), text
        assert nk.value == int((want > 0).sum())


def test_kernel_rejects_malformed_programs():
    filt = bf.compile_filter("maxdepth > 0.05").struct(1.0)
    t = torch.zeros(4, dtype=torch.float64, device="cuda")
    c = torch.zeros(4, dtype=torch.int64, device="cuda")
    lut = torch.zeros(4, dtype=torch.int32, device="cuda")
    L, nk = _lib.lib(), ctypes.c_int64(0)

    def call(f):
        _lib.check(L.ms_bluespot_filter_dev(ctypes.byref(f), 3, t.data_ptr(), t.data_ptr(), c.data_ptr(),
                                            lut.data_ptr(), ctypes.byref(nk), _stream()), "ms_bluespot_filter_dev")

    for mutate, match in ((lambda f: setattr(f, "n_ops", 2), "leaves"), (lambda f: setattr(f, "n_ops", 0), "operations"),
                          (lambda f: f.op.__setitem__(2, 99), "op code"), (lambda f: f.op.__setitem__(0, bf.GT), "underflow"),
                          (lambda f: setattr(f, "cell_area", 0.0), "cell_area")):
        f = bf.compile_filter("maxdepth > 0.05").struct(1.0)
        mutate(f)
        with pytest.raises(ValueError, match=match):
            call(f)
    call(filt)


@pytest.mark.parametrize("offset", [0, 1, 2, 3])
def test_relabel_in_place(offset):
    rng = np.random.default_rng(offset)
    n, nl = 100003, 900
    lab = rng.integers(0, nl + 1, n + offset).astype(np.int32)
    lut = _rank_table(rng.random(nl + 1) < 0.4)
    t = torch.from_numpy(lab).cuda()
    view = t[offset:]                                       # unaligned starts take the head path
    lt = torch.from_numpy(lut).cuda()
    _lib.check(_lib.lib().ms_relabel_dev(view.data_ptr(), n, nl, lt.data_ptr(), _stream()), "ms_relabel_dev")
    got = t.cpu().numpy()
    assert np.array_equal(got[offset:], lut[lab[offset:]]) and np.array_equal(got[:offset], lab[:offset])
    bad = torch.from_numpy(np.array([0, 1, nl + 1, 2], np.int32)).cuda()
    with pytest.raises(IndexError):
        _lib.check(_lib.lib().ms_relabel_dev(bad.data_ptr(), 4, nl, lt.data_ptr(), _stream()), "ms_relabel_dev")


# ------------------------------------------------------------------------------------- single GPU vs the oracle
def _oracle_chain(dem, text, ca):
    """BluespotTool.process's sequence (bluespots.py:158-206) with the oracle's functions."""
    filled = port.fill_terrain(dem)
    depths = filled - dem
    short, diag = port.minimum_safe_short_and_diag(dem)
    fnf = port.fill_terrain_no_flats(dem, short, diag)
    fd = port.terrain_flowdirection(fnf)
    acc = port.accumulated_flow(fd, fast=True)
    raw, nraw = port.connected_components(depths)
    st = port.label_stats(depths, raw, nraw)
    keep = [False] + list(reference_decisions(text, st["count"][1:], st["max"][1:], st["sum"][1:], ca))
    lab, n = port.connected_components(port.keep_labels(raw, keep))
    ws = lab.copy()
    port.watersheds_from_labels(fd, ws, 0)
    return dict(filled=filled, depths=depths, fnf=fnf, flowdir=fd, accum=acc, raw=raw, nraw=nraw, labels=lab,
                wsheds=ws, n=n, stats=port.label_stats(depths, lab, n), count=port.label_count(ws),
                ppmin=port.label_min_index(fnf, lab, n), ppmax=port.label_max_index(acc, lab, n))


def _check_tables(t, want):
    n = want["n"]
    for k in ("min", "max", "count"):
        assert np.array_equal(t["st_" + k], want["stats"][k]), k
    np.testing.assert_allclose(t["st_sum"], want["stats"]["sum"], rtol=1e-6, atol=1e-300)
    cnt = np.zeros(n + 1, np.int64)
    cnt[:want["count"].size] = want["count"][: n + 1]
    assert np.array_equal(t["ws_count"], cnt)
    for key in ("ppmin", "ppmax"):
        for f in ("value", "row", "col"):
            assert np.array_equal(t[key + "_" + f], want[key][f]), key + f


def test_golden_dtm188_cli_filter(dtm188):
    dem = dtm188["dtm"]
    p = RasterPipeline(*dem.shape)
    p.run(torch.from_numpy(dem).cuda(), bluespot_filter=CLI, cell_area=CA188)
    got = _snapshot(p)
    assert p.nlabels == 486 and p.stats["bluespots_raw"] == 523
    keep = [False] + [bool(parse_filter(CLI)({"area": np.int64(c) * CA188, "max": m, "volume": s * CA188}))
                      for c, m, s in zip(dtm188["raw_stats_count"][1:], dtm188["raw_stats_max"][1:],
                                         dtm188["raw_stats_sum"][1:])]
    lab = _rank_table(keep)[dtm188["raw_labels"]]
    assert np.array_equal(got["labels"], lab)
    ws = lab.copy()
    port.watersheds_from_labels(dtm188["flowdir_noflats"], ws, 0)
    assert np.array_equal(got["wsheds"], ws)
    depths = dtm188["depths"]
    want = dict(n=486, stats=port.label_stats(depths, lab, 486), count=port.label_count(ws),
                ppmin=port.label_min_index(dtm188["filled_no_flats"], lab, 486),
                ppmax=port.label_max_index(dtm188["accum"], lab, 486))
    _check_tables(got, want)


def _network_and_flood_check(p, want, ca, mm):
    net = p.network(cell_area=ca, events_mm=mm)
    fl = p.flood(net, ca)
    torch.cuda.synchronize()
    lab, n = want["labels"], want["n"]
    mi = want["ppmin"]
    nodes = port.pourpoint_network(want["flowdir"], lab, list(zip(mi["row"].tolist(), mi["col"].tolist())), 0)
    parent = np.array([-1 if d["downstream_id"] is None else d["downstream_id"] for d in nodes])
    assert np.array_equal(net["parent"].cpu().numpy(), parent)
    area = np.zeros(n + 1)
    area[: want["count"].size] = want["count"][: n + 1]
    st_sum = p.table("st_sum").cpu().numpy()
    ref = port.rain_events(parent, area * ca, st_sum * ca, mm, mnetwork.SUM_MODE)
    v = net["v"].cpu().numpy()
    for k in ("rainv", "spillv", "v"):
        assert np.array_equal(net[k].cpu().numpy(), ref[k]), k
    wl = oflood.water_levels(p.dem.cpu().numpy(), want["filled"], lab, v, ca, st_sum)
    level, wet = fl["level"].cpu().numpy(), fl["wet"].cpu().numpy()
    assert np.array_equal(np.isnan(level), np.isnan(wl["level"]))
    m = ~np.isnan(level)
    assert (np.abs(level[m] - wl["level"][m]) <= 1e-12 * np.maximum(1.0, np.abs(wl["level"][m]))).all()
    same = level == wl["level"]
    assert np.array_equal(wet[same], wl["wet"][same]) and same.mean() > 0.9
    d = p.water_depth(fl["level"][0]).cpu().numpy()
    assert np.array_equal(d, oflood.water_depth(p.dem.cpu().numpy(), want["filled"], lab, level[0]))


@pytest.mark.parametrize("size,text", [(1024, "maxdepth > 0.05"), (1024, MIXED), (2048, "maxdepth > 0.05"),
                                       (2048, MIXED)])
def test_fractal_against_the_reference_sequence(size, text):
    dem = synth.fractal_dem(size, size, seed=2)
    want = _oracle_chain(dem, text, CA)
    p = RasterPipeline(size, size)
    p.run(torch.from_numpy(dem).cuda(), bluespot_filter=text, cell_area=CA)
    got = _snapshot(p)
    assert p.stats["bluespots_raw"] == want["nraw"] and 0 < p.nlabels == want["n"] < want["nraw"]
    for name in ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds"):
        assert np.array_equal(got[name], want[name]), name
    _check_tables(got, want)
    _network_and_flood_check(p, want, CA, [10.0, 30.0, 100.0])


# --------------------------------------------------------------------------------------------- edge filters
def test_edge_filters():
    dem = torch.from_numpy(synth.fractal_dem(512, 640, seed=2)).cuda()
    p = RasterPipeline(512, 640)
    base = _snapshot(p.run(dem))
    assert "bluespots_raw" not in p.stats
    _same(_snapshot(p.run(dem, bluespot_filter="")), base)
    assert "bluespots_raw" not in p.stats
    _same(_snapshot(p.run(dem, bluespot_filter=None, cell_area=3.0)), base)
    for keep_all in ("1", "maxdepth > 0", "area >= 1"):
        _same(_snapshot(p.run(dem, bluespot_filter=keep_all, cell_area=2.0)), base)
        assert p.stats["bluespots_raw"] == base["n"]
    got = _snapshot(p.run(dem, bluespot_filter="maxdepth < 0", cell_area=2.0))
    assert p.nlabels == 0 and p.stats["bluespots_raw"] == base["n"]
    assert not got["labels"].any() and not got["wsheds"].any()
    for k in TABLES:
        assert got[k].shape == (1,), k
    assert got["st_count"][0] == 512 * 640 and got["ws_count"][0] == 512 * 640
    net = p.network(cell_area=CA, events_mm=[10.0])
    fl = p.flood(net, CA)
    torch.cuda.synchronize()
    assert net["parent"].shape == (1,) and fl["level"].shape == (1, 1) and np.isnan(fl["level"].cpu().numpy()).all()
    assert not p.water_depth(fl["level"][0]).any()
    with pytest.raises(ValueError, match="unknown name"):
        p.run(dem, bluespot_filter="depth > 1")
    with pytest.raises(ValueError, match="cell_area"):
        p.run(dem, bluespot_filter="area > 1", cell_area=0.0)


def test_run_host_ships_the_filtered_rasters():
    dem = synth.fractal_dem(640, 512, seed=2)
    p = RasterPipeline(640, 512)
    want = _snapshot(p.run(torch.from_numpy(dem).cuda(), bluespot_filter=MIXED, cell_area=CA))
    q = RasterPipeline(640, 512)
    h = q.run_host(dem, bluespot_filter=MIXED, cell_area=CA)
    assert q.nlabels == want["n"] and q.stats["bluespots_raw"] > q.nlabels
    for name in RasterPipeline.HOST_RASTERS:
        assert np.array_equal(h[name].numpy(), want[name]), name
    for k in TABLES:
        if k != "st_sum":
            assert np.array_equal(h[k][: q.nlabels + 1].numpy(), want[k]), k


# -------------------------------------------------------------------------------------------------- row bands
def _band_case(kind):
    if kind == "fractal":
        return synth.fractal_dem(640, 384, seed=2), MIXED, CA
    # 640 rows: band edges on rows 128 / 256 / 384 / 512 at five bands; the r = 100 lake crosses the edge of two bands
    return _pits(640, 512, EDGE_PITS), "area > 300 and not 55 < maxdepth < 65 or area < 2", 1.0


@pytest.mark.parametrize("kind,nb", [("fractal", 2), ("fractal", 3), ("fractal", 5), ("pits", 2), ("pits", 3),
                                     ("pits", 5)])
def test_bands_equal_the_single_gpu_filtered_run(kind, nb):
    dem, text, ca = _band_case(kind)
    rows, cols = dem.shape
    single = RasterPipeline(rows, cols)
    want = _snapshot(single.run(torch.from_numpy(dem).cuda(), bluespot_filter=text, cell_area=ca))
    assert 0 < single.nlabels < single.stats["bluespots_raw"]

    def after(p):
        net = p.network(cell_area=ca, events_mm=[10.0, 30.0, 100.0])
        res = p.flood({"v": net["v"]}, ca)
        return net["v"].clone(), res["level"].cpu().numpy(), res["wet"].cpu().numpy()

    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb, after=after, bluespot_filter=text, cell_area=ca)
    try:
        for name in ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds"):
            got = torch.cat([p.out[name] for p in pipes]).cpu().numpy()
            assert np.array_equal(got, want[name]), name
        lab = want["labels"]
        if kind == "pits":
            assert any(np.intersect1d(lab[p.r0][lab[p.r0] > 0], lab[p.r0 - 1]).size for p in pipes[1:]), \
                "no kept bluespot crosses a band edge"
        for p in pipes:
            assert p.nlabels == want["n"] and p.stats["bluespots_raw"] == single.stats["bluespots_raw"]
            assert sum(c for _, c in p.label_ranges) == p.nlabels
            for k in TABLES:
                t = p.tables[k][: p.nlabels + 1].cpu().numpy()
                if k == "st_sum":
                    np.testing.assert_allclose(t, want[k], rtol=1e-12, atol=1e-300)
                else:
                    assert np.array_equal(t, want[k]), k
        # every label lies in the range of the band holding its first cell
        first = {}
        for g, p in enumerate(pipes):
            for l in np.unique(lab[p.r0:p.r1]):
                first.setdefault(int(l), g)
        for l, g in first.items():
            if l:
                o, c = pipes[0].label_ranges[g]
                assert o < l <= o + c, (l, g, pipes[0].label_ranges)
        # flood levels bitwise the single-GPU flood's on the filtered labels, given the same st_sum and v
        m = want["n"] + 1
        single.tables["st_sum"][:m].copy_(pipes[0].tables["st_sum"][:m])
        v = pipes[0].after_result[0]
        ref = single.flood({"v": v.to(single.device)}, ca)
        rl, rw = ref["level"].cpu().numpy(), ref["wet"].cpu().numpy()
        for p in pipes:
            _, level, wet = p.after_result
            assert np.array_equal(level.view(np.int64), rl.view(np.int64)) and np.array_equal(wet, rw)
    finally:
        for p in pipes:
            p.close()


def test_bands_keep_nothing():
    dem = synth.fractal_dem(384, 256, seed=2)
    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), 3, bluespot_filter="maxdepth < 0", cell_area=CA,
                               after=lambda p: p.flood({"v": p.network(CA, [10.0])["v"]}, CA)["level"].cpu().numpy())
    try:
        for p in pipes:
            assert p.nlabels == 0 and p.label_ranges == [(0, 0)] * 3 and not p.out["labels"].any()
            assert np.isnan(p.after_result).all()
    finally:
        for p in pipes:
            p.close()

