"""Water levels and depth rasters across row bands (BandPipeline.flood / water_depth), bands as threads on one GPU:
every rank's `level` (compared as int64 bits) and `wet` must equal malstroem_b200.flood.water_levels on the WHOLE
raster given the band run's own st_sum and v, and the bands' depth rasters put together must equal
flood.water_depth bitwise.  Fixtures put lakes of every solve path (one warp, one CTA, the global sort) across band
edges, one lake across three bands, and a band that owns no label."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from malstroem_b200 import bands, flood, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CA = 0.16


def _pits(rows, cols, pits, plateau=1000):
    """Conical integer pits (cy, cx, r) on a flat plateau: pit r holds the cells with floor(dist) < r."""
    dem = np.full((rows, cols), plateau, np.float32)
    rr, cc = np.mgrid[0:rows, 0:cols]
    for cy, cx, r in pits:
        dist = np.floor(np.hypot(rr - cy, cc - cx))
        dem = np.where(dist < r, np.float32(plateau - (r - dist)), dem)
    return dem


# centred on rows 128 / 256 / 384 (band edges at 4 and at 8 bands): crossing lakes of <= 512, 513-8192 and > 8192
# cells; the r = 100 lake spans four of the 64-row bands; the rest are inside one band
EDGE_PITS = [(128, 10, 2), (128, 20, 5), (128, 45, 12), (256, 80, 20), (384, 130, 40), (128, 470, 30),
             (256, 300, 100), (448, 445, 60), (30, 200, 10), (60, 470, 3), (20, 100, 1), (500, 20, 1), (480, 100, 7)]


def _whole(pipes):
    cat = lambda name: torch.cat([p.out[name] for p in pipes]).cpu().numpy()      # noqa: E731
    dem = torch.cat([p.dem for p in pipes]).cpu().numpy()
    return dem, cat("filled"), cat("labels")


def _spans(lab, pipes):
    """label -> number of bands holding cells of it"""
    n = pipes[0].nlabels
    seen = np.zeros((len(pipes), n + 1), bool)
    for g, p in enumerate(pipes):
        seen[g, np.unique(lab[p.r0:p.r1])] = True
    return seen[:, 1:].sum(0)


def _check(pipes, results, events):
    """results[g] = (level, wet, depth rasters of every event) of rank g; events: the v the flood ran on."""
    dem, filled, lab = _whole(pipes)
    st_sum = pipes[0].tables["st_sum"].cpu().numpy()
    want = flood.water_levels(dem, filled, lab, events, CA, st_sum=st_sum)
    for level, wet, _ in results:
        assert np.array_equal(level.view(np.int64), want["level"].view(np.int64))
        assert np.array_equal(wet, want["wet"])
    for e in range(events.shape[0]):
        got = np.concatenate([r[2][e] for r in results])
        assert np.array_equal(got.view(np.int32), flood.water_depth(dem, filled, lab, want["level"][e]).view(np.int32))
    return want


def _run(dem, nb, volumes):
    """The banded run, then flood + water_depth on every rank; volumes(p) -> the v tensor the flood gets."""
    def after(p):
        v = volumes(p)
        res = p.flood({"v": v}, CA)
        depth = [p.water_depth(res["level"][e]).cpu().numpy() for e in range(v.shape[0])]
        return v.cpu().numpy(), res["level"].cpu().numpy(), res["wet"].cpu().numpy(), depth

    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb, after=after)
    vs = [p.after_result[0] for p in pipes]
    assert all(np.array_equal(v.view(np.int64), vs[0].view(np.int64)) for v in vs)
    return pipes, vs[0], [p.after_result[1:] for p in pipes]


def _volumes(seed):
    def make(p):
        cap = p.tables["st_sum"] * CA
        g = torch.Generator(device="cpu").manual_seed(seed)
        frac = torch.rand((5, cap.numel()), generator=g, dtype=torch.float64).to(p.device)
        v = torch.floor(frac * cap * 64) / 64
        v[1] = 0.0
        v[2] = cap
        v[3, 1::3] = float("nan")
        v[4] = cap * 0.999
        return v.contiguous()
    return make


@pytest.mark.parametrize("nb", [4, 8])
def test_every_solve_path_across_band_edges(nb):
    dem = _pits(512, 512, EDGE_PITS)
    pipes, v, results = _run(dem, nb, _volumes(nb))
    try:
        _, _, lab = _whole(pipes)
        cnt = np.bincount(lab.ravel())[1:]
        spans = _spans(lab, pipes)
        cross = spans > 1
        assert (cross & (cnt <= 512)).any() and (cross & (cnt > 512) & (cnt <= 8192)).any() and (cross & (cnt > 8192)).any()
        if nb == 8:
            assert spans.max() >= 3
        want = _check(pipes, results, v)
        assert np.isnan(want["level"][3, 1::3]).all() and (want["wet"][1] == 0).all()
    finally:
        for p in pipes:
            p.close()


def test_band_that_owns_no_label():
    rows, cols = 384, 192
    y, x = np.mgrid[0:rows, 0:cols].astype(np.float64)
    bowl = ((y - rows / 2) / rows) ** 2 + ((x - cols / 2) / cols) ** 2
    dem = (50.0 + 40.0 * bowl).astype(np.float32)
    dem[:, :3] = dem[:, -3:] = 80.0
    dem[:3, :] = dem[-3:, :] = 80.0
    dem[rows // 3, :40] = 55.0
    dem[200:260, 100:150] = np.float32(52.0)
    dem = (np.round(dem * 1000) / 1000).astype(np.float32)
    pipes, v, results = _run(dem, 6, _volumes(5))
    try:
        assert any(c == 0 for _, c in pipes[0].label_ranges)
        _check(pipes, results, v)
    finally:
        for p in pipes:
            p.close()


@pytest.mark.parametrize("kind,nb", [("fractal", 4), ("pathological", 2), ("pathological", 8)])
def test_driven_by_the_network(kind, nb):
    dem = synth.fractal_dem(512, 384, seed=3) if kind == "fractal" else synth.pathological_dem(512, 384)
    pipes, v, results = _run(dem, nb, lambda p: p.network(CA, [10.0, 30.0, 100.0])["v"])
    try:
        assert pipes[0].nlabels > 0
        _check(pipes, results, v)
    finally:
        for p in pipes:
            p.close()


def _run_error(dem, nb, prepare):
    def after(p):
        try:
            v = prepare(p)
            p.flood({"v": v}, CA)
        except Exception as e:      # noqa: BLE001 - every rank's outcome is asserted by the test
            return e
        return None

    pipes = bands.run_threaded(torch.from_numpy(dem).cuda(), nb, after=after)
    for p in pipes:
        p.close()
    return [p.after_result for p in pipes]


def test_negative_volume_reaches_every_rank():
    def prepare(p):
        v = p.network(CA, [30.0])["v"].clone()
        lo, c = p.label_ranges[-1]
        assert c > 0
        v[0, lo + 1] = -1.0
        return v

    errs = _run_error(synth.fractal_dem(512, 384, seed=3), 4, prepare)
    assert all(isinstance(e, ValueError) and "negative" in str(e) for e in errs), errs


def test_non_uniform_fill_in_a_non_owner_band_reaches_every_rank():
    def prepare(p):
        if p.comm.rank == p.comm.size - 1:
            lo = p.label_ranges[p.comm.rank][0]
            lab = p.out["labels"]
            cells = torch.nonzero(((lab > 0) & (lab <= lo)).view(-1))
            assert cells.numel() > 0              # a lake that crosses into this band from a lower one
            p.out["filled"].view(-1)[cells[0, 0]] += 1.0
        return p.tables["st_sum"].view(1, -1) * CA * 0.5

    errs = _run_error(_pits(512, 512, EDGE_PITS), 4, prepare)
    assert all(isinstance(e, ValueError) and "uniform" in str(e) for e in errs), errs


def test_two_gpus_equal_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "band_flood_bench.py"), "--size", "2048",
           "--reps", "1", "--no-c5"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "bitwise equal to the single-GPU flood: True" in r.stdout, r.stdout[-3000:]
    assert "RESULT OK" in r.stdout, r.stdout[-3000:]
