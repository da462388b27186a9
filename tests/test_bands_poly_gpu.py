"""vector.polygonize_band (label polygonisation on row bands, csrc/polygon.cu ms_band_poly_*) against
polygonize_labels_device on the whole raster: bands as ThreadComm threads on one GPU at 2, 4 and 8 bands, both
connectivities, with and without nodata.  Concatenated over the ranks, the polygons (value, region, rings, start vertex
and vertices) must be the single-GPU ones in the same order, each rank's rings in leader order, feature ids global."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

from malstroem_b200 import bands, vector
from poly_cases import cases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 500                      # 8 bands of 64 rows, 4 of 128, 2 of 256 (the last one short)


def run_bands(n, fn):
    grp = bands.ThreadGroup(n)
    out, errs = [None] * n, [None] * n

    def work(rank):
        try:
            torch.cuda.set_device(0)
            out[rank] = fn(bands.ThreadComm(grp, rank))
        except BaseException as e:      # noqa: BLE001
            errs[rank] = e
            grp.barrier.abort()

    ts = [threading.Thread(target=work, args=(r,)) for r in range(n)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(300)
        assert not t.is_alive(), "a rank hangs"
    return out, errs


def as_polys(rings):
    out = []
    for value, ks in rings.polygons():
        out.append((value, int(rings.region[ks[0]]),
                    [list(zip(*[x.tolist() for x in rings.ring_lattice(k)])) for k in ks]))
    return out


def banded(lab, n, connect8, nodata):
    rows = lab.shape[0]
    bounds = bands.band_rows(rows, n)

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        return vector.polygonize_band(comm, lab[r0:r1].clone(), r0, rows, connect8=connect8, nodata=nodata)

    out, errs = run_bands(n, fn)
    assert errs == [None] * n, errs
    return out


def check(a, n, connect8, nodata):
    lab = torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda() if isinstance(a, np.ndarray) else a
    one = vector.polygonize_labels_device(lab, connect8=connect8, nodata=nodata)
    parts = banded(lab, n, connect8, nodata)
    got = [p for r in parts for p in as_polys(r)]
    assert got == as_polys(one)
    for r in parts:
        # leader = lowest global edge number: its cell first, then its side (top of the cell before its bottom)
        key = r.cell * 4 + np.where(r.hole != 0, 2, 0)
        assert np.all(np.diff(key) > 0)
    assert sum(r.nedges for r in parts) == one.nedges
    ids = [f["id"] for r in parts for f in r.features()]
    assert ids == list(range(len(ids)))
    return parts


def scaled():
    out = {}
    for name, a in cases().items():
        k = -(-ROWS // a.shape[0])
        b = np.kron(a, np.ones((k, 1 + k // 4), dtype=np.int32))
        if name.startswith("random") or name in ("checkerboard", "negative_values"):
            b = np.tile(a, (k, max(1, 200 // a.shape[1])))        # keep the fine structure
        out["kron_" + name] = b[:ROWS]
    return out


def special():
    out = {}
    out["checkerboard"] = (np.add.outer(np.arange(ROWS), np.arange(131)) % 2).astype(np.int32)
    d = np.zeros((ROWS, 120), dtype=np.int32)
    for e in range(64, ROWS, 64):                      # diagonal pairs that join only across a band edge
        c = 3 + e // 16
        d[e - 1, c] = d[e, c + 1] = 7
        d[e - 1, c + 40] = d[e, c + 39] = 7
        d[e - 1, c + 80] = 5
        d[e, c + 81] = 5
    d[10, 3:100] = 7                                   # ... and one region they hang on
    out["diagonals_across_edges"] = d
    r, c = np.meshgrid(np.arange(ROWS), np.arange(300), indexing="ij")
    out["nested_all_bands"] = ((np.minimum(np.minimum(r, c), np.minimum(ROWS - 1 - r, 299 - c)) // 3) % 4).astype(
        np.int32)
    t = np.zeros((ROWS, 64), dtype=np.int32)
    t[1:ROWS - 1, 5] = 3                               # a tall thin region through every band
    t[2:ROWS - 2, 20:22] = 4
    t[::7, 40] = 9
    out["tall_thin"] = t
    h = np.zeros((ROWS, 100), dtype=np.int32)          # band 0 owns the exterior; holes far down
    for k, r0 in enumerate(range(140, ROWS - 10, 45)):
        h[r0:r0 + 5, 10 + k:20 + 2 * k] = k + 1
        h[r0 + 2, 60:90] = 50 + k
    out["holes_far_below"] = h
    e = np.zeros((ROWS, 90), dtype=np.int32)
    e[5:30, 5:30] = 1
    e[8:12, 8:12] = 2
    out["later_bands_own_nothing"] = e
    rng = np.random.default_rng(5)
    nd = rng.integers(0, 3, size=(ROWS, 77)).astype(np.int32)
    for b in range(63, ROWS, 64):
        nd[b] = -9999
        nd[b + 1 if b + 1 < ROWS else b] = -9999
    out["nodata_rows_at_edges"] = nd
    out["negative"] = ((rng.integers(0, 3, size=(ROWS, 50)) - 1) * 1000000).astype(np.int32)
    return out


ALL = dict(scaled(), **special())


@pytest.mark.parametrize("name", sorted(ALL))
@pytest.mark.parametrize("n", [2, 4, 8])
@pytest.mark.parametrize("connect8", [True, False])
def test_bands_equal_one_gpu(name, n, connect8):
    a = ALL[name]
    check(a, n, connect8, None)
    nd = -9999 if name == "nodata_rows_at_edges" else int(np.bincount((a - a.min()).ravel()).argmax() + a.min())
    check(a, n, connect8, nd)


@pytest.mark.parametrize("n", [2, 4, 8])
def test_pipeline_labels_fractal(n):
    from malstroem_b200 import pipeline, synth
    p = pipeline.RasterPipeline(1024, 700)
    p.dem.copy_(torch.from_numpy(synth.fractal_dem(1024, 700, seed=1)).cuda())
    p.run()
    for which in ("labels", "wsheds"):
        for connect8 in (True, False):
            parts = check(p.out[which], n, connect8, None)
            assert sum(r.band_stats["segments"] for r in parts) > 0          # rings do cross the band edges
    check(p.out["labels"], n, True, 0)


def test_vectorize_labels_band_equals_the_file(tmp_path):
    from malstroem_b200 import io as mio
    from test_gpu_band_io import write_banded, TRANSFORM
    a = ALL["holes_far_below"] + ALL["kron_blobs"][:, :100]
    path = str(tmp_path / "labels.tif")
    write_banded(path, a, 4)
    want = list(vector.vectorize_labels_file(path, "bspot_id"))
    assert len(want) > 10
    out, errs = run_bands(4, lambda comm: list(vector.vectorize_labels_band(comm, path, "bspot_id")))
    assert errs == [None] * 4, errs
    assert [f for part in out for f in part] == want
    assert mio.RasterReader(path).transform == TRANSFORM


def test_an_error_on_one_rank_reaches_every_rank():
    lab = torch.zeros((ROWS, 40), dtype=torch.int32, device="cuda")
    bounds = bands.band_rows(ROWS, 4)

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        mine = lab[r0:r1] if comm.rank != 2 else lab[r0:r1, :30]            # one band of another width
        return vector.polygonize_band(comm, mine.contiguous(), r0, ROWS)

    out, errs = run_bands(4, fn)
    assert all(isinstance(e, ValueError) for e in errs), errs


def test_two_gpus_equal_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29553", os.path.join(ROOT, "tools", "band_poly_bench.py"), "--size", "1024"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "equal to one GPU: True" in r.stdout, r.stdout[-3000:]
    assert "RESULT OK" in r.stdout, r.stdout[-3000:]
