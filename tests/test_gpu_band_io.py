"""GeoTIFF files of a banded run (RasterWriter.write_band, RasterReader.read_rows, ms_tiff_decode_rows_dev), bands as
ThreadComm threads on one GPU:
  * write_band writes the same bytes as RasterWriter.write of the whole raster, for the four dtypes the reference
    writes and band splits whose edges cut tile rows (one tile row spanning four bands, bands owning none) or not;
  * read_rows gives the rows of read_device for our files, real-zlib tiles and strips, uncompressed files and the
    reference's GDAL fixtures, for windows of one row, windows starting and ending inside a block, with and without
    the short last strip, and with nodata substitution (a value, 0 - never substituted - and NaN);
  * a DEM file read band by band, the banded run and write_band of the six result rasters give the files
    RasterPipeline + RasterWriter.write give;
  * errors reach every rank: a malformed stream in one band's window, an unwritable path (no rank hangs, no file is
    left behind)."""
import os
import struct
import subprocess
import sys
import threading

import cv2
import numpy as np
import pytest
import torch

from malstroem_b200 import bands, io as mio, synth
from malstroem_b200.pipeline import RasterPipeline
from test_gpu_io import TIF, TRANSFORM, rasters, reference_tiff

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPLITS = [((700, 517), 4), ((500, 300), 8), ((1024, 1000), 4), ((257, 5), 2), ((188, 250), 2)]
TORCH = {"f32": torch.float32, "f64": torch.float64, "i32": torch.int32, "u8": torch.uint8}


def run_bands(n, fn):
    """fn(comm) in n threads; returns (results, errors) per rank; fails if a rank does not come back"""
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
    torch.cuda.synchronize()
    return out, errs


def write_banded(path, arr, n, **kw):
    rows = arr.shape[0]
    d = torch.from_numpy(arr).cuda() if isinstance(arr, np.ndarray) else arr
    bounds = bands.band_rows(rows, n)

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        w = mio.RasterWriter(path, TRANSFORM, "EPSG:25832", **kw)
        w.write_band(comm, d[r0:r1].clone(), r0, rows)
        return w.stats

    out, errs = run_bands(n, fn)
    assert errs == [None] * n, errs
    return out


@pytest.mark.parametrize("shape,n", SPLITS)
def test_write_band_files_equal_the_whole_raster_writer(tmp_path, shape, n):
    for name, arr in rasters(shape[0], shape[1], 5).items():
        whole, banded = str(tmp_path / ("w_" + name + ".tif")), str(tmp_path / ("b_" + name + ".tif"))
        mio.RasterWriter(whole, TRANSFORM, "EPSG:25832", nodata=-999).write(arr)
        stats = write_banded(banded, arr, n, nodata=-999)
        assert open(banded, "rb").read() == open(whole, "rb").read(), (name, shape, n)
        got = cv2.imread(banded, cv2.IMREAD_UNCHANGED)
        assert got is not None and np.array_equal(got.reshape(arr.shape), arr), name
        plan = mio.band_tile_plan(bands.band_rows(shape[0], n), shape[0])
        want = [sum(b - a for _, a, b in p["recv"]) * shape[1] * arr.dtype.itemsize for p in plan]
        assert [s["exchanged_bytes"] for s in stats] == want
        assert sum(s["band_tiles"] for s in stats) == stats[0]["tiles"]


def windows(rows, block_h):
    w = {(r, r + 1) for r in (0, 1, block_h - 1, block_h, rows // 2, rows - 2, rows - 1) if 0 <= r < rows}
    w |= {(0, rows), (3, rows), (0, rows - 3), (block_h // 2, min(rows, block_h + block_h // 2 + 1))}
    last = ((rows - 1) // block_h) * block_h           # first row of the last block row
    w |= {(max(0, last - 5), rows), (max(0, last - 5), max(1, last)), (max(0, last - 1), last + 1)}
    return sorted((a, b) for a, b in w if 0 <= a < b <= rows)


def check_windows(path, **kw):
    r = mio.RasterReader(path, **kw)
    whole = r.read_device()
    for a, b in windows(r._info.rows, r._info.block_h):
        got = r.read_rows(a, b)
        assert got.dtype == whole.dtype and got.shape == (b - a, whole.shape[1])
        assert torch.equal(got.view(torch.uint8), whole[a:b].view(torch.uint8)), (path, a, b)
    return whole


@pytest.mark.parametrize("shape,n", SPLITS)
def test_read_rows_of_write_band_files(tmp_path, shape, n):
    for name, arr in rasters(shape[0], shape[1], 6).items():
        p = str(tmp_path / (name + ".tif"))
        write_banded(p, arr, n)
        whole = check_windows(p)
        assert np.array_equal(whole.cpu().numpy(), arr)
        # every band's rows, into a preallocated tensor
        for r0, r1 in bands.band_rows(shape[0], n):
            out = torch.empty((r1 - r0, shape[1]), dtype=TORCH[name], device="cuda")
            assert mio.RasterReader(p).read_rows(r0, r1, out=out) is out
            assert np.array_equal(out.cpu().numpy(), arr[r0:r1])


@pytest.mark.parametrize("level", [0, 6])
@pytest.mark.parametrize("strips", [0, 8])
def test_read_rows_of_real_zlib_files(tmp_path, level, strips):
    for name, arr in rasters(300, 517, 4).items():
        for predictor in (1, 2):
            p = str(tmp_path / ("%s_%d.tif" % (name, predictor)))
            reference_tiff(p, arr, predictor, level, strips)
            assert np.array_equal(check_windows(p).cpu().numpy(), arr)


def uncompressed_tiff(path, arr, strips):
    """reference_tiff's strip layout with the raw rows as blocks (compression 1): the last strip is short"""
    blocks = [arr[r0:r0 + strips].tobytes() for r0 in range(0, arr.shape[0], strips)]
    reference_tiff(path, arr, 1, 0, strips)
    info = mio.TiffInfo(path)
    raw = bytearray(open(path, "rb").read())
    pos = 8
    offs = []
    for b in blocks:
        offs.append(pos)
        pos += len(b)
    # same sizes as zlib level 0 would not be: rewrite the file with the raw blocks, patching offsets / counts / 259
    head_len = 8
    data = b"".join(blocks)
    ifd_off = struct.unpack("<I", raw[4:8])[0]
    old_data_end = ifd_off
    tail = bytes(raw[old_data_end:])
    shift = head_len + len(data) + ((head_len + len(data)) & 1) - old_data_end
    n = struct.unpack("<H", tail[:2])[0]
    tail = bytearray(tail)
    extra = {}
    for k in range(n):
        o = 2 + 12 * k
        tag, typ, count = struct.unpack("<HHI", tail[o:o + 8])
        size = mio._TYPE_SIZE[typ] * count
        if size > 4:
            at = struct.unpack("<I", tail[o + 8:o + 12])[0]
            tail[o + 8:o + 12] = struct.pack("<I", at + shift)
            extra[tag] = (typ, at - old_data_end, count)
        if tag == 259:
            tail[o + 8:o + 10] = struct.pack("<H", 1)
    for tag, vals in ((273, offs), (279, [len(b) for b in blocks])):
        typ, at, count = extra[tag] if tag in extra else (None, None, None)
        assert count == len(vals)
        tail[at:at + 4 * count] = struct.pack("<%dI" % count, *vals)
    new_ifd = head_len + len(data) + ((head_len + len(data)) & 1)
    out = b"II" + struct.pack("<HI", 42, new_ifd) + data + (b"\0" if (head_len + len(data)) & 1 else b"") + bytes(tail)
    with open(path, "wb") as f:
        f.write(out)
    assert mio.TiffInfo(path).compression == 1 and info.block_h == strips


def test_read_rows_of_an_uncompressed_file(tmp_path):
    for name, arr in rasters(300, 517, 7).items():
        p = str(tmp_path / (name + ".tif"))
        uncompressed_tiff(p, arr, 8)
        assert np.array_equal(check_windows(p).cpu().numpy(), arr), name


def test_read_rows_of_the_references_own_files(dtm188):
    # dtm.tif: 188 = 23 * 8 + 4 rows in strips of 8, the last one short; the others are one tile
    for name in ("labelled", "flowdir_noflats", "dtm", "filled_no_flats"):
        whole = check_windows(os.path.join(TIF, name + ".tif"))
        assert np.array_equal(whole.cpu().numpy(), dtm188[name])


def test_read_rows_nodata_substitution(tmp_path):
    arr = synth.fractal_dem(600, 300, seed=2)
    arr[250:262, 7:40] = -9999.0
    q = arr.copy()
    q[100:300, 50:60] = np.nan
    z = arr.copy()
    z[z < 20] = 0
    for nodata, a in ((-9999, arr), (float("nan"), q), (0, z)):
        p = str(tmp_path / "n.tif")
        write_banded(p, a, 3, nodata=nodata)
        got = check_windows(p, nodatasubst=-999).cpu().numpy()
        if nodata == 0:
            want = z                                        # io.py:69: a nodata of 0 is never substituted
        elif nodata == -9999:
            want = np.where(np.isclose(arr, -9999.0), np.float32(-999), arr)
        else:
            want = np.where(np.isnan(q), np.float32(-999), q)
        assert np.array_equal(got, want), nodata


def test_malformed_stream_in_one_bands_window(tmp_path):
    arr = synth.fractal_dem(1024, 300, seed=3)
    p = str(tmp_path / "bad.tif")
    reference_tiff(p, arr, 2, 6)
    info = mio.TiffInfo(p)
    bad = 2 * 2                                             # tile row 2 (rows 512..767), first tile
    raw = bytearray(open(p, "rb").read())
    o = info.offsets[bad]
    raw[o + 2:o + 40] = b"\xff" * 38
    open(p, "wb").write(bytes(raw))
    bounds = bands.band_rows(1024, 4)

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        return mio.RasterReader(p).read_rows(r0, r1).cpu().numpy()

    out, errs = run_bands(4, fn)
    for g, (r0, r1) in enumerate(bounds):
        if r0 <= 512 < r1:
            assert isinstance(errs[g], ValueError), errs
        else:
            assert errs[g] is None and np.array_equal(out[g], arr[r0:r1]), errs


def test_write_band_to_an_unwritable_path(tmp_path):
    arr = synth.fractal_dem(700, 517, seed=4)
    for path in (str(tmp_path / "missing" / "x.tif"), str(tmp_path)):     # no such directory; a directory
        bounds = bands.band_rows(700, 4)
        d = torch.from_numpy(arr).cuda()

        def fn(comm):
            r0, r1 = bounds[comm.rank]
            mio.RasterWriter(path, TRANSFORM, None).write_band(comm, d[r0:r1], r0, 700)

        _, errs = run_bands(4, fn)
        assert all(e is not None for e in errs), errs
        assert isinstance(errs[0], OSError) and all(isinstance(e, RuntimeError) for e in errs[1:]), errs
    assert os.listdir(str(tmp_path)) == []


@pytest.mark.parametrize("shape,n", [((700, 517), 4), ((500, 300), 8)])
def test_dem_file_through_the_bands_to_result_files(tmp_path, shape, n):
    rows, cols = shape
    dem = synth.fractal_dem(rows, cols, seed=8)
    src = str(tmp_path / "dem.tif")
    mio.RasterWriter(src, TRANSFORM, "EPSG:25832").write(dem)
    q = RasterPipeline(rows, cols)
    q.run(mio.RasterReader(src).read_device())
    names = RasterPipeline.HOST_RASTERS
    for name in names:
        mio.RasterWriter(str(tmp_path / ("w_" + name + ".tif")), TRANSFORM, "EPSG:25832").write(q.out[name])

    def fn(comm):
        p = bands.BandPipeline(rows, cols, comm)
        try:
            mio.RasterReader(src).read_rows(p.r0, p.r1, out=p.dem)
            p.run()
            for name in names:
                w = mio.RasterWriter(str(tmp_path / ("b_" + name + ".tif")), TRANSFORM, "EPSG:25832")
                w.write_band(comm, p.out[name], p.r0, rows)
        finally:
            p.close()

    _, errs = run_bands(n, fn)
    assert errs == [None] * n, errs
    for name in names:
        a = open(str(tmp_path / ("b_" + name + ".tif")), "rb").read()
        b = open(str(tmp_path / ("w_" + name + ".tif")), "rb").read()
        assert a == b, name


def test_two_gpus_write_and_read_across_a_tile_row():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    # 700 rows in 2 bands: 0-384 and 384-700, so the second tile row (256-512) crosses the band edge
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "band_io_bench.py"), "--size", "700"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "tile rows that cross a band edge: 1" in r.stdout, r.stdout[-3000:]
    assert "all files byte-identical to the single-GPU writer: True" in r.stdout, r.stdout[-3000:]
    assert "RESULT OK" in r.stdout, r.stdout[-3000:]
