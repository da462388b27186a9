"""Row-band GeoTIFF writing, the host half (no GPU): how bands share the file's 256-row tile rows
(io.band_tile_plan), where each band's tiles go in the file (io.band_file_offsets, against build_tiff's own offsets,
classic and BigTIFF), and RasterWriter.write_band's collective check of the bands, which every rank fails alike and
before any device work."""
import struct
import threading

import numpy as np
import pytest
import torch

from malstroem_b200 import bands, io as mio

T = mio.TILE


def check_plan(bounds, rows):
    plans = mio.band_tile_plan(bounds, rows)
    assert len(plans) == len(bounds)
    owner = {}
    for g, (p, (r0, r1)) in enumerate(zip(plans, bounds)):
        t0, t1 = p["own"]
        for t in range(t0, t1):
            assert t not in owner
            owner[t] = g
            assert r0 <= t * T < r1                                    # the band of the tile row's first row
        i0, i1 = p["inner"]
        assert i0 == t0 and i1 <= t1
        for t in range(i0, i1):
            assert min((t + 1) * T, rows) <= r1                        # encoded from the band's own rows
        if p["cross"] is None:
            assert i1 == t1
        else:
            assert p["cross"] == t1 - 1 == i1 and min(t1 * T, rows) > r1
            # the received rows are exactly those of the crossing tile row past the band's end, in order
            got = []
            for src, a, b in p["recv"]:
                assert src > g and bounds[src][0] <= a < b <= bounds[src][1]
                got.extend(range(a, b))
            assert got == list(range(r1, min(t1 * T, rows)))
        if p["cross"] is None:
            assert p["recv"] == []
        if p["send"] is not None:
            dest, a, b = p["send"]
            assert dest < g and a == r0 and b <= r1
            assert plans[dest]["cross"] == r0 // T
            if t1 == t0:
                assert b == min(r1, (r0 // T + 1) * T)                # nothing beyond the tile row it lacks
        else:
            assert r0 % T == 0 or r1 == r0
        if t1 == t0 and r1 > r0:
            assert p["cross"] is None and p["recv"] == []              # a band without a tile row owns nothing
    assert sorted(owner) == list(range(-(-rows // T)))
    return plans


@pytest.mark.parametrize("rows,n", [(500, 8), (700, 4), (11000, 8), (1000, 3), (65536, 8), (257, 2)])
def test_plan_of_the_band_split(rows, n):
    bounds = bands.band_rows(rows, n)
    plans = check_plan(bounds, rows)
    if rows % (T * n) == 0:
        assert all(p["send"] is None for p in plans)                   # aligned edges exchange nothing
    if (rows, n) == (500, 8):
        # bands of 64 rows: the first tile row spans bands 0-3, three bands own no tile row
        assert [p["own"][1] - p["own"][0] for p in plans] == [1, 0, 0, 0, 1, 0, 0, 0][:len(plans)]
        assert plans[0]["recv"] == [(1, 64, 128), (2, 128, 192), (3, 192, 256)]
    if (rows, n) == (700, 4):
        assert bounds[:2] == [(0, 192), (192, 384)]


@pytest.mark.parametrize("bounds,rows", [
    ([(0, 100), (100, 101), (101, 700)], 700),
    ([(0, 300), (300, 300), (300, 310), (310, 1000)], 1000),              # an empty band
    ([(0, 10), (10, 20), (20, 30), (30, 40), (40, 600)], 600),
    ([(0, 256), (256, 512), (512, 513)], 513),
    ([(0, 5)], 5),
    ([(0, 1), (1, 1000), (1000, 1001)], 1001),
    ([(0, 255), (255, 257), (257, 258)], 258),
])
def test_plan_of_uneven_bands(bounds, rows):
    check_plan(bounds, rows)


def directory_offsets(head, tail, tile_sizes):
    """Tag 324 (tile offsets) of build_tiff's directory, read from the tail alone"""
    big = head[2:4] == struct.pack("<H", 43)
    pos = len(head) + sum(tile_sizes)
    ifd = tail[pos & 1:]
    n = struct.unpack("<Q" if big else "<H", ifd[:8 if big else 2])[0]
    entry, base = (20, 8) if big else (12, 2)
    for k in range(n):
        e = ifd[base + entry * k: base + entry * (k + 1)]
        tag, typ = struct.unpack("<HH", e[:4])
        if tag == 324:
            count = struct.unpack("<Q" if big else "<I", e[4:12] if big else e[4:8])[0]
            field = e[12:20] if big else e[8:12]
            w = 8 if big else 4
            if count * w <= len(field):
                raw = field[:count * w]
            else:
                at = struct.unpack("<Q" if big else "<I", field)[0] - pos
                raw = tail[at:at + count * w]
            return list(struct.unpack("<%d%s" % (count, "Q" if big else "I"), raw))
    raise AssertionError("no tile offsets")


@pytest.mark.parametrize("sizes,band_tiles,big", [
    ([100 + 7 * k for k in range(12)], [3, 0, 6, 3], False),
    ([1 << 30] * 5, [2, 0, 3], True),                                        # BigTIFF, as test_bigtiff_directory
    ([(1 << 30) + 3, 5, 1 << 30, 7, 1 << 30, 11, 1 << 30], [1, 1, 4, 1], True),
    ([(1 << 30) + 3, 5, 1 << 30, 7, 1 << 30, 11, 1 << 29], [1, 1, 4, 1], False),       # just below the switch
    ([33], [1], False),
])
def test_offsets_from_gathered_sizes_equal_the_directory(sizes, band_tiles, big):
    head, tail = mio.build_tiff(70000, 70000, np.float32, 2, sizes, None, None)
    assert (len(head) == 16) == big == (mio.tiff_head_len(sizes) == 16)
    offs = directory_offsets(head, tail, sizes)
    first = np.concatenate([[0], np.cumsum(band_tiles)])[:-1]
    got = mio.band_file_offsets(sizes, band_tiles)
    assert got == [offs[k] if k < len(offs) else len(head) + sum(sizes) for k in first]


def run_ranks(n, fn):
    grp = bands.ThreadGroup(n)
    out, errs = [None] * n, [None] * n

    def work(rank):
        try:
            out[rank] = fn(bands.ThreadComm(grp, rank))
        except BaseException as e:      # noqa: BLE001
            errs[rank] = e

    ts = [threading.Thread(target=work, args=(r,)) for r in range(n)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(60)
        assert not t.is_alive(), "a rank hangs"
    return out, errs


@pytest.mark.parametrize("case", ["gap", "overlap", "short", "cols", "dtype", "order", "rows"])
def test_write_band_rejects_bands_that_do_not_tile_the_raster(tmp_path, case):
    rows, cols = 700, 33
    bounds = bands.band_rows(rows, 3)
    path = str(tmp_path / "x.tif")

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        c, dt, rr = cols, torch.float32, rows
        if case == "gap" and comm.rank == 1:
            r0 += 1
        if case == "overlap" and comm.rank == 2:
            r0 -= 1
        if case == "short" and comm.rank == 2:
            r1 -= 1
        if case == "cols" and comm.rank == 1:
            c += 1
        if case == "dtype" and comm.rank == 0:
            dt = torch.float64
        if case == "order":
            r0, r1 = bounds[comm.size - 1 - comm.rank]
        if case == "rows" and comm.rank == 0:
            rr += 1
        band = torch.zeros((r1 - r0, c), dtype=dt)
        mio.RasterWriter(path, None, None).write_band(comm, band, r0, rr)

    _, errs = run_ranks(3, fn)
    for e in errs:
        assert isinstance(e, ValueError) and "do not tile" in str(e), errs
    assert not (tmp_path / "x.tif").exists()


def test_write_band_without_gpu_fails_loudly_after_the_band_check(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    bounds = bands.band_rows(300, 2)

    def fn(comm):
        r0, r1 = bounds[comm.rank]
        mio.RasterWriter(str(tmp_path / "x.tif"), None, None).write_band(comm, torch.zeros((r1 - r0, 9)), r0, 300)

    _, errs = run_ranks(2, fn)
    for e in errs:
        assert isinstance(e, RuntimeError) and "no CPU fallback" in str(e), errs
