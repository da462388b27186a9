"""Mirror of malstroem/io.py's raster half (RasterReader io.py:21-72, RasterWriter io.py:75-139) without GDAL:
GeoTIFF files — tiled 256 x 256, deflate, predictor 2 for float32 / int32 / uint8, exactly the options the reference's
writer passes to GDAL (io.py:112, :127-136) — are written and read with the codec kernels of csrc/tiff.cu
(SURVEY.md 8(f3)).  The byte-heavy halves (predictor + deflate, inflate + predictor + nodata substitution) run on the
device; this module is the container: header, tag directory, tile offsets (a few hundred bytes per file).

Same constructor arguments, attributes and methods as the reference classes, so `DemTool` / `BluespotTool` accept them
as duck-typed readers / writers.  Differences, all forced by the absence of GDAL's CRS database: `crs` is carried as
the GeoTIFF citation string (written to and read from GTCitationGeoKey) instead of being translated to EPSG geokeys;
readers without GDAL's WKT parser (cv2, tifffile) are unaffected.  The vector half of io.py (OGR) is out of scope.
There is no CPU fallback: read() / write() need the CUDA library.
"""
import bisect
import ctypes
import os
import struct

import numpy as np

from . import _lib

TILE = 256
# TIFF field types
_BYTE, _ASCII, _SHORT, _LONG, _RATIONAL, _DOUBLE, _LONG8 = 1, 2, 3, 4, 5, 12, 16
_TYPE_SIZE = {1: 1, 2: 1, 3: 2, 4: 4, 5: 8, 6: 1, 7: 1, 8: 2, 9: 4, 10: 8, 11: 4, 12: 8, 16: 8, 17: 8, 18: 8}
_TYPE_FMT = {1: "B", 2: "c", 3: "H", 4: "I", 6: "b", 7: "B", 8: "h", 9: "i", 11: "f", 12: "d", 16: "Q", 17: "q", 18: "Q"}
# numpy dtype <-> (sample format, bits)
_DTYPES = {np.dtype(np.uint8): (1, 8), np.dtype(np.uint16): (1, 16), np.dtype(np.uint32): (1, 32),
           np.dtype(np.int8): (2, 8), np.dtype(np.int16): (2, 16), np.dtype(np.int32): (2, 32), np.dtype(np.int64): (2, 64),
           np.dtype(np.uint64): (1, 64), np.dtype(np.float32): (3, 32), np.dtype(np.float64): (3, 64)}
_FROM_TIFF = {v: k for k, v in _DTYPES.items()}


# ------------------------------------------------------------------------------------------------ container: write
def _geo_tags(transform, crs):
    """ModelPixelScale / ModelTiepoint (or ModelTransformation for a rotated grid) + a minimal GeoKey directory."""
    tags = []
    if transform is not None:
        x0, sx, rx, y0, ry, sy = [float(v) for v in transform]
        if rx == 0.0 and ry == 0.0:
            tags.append((33550, _DOUBLE, [abs(sx), abs(sy), 0.0]))
            tags.append((33922, _DOUBLE, [0.0, 0.0, 0.0, x0, y0, 0.0]))
        else:
            tags.append((34264, _DOUBLE, [sx, rx, 0.0, x0, ry, sy, 0.0, y0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0]))
    cit = (str(crs) + "|") if crs else ""
    keys = [1, 1, 0, 0]
    entries = [(1024, 0, 1, 1 if crs else 32767), (1025, 0, 1, 1)]       # GTModelType (projected / user), RasterType area
    if cit:
        entries.append((1026, 34737, len(cit), 0))                       # GTCitationGeoKey -> GeoAsciiParams
    keys[3] = len(entries)
    for e in entries:
        keys.extend(e)
    tags.append((34735, _SHORT, keys))
    if cit:
        tags.append((34737, _ASCII, cit))
    return tags


def _pack_value(typ, values):
    if typ == _ASCII:
        b = values.encode("latin-1", "replace") + b"\0"
        return b, len(b)
    vals = list(values)
    return struct.pack("<%d%s" % (len(vals), _TYPE_FMT[typ]), *vals), len(vals)


def tiff_head_len(tile_sizes):
    """Bytes before the first tile in build_tiff's file: 8 (classic TIFF) or 16 (BigTIFF, for 4 GB of data and up)."""
    total = int(sum(int(s) for s in tile_sizes))
    return 16 if total + 65536 + 16 * len(tile_sizes) >= (1 << 32) - (1 << 20) else 8


def build_tiff(rows, cols, dtype, predictor, tile_sizes, transform=None, crs=None, nodata=None):
    """Header and tag directory of a tiled, deflate-compressed single-band TIFF whose tile data (the zlib streams, in
    tile order, one after the other) follows the header directly.  Returns (head bytes, tail bytes): the file is
    head + data + tail.  Classic TIFF below 4 GB, BigTIFF above (the reference's bigtiff='if_safer')."""
    fmt, bits = _DTYPES[np.dtype(dtype)]
    head_len = tiff_head_len(tile_sizes)
    big = head_len == 16
    offsets, pos = [], head_len
    for s in tile_sizes:
        offsets.append(pos)
        pos += int(s)
    data_end = pos + (pos & 1)
    off_type = _LONG8 if big else _LONG
    tags = [(256, _LONG, [cols]), (257, _LONG, [rows]), (258, _SHORT, [bits]), (259, _SHORT, [8]), (262, _SHORT, [1]),
            (277, _SHORT, [1]), (284, _SHORT, [1]), (317, _SHORT, [predictor]), (322, _SHORT, [TILE]), (323, _SHORT, [TILE]),
            (324, off_type, offsets), (325, off_type, [int(s) for s in tile_sizes]), (339, _SHORT, [fmt])]
    tags += _geo_tags(transform, crs)
    if nodata is not None:
        tags.append((42113, _ASCII, "%.17g" % float(nodata)))
    tags.sort(key=lambda t: t[0])
    # the directory sits after the data; values that do not fit the entry go after the directory
    entry = 20 if big else 12
    ifd_off = data_end
    ifd_len = (8 if big else 2) + entry * len(tags) + (8 if big else 4)
    extra_off = ifd_off + ifd_len
    ifd = struct.pack("<Q" if big else "<H", len(tags))
    extra = b""
    inline = 8 if big else 4
    for tag, typ, values in tags:
        raw, count = _pack_value(typ, values)
        if len(raw) <= inline:
            field = raw + b"\0" * (inline - len(raw))
        else:
            if (extra_off + len(extra)) & 1:
                extra += b"\0"
            field = struct.pack("<Q" if big else "<I", extra_off + len(extra))
            extra += raw
        ifd += struct.pack("<HH", tag, typ) + struct.pack("<Q" if big else "<I", count) + field
    ifd += struct.pack("<Q" if big else "<I", 0)
    head = (b"II" + struct.pack("<HHHQ", 43, 8, 0, ifd_off)) if big else (b"II" + struct.pack("<HI", 42, ifd_off))
    tail = (b"\0" if (pos & 1) else b"") + ifd + extra
    return head, tail


# ---------------------------------------------------------------------------------------- container: row bands
def band_tile_plan(bands, rows):
    """How row bands share the 256-row tile rows of one file.  bands: [(r0, r1)] in rank order, tiling [0, rows).
    Tile row t belongs to the band that holds its first row 256 t.  Per rank a dict:
      own    (t0, t1): the tile rows the band encodes;
      inner  (t0, t1): those of `own` whose rows all lie in the band (encoded straight from the band's rows);
      cross  the last tile row of `own` when it runs past the band's last row, else None;
      send   (dest, a, b): rows [a, b) of the band, which the owner `dest` of the tile row that crosses the band's
             first row lacks; None when the band starts on a tile row;
      recv   [(src, a, b)] in rank order: the `send`s addressed to this band, together the rows of `cross` past the
             band's last row.
    Rows only travel towards lower ranks and may skip bands that own no tile row."""
    ends = [int(b) for _, b in bands]
    plans = []
    for r0, r1 in bands:
        t0, t1 = -(-r0 // TILE), -(-r1 // TILE)
        cross = t1 - 1 if t1 > t0 and min(t1 * TILE, rows) > r1 else None
        send = None
        first = (r0 // TILE) * TILE
        if r1 > r0 and first < r0:
            send = (bisect.bisect_right(ends, first), r0, min(r1, first + TILE))
        plans.append({"own": (t0, t1), "inner": (t0, t1 if cross is None else cross), "cross": cross, "send": send,
                      "recv": []})
    for g, p in enumerate(plans):
        if p["send"] is not None:
            plans[p["send"][0]]["recv"].append((g,) + p["send"][1:])
    return plans


def band_file_offsets(tile_sizes, band_tiles):
    """File offset of every band's first tile in build_tiff's layout: tile_sizes of the whole file in tile order,
    band_tiles = the number of tiles of each band, in rank order."""
    cum = np.concatenate([[0], np.cumsum(np.asarray(tile_sizes, dtype=np.int64))])
    first = np.concatenate([[0], np.cumsum(np.asarray(band_tiles, dtype=np.int64))])[:-1]
    head = tiff_head_len(tile_sizes)
    return [head + int(cum[k]) for k in first]


# ------------------------------------------------------------------------------------------------- container: read
class TiffInfo(object):
    """The tags of the first image of a (Big)TIFF file that matter for a single-band raster."""

    def __init__(self, filepath):
        self.filepath = filepath
        with open(filepath, "rb") as f:
            head = f.read(16)
            if head[:2] == b"II":
                bo = "<"
            elif head[:2] == b"MM":
                bo = ">"
            else:
                raise ValueError("%s: not a TIFF file" % filepath)
            magic = struct.unpack(bo + "H", head[2:4])[0]
            if magic == 42:
                big, ifd_off = False, struct.unpack(bo + "I", head[4:8])[0]
            elif magic == 43:
                big, ifd_off = True, struct.unpack(bo + "Q", head[8:16])[0]
            else:
                raise ValueError("%s: not a TIFF file (magic %d)" % (filepath, magic))
            self.bo, self.big = bo, big
            f.seek(ifd_off)
            n = struct.unpack(bo + ("Q" if big else "H"), f.read(8 if big else 2))[0]
            entry = 20 if big else 12
            raw = f.read(entry * n)
            self.tags = {}
            for k in range(n):
                e = raw[k * entry:(k + 1) * entry]
                tag, typ = struct.unpack(bo + "HH", e[:4])
                count = struct.unpack(bo + ("Q" if big else "I"), e[4:12] if big else e[4:8])[0]
                field = e[12:20] if big else e[8:12]
                size = _TYPE_SIZE.get(typ, 1) * count
                if size <= len(field):
                    data = field[:size]
                else:
                    off = struct.unpack(bo + ("Q" if big else "I"), field)[0]
                    here = f.tell()
                    f.seek(off)
                    data = f.read(size)
                    f.seek(here)
                if typ == _ASCII:
                    self.tags[tag] = data.split(b"\0")[0].decode("latin-1")
                elif typ in _TYPE_FMT:
                    self.tags[tag] = list(struct.unpack(bo + "%d%s" % (count, _TYPE_FMT[typ]), data))
        t = self.tags
        self.cols, self.rows = int(t[256][0]), int(t[257][0])
        if int(t.get(277, [1])[0]) != 1:
            raise NotImplementedError("%s: only single-band rasters" % filepath)
        bits, fmt = int(t.get(258, [1])[0]), int(t.get(339, [1])[0])
        if (fmt, bits) not in _FROM_TIFF:
            raise NotImplementedError("%s: sample format %d with %d bits" % (filepath, fmt, bits))
        self.dtype, self.sample_format, self.sample_bytes = _FROM_TIFF[(fmt, bits)], fmt, bits // 8
        self.compression = int(t.get(259, [1])[0])
        if self.compression not in (1, 8, 32946):
            raise NotImplementedError("%s: compression %d (none and deflate are supported)" % (filepath, self.compression))
        self.predictor = int(t.get(317, [1])[0])
        if self.predictor not in (1, 2):
            raise NotImplementedError("%s: predictor %d" % (filepath, self.predictor))
        if bo == ">" and self.sample_bytes > 1:
            raise NotImplementedError("%s: big-endian samples" % filepath)
        if 322 in t:
            self.block_w, self.block_h = int(t[322][0]), int(t[323][0])
            self.offsets, self.counts = [int(v) for v in t[324]], [int(v) for v in t[325]]
        else:
            self.block_w = self.cols
            self.block_h = min(int(t.get(278, [self.rows])[0]), self.rows)
            self.offsets, self.counts = [int(v) for v in t[273]], [int(v) for v in t[279]]
        nd = t.get(42113)
        try:
            self.nodata = float(nd) if nd is not None and nd.strip() != "" else None
        except ValueError:
            self.nodata = None
        # GDAL style affine transform
        if 34264 in t:
            m = t[34264]
            self.transform = (m[3], m[0], m[1], m[7], m[4], m[5])
        elif 33550 in t and 33922 in t:
            sx, sy = t[33550][0], t[33550][1]
            i, j, _, x, y, _ = t[33922][:6]
            self.transform = (x - i * sx, sx, 0.0, y + j * sy, 0.0, -sy)
        else:
            self.transform = (0.0, 1.0, 0.0, 0.0, 0.0, 1.0)
        cit = t.get(34737)
        self.crs = cit.rstrip("|") if cit else ""


# ------------------------------------------------------------------------------------------------------- the classes
def _np_dtype(data):
    if isinstance(data, np.ndarray):
        return data.dtype
    return np.dtype(str(data.dtype).replace("torch.", ""))


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("malstroem_b200.io needs a CUDA device (there is no CPU fallback)")
    return torch


class RasterReader(object):
    """io.RasterReader (io.py:21-72): a single-band GeoTIFF into a 2-D numpy array, nodata replaced by
    `nodatasubst`.  read_device() returns the raster as a cuda tensor (for the device-resident pipeline)."""

    def __init__(self, filepath, nodatasubst=None):
        self.filepath = filepath
        self._info = TiffInfo(filepath)
        self.transform = self._info.transform
        self.crs = self._info.crs
        self.nodata = self._info.nodata
        self.nodatasubst = nodatasubst

    def _blocks(self, b0, b1, dev):
        """Block rows [b0, b1) of the file on `dev`: (the compressed blocks one after the other, their offsets, their
        lengths, the scratch the decode inflates into, the number of blocks).  Only these blocks are read, with seek +
        readinto into one pinned buffer."""
        torch = _torch()
        t = self._info
        bx = -(-t.cols // t.block_w)
        k0, k1 = b0 * bx, b1 * bx
        if len(t.offsets) < k1 or len(t.counts) < k1:
            raise ValueError("%s: %d blocks listed, %d needed" % (self.filepath, min(len(t.offsets), len(t.counts)), k1))
        counts = t.counts[k0:k1]
        nblocks = k1 - k0
        # the compressed blocks, one after the other, in one pinned buffer
        total = sum(counts)
        host = torch.empty(max(total, 1), dtype=torch.uint8).pin_memory()
        hv = host.numpy()
        offs = np.zeros(nblocks, np.uint64)
        pos = 0
        with open(self.filepath, "rb") as f:
            for k in range(nblocks):
                f.seek(t.offsets[k0 + k])
                f.readinto(memoryview(hv)[pos:pos + counts[k]])
                offs[k] = pos
                pos += counts[k]
        block_bytes = t.block_w * t.block_h * t.sample_bytes
        d_in = host.to(dev, non_blocking=True)
        d_off = torch.from_numpy(offs.view(np.int64)).to(dev)
        d_len = torch.from_numpy(np.asarray(counts, dtype=np.uint32).view(np.int32)).to(dev)
        scratch = torch.empty(nblocks * block_bytes, dtype=torch.uint8, device=dev)
        if t.compression == 1:
            # raw blocks: lined up at the block stride (the last strip may be short)
            for k in range(nblocks):
                o = int(offs[k])
                scratch[k * block_bytes:k * block_bytes + counts[k]] = d_in[o:o + counts[k]]
        return d_in, d_off, d_len, scratch, nblocks

    def _subst(self):
        """(subst_mode, nodata, subst) of the decode.  `if self.nodata and self.nodatasubst is not None` (io.py:69):
        a nodata value of 0 is never substituted."""
        mode = 0
        if self.nodata and self.nodatasubst is not None:
            mode = 2 if np.isnan(self.nodata) else 1
        return (mode, float(self.nodata) if self.nodata is not None else 0.0,
                float(self.nodatasubst) if self.nodatasubst is not None else 0.0)

    def read_device(self, device=0):
        torch = _torch()
        t = self._info
        dev = torch.device("cuda", device)
        d_in, d_off, d_len, scratch, nblocks = self._blocks(0, -(-t.rows // t.block_h), dev)
        out = torch.empty((t.rows, t.cols), dtype=getattr(torch, np.dtype(t.dtype).name), device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with _lib.lock:
            _lib.check(_lib.lib().ms_init(dev.index or 0), "ms_init")
            _lib.check(_lib.lib().ms_tiff_decode_dev(
                d_in.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), nblocks, t.block_w, t.block_h, t.sample_bytes,
                t.sample_format, t.predictor, scratch.data_ptr(), out.data_ptr(), t.rows, t.cols, *self._subst(),
                1 if t.compression != 1 else 0, ctypes.c_void_p(stream)), "RasterReader.read")
        return out

    def read_rows(self, r0, r1, device=0, out=None):
        """Rows [r0, r1) of the raster as a cuda tensor, the same values as read_device()[r0:r1], nodata substituted
        alike.  Only the blocks (tiles or strips) that meet those rows are read from the file and decoded, so a row
        band of a raster that no single device holds reads its own share of the file.  out: a contiguous tensor of
        shape (r1 - r0, cols) and the file's dtype on `device` to decode into (for example BandPipeline.dem).  Not a
        collective: every band reads on its own."""
        t = self._info
        r0, r1 = int(r0), int(r1)
        if not 0 <= r0 < r1 <= t.rows:
            raise ValueError("read_rows: rows [%d, %d) are not inside [0, %d)" % (r0, r1, t.rows))
        torch = _torch()
        dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        dt = getattr(torch, np.dtype(t.dtype).name)
        if out is None:
            out = torch.empty((r1 - r0, t.cols), dtype=dt, device=dev)
        elif (tuple(out.shape) != (r1 - r0, t.cols) or out.dtype != dt or not out.is_contiguous()
              or out.device != dev):
            raise ValueError("read_rows: out must be a contiguous %s tensor of shape (%d, %d) on %s"
                             % (dt, r1 - r0, t.cols, dev))
        b0, b1 = r0 // t.block_h, -(-r1 // t.block_h)
        d_in, d_off, d_len, scratch, nblocks = self._blocks(b0, b1, dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        with _lib.lock:
            _lib.check(_lib.lib().ms_init(dev.index or 0), "ms_init")
            _lib.check(_lib.lib().ms_tiff_decode_rows_dev(
                d_in.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), nblocks, t.block_w, t.block_h, t.sample_bytes,
                t.sample_format, t.predictor, scratch.data_ptr(), out.data_ptr(), t.rows, t.cols, b0, r0, r1 - r0,
                *self._subst(), 1 if t.compression != 1 else 0, ctypes.c_void_p(stream)), "RasterReader.read_rows")
        return out

    def read(self):
        return self.read_device().cpu().numpy()


class RasterWriter(object):
    """io.RasterWriter (io.py:75-139): a 2-D array (numpy, or a cuda tensor) as a tiled, deflate-compressed GeoTIFF,
    predictor 2 for float32 / int32 / uint8 and none for float64, as the reference configures GDAL."""

    def __init__(self, filepath, transform, crs, nodata=None):
        self.filepath = filepath
        self.transform = transform
        self.crs = crs
        self.driver = 'gtiff'
        self.options = dict(tiled='yes', compress='deflate', bigtiff='if_safer')
        self.datatype = None
        self.nodata = nodata
        self.stats = {}

    def _predictor(self, dtype):
        """The GDAL datatype (set on the first write) and the predictor the reference gives GDAL for `dtype`."""
        if not self.datatype:
            # io.py:124-136: the four types the reference knows, predictor 2 for all but float64
            if dtype == np.float64:
                self.datatype = 'Float64'
            elif dtype == np.float32:
                self.datatype = 'Float32'
                self.options['predictor'] = 2
            elif dtype == np.int32:
                self.datatype = 'Int32'
                self.options['predictor'] = 2
            elif dtype == np.uint8:
                self.datatype = 'Byte'
                self.options['predictor'] = 2
            else:
                raise NotImplementedError("Cannot determine GDAL datatype for numpy datatype {}".format(dtype))
        return int(self.options.get('predictor', 1))

    def write(self, data, device=0):
        torch = _torch()
        dtype = _np_dtype(data)
        predictor = self._predictor(dtype)
        if len(data.shape) != 2:
            raise ValueError("RasterWriter.write: a 2-D array is required")
        dev = torch.device("cuda", device)
        d = torch.from_numpy(np.ascontiguousarray(data)).to(dev) if isinstance(data, np.ndarray) else data.contiguous()
        rows, cols = int(d.shape[0]), int(d.shape[1])
        es = d.element_size()
        L = _lib.lib()
        tiles = (-(-rows // TILE)) * (-(-cols // TILE))
        with _lib.lock:
            _lib.check(L.ms_init(dev.index or 0), "ms_init")
            slot = int(L.ms_tiff_tile_slot(es))
        slots = torch.empty(tiles * slot, dtype=torch.uint8, device=dev)
        sizes = torch.empty(tiles, dtype=torch.int32, device=dev)
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with _lib.lock:
            _lib.check(L.ms_tiff_encode_dev(d.data_ptr(), es, rows, cols, predictor, slots.data_ptr(), slot,
                                            sizes.data_ptr(), stream), "RasterWriter.write")
        offs = torch.cumsum(sizes.long(), 0) - sizes.long()
        total = int(offs[-1] + sizes[-1])
        packed = torch.empty(total, dtype=torch.uint8, device=dev)
        with _lib.lock:
            _lib.check(L.ms_tiff_pack_dev(slots.data_ptr(), slot, sizes.data_ptr(), offs.data_ptr(), tiles,
                                          packed.data_ptr(), stream), "RasterWriter.write")
        host = torch.empty(total, dtype=torch.uint8).pin_memory()
        host.copy_(packed, non_blocking=True)
        tile_sizes = sizes.cpu().numpy().astype(np.int64)
        torch.cuda.current_stream(dev).synchronize()
        head, tail = build_tiff(rows, cols, dtype, predictor, tile_sizes, self.transform, self.crs, self.nodata)
        with open(self.filepath, "wb") as f:
            f.write(head)
            f.write(memoryview(host.numpy()))
            f.write(tail)
        self.stats = {"raw_bytes": rows * cols * es, "file_bytes": len(head) + total + len(tail), "tiles": tiles}

    STAGE_BYTES = 64 << 20          # each of write_band's two pinned staging buffers
    ENCODE_SLOT_BYTES = 1 << 30     # write_band's tile slots per encode call (at least one tile row)

    def write_band(self, comm, band, r0, rows, device=0):
        """Collective over `comm` (bands.ThreadComm or bands.DistComm): every rank passes its own `band`, rows
        [r0, r0 + band.shape[0]) of a rows x cols raster, and together they write ONE file, byte for byte what write()
        writes for the whole raster.  No rank holds more than its band:
          * tile row t belongs to the band holding row 256 t (band_tile_plan); the band that owns the tile row across
            its last row receives the rows it lacks (fewer than 256) from the following bands, all other tile rows are
            encoded straight from the band's rows;
          * the tile sizes (one int per tile) are gathered, every rank computes the same container and its own offset;
            rank 0 creates the file with the header and its final size, then every rank writes its tiles at its
            offset and rank 0 the tag directory.
        Memory per rank: on the device, the band, its compressed tiles and at most ENCODE_SLOT_BYTES of tile slots; on
        the host, two pinned staging buffers of STAGE_BYTES (the device-to-host copy of one overlaps the file write of
        the other) and O(tiles of the file) for the sizes and the tag directory - independent of the raster's size
        otherwise.  All ranks must see the same file system (one host).
        Bands that do not tile [0, rows) in rank order, or disagree on cols or dtype, make every rank raise ValueError
        before any device work; a failure on one rank (allocation, encode, an unwritable path, a short write) makes
        every rank raise, and rank 0 removes the partial file."""
        import torch
        try:
            dtype = _np_dtype(band)
            code = list(_DTYPES).index(dtype) if dtype in _DTYPES else len(_DTYPES)
        except TypeError:
            dtype, code = None, -1
        two_d = len(band.shape) == 2
        r0, rows = int(r0), int(rows)
        mine = [r0, r0 + int(band.shape[0]) if two_d else -1, int(band.shape[1]) if two_d else -1, code, rows]
        where = band.device if isinstance(band, torch.Tensor) else torch.device("cpu")
        got = comm.all_gather(torch.tensor(mine, dtype=torch.int64, device=where)).cpu().tolist()
        bounds = [(a, b) for a, b, _, _, _ in got]
        ok = (got[0][0] == 0 and got[-1][1] == rows and rows >= 1
              and all(g[1] >= g[0] and g[2] >= 1 and g[2:] == got[0][2:] for g in got)
              and all(got[k][0] == got[k - 1][1] for k in range(1, len(got))))
        if not ok:
            raise ValueError("write_band: the bands (r0, r1, cols, dtype, rows) %s do not tile the rows of one raster "
                             "in rank order" % got)
        torch = _torch()
        predictor = self._predictor(dtype)
        cols, r1, rank = got[0][2], bounds[comm.rank][1], comm.rank
        dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        plans = band_tile_plan(bounds, rows)
        plan = plans[rank]
        tiles_x = -(-cols // TILE)
        fail, made = [None], [False]

        def agree():
            """all ranks learn whether any rank failed; every rank raises (rank 0 removes the file it made first)"""
            bad = comm.all_reduce(torch.tensor([0 if fail[0] is None else 1], dtype=torch.int32, device=dev), "max")
            if int(bad.item()):
                if made[0]:
                    os.remove(self.filepath)
                if fail[0] is not None:
                    raise fail[0]
                raise RuntimeError("write_band: %s: the write failed on another rank" % self.filepath)

        L = _lib.lib()
        try:
            d = (torch.from_numpy(np.ascontiguousarray(band)) if isinstance(band, np.ndarray) else band)
            d = d.to(dev).contiguous()
            es = d.element_size()
            u8 = d.view(torch.uint8)
            with _lib.lock:
                _lib.check(L.ms_init(dev.index or 0), "ms_init")
                slot = int(L.ms_tiff_tile_slot(es))
        except (RuntimeError, ValueError, OSError, MemoryError) as e:
            fail[0] = e
        agree()
        # the rows of the tile row across each band's last row, from the bands that hold them
        recv = None
        if any(p["send"] is not None for p in plans):
            chunks = [u8[:0]] * comm.size
            if plan["send"] is not None:
                dest, a, b = plan["send"]
                chunks[dest] = u8[a - r0:b - r0]
            got = comm.all_to_all_var(chunks)
            if plan["recv"]:
                recv = torch.cat([got[src] for src, _, _ in plan["recv"]])
        stream = torch.cuda.current_stream(dev)
        sizes_h, packed = [], []
        ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
        try:
            ev[0].record(stream)
            per = max(1, self.ENCODE_SLOT_BYTES // (tiles_x * slot))         # tile rows per encode call
            slots = None

            def encode(src):
                nonlocal slots
                n = -(-int(src.shape[0]) // TILE) * tiles_x
                if slots is None or slots.numel() < n * slot:
                    slots = torch.empty(min(per, plan["own"][1] - plan["own"][0]) * tiles_x * slot, dtype=torch.uint8,
                                        device=dev)
                sizes = torch.empty(n, dtype=torch.int32, device=dev)
                st = ctypes.c_void_p(stream.cuda_stream)
                with _lib.lock:
                    _lib.check(L.ms_tiff_encode_dev(src.data_ptr(), es, int(src.shape[0]), cols, predictor,
                                                    slots.data_ptr(), slot, sizes.data_ptr(), st), "write_band")
                offs = torch.cumsum(sizes.long(), 0) - sizes.long()
                h = sizes.cpu().numpy().astype(np.int64)
                out = torch.empty(int(h.sum()), dtype=torch.uint8, device=dev)
                with _lib.lock:
                    _lib.check(L.ms_tiff_pack_dev(slots.data_ptr(), slot, sizes.data_ptr(), offs.data_ptr(), n,
                                                  out.data_ptr(), st), "write_band")
                sizes_h.append(h)
                packed.append(out)

            t0, t1 = plan["inner"]
            for t in range(t0, t1, per):
                a, b = t * TILE, min(min(t + per, t1) * TILE, rows)
                encode(d[a - r0:b - r0])
            if plan["cross"] is not None:
                a = plan["cross"] * TILE
                slab = torch.empty((min(a + TILE, rows) - a, cols), dtype=d.dtype, device=dev)
                slab[:r1 - a] = d[a - r0:]
                slab.view(torch.uint8)[r1 - a:] = recv
                encode(slab)
            ev[1].record(stream)
        except (RuntimeError, ValueError, OSError, MemoryError) as e:
            fail[0] = e
        agree()
        # the container: every rank computes the same one from the gathered sizes
        mine = np.concatenate(sizes_h) if sizes_h else np.zeros(0, np.int64)
        parts = comm.all_gather_var(torch.from_numpy(mine).to(dev))
        band_tiles = [int(x.numel()) for x in parts]
        tile_sizes = torch.cat(parts).cpu().numpy()
        head, tail = build_tiff(rows, cols, dtype, predictor, tile_sizes, self.transform, self.crs, self.nodata)
        data = int(tile_sizes.sum())
        size = len(head) + data + len(tail)
        offset = band_file_offsets(tile_sizes, band_tiles)[rank]
        if rank == 0:
            try:
                with open(self.filepath, "wb") as f:
                    made[0] = True
                    f.write(head)
                    f.truncate(size)
            except OSError as e:
                fail[0] = e
        agree()
        try:
            fd = os.open(self.filepath, os.O_WRONLY)
            try:
                self._pwrite_device(fd, packed, offset, dev)
                if rank == 0:
                    _pwrite_all(fd, memoryview(tail), len(head) + data)
            finally:
                os.close(fd)
        except (RuntimeError, ValueError, OSError, MemoryError) as e:
            fail[0] = e
        agree()
        ev[1].synchronize()
        self.stats = {"raw_bytes": rows * cols * es, "file_bytes": size, "tiles": len(tile_sizes),
                      "band_tiles": band_tiles[rank], "band_bytes": int(mine.sum()),
                      "exchanged_bytes": 0 if recv is None else recv.numel(), "encode_ms": ev[0].elapsed_time(ev[1])}

    def _pwrite_device(self, fd, parts, offset, dev):
        """The device tensors `parts` (uint8), one after the other, to `fd` at `offset`: device-to-host copies into two
        pinned buffers of at most STAGE_BYTES taking turns, each copy overlapping the file write of the other buffer."""
        import torch
        total = sum(int(p.numel()) for p in parts)
        if total == 0:
            return
        cap = min(self.STAGE_BYTES, total)
        bufs = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        pieces = [(p, a, min(a + cap, int(p.numel()))) for p in parts for a in range(0, int(p.numel()), cap)]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        done = [None, None]

        def issue(i):
            p, a, b = pieces[i]
            with torch.cuda.stream(side):
                bufs[i % 2][:b - a].copy_(p[a:b], non_blocking=True)
                done[i % 2] = torch.cuda.Event()
                done[i % 2].record(side)

        issue(0)
        pos = offset
        for i, (p, a, b) in enumerate(pieces):
            if i + 1 < len(pieces):
                issue(i + 1)            # the buffer of piece i - 1, whose write has returned
            done[i % 2].synchronize()
            _pwrite_all(fd, memoryview(bufs[i % 2].numpy())[:b - a], pos)
            pos += b - a


def _pwrite_all(fd, view, pos):
    while len(view):
        n = os.pwrite(fd, view, pos)
        if n <= 0:
            raise OSError("short write at byte %d" % pos)
        view, pos = view[n:], pos + n
