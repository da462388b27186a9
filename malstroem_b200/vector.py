"""SURVEY.md §8(f4): the raster half of malstroem/vector.py on the device.

`vectorize_labels_file` (vector.py:42-87) runs `gdal.Polygonize(band, band.GetMaskBand(), layer, 0, ['8CONNECTED=8'])`
on a label raster and yields one GeoJSON feature per polygon.  Here the file is decoded on the device (io.py), the
rings are built by csrc/polygon.cu (ms_polygonize*: boundary edges, ring leaders and positions by pointer doubling,
corner compaction, regions by union-find) and this module groups rings into features and applies the geotransform.

Same features as GDAL's: one polygon per 8-connected region of equal value (value 0 included: the reference's fixture
gives 113 = 104 labels + 9 background regions, tests/test_vector.py:18-20), holes as inner rings, vertices at pixel
corners in world coordinates, only where the outline turns.  NOT pinned against GDAL (absent here): the order of the
features (here: by the region's first cell in raster order; GDAL: by the row that completes the polygon), the start
vertex and the winding of each ring.  What the tests pin instead: the reference's own feature count, exact equality of
the rasterised features with the raster, and ring-for-ring equality with an independent CPU walk (oracle/polygonize.py).
"""
import numpy as np

from . import _lib


def transform_cell_to_world(cell, geotransform):
    """vector.py:21-39 — world coordinates of the centre of cell (row, col); `gdal.ApplyGeoTransform`'s arithmetic."""
    row, col = cell[:2]
    px, ln = col + 0.5, row + 0.5
    x = geotransform[0] + px * geotransform[1] + ln * geotransform[2]
    y = geotransform[3] + px * geotransform[4] + ln * geotransform[5]
    return (x, y)


class Rings(object):
    """Rings of a polygonised raster: ring k owns vertices offset[k]:offset[k+1] of (vrow, vcol) — lattice corners,
    the region on the right-hand side walking the ring on the screen, no repeated closing vertex."""

    def __init__(self, shape, offset, value, cell, region, hole, vrow, vcol, nedges, first_id=0):
        """first_id: the id of the first feature (polygonize_band: the polygons of the lower ranks come first)."""
        self.shape = shape
        self.offset, self.value, self.cell, self.region, self.hole = offset, value, cell, region, hole
        self.vrow, self.vcol = vrow, vcol
        self.nedges = nedges
        self.first_id = first_id

    def __len__(self):
        return len(self.value)

    def polygons(self):
        """[(value, [exterior ring index, hole ring index, ...]), ...] ordered by the region's first cell."""
        ext = np.flatnonzero(self.hole == 0)
        holes = np.flatnonzero(self.hole != 0)
        # an exterior ring's leader cell IS its region's first cell, and the rings come sorted by leader cell
        ext_region = self.region[ext]
        if len(ext) > 1 and not np.all(np.diff(ext_region) > 0):
            raise RuntimeError("polygonize: exterior rings are not one per region")
        where = np.searchsorted(ext_region, self.region[holes])
        if len(holes) and (np.any(where >= len(ext)) or np.any(ext_region[np.minimum(where, len(ext) - 1)] != self.region[holes])):
            raise RuntimeError("polygonize: a hole without an exterior ring")
        order = np.argsort(where, kind="stable")
        first = np.searchsorted(where[order], np.arange(len(ext) + 1))
        out = []
        for k in range(len(ext)):
            out.append((int(self.value[ext[k]]), [int(ext[k])] + [int(h) for h in holes[order[first[k]:first[k + 1]]]]))
        return out

    def ring_lattice(self, k):
        a, b = int(self.offset[k]), int(self.offset[k + 1])
        return self.vrow[a:b], self.vcol[a:b]

    def features(self, geotransform=None, id_attribute="bspot_id"):
        """GeoJSON features as OGR's Feature.ExportToJson gives them (vector.py:78-80)."""
        gt = geotransform if geotransform is not None else (0.0, 1.0, 0.0, 0.0, 0.0, 1.0)
        c, r = self.vcol.astype(np.float64), self.vrow.astype(np.float64)
        x = gt[0] + c * gt[1] + r * gt[2]
        y = gt[3] + c * gt[4] + r * gt[5]
        for fid, (value, rings) in enumerate(self.polygons(), start=self.first_id):
            coords = []
            for k in rings:
                a, b = int(self.offset[k]), int(self.offset[k + 1])
                ring = [[float(x[i]), float(y[i])] for i in range(a, b)]
                ring.append(ring[0])
                coords.append(ring)
            yield {"type": "Feature", "geometry": {"type": "Polygon", "coordinates": coords},
                   "properties": {id_attribute: value}, "id": fid}


def _fetch(shape, counts):
    nr, nv, ne = int(counts[0]), int(counts[1]), int(counts[2])
    offset = np.zeros(nr + 1, dtype=np.int64)
    value = np.zeros(nr, dtype=np.int32)
    cell = np.zeros(nr, dtype=np.int64)
    region = np.zeros(nr, dtype=np.int64)
    hole = np.zeros(nr, dtype=np.uint8)
    vrow = np.zeros(nv, dtype=np.int32)
    vcol = np.zeros(nv, dtype=np.int32)
    _lib.check(_lib.lib().ms_polygonize_fetch(_lib.ptr(offset), _lib.ptr(value), _lib.ptr(cell), _lib.ptr(region),
                                              _lib.ptr(hole), _lib.ptr(vrow), _lib.ptr(vcol)), "polygonize")
    return Rings(shape, offset, value, cell, region, hole, vrow, vcol, ne)


def _nodata_args(nodata):
    if nodata is None:
        return 0, 0
    if float(nodata) != int(nodata) or not (-2 ** 31 <= int(nodata) < 2 ** 31):
        return 0, 0          # no int32 cell can equal it
    return 1, int(nodata)


def polygonize_labels(labels, connect8=True, nodata=None):
    """Rings of a 2-D int32 label raster (numpy).  gdal.Polygonize's region rule; see the module docstring."""
    if not isinstance(labels, np.ndarray) or labels.ndim != 2:
        raise ValueError("polygonize_labels: a 2-D numpy array is required")
    if labels.dtype != np.int32:
        if not np.issubdtype(labels.dtype, np.integer) and labels.dtype != np.bool_:
            raise ValueError("Buffer dtype mismatch, expected an integer raster but got %s" % labels.dtype)
        labels = labels.astype(np.int32)
    labels = np.ascontiguousarray(labels)
    if labels.size == 0:
        raise ValueError("Width or height of processing area is zero")
    has, nd = _nodata_args(nodata)
    counts = np.zeros(3, dtype=np.int64)
    with _lib.lock:
        _lib.check(_lib.lib().ms_polygonize(_lib.ptr(labels), labels.shape[0], labels.shape[1], 1 if connect8 else 0,
                                            has, nd, _lib.ptr(counts)), "polygonize")
        _lib.track(labels)
        return _fetch(labels.shape, counts)


def polygonize_labels_device(labels, connect8=True, nodata=None):
    """The same for a 2-D int32 CUDA tensor (e.g. RasterReader.read_device or RasterPipeline's labels)."""
    import torch
    if labels.dim() != 2 or labels.dtype != torch.int32 or not labels.is_cuda:
        raise ValueError("polygonize_labels_device: a 2-D int32 CUDA tensor is required")
    labels = labels.contiguous()
    has, nd = _nodata_args(nodata)
    counts = np.zeros(3, dtype=np.int64)
    stream = torch.cuda.current_stream(labels.device).cuda_stream
    with _lib.lock:
        _lib.check(_lib.lib().ms_polygonize_dev(labels.data_ptr(), labels.shape[0], labels.shape[1],
                                                1 if connect8 else 0, has, nd, _lib.ptr(counts), stream), "polygonize")
        return _fetch(tuple(labels.shape), counts)


def vectorize_labels_file(labeled_file, id_attribute="bspot_id"):
    """vector.py:42-87 — yields one GeoJSON feature per polygon of the label raster in `labeled_file` (GeoTIFF)."""
    from . import io
    reader = io.RasterReader(labeled_file)
    labels = reader.read_device()
    import torch
    if labels.dtype != torch.int32:
        if labels.dtype.is_floating_point:
            raise ValueError("vectorize_labels_file: an integer raster is required, got %s" % labels.dtype)
        labels = labels.to(torch.int32)
    rings = polygonize_labels_device(labels, connect8=True, nodata=reader.nodata)
    del labels
    for feature in rings.features(reader.transform, id_attribute):
        yield feature


# ---- row bands (DESIGN.md §8(f4)) ------------------------------------------------------------------------------------
class _Phases(object):
    """Library calls and allocations of one phase; a failure on any rank makes every rank raise after the phase
    (a max all-reduce of the flag), so that no rank waits in a collective the failed one never reaches."""

    def __init__(self, comm, dev):
        self.comm, self.dev, self.err = comm, dev, None

    def run(self, fn, *args):
        if self.err is None:
            try:
                return fn(*args)
            except (RuntimeError, ValueError, IndexError) as e:       # torch's out-of-memory error is a RuntimeError
                self.err = e
        return None

    def call(self, name, *args):
        def go():
            with _lib.lock:
                _lib.check(getattr(_lib.lib(), name)(*args), name)
        self.run(go)

    def sync(self, extra=None):
        import torch
        flags = torch.tensor([1 if self.err is not None else 0] + ([] if extra is None else [int(extra)]),
                             dtype=torch.int64, device=self.dev)
        got = self.comm.all_reduce(flags, "max").tolist()
        if got[0]:
            if self.err is not None:
                raise self.err
            raise RuntimeError("polygonize_band: a phase failed on another band")
        return got[1:]


def polygonize_band(comm, labels, r0, rows, connect8=True, nodata=None):
    """Rings of a label raster split into row bands, one per rank of `comm` (bands.ThreadComm or bands.DistComm);
    collective.  labels: this band's rows [r0, r0 + labels.shape[0]) as an int32 CUDA tensor; rows: the raster's row
    count; the bands must tile the raster in rank order.  Returns this rank's Rings: every polygon whose region's first
    cell lies in the band, its exterior ring and all of its holes, sorted by leader (the ring's lowest global edge
    number), with global `cell`, `region` and `vrow` and `first_id` after the lower ranks' polygons.  Concatenated
    over the ranks in rank order, polygons() and the rings' vertices are those of polygonize_labels_device on the
    whole raster.  The phases (DESIGN.md §8(f4)): edges counted and numbered in the band (halo label rows; one gather
    of the counts), successors (the neighbours' first edge numbers and side masks of their edge rows), rings closed in
    the band resolved as on one GPU and the others cut into segments, the segments of all bands gathered and linked
    into rings on every rank, regions merged across band edges, and every ring's vertices sent to the band that owns
    its polygon (always the same or a lower rank)."""
    import ctypes
    import torch
    from . import bands
    if labels.dim() != 2 or labels.dtype != torch.int32 or not labels.is_cuda:
        raise ValueError("polygonize_band: a 2-D int32 CUDA tensor is required")
    labels = labels.contiguous()
    dev = labels.device
    i64, i32, u8 = torch.int64, torch.int32, torch.uint8
    h, C = int(labels.shape[0]), int(labels.shape[1])
    r0, R, G, g = int(r0), int(rows), comm.size, comm.rank
    got = comm.all_gather(torch.tensor([r0, r0 + h, C], dtype=i64, device=dev)).cpu().tolist()
    if not (got[0][0] == 0 and got[-1][1] == R and all(x[1] > x[0] and x[2] == C and C >= 1 for x in got)
            and all(got[k][0] == got[k - 1][1] for k in range(1, G))):
        raise ValueError("polygonize_band: the bands (r0, r1, cols) %s do not tile the rows of one raster in rank order"
                         % got)
    starts = torch.tensor([x[0] for x in got], dtype=i64, device=dev)
    has, nd = _nodata_args(nodata)
    c8 = 1 if connect8 else 0
    halo = (1 if g > 0 else 0) | (2 if g + 1 < G else 0)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    ph = _Phases(comm, dev)
    P = ctypes.c_void_p

    def p(t):
        return P(t.data_ptr())

    # 1. count and number: halo label rows, edges per cell, the global base of the band's edge numbers
    ext = torch.empty((h + 2, C), dtype=i32, device=dev)
    ext[1:h + 1] = labels
    above, below = comm.exchange(labels[0].contiguous(), labels[h - 1].contiguous())
    if above is not None:
        ext[0] = above
    if below is not None:
        ext[h + 1] = below
    lab = P(ext[1].data_ptr())
    grid = (lab, h, C, halo, c8, has, nd)
    ne = ctypes.c_int64(0)
    bufs = ph.run(lambda: (torch.empty(h * C, dtype=i32, device=dev), torch.empty(2 * C, dtype=i32, device=dev),
                           torch.empty(2 * C, dtype=u8, device=dev)))
    if bufs is not None:
        eoff, row_eoff, row_mask = bufs
        ph.call("ms_band_poly_count_dev", *grid, p(eoff), ctypes.byref(ne), p(row_eoff), p(row_mask), st)
    ph.sync()
    E = ne.value
    counts = comm.all_gather(torch.tensor([E], dtype=i64, device=dev)).view(-1).tolist()
    base = sum(counts[:g])
    nb = (1 if g > 0 else 0) + (1 if g + 1 < G else 0)
    stats = {"edges": E, "exchange_bytes": {"halo_labels": nb * C * 4, "edge_rows": nb * C * 16}}    # sent by this rank
    # 2. successors: the neighbours' (global first edge, side mask) of their edge rows
    up = torch.stack([row_eoff[:C].long() + base, row_mask[:C].long()])
    down = torch.stack([row_eoff[C:].long() + base, row_mask[C:].long()])
    a, b = comm.exchange(up, down)
    halo_eoff = torch.zeros(2 * C, dtype=i64, device=dev)
    halo_mask = torch.zeros(2 * C, dtype=u8, device=dev)
    for k, x in ((0, a), (1, b)):
        if x is not None:
            halo_eoff[k * C:(k + 1) * C] = x[0]
            halo_mask[k * C:(k + 1) * C] = x[1].to(u8)
    S4 = 4 * C
    exit_edge = torch.full((S4,), -1, dtype=i32, device=dev)
    exit_next = torch.zeros(S4, dtype=i64, device=dev)
    exit_corner = torch.zeros(S4, dtype=u8, device=dev)
    seg_entry = torch.zeros(S4, dtype=i32, device=dev)
    seg_min = torch.zeros(S4, dtype=i32, device=dev)
    seg_tmin = torch.zeros(S4, dtype=i32, device=dev)
    counts2 = np.zeros(2, dtype=np.int64)
    if E:
        bufs = ph.run(lambda: [torch.empty(E, dtype=t, device=dev) for t in (i32, i32, i64, i64)])
        if bufs is not None:
            ecell, succ, lead, rank = bufs
            ph.call("ms_band_poly_edges_dev", *grid, p(eoff), E, p(halo_eoff), p(halo_mask), p(ecell), p(succ), p(lead),
                    p(rank), p(exit_edge), p(exit_next), p(exit_corner), st)
    ph.sync()
    del eoff
    # 3. local resolve: closed rings as on one GPU, the rest cut into segments
    if E:
        bufs = ph.run(lambda: [torch.empty(E, dtype=i32, device=dev) for _ in range(7)])
        if bufs is not None:
            ishead, uidx, ulen, ustart, placed, corner, vidx = bufs
            ph.call("ms_band_poly_place_dev", C, E, p(ecell), p(succ), p(lead), p(rank), p(ishead), p(uidx), p(ulen),
                    p(ustart), p(placed), p(corner), p(vidx), p(seg_entry), p(seg_min), p(seg_tmin),
                    _lib.ptr(counts2), st)
    ph.sync()
    U, NV = int(counts2[0]), int(counts2[1])
    unit = {}
    root_rows = torch.full((2 * C,), -1, dtype=i64, device=dev)
    vloc = torch.zeros(0, dtype=i64, device=dev)
    if E:
        def alloc():
            vr = torch.empty(max(NV, 1), dtype=i32, device=dev)
            vc = torch.empty(max(NV, 1), dtype=i32, device=dev)
            for k, t in (("head", i32), ("len", i32), ("vstart", i32), ("vcount", i32), ("value", i32), ("root", i64),
                         ("slot", i32)):
                unit[k] = torch.empty(U, dtype=t, device=dev)
            return vr, vc
        got_v = ph.run(alloc)
        if got_v is not None:
            vr, vc = got_v
            ph.call("ms_band_poly_emit_dev", *grid, r0, E, p(ecell), p(lead), p(ishead), p(uidx), p(ulen), p(ustart),
                    p(placed), p(corner), p(vidx), NV, p(vr), p(vc), p(unit["head"]), p(unit["len"]), p(unit["vstart"]),
                    p(unit["vcount"]), p(unit["value"]), p(unit["root"]), p(unit["slot"]), p(root_rows), st)
    ph.sync()
    if E:
        vloc = (vr[:NV].long() << 32) | vc[:NV].long()
        del vr, vc, placed, corner, ishead, uidx, ulen, succ, lead, rank
    # 5. regions across band edges (the merge runs on the host of every rank, O(bands * cols))
    rows_all = comm.all_gather(torch.cat([root_rows, torch.stack([labels[0], labels[h - 1]]).view(-1).long()])).cpu()
    rows_all = rows_all.numpy()
    top = np.ascontiguousarray(rows_all[:, :C])
    bot = np.ascontiguousarray(rows_all[:, C:2 * C])
    vtop = np.ascontiguousarray(rows_all[:, 2 * C:3 * C].astype(np.int32))
    vbot = np.ascontiguousarray(rows_all[:, 3 * C:].astype(np.int32))
    capn = 2 * G * C
    m_root, m_glob, nm = np.empty(capn, dtype=np.int64), np.empty(capn, dtype=np.int64), ctypes.c_int64(0)
    with _lib.lock:
        _lib.check(_lib.lib().ms_cc_boundary_merge_values(G, C, _lib.ptr(top), _lib.ptr(bot), _lib.ptr(vtop),
                                                           _lib.ptr(vbot), c8, _lib.ptr(m_root), _lib.ptr(m_glob), capn,
                                                           ctypes.byref(nm)), "ms_cc_boundary_merge_values")
    mr = torch.from_numpy(m_root[:nm.value]).to(dev)
    mg = torch.from_numpy(m_glob[:nm.value]).to(dev)

    def region_of(x):
        if mr.numel() == 0:
            return x
        at = torch.searchsorted(mr, x).clamp(max=mr.numel() - 1)
        return torch.where(mr[at] == x, mg[at], x)

    def owner_of(region):
        return torch.searchsorted(starts, region // C, right=True) - 1

    # 4. crossing rings: every band's segments, linked into rings on every rank
    if U:
        ec = ecell[unit["head"].long()].long() & 0xffffffff
        head_gid = unit["head"].long() + base
        hcell = ec >> 2
        hside = ec & 3
        region = region_of(unit["root"])
        seg = unit["slot"] >= 0
        sl = unit["slot"][seg].long()
        mnl = seg_min[sl].long()
        mec = ecell[mnl].long() & 0xffffffff
        tmin = seg_tmin[sl].long()
        kmin = vidx[ustart[unit["head"][seg].long()].long() + tmin].long() - unit["vstart"][seg].long()
        rec = torch.stack([head_gid[seg], exit_next[sl], unit["len"][seg].long(), mnl + base, tmin,
                           unit["vcount"][seg].long(), kmin, exit_corner[sl].long(), unit["value"][seg].long(),
                           region[seg], r0 * C + (mec >> 2), mec & 3], dim=1)
    else:
        rec = torch.zeros((0, 12), dtype=i64, device=dev)
    allrec = comm.all_gather_var(rec)
    myfirst = sum(x.shape[0] for x in allrec[:g])
    allrec = torch.cat(allrec)
    stats["exchange_bytes"]["segments"] = int(rec.numel()) * 8 * (G - 1)
    stats["segments"] = int(allrec.shape[0])
    sol = ph.run(bands.ring_segments, *[allrec[:, k].contiguous() for k in range(8)])
    ph.sync()
    fs = sol["first"]
    # ring records (leader, L, V, value, cell, region, hole) of the crossing rings, complete on every rank
    xring = torch.stack([sol["leader"], sol["L"], sol["V"], allrec[fs, 8], allrec[fs, 10], allrec[fs, 9],
                         (allrec[fs, 11] != 0).long()], dim=1)
    xowner = owner_of(xring[:, 5])
    # 6. assemble at the owner: closed rings' records and every unit's vertices go to the band owning the polygon
    chunks = [[] for _ in range(G)]
    if U:
        closed = ~seg
        uV = unit["vcount"].long()
        lead_of = head_gid.clone()
        start_of = torch.zeros(U, dtype=i64, device=dev)
        dest = owner_of(region)
        mine = sol["ring"][myfirst:myfirst + int(seg.sum())]
        if mine.numel():
            my_ce = sol["centry"][myfirst:myfirst + mine.numel()]
            my_vo = sol["voff"][myfirst:myfirst + mine.numel()]
            Vm = sol["V"][mine].clamp(min=1)
            lead_of[seg] = sol["leader"][mine]
            start_of[seg] = (my_vo + my_ce) % Vm
            dest[seg] = xowner[mine]
            # the entry's start vertex, where the ring turns onto the entry edge
            eh, es = hcell[seg], hside[seg]
            evert = ((r0 + eh // C + (es >= 2).long()) << 32) | (eh % C + ((es == 1) | (es == 2)).long())
            ent = my_ce != 0
            ent_blk = torch.stack([sol["leader"][mine], my_vo % Vm, torch.ones_like(my_vo)], dim=1)[ent]
            ent_dest, ent_vert = dest[seg][ent], evert[ent]
        else:
            ent_blk = torch.zeros((0, 3), dtype=i64, device=dev)
            ent_dest = ent_vert = torch.zeros(0, dtype=i64, device=dev)
        crec = torch.stack([head_gid, unit["len"].long(), uV, unit["value"].long(), r0 * C + hcell, region,
                            (hside != 0).long()], dim=1)
        blk = torch.stack([lead_of, start_of, uV], dim=1)
        vdest = torch.repeat_interleave(dest, uV)
        for r in range(G):
            cr = crec[closed & (dest == r)]
            bk = torch.cat([blk[dest == r], ent_blk[ent_dest == r]])
            vv = torch.cat([vloc[vdest == r], ent_vert[ent_dest == r]])
            chunks[r] = torch.cat([torch.tensor([cr.shape[0], bk.shape[0]], dtype=i64, device=dev), cr.reshape(-1),
                                   bk.reshape(-1), vv])
    else:
        chunks = [torch.zeros(2, dtype=i64, device=dev) for _ in range(G)]
    recv = comm.all_to_all_var(chunks)
    stats["exchange_bytes"]["to_owner"] = sum(int(c.numel()) * 8 for r, c in enumerate(chunks) if r != g)
    recs, blks, verts = [xring[xowner == g]], [], []
    for c in recv:
        nr_, nb_ = int(c[0]), int(c[1])
        recs.append(c[2:2 + 7 * nr_].view(nr_, 7))
        blks.append(c[2 + 7 * nr_:2 + 7 * nr_ + 3 * nb_].view(nb_, 3))
        verts.append(c[2 + 7 * nr_ + 3 * nb_:])
    recs, blks, verts = torch.cat(recs), torch.cat(blks), torch.cat(verts)
    recs = recs[torch.argsort(recs[:, 0])]
    nrings = recs.shape[0]
    voff = torch.zeros(nrings + 1, dtype=i64, device=dev)
    voff[1:] = torch.cumsum(recs[:, 2], 0)
    out = torch.zeros(int(voff[-1]), dtype=i64, device=dev)
    bad = int(blks[:, 2].sum()) != out.numel() if blks.numel() else out.numel() != 0
    if blks.shape[0] and nrings:
        k = torch.searchsorted(recs[:, 0].contiguous(), blks[:, 0].contiguous()).clamp(max=nrings - 1)
        bad = bad or not bool((recs[k, 0] == blks[:, 0]).all())
        bid = torch.repeat_interleave(torch.arange(blks.shape[0], device=dev), blks[:, 2])
        first = torch.cumsum(blks[:, 2], 0) - blks[:, 2]
        j = torch.arange(verts.numel(), device=dev) - first[bid]
        kb = k[bid]
        out[voff[kb] + (blks[bid, 1] + j) % recs[kb, 2].clamp(min=1)] = verts
    npoly = int((recs[:, 6] == 0).sum())
    polys = comm.all_gather(torch.tensor([npoly, 1 if bad else 0], dtype=i64, device=dev)).cpu()
    if int(polys[:, 1].max()):
        raise RuntimeError("polygonize_band: the ring pieces received do not fill the rings (rank %s)"
                           % polys[:, 1].tolist())
    recs_h, out_h = recs.cpu().numpy(), out.cpu().numpy()
    rings = Rings((R, C), voff.cpu().numpy(), recs_h[:, 3].astype(np.int32), recs_h[:, 4].copy(), recs_h[:, 5].copy(),
                  recs_h[:, 6].astype(np.uint8), (out_h >> 32).astype(np.int32), (out_h & 0xffffffff).astype(np.int32),
                  int(recs_h[:, 1].sum()), first_id=int(polys[:g, 0].sum()))
    rings.band_stats = stats
    return rings


def vectorize_labels_band(comm, labeled_file, id_attribute="bspot_id", device=0):
    """vectorize_labels_file on row bands, collective over `comm`: every rank reads its rows
    (bands.band_rows(rows, comm.size)) of `labeled_file` and yields the GeoJSON features of the polygons it owns,
    with global ids; concatenated in rank order they are vectorize_labels_file's features."""
    import torch
    from . import bands, io
    reader = io.RasterReader(labeled_file)
    r0, r1 = bands.band_rows(reader._info.rows, comm.size)[comm.rank]
    labels = reader.read_rows(r0, r1, device=device)
    if labels.dtype != torch.int32:
        if labels.dtype.is_floating_point:
            raise ValueError("vectorize_labels_band: an integer raster is required, got %s" % labels.dtype)
        labels = labels.to(torch.int32)
    rings = polygonize_band(comm, labels, r0, reader._info.rows, connect8=True, nodata=reader.nodata)
    del labels
    for feature in rings.features(reader.transform, id_attribute):
        yield feature
