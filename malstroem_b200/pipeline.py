"""Device-resident whole path: DEM in HBM -> every raster and per-label table of the hot path in HBM
(`ms_pipeline_dev`), plus a host-buffer front end that adds the H2D / D2H copies.

torch is used for what it is good at here — owning device / pinned memory and the CUDA stream; every
kernel that runs is from libmalstroem_b200.so.
"""
import ctypes

import numpy as np
import torch

from . import _lib

RASTERS = (("filled", torch.float32), ("depths", torch.float32), ("fnf", torch.float64), ("flowdir", torch.uint8),
           ("accum", torch.float64), ("labels", torch.int32), ("wsheds", torch.int32))
TABLES = (("st_min", torch.float64), ("st_max", torch.float64), ("st_sum", torch.float64), ("st_count", torch.int64),
          ("ws_count", torch.int64), ("ppmin_value", torch.float64), ("ppmin_row", torch.int64),
          ("ppmin_col", torch.int64), ("ppmax_value", torch.float64), ("ppmax_row", torch.int64),
          ("ppmax_col", torch.int64))
STAT_NAMES = ("boruvka_rounds", "catchments", "noflat_rounds", "noflat_tile_visits", "noflat_reverify",
              "fill_jump_rounds", "wshed_jump_rounds", "noflat_sweep_rounds")


class RasterPipeline(object):
    """Buffers for one `rows x cols` raster on one GPU and the call that fills them."""

    # rasters the host-buffer front end brings back: what the reference's tools write (dem.py:67-93: filled, flowdir,
    # depths, accum; bluespots.py:169,189: bluespot labels, watersheds).  The no-flats surface is an intermediate there
    # (dem.py:80-86 computes it for the flow directions and drops it), so it stays in HBM unless asked for.
    HOST_RASTERS = ("filled", "depths", "flowdir", "accum", "labels", "wsheds")

    def __init__(self, rows, cols, device=0, with_accum=True, table_capacity=None):
        if not torch.cuda.is_available():
            raise RuntimeError("malstroem_b200.pipeline needs a CUDA device (there is no CPU fallback)")
        self.rows, self.cols = int(rows), int(cols)
        self.device = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        self.with_accum = with_accum
        n = self.rows * self.cols
        # 8-connected components of a raster: at most ceil(rows/2)*ceil(cols/2)
        cap = ((self.rows + 1) // 2) * ((self.cols + 1) // 2) + 1
        self.table_capacity = int(table_capacity) if table_capacity else cap
        with _lib.lock:
            _lib.check(_lib.lib().ms_init(self.device.index or 0), "ms_init")
        self.dem = torch.empty((self.rows, self.cols), dtype=torch.float32, device=self.device)
        self.out = {}
        for name, dt in RASTERS:
            if name == "accum" and not with_accum:
                continue
            self.out[name] = torch.empty((self.rows, self.cols), dtype=dt, device=self.device)
        self.tables = {}
        for name, dt in TABLES:
            if name.startswith("ppmax") and not with_accum:
                continue
            self.tables[name] = torch.empty((self.table_capacity,), dtype=dt, device=self.device)
        self.io = _lib.MsRasters()
        self.io.rows, self.io.cols = self.rows, self.cols
        self.io.dem = self.dem.data_ptr()
        for name, t in self.out.items():
            setattr(self.io, name, t.data_ptr())
        for name, t in self.tables.items():
            setattr(self.io, name, t.data_ptr())
        self.io.table_capacity = self.table_capacity
        self.nlabels = 0
        self.stats = {}
        self._host = None

    # ---- device-resident run (bench `value`) ---------------------------------------------------------
    def run(self, dem=None, host_out=None, bluespot_filter=None, cell_area=1.0):
        """dem: optional cuda float32 tensor of the pipeline's shape (else self.dem is used as is).
        host_out: optional _lib.MsHostOut of pinned host buffers the finished rasters are shipped to while the later
        stages run (complete after ms_copies_wait).
        bluespot_filter: optional `-filter` text of the reference's CLI (malstroem_b200.bluespot_filter), evaluated on
        the raw bluespots with `cell_area` (the area of one cell, for `area` and `volume`); every raster and table
        from the labels on is then the filtered one (bluespots.py:158-206), and stats["bluespots_raw"] holds the raw
        count.  None or "" runs without a filter."""
        from . import bluespot_filter as _bf
        prog = _bf.compile_filter(bluespot_filter)
        filt = prog.struct(cell_area) if prog is not None else None
        if dem is not None and dem.data_ptr() != self.dem.data_ptr():
            self.dem.copy_(dem)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        nraw = ctypes.c_int64(0)
        with _lib.lock:
            if filt is not None:
                _lib.check(_lib.lib().ms_pipeline_filtered_host_dev(
                    ctypes.byref(self.io), ctypes.byref(host_out) if host_out is not None else None, ctypes.byref(filt),
                    ctypes.byref(nraw), ctypes.c_void_p(stream)), "ms_pipeline_filtered_host_dev")
            elif host_out is None:
                _lib.check(_lib.lib().ms_pipeline_dev(ctypes.byref(self.io), ctypes.c_void_p(stream)), "ms_pipeline_dev")
            else:
                _lib.check(_lib.lib().ms_pipeline_host_dev(ctypes.byref(self.io), ctypes.byref(host_out),
                                                           ctypes.c_void_p(stream)), "ms_pipeline_host_dev")
        self.nlabels = int(self.io.nlabels)
        self.stats = dict(zip(STAT_NAMES, [int(v) for v in self.io.stats]))
        if filt is not None:
            self.stats["bluespots_raw"] = int(nraw.value)
        self.short, self.diag = float(self.io.short_eps), float(self.io.diag_eps)
        return self

    def table(self, name):
        return self.tables[name][: self.nlabels + 1]

    # ---- the bluespot network and rain events on the finished tables (SURVEY.md §8(f1,f2)) -----------
    def network(self, cell_area=1.0, events_mm=(), use_accum_pourpoints=False, sum_mode=None):
        """What StreamTool + RainTool compute from BluespotTool's output (streams.py:66-100, rain.py:60-79), device
        resident: returns dict of cuda tensors — `parent` int32 [nlabels+1] (downstream bluespot, -1 = none) and
        rainv / spillv / v / pctv float64 [n_events, nlabels+1] (pctv NaN where the capacity is 0)."""
        from . import network as _network
        n = self.nlabels + 1
        mm = np.ascontiguousarray(np.atleast_1d(np.asarray(events_mm, dtype=np.float64)))
        ne = int(mm.size)
        if ne > 16:
            raise ValueError("network: at most 16 rain events per pass")
        res = {"parent": torch.empty((n,), dtype=torch.int32, device=self.device)}
        for k in ("rainv", "spillv", "v", "pctv"):
            res[k] = torch.empty((ne, n), dtype=torch.float64, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with _lib.lock:
            _lib.check(_lib.lib().ms_bluespot_network_dev(
                ctypes.byref(self.io), float(cell_area), 1 if use_accum_pourpoints else 0, ne, _lib.ptr(mm),
                _network.SUM_MODE if sum_mode is None else sum_mode, res["parent"].data_ptr(),
                res["rainv"].data_ptr(), res["spillv"].data_ptr(), res["v"].data_ptr(), res["pctv"].data_ptr(),
                ctypes.c_void_p(stream)), "ms_bluespot_network_dev")
        return res

    # ---- water levels and depth rasters after the rain events (csrc/flood.cu) -------------------------
    def flood(self, net, cell_area):
        """Water level and wet-cell count of every bluespot per event of `net` (the dict `network()` returned, with
        the same cell_area), device resident: dict of cuda tensors `level` float64 and `wet` int64 [n_events,
        nlabels+1].  Level-pool approximation, see malstroem_b200.flood."""
        v = net["v"].contiguous()
        n = self.nlabels + 1
        if v.dim() != 2 or v.shape[1] != n or v.dtype != torch.float64 or v.device != self.device:
            raise ValueError("flood: net['v'] must be a float64 tensor [n_events, %d] on %s" % (n, self.device))
        ne = int(v.shape[0])
        res = {"level": torch.empty((ne, n), dtype=torch.float64, device=self.device),
               "wet": torch.empty((ne, n), dtype=torch.int64, device=self.device)}
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with _lib.lock:
            _lib.check(_lib.lib().ms_flood_levels_dev(
                self.dem.data_ptr(), self.out["filled"].data_ptr(), self.out["labels"].data_ptr(), self.rows,
                self.cols, self.nlabels, self.tables["st_sum"].data_ptr(), float(cell_area), ne, v.data_ptr(),
                res["level"].data_ptr(), res["wet"].data_ptr(), ctypes.c_void_p(stream)), "ms_flood_levels_dev")
        return res

    def water_depth(self, level_row, out=None):
        """Water depth raster (cuda float32, rows x cols) of one event: `level_row` is one row of flood()'s `level`.
        Rasters are made one event at a time: at 32768^2 each is 4 GB."""
        n = self.nlabels + 1
        level_row = level_row.contiguous()
        if level_row.shape != (n,) or level_row.dtype != torch.float64 or level_row.device != self.device:
            raise ValueError("water_depth: level_row must be a float64 tensor [%d] on %s" % (n, self.device))
        if out is None:
            out = torch.empty((self.rows, self.cols), dtype=torch.float32, device=self.device)
        elif (out.shape != (self.rows, self.cols) or out.dtype != torch.float32 or not out.is_contiguous()
              or out.device != self.device):
            raise ValueError("water_depth: out must be a contiguous float32 tensor of the raster's shape on %s" % self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with _lib.lock:
            _lib.check(_lib.lib().ms_water_depth_dev(
                self.dem.data_ptr(), self.out["filled"].data_ptr(), self.out["labels"].data_ptr(), self.rows,
                self.cols, self.nlabels, level_row.data_ptr(), out.data_ptr(), ctypes.c_void_p(stream)),
                "ms_water_depth_dev")
        return out

    # ---- host-buffer run (bench `e2e`): H2D of the DEM, the run, D2H of every raster + table ---------
    def host_rasters(self):
        return [k for k in self.out if k in self.HOST_RASTERS or (k == "fnf" and self.host_fnf)]

    host_fnf = False      # set True to also ship the float64 no-flats surface to the host

    def host_buffers(self):
        if self._host is None:
            h = {"dem": torch.empty((self.rows, self.cols), dtype=torch.float32).pin_memory()}
            for name in self.host_rasters():
                t = self.out[name]
                h[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
            for name, t in self.tables.items():
                h[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
            self._host = h
        return self._host

    def run_host(self, dem_host=None, bluespot_filter=None, cell_area=1.0):
        """dem_host: pinned (or pageable) float32 CPU tensor / ndarray.  Returns the dict of pinned host
        tensors holding the output rasters (HOST_RASTERS) and the first nlabels+1 entries of every table.
        bluespot_filter, cell_area: as for run()."""
        h = self.host_buffers()
        if dem_host is not None:
            src = torch.from_numpy(dem_host) if isinstance(dem_host, np.ndarray) else dem_host
            if src.data_ptr() != h["dem"].data_ptr():
                h["dem"].copy_(src)
        self.dem.copy_(h["dem"], non_blocking=True)
        ho = _lib.MsHostOut()
        for name in self.host_rasters():
            setattr(ho, name, h[name].data_ptr())
        self.run(host_out=ho, bluespot_filter=bluespot_filter, cell_area=cell_area)          # rasters leave through the copy stream while the later stages run
        m = self.nlabels + 1
        for name, t in self.tables.items():
            h[name][:m].copy_(t[:m], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        with _lib.lock:
            _lib.check(_lib.lib().ms_copies_wait(), "ms_copies_wait")
        return h

    def bytes_h2d(self):
        return self.rows * self.cols * 4

    def bytes_d2h(self):
        n = self.rows * self.cols
        per_cell = sum(self.out[k].element_size() for k in self.host_rasters())
        per_label = sum(t.element_size() for t in self.tables.values())
        return n * per_cell + (self.nlabels + 1) * per_label


def synth_fractal(rows, cols, seed=1, row0=0, col0=0, device=0, out=None):
    """The synthetic fractal DEM (malstroem_b200/synth.py, bit-identical) generated on the device."""
    dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    with _lib.lock:
        _lib.check(_lib.lib().ms_init(dev.index or 0), "ms_init")
        _lib.check(_lib.lib().ms_synth_fractal_dev(out.data_ptr(), rows, cols, row0, col0, seed,
                                                   ctypes.c_void_p(stream)), "ms_synth_fractal_dev")
    return out
