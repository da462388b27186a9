"""Row-band driver: ONE raster split by rows across GPUs (SURVEY.md §8(e)), one band per rank.

Every stage of the hot path runs as "band-local kernel phase -> small exchange -> band-local kernel phase":

    stage                     exchanged between the phases
    K0 min/max                2 floats (all-reduce)
    K1 fill                   halo row of the DEM; counts + ids of the components that wait for a neighbour; the
                              boundary graph (lowest edge between such components), solved redundantly on every rank
    K2 no-flats fill          halo rows of the plain fill and of the surface, repeated until no band changes
    K3 D8                     halo rows of the surface (already there)
    K4 accumulation           per edge cell: where it leaves / which exit it ends at / the count it carries;
                              totals over the forest of all band exits
    K5/6 bluespot labels      roots of the edge rows; merged on the host (CPU, O(cols)); per-band counts
    K7 watersheds             per edge cell what it resolves to; chains followed across bands
    K8-K10 tables             all-reduces of the per-label tables (min / max / sum)

The kernels are the library's (`ms_band_*` of include/malstroem_b200.h); torch is used for device memory, the
stream, index arithmetic on the O(cols) boundary arrays and torch.distributed (NCCL on GPUs; gloo in the CPU tests
of the exchange layer).  `ThreadComm` runs G bands as G threads of one process on one GPU — the same code path, used
by the single-GPU tests of the decomposition.  Results are bit-identical to the single-GPU path.
"""
import ctypes
import threading

import numpy as np
import torch

from . import _lib

OPEN_TOP, OPEN_BOTTOM = 1, 2
BAND_ALIGN = 64


def band_rows(rows, size):
    """Row ranges [(r0, r1)] of the bands: boundaries on multiples of 64 rows, every band non-empty."""
    per = -(-rows // size)
    per = -(-per // BAND_ALIGN) * BAND_ALIGN
    out = []
    for g in range(size):
        r0, r1 = g * per, min(rows, (g + 1) * per)
        if r1 - r0 < 2:
            raise ValueError("raster of %d rows is too small for %d bands of a multiple of %d rows"
                             % (rows, size, BAND_ALIGN))
        out.append((r0, r1))
    return out


# ------------------------------------------------------------------------------------------- communicators
class ThreadGroup(object):
    """Shared state of `size` ThreadComm ranks living in one process."""

    def __init__(self, size):
        self.size = size
        self.barrier = threading.Barrier(size)
        self.slots = [None] * size


class ThreadComm(object):
    def __init__(self, group, rank):
        self.g, self.rank, self.size = group, rank, group.size

    def _swap(self, item):
        self.g.slots[self.rank] = item
        self.g.barrier.wait()
        got = list(self.g.slots)
        self.g.barrier.wait()
        return got

    def all_gather(self, t):
        return torch.stack([x.clone() for x in self._swap(t)])

    def all_gather_var(self, t):
        return [x.clone() for x in self._swap(t)]

    def all_reduce(self, t, op):
        got = torch.stack(self._swap(t.clone()))
        r = {"sum": got.sum(0), "min": got.min(0).values, "max": got.max(0).values}[op]
        t.copy_(r.to(t.dtype))
        return t

    def all_to_all_var(self, chunks):
        """chunks[j] goes to rank j; returns what every rank sent to this one (tensors of one dtype, any first dim)."""
        got = self._swap(list(chunks))
        return [x[self.rank].clone() for x in got]

    def exchange(self, up, down):
        got = self._swap((up, down))
        a = got[self.rank - 1][1].clone() if self.rank > 0 else None
        b = got[self.rank + 1][0].clone() if self.rank + 1 < self.size else None
        return a, b


class DistComm(object):
    """torch.distributed (NCCL on GPUs, gloo on CPU tensors)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.size = dist.get_rank(group), dist.get_world_size(group)

    def all_gather(self, t):
        t = t.contiguous()
        out = torch.empty(self.size * t.numel(), dtype=t.dtype, device=t.device)
        self.dist.all_gather_into_tensor(out, t.view(-1), group=self.group)
        return out.view((self.size,) + tuple(t.shape))

    def all_gather_var(self, t):
        n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
        ns = self.all_gather(n).view(-1).tolist()
        m = max(max(ns), 1)
        pad = torch.zeros((m,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        pad[: t.shape[0]] = t
        got = self.all_gather(pad)
        return [got[i, : ns[i]] for i in range(self.size)]

    def all_to_all_var(self, chunks):
        n = torch.tensor([c.shape[0] for c in chunks], dtype=torch.int64, device=chunks[0].device)
        got = torch.empty_like(n)
        self.dist.all_to_all_single(got, n, group=self.group)
        ns = got.tolist()
        tail = tuple(chunks[0].shape[1:])
        row = int(np.prod(tail))
        send = torch.cat([c.reshape(-1) for c in chunks])
        out = torch.empty(sum(ns) * row, dtype=send.dtype, device=send.device)
        self.dist.all_to_all_single(out, send, output_split_sizes=[k * row for k in ns],
                                    input_split_sizes=[c.shape[0] * row for c in chunks], group=self.group)
        return [x.view((-1,) + tail) for x in out.split([k * row for k in ns])]

    def all_reduce(self, t, op):
        d = self.dist
        self.dist.all_reduce(t, op={"sum": d.ReduceOp.SUM, "min": d.ReduceOp.MIN, "max": d.ReduceOp.MAX}[op],
                             group=self.group)
        return t

    def exchange(self, up, down):
        d, ops = self.dist, []
        a = torch.empty_like(up) if self.rank > 0 else None
        b = torch.empty_like(down) if self.rank + 1 < self.size else None
        if self.rank > 0:
            ops += [d.P2POp(d.isend, up.contiguous(), self.rank - 1, self.group),
                    d.P2POp(d.irecv, a, self.rank - 1, self.group)]
        if self.rank + 1 < self.size:
            ops += [d.P2POp(d.isend, down.contiguous(), self.rank + 1, self.group),
                    d.P2POp(d.irecv, b, self.rank + 1, self.group)]
        if ops:
            for w in d.batch_isend_irecv(ops):
                w.wait()
        return a, b


# -------------------------------------------------------------------------------------- boundary arithmetic
# (device-agnostic torch code on O(cols) arrays; unit-tested on CPU in tests/test_bands_cpu.py)
def accum_forest(exit_to, entry_root, cols):
    """Parent index of every node (band g, side s, column c) -> node id (g*2+s)*cols+c in the forest of band exits.
    exit_to, entry_root: int tensors [G, 2*cols] as produced by ms_band_accum_local_dev."""
    G = exit_to.shape[0]
    dev = exit_to.device
    e = exit_to.view(G, 2, cols).long()
    root = entry_root.view(G, 2, cols).long()
    g = torch.arange(G, device=dev).view(G, 1, 1).expand(G, 2, cols)
    s = torch.arange(2, device=dev).view(1, 2, 1).expand(G, 2, cols)
    gn = torch.where(s == 0, g - 1, g + 1)                 # the band the exit leads into
    valid = (e >= 0) & (gn >= 0) & (gn < G)
    gn_c, to_c = gn.clamp(0, G - 1), e.clamp(0, cols - 1)
    r = root[gn_c, 1 - s, to_c]                            # exit (side*cols+col) of band gn the entry's path ends at
    parent = torch.where(valid & (r >= 0), gn_c * 2 * cols + r, torch.full_like(r, -1))
    return parent.reshape(-1).to(torch.int32)


def watershed_chain(edge_res, exit_to, cols):
    """Reference array for ms_chain_resolve_dev over nodes (g, s, c): >= 0 final label, < 0 -> -(1 + node)."""
    G = edge_res.shape[0]
    dev = edge_res.device
    res = edge_res.view(G, 2, cols).long()
    e = exit_to.view(G, 2, cols).long()
    g = torch.arange(G, device=dev).view(G, 1, 1).expand(G, 2, cols)
    k = (-(res + 1)).clamp(min=0)                          # side'*cols + col' of the band's own exit
    s2, c2 = k // cols, k % cols
    to = e[g, s2, c2]
    gn = torch.where(s2 == 0, g - 1, g + 1)
    ok = (res < 0) & (to >= 0) & (gn >= 0) & (gn < G)
    node = (gn.clamp(0, G - 1) * 2 + (1 - s2)) * cols + to.clamp(0, cols - 1)
    arr = torch.where(res >= 0, res, torch.where(ok, -(1 + node), torch.zeros_like(res)))
    return arr.reshape(-1).to(torch.int32)


def exit_targets(exit_to, cols, g):
    """For band g: node ids (in the (G,2,cols) numbering) its exits lead into, and a mask of real exits."""
    G = exit_to.shape[0]
    e = exit_to.view(G, 2, cols)[g].long()
    s = torch.arange(2, device=e.device).view(2, 1).expand(2, cols)
    gn = torch.where(s == 0, torch.full_like(s, g - 1), torch.full_like(s, g + 1))
    ok = (e >= 0) & (gn >= 0) & (gn < G)
    node = (gn.clamp(0, G - 1) * 2 + (1 - s)) * cols + e.clamp(0, cols - 1)
    return node.reshape(-1), ok.reshape(-1)


def label_owner(labels, offsets):
    """The band that owns each label (ascending `offsets`: the label offsets of the bands, band g numbering offsets[g]
    + 1 ... offsets[g] + count[g]): the last band whose offset lies below the label."""
    return torch.searchsorted(offsets, labels, right=False) - 1


def cc_plan(roots, globals_, cell_lo, cell_hi):
    """From the merged boundary roots (numpy int64, ascending `roots`, their component's smallest root `globals_`):
    the band's re-rooted local roots, the component roots it owns, and the sorted list of all component roots."""
    comp_roots = np.unique(globals_)
    mine = (roots >= cell_lo) & (roots < cell_hi)
    rer = mine & (globals_ != roots)
    own = (comp_roots >= cell_lo) & (comp_roots < cell_hi)
    return {"rerooted_local": (roots[rer] - cell_lo).astype(np.int32),
            "rerooted_global": globals_[rer],
            "comp_roots": comp_roots,
            "owned_pos": np.nonzero(own)[0],
            "owned_local": (comp_roots[own] - cell_lo).astype(np.int32)}


# ------------------------------------------------------------------------------------------------ pipeline
def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class BandPipeline(object):
    """Buffers of one band of a `rows x cols` raster and the staged run over `comm`."""

    RASTERS = (("filled", torch.float32, True), ("depths", torch.float32, False), ("fnf", torch.float64, True),
               ("flowdir", torch.uint8, True), ("accum", torch.float64, False), ("labels", torch.int32, False),
               ("wsheds", torch.int32, False))

    def __init__(self, rows, cols, comm, device=0, eps=None):
        """eps: optional (short, diag) for the no-flats fill instead of fill.minimum_safe_short_and_diag's values
        (fill_terrain_no_flats takes them as arguments, fill.py:174)."""
        if not torch.cuda.is_available():
            raise RuntimeError("malstroem_b200.bands needs a CUDA device (there is no CPU fallback)")
        self.R, self.cols, self.comm = int(rows), int(cols), comm
        self.eps = eps
        self.device = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        self.r0, self.r1 = band_rows(self.R, comm.size)[comm.rank]
        self.rows = self.r1 - self.r0
        self.open = (OPEN_TOP if comm.rank > 0 else 0) | (OPEN_BOTTOM if comm.rank + 1 < comm.size else 0)
        self.cell_offset = self.r0 * self.cols
        L = _lib.lib()
        with _lib.lock:
            _lib.check(L.ms_init(self.device.index or 0), "ms_init")
            h = ctypes.c_void_p()
            _lib.check(L.ms_band_create(self.rows, self.cols, self.open, ctypes.byref(h)), "ms_band_create")
        self.h = h
        dev = self.device
        self.dem_ext = torch.zeros((self.rows + 2, self.cols), dtype=torch.float32, device=dev)
        self.ext, self.out = {}, {}
        for name, dt, halo in self.RASTERS:
            if halo:
                self.ext[name] = torch.zeros((self.rows + 2, self.cols), dtype=dt, device=dev)
                self.out[name] = self.ext[name][1:1 + self.rows]
            else:
                self.out[name] = torch.empty((self.rows, self.cols), dtype=dt, device=dev)
        self.dem = self.dem_ext[1:1 + self.rows]
        self.tables, self.nlabels, self.stats = {}, 0, {}
        self._flowdir_done = False
        self._cc_allr = self._cc_plan = None
        self.p2p = self._p2p_setup()

    def _p2p_setup(self):
        """Bands on different GPUs of one node (torch.distributed / NCCL): map every band's no-flats solver state
        into every rank through CUDA IPC, so that the solver kernels can feed each other over NVLink."""
        import os
        comm = self.comm
        if not isinstance(comm, DistComm) or comm.size < 2 or os.environ.get("MS_BAND_P2P", "1") == "0":
            return False
        if comm.dist.get_backend(comm.group) != "nccl":
            return False
        info = np.zeros(80, dtype=np.uint8)
        self._call("ms_band_nf_shared_create", self.h, _lib.ptr(info))
        infos = comm.all_gather(torch.from_numpy(info).to(self.device)).cpu().numpy().copy()
        rows_all = np.array([b - a for a, b in band_rows(self.R, comm.size)], dtype=np.int64)
        self._call("ms_band_nf_shared_open", self.h, comm.rank, comm.size, _lib.ptr(infos), _lib.ptr(rows_all))
        return True

    def close(self):
        if self.h is not None:
            with _lib.lock:
                _lib.lib().ms_band_destroy(self.h)
            self.h = None

    # ---- helpers
    def _call(self, name, *args):
        with _lib.lock:
            _lib.check(getattr(_lib.lib(), name)(*args), name)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _halo(self, ext):
        """Send the first / last own row to the neighbours, receive their rows into the halo rows."""
        a, b = self.comm.exchange(ext[1], ext[self.rows])
        if a is not None:
            ext[0].copy_(a)
        if b is not None:
            ext[self.rows + 1].copy_(b)

    # ---- the staged run (order and operands: DemTool.process dem.py:53-93, BluespotTool.process bluespots.py:138-216)
    def _tick(self, name):
        """MS_BAND_TIMING=1: wall time per stage (with a device synchronisation at every stage boundary)."""
        if not self._timing:
            return
        import time
        torch.cuda.synchronize(self.device)
        now = time.perf_counter()
        self.timing[name] = self.timing.get(name, 0.0) + (now - self._t_last) * 1e3
        self._t_last = now

    def run(self, ship=None):
        """ship(names), if given, is called after the stage that finishes the rasters `names` (run_host: D2H copies)."""
        import os
        import time
        ship = ship or (lambda names: None)
        L, comm, dev, cols, rows, n = _lib.lib(), self.comm, self.device, self.cols, self.rows, self.rows * self.cols
        st = self._stream()
        i64 = ctypes.c_int64
        self._timing = os.environ.get("MS_BAND_TIMING") == "1"
        if self._timing:
            self.timing = getattr(self, "timing", {})
            torch.cuda.synchronize(self.device)
            self._t_last = time.perf_counter()
        # K1 fill (+ depths)
        self._halo(self.dem_ext)
        nF = i64(0)
        self._call("ms_band_fill_local_dev", self.h, _p(self.dem), ctypes.byref(nF), st)
        counts = comm.all_gather(torch.tensor([nF.value], dtype=torch.int64, device=dev)).view(-1)
        total_f = int(counts.sum())
        graph_x = None
        if total_f:
            base = int(counts[: comm.rank].sum())
            gids = torch.zeros((2, cols), dtype=torch.int32, device=dev)
            self._call("ms_band_fill_edge_ids_dev", self.h, base, _p(gids[0]), _p(gids[1]), st)
            h_top, h_bot = comm.exchange(gids[0], gids[1])
            cap = 16 * (nF.value + cols) + 1024
            ea = torch.empty(cap, dtype=torch.int32, device=dev)
            eb = torch.empty(cap, dtype=torch.int32, device=dev)
            ew = torch.empty(cap, dtype=torch.float32, device=dev)
            ne = i64(0)
            self._call("ms_band_fill_edges_dev", self.h, _p(self.dem), _p(h_top), _p(h_bot), _p(ea), _p(eb), _p(ew), cap,
                       ctypes.byref(ne), st)
            k = ne.value
            packed = torch.stack([ea[:k], eb[:k], ew[:k].view(torch.int32)], dim=1)      # one gather for the graph
            packed = torch.cat(comm.all_gather_var(packed))
            ea, eb = packed[:, 0].contiguous(), packed[:, 1].contiguous()
            ew = packed[:, 2].contiguous().view(torch.float32)
            graph_x = torch.empty(total_f + 1, dtype=torch.float32, device=dev)
            self._call("ms_graph_minimax_dev", total_f + 1, _p(ea), _p(eb), _p(ew), ea.numel(), _p(graph_x), st)
            self.stats["fill_graph_edges"] = int(ea.numel())
        self.stats["fill_frozen"] = total_f
        self._call("ms_band_fill_finish_dev", self.h, _p(self.dem), _p(graph_x), _p(self.out["filled"]),
                   _p(self.out["depths"]), st)
        self._halo(self.ext["filled"])
        ship(("filled", "depths"))
        self._tick("fill")
        # short / diag (fill.py:235-250)
        mm = torch.empty(2, dtype=torch.float32, device=dev)
        self._call("ms_minmax_f32_dev", _p(self.dem), n, _p(mm), st)
        lo, hi = mm[:1].clone(), mm[1:].clone()
        comm.all_reduce(lo, "min")
        comm.all_reduce(hi, "max")
        maxval = np.float64(max(abs(np.float32(hi.item())), abs(np.float32(lo.item()))))
        self.short = float((np.nextafter(maxval, np.inf) - maxval) * 1024.0)
        self.diag = float(self.short * 2 ** 0.5)
        if self.eps is not None:
            self.short, self.diag = float(self.eps[0]), float(self.eps[1])
        self._tick("minmax")
        # K5/K6 phase 1 (needs the depths only): its host-side merge then overlaps the no-flats solver kernel
        self._cc_allr = None
        if self.p2p:
            self._labels_local(st)
            self._tick("labels_local")
        # K2 no-flats fill
        self._noflats(st)
        self._tick("noflats")
        # K3 D8 (written by the no-flats finishing pass when the integer-raster solve ran)
        if not self._flowdir_done:
            self._call("ms_band_flowdir_dev", self.h, _p(self.out["fnf"]), _p(self.out["flowdir"]), 1, st)
        self._halo(self.ext["flowdir"])
        ship(("flowdir",))
        self._tick("flowdir")
        # K4 accumulation
        self._accum(st)
        ship(("accum",))
        self._tick("accum")
        # K5/K6 bluespot labels, K8 stats
        self._labels(st)
        ship(("labels",))
        self._tick("labels")
        # K7 watersheds, then every per-label table (K8, K10, K8', K8'') in two fused passes and three all-reduces
        self._watersheds(st)
        ship(("wsheds",))
        self._tick("watersheds")
        self._tables(st)
        self._tick("tables")
        return self

    def _noflats(self, st):
        comm, dev, cols = self.comm, self.device, self.cols
        fnf = self.ext["fnf"]
        i64 = ctypes.c_int64
        self._flowdir_done = False
        if self.p2p and self._noflats_ir(st):
            return
        if self.p2p and self._noflats_p2p(st):
            return
        self._call("ms_band_nf_ban_dev", self.h, None, None, 0.0, 0.0, 1, None, st)      # no bans from an earlier run

        def attempt(cap):
            ns = i64(0)
            self._call("ms_band_nf_init_dev", self.h, _p(self.dem), _p(self.out["filled"]), _p(self.out["fnf"]),
                       ctypes.byref(ns), st)
            cap_bound = float(_lib.lib().ms_nf_cap_bound(self.R, self.cols, self.diag))
            self._halo(fnf)
            self._tick("nf_init")
            visits = i64(0)
            self._call("ms_band_nf_solve_dev", self.h, _p(self.dem), _p(self.out["filled"]), _p(self.out["fnf"]),
                       self.short, self.diag, cap_bound, cap, 0, 0, ctypes.byref(visits), st)
            total_visits, sweeps = visits.value, 0
            self._tick("nf_first_solve")
            for sweeps in range(1, 100000):
                old_top, old_bot = fnf[0].clone(), fnf[self.rows + 1].clone()
                self._halo(fnf)
                # which of my halo rows changed — decided on the device, one small gather tells every rank everything
                flags = torch.zeros(2, dtype=torch.int32, device=dev)
                if self.open & OPEN_TOP:
                    flags[0] = (old_top != fnf[0]).any()
                if self.open & OPEN_BOTTOM:
                    flags[1] = (old_bot != fnf[self.rows + 1]).any()
                allf = comm.all_gather(flags).cpu().numpy()
                if not allf.any():
                    break
                ch = int(allf[comm.rank, 0]) | (int(allf[comm.rank, 1]) << 1)
                if ch:
                    self._call("ms_band_nf_solve_dev", self.h, _p(self.dem), _p(self.out["filled"]), _p(self.out["fnf"]),
                               self.short, self.diag, cap_bound, cap, 1, ch, ctypes.byref(visits), st)
                    total_visits += visits.value
            self._tick("nf_exchange_loop")
            nv = i64(0)
            self._call("ms_band_nf_verify_dev", self.h, _p(self.dem), _p(self.out["fnf"]), self.short, self.diag,
                       ctypes.byref(nv), st)
            bad = comm.all_reduce(torch.tensor([nv.value], dtype=torch.int64, device=dev), "sum")
            self._tick("nf_verify")
            self.stats.update(noflat_exchanges=sweeps, noflat_tile_visits=total_visits, noflat_capped=cap)
            return int(bad.item())

        for cap in (1, 0):
            if attempt(cap) == 0:
                return
        # Seed repair, as on one GPU (fill_no_flats_dev_impl): a "seed" the stencil rejects (the lake next to it has
        # risen above it) is banned - relaxed like a lake cell from then on - and the uncapped solve is repeated.
        # Every band bans its own cells; the decision to go on is taken on the all-reduced count.
        for repairs in range(1, 1001):
            nv = i64(0)
            self._call("ms_band_nf_ban_dev", self.h, _p(self.dem), _p(self.out["fnf"]), self.short, self.diag, 0,
                       ctypes.byref(nv), st)
            self.stats["noflat_repairs"] = repairs
            if attempt(0) == 0:
                return
        raise RuntimeError("band no-flats fill: seed verification did not settle")

    def _noflats_ir(self, st):
        """The capped solve on the integer raster (the single-GPU solver k_nf_solve_ir), every band's kernel running
        at once and exchanging edge rows and tile activations over NVLink peer memory; the finishing pass writes the
        surface once, verifies it with the halo rows and writes the D8 codes on the way.  Every decision is taken on
        values all ranks share (gathered / reduced), so the ranks stay in step; returns False when the raster does
        not fit the integer form or the verification rejects the result (the W-based paths take over)."""
        comm, dev, cols = self.comm, self.device, self.cols
        i64, cint = ctypes.c_int64, ctypes.c_int
        cap_bound = float(_lib.lib().ms_nf_cap_bound(self.R, self.cols, self.diag))
        dem, filled = self.dem, self.out["filled"]
        fix = torch.empty((2, cols), dtype=torch.uint8, device=dev)
        self._call("ms_band_nf_ir_edgefix_dev", self.h, _p(dem), _p(filled), _p(fix[0]), _p(fix[1]), st)
        halo_top, halo_bot = comm.exchange(fix[0], fix[1])
        q, bad, err = i64(0), cint(0), 0
        try:
            self._call("ms_band_nf_ir_prepare_dev", self.h, _p(dem), _p(filled), self.short, self.diag, cap_bound,
                       _p(halo_top), _p(halo_bot), ctypes.byref(q), ctypes.byref(bad), st)
        except RuntimeError:
            err = 1
        self._tick("nf_init")
        # one gather: also the barrier after which every band's edge rows are in its neighbours' mailboxes
        allq = comm.all_gather(torch.tensor([q.value, bad.value + err], dtype=torch.int64, device=dev)).cpu()
        if int(allq[:, 1].sum()) > 0:
            return False
        visits = i64(0)
        if int(allq[:, 0].sum()) > 0:
            self._call("ms_band_nf_p2p_arm_dev", self.h, st)
            comm.all_reduce(torch.zeros(1, dtype=torch.int32, device=dev), "sum").cpu()           # barrier
            try:
                self._call("ms_band_nf_ir_solve_launch_dev", self.h, _p(filled), self.short, self.diag, st)
                if self._cc_allr is not None:
                    self._labels_merge()          # CPU work while the solver kernels of all bands run
                self._call("ms_band_nf_ir_solve_wait_dev", self.h, ctypes.byref(visits), ctypes.byref(bad), st)
            except RuntimeError:
                err = 1
        self._tick("nf_p2p_solve")
        nv = i64(0)
        if not err and not bad.value:
            self._call("ms_band_nf_ir_finish_dev", self.h, _p(dem), _p(filled), _p(self.out["fnf"]),
                       _p(self.out["flowdir"]), self.short, self.diag, ctypes.byref(nv), st)
        res = comm.all_reduce(torch.tensor([nv.value, bad.value + err], dtype=torch.int64, device=dev), "sum").cpu()
        self._tick("nf_verify")
        ok = int(res[0]) == 0 and int(res[1]) == 0
        self.stats.update(noflat_exchanges=0, noflat_tile_visits=visits.value, noflat_capped=1, noflat_p2p=1,
                          noflat_ir=1 if ok else 0, noflat_p2p_violations=int(res[0]),
                          noflat_p2p_queued=allq[:, 0].tolist())
        if ok:
            self._flowdir_done = True
        return ok

    def _noflats_p2p(self, st):
        """The capped solve with all bands' solver kernels running at once and exchanging over NVLink peer memory.
        Returns False if the verification stencil rejects the result (the host-driven generic path takes over)."""
        comm, dev = self.comm, self.device
        fnf = self.ext["fnf"]
        i64 = ctypes.c_int64
        cap_bound = float(_lib.lib().ms_nf_cap_bound(self.R, self.cols, self.diag))
        ns = i64(0)
        self._call("ms_band_nf_init_dev", self.h, _p(self.dem), _p(self.out["filled"]), _p(self.out["fnf"]),
                   ctypes.byref(ns), st)
        self._halo(fnf)
        self._call("ms_band_nf_seedcand_dev", self.h, _p(self.out["filled"]), _p(self.out["fnf"]), self.short, self.diag,
                   cap_bound, st)
        self._halo(fnf)
        self._tick("nf_init")
        q = i64(0)
        self._call("ms_band_nf_p2p_prepare_dev", self.h, _p(self.out["fnf"]), ctypes.byref(q), st)
        torch.cuda.synchronize(dev)
        allq = comm.all_gather(torch.tensor([q.value], dtype=torch.int64, device=dev)).cpu()      # also a barrier
        visits = i64(0)
        if int(allq.sum()) > 0:
            self._call("ms_band_nf_p2p_arm_dev", self.h, st)
            comm.all_reduce(torch.zeros(1, dtype=torch.int32, device=dev), "sum").cpu()           # barrier
            self._call("ms_band_nf_p2p_solve_dev", self.h, _p(self.out["filled"]), _p(self.out["fnf"]), self.short,
                       self.diag, cap_bound, ctypes.byref(visits), st)
        self._tick("nf_p2p_solve")
        self._halo(fnf)
        nv = i64(0)
        self._call("ms_band_nf_verify_dev", self.h, _p(self.dem), _p(self.out["fnf"]), self.short, self.diag,
                   ctypes.byref(nv), st)
        bad = comm.all_reduce(torch.tensor([nv.value], dtype=torch.int64, device=dev), "sum")
        self._tick("nf_verify")
        nbad = int(bad.item())
        self.stats.update(noflat_exchanges=0, noflat_tile_visits=visits.value, noflat_capped=1, noflat_p2p=1,
                          noflat_p2p_violations=nbad, noflat_p2p_queued=allq.view(-1).tolist())
        return nbad == 0

    def _accum(self, st):
        comm, dev, cols = self.comm, self.device, self.cols
        G, g = comm.size, comm.rank
        exit_to = torch.empty(2 * cols, dtype=torch.int32, device=dev)
        exit_val = torch.empty(2 * cols, dtype=torch.float64, device=dev)
        entry_root = torch.empty(2 * cols, dtype=torch.int32, device=dev)
        self._call("ms_band_accum_local_dev", self.h, _p(self.out["flowdir"]), _p(exit_to), _p(exit_val),
                   _p(entry_root), st)
        packed = comm.all_gather(torch.stack([exit_to.double(), exit_val, entry_root.double()]))     # [G, 3, 2*cols]
        all_to, all_val, all_root = packed[:, 0].to(torch.int32), packed[:, 1].contiguous(), packed[:, 2].to(torch.int32)
        parent = accum_forest(all_to, all_root, cols).contiguous()
        totals = all_val.reshape(-1).clone()
        self._call("ms_forest_accumulate_dev", totals.numel(), _p(parent), _p(totals), st)
        totals = totals.view(G, 2, cols)
        top = totals[g - 1, 1].contiguous() if g > 0 else None
        bot = totals[g + 1, 0].contiguous() if g + 1 < G else None
        self._call("ms_band_accum_finish_dev", self.h, _p(self.out["flowdir"]), _p(top), _p(bot), _p(self.out["accum"]),
                   st)

    def _labels_local(self, st):
        """K5/K6 phase 1: the band's own components (kernels) and the roots of every band's edge rows on the host."""
        comm, dev, cols = self.comm, self.device, self.cols
        roots_tb = torch.empty((2, cols), dtype=torch.int64, device=dev)
        self._call("ms_band_cc_local_dev", self.h, _p(self.out["depths"]), _lib.MS_F32, self.cell_offset,
                   _p(roots_tb[0]), _p(roots_tb[1]), st)
        self._cc_allr = comm.all_gather(roots_tb).cpu().numpy()              # [G, 2, cols]
        self._cc_plan = None

    def _labels_merge(self):
        """K5/K6 phase 2, host only (O(G * cols)): components that touch across band edges.  Runs while the no-flats
        solver kernel is busy on the device when the integer-raster path is taken."""
        if self._cc_plan is not None:
            return
        G, cols = self.comm.size, self.cols
        L = _lib.lib()
        allr = self._cc_allr
        top = np.ascontiguousarray(allr[:, 0, :])
        bot = np.ascontiguousarray(allr[:, 1, :])
        capn = 2 * G * cols
        out_root = np.empty(capn, dtype=np.int64)
        out_glob = np.empty(capn, dtype=np.int64)
        k = ctypes.c_int64(0)
        with _lib.lock:
            _lib.check(L.ms_cc_boundary_merge(G, cols, _lib.ptr(top), _lib.ptr(bot), _lib.ptr(out_root),
                                              _lib.ptr(out_glob), capn, ctypes.byref(k)), "ms_cc_boundary_merge")
        self._cc_plan = cc_plan(out_root[: k.value], out_glob[: k.value], self.cell_offset,
                                self.cell_offset + self.rows * cols)
        self._cc_nroots = int(k.value)

    def _labels(self, st):
        comm, dev, cols = self.comm, self.device, self.cols
        if self._cc_allr is None:
            self._labels_local(st)
        self._labels_merge()
        plan = self._cc_plan
        k = ctypes.c_int64(self._cc_nroots)
        self._cc_allr = None
        rer = torch.from_numpy(plan["rerooted_local"]).to(dev)
        cnt = ctypes.c_int64(0)
        self._call("ms_band_cc_count_dev", self.h, _p(rer) if rer.numel() else None, rer.numel(), ctypes.byref(cnt), st)
        counts = comm.all_gather(torch.tensor([cnt.value], dtype=torch.int64, device=dev)).view(-1)
        label_offset = int(counts[: comm.rank].sum())
        self.nlabels = int(counts.sum())
        cl = counts.tolist()
        self.label_ranges = [(sum(cl[:g]), c) for g, c in enumerate(cl)]      # (offset, count) of every band
        # labels of the component roots that touch a band edge, published by their owners
        ncomp = len(plan["comp_roots"])
        lab_of = torch.zeros(max(ncomp, 1), dtype=torch.int64, device=dev)
        if len(plan["owned_local"]):
            idx = torch.from_numpy(plan["owned_local"]).to(dev)
            lab = torch.empty(idx.numel(), dtype=torch.int32, device=dev)
            self._call("ms_band_cc_root_labels_dev", self.h, _p(idx), idx.numel(), label_offset, _p(lab), st)
            lab_of[torch.from_numpy(plan["owned_pos"]).to(dev)] = lab.long()
        comm.all_reduce(lab_of, "sum")
        rer_lab = None
        if rer.numel():
            pos = np.searchsorted(plan["comp_roots"], plan["rerooted_global"])
            rer_lab = lab_of[torch.from_numpy(pos).to(dev)].to(torch.int32).contiguous()
        self._call("ms_band_cc_finish_dev", self.h, _p(rer) if rer.numel() else None, _p(rer_lab), rer.numel(),
                   label_offset, _p(self.out["labels"]), st)
        self.stats["cc_boundary_roots"] = int(k.value)

    def _tables(self, st):
        """label_stats(depths, labels), label_count(wsheds), label_min_index(fnf, labels), label_max_index(accum,
        labels) (bluespots.py:160-205) for the whole raster, complete on every rank."""
        comm, dev, n, cols, m = self.comm, self.device, self.rows * self.cols, self.cols, self.nlabels + 1
        lohi = torch.empty(4 * m, dtype=torch.float64, device=dev)       # st_min, st_max, ppmin value, ppmax value
        sums = torch.empty(m, dtype=torch.float64, device=dev)           # st_sum
        cnts = torch.empty(2 * m, dtype=torch.int64, device=dev)         # st_count, ws_count
        self._call("ms_band_tables_a_dev", _p(self.out["depths"]), _p(self.out["labels"]), _p(self.out["fnf"]),
                   _p(self.out["accum"]), _p(self.out["wsheds"]), n, cols, self.nlabels, _p(lohi[0:]), _p(lohi[m:]),
                   _p(sums[0:]), _p(cnts[0:]), _p(cnts[m:]), _p(lohi[2 * m:]), _p(lohi[3 * m:]), st)
        lohi[m:2 * m].neg_()                                 # max(x) = -min(-x): one min all-reduce for all four
        lohi[3 * m:].neg_()
        comm.all_reduce(lohi, "min")
        lohi[m:2 * m].neg_()
        lohi[3 * m:].neg_()
        comm.all_reduce(cnts, "sum")
        comm.all_reduce(sums, "sum")
        idx = torch.empty(2 * m, dtype=torch.int64, device=dev)
        self._call("ms_band_tables_b_dev", _p(self.out["labels"]), _p(self.out["fnf"]), _p(self.out["accum"]), n,
                   self.nlabels, _p(lohi[2 * m:]), _p(lohi[3 * m:]), self.cell_offset, _p(idx[0:]), _p(idx[m:]), st)
        comm.all_reduce(idx, "min")
        none = idx == torch.iinfo(torch.int64).max
        rows_ = torch.where(none, torch.full_like(idx, -1), idx // cols)
        cols_ = torch.where(none, torch.full_like(idx, -1), idx % cols)
        t = self.tables
        t["st_min"], t["st_max"], t["st_sum"] = lohi[:m], lohi[m:2 * m], sums
        t["st_count"], t["ws_count"] = cnts[:m], cnts[m:]
        for k, key in enumerate(("ppmin", "ppmax")):
            t[key + "_value"] = lohi[(2 + k) * m:(3 + k) * m]
            t[key + "_row"] = rows_[k * m:(k + 1) * m]
            t[key + "_col"] = cols_[k * m:(k + 1) * m]

    def _watersheds(self, st):
        comm, dev, cols = self.comm, self.device, self.cols
        G, g = comm.size, comm.rank
        ws = self.out["wsheds"]
        ws.copy_(self.out["labels"])
        edge_res = torch.empty(2 * cols, dtype=torch.int32, device=dev)
        exit_to = torch.empty(2 * cols, dtype=torch.int32, device=dev)
        self._call("ms_band_ws_local_dev", self.h, _p(self.out["flowdir"]), _p(ws), 0, _p(edge_res), _p(exit_to), st)
        packed = comm.all_gather(torch.stack([edge_res, exit_to]))                                   # [G, 2, 2*cols]
        all_res, all_to = packed[:, 0].contiguous(), packed[:, 1].contiguous()
        arr = watershed_chain(all_res, all_to, cols).contiguous()
        final = torch.empty_like(arr)
        self._call("ms_chain_resolve_dev", arr.numel(), _p(arr), _p(final), st)
        node, ok = exit_targets(all_to, cols, g)
        exit_label = torch.where(ok, final[node.clamp(0, arr.numel() - 1)], torch.zeros_like(final[:1])).to(torch.int32)
        self._call("ms_band_ws_finish_dev", self.h, _p(self.out["flowdir"]), _p(ws), 0, _p(exit_label.contiguous()), st)

    # ---- the bluespot network and rain events on the finished tables (SURVEY.md §8(f1,f2)) -----------------------
    def network(self, cell_area=1.0, events_mm=(), use_accum_pourpoints=False, sum_mode=None):
        """RasterPipeline.network for a banded run: every rank ends up with the complete tables — `parent` int32
        [nlabels+1] and rainv / spillv / v / pctv float64 [n_events, nlabels+1].  Each band answers for the pour
        points it owns (one lookup in the watershed raster, halo rows exchanged with the neighbours), a max
        all-reduce combines them, and the rain events are evaluated on every rank from the replicated tables."""
        from . import network as _network
        comm, dev, n, st = self.comm, self.device, self.nlabels + 1, self._stream()
        key = "ppmax" if use_accum_pourpoints else "ppmin"
        ws = self.out["wsheds"]
        above, below = comm.exchange(ws[0].contiguous(), ws[self.rows - 1].contiguous())
        parent = torch.empty(n, dtype=torch.int32, device=dev)
        self._call("ms_band_pp_parent_dev", _p(self.out["flowdir"]), _p(ws), _p(above) if above is not None else None,
                   _p(below) if below is not None else None, self.rows, self.cols, self.r0, self.R, n,
                   _p(self.tables[key + "_row"].contiguous()), _p(self.tables[key + "_col"].contiguous()), _p(parent), st)
        comm.all_reduce(parent, "max")
        parent.clamp_(min=-1)                                # a label without a pour point: no downstream node
        mm = np.ascontiguousarray(np.atleast_1d(np.asarray(events_mm, dtype=np.float64)))
        ne = int(mm.size)
        res = {"parent": parent}
        area = (self.tables["ws_count"].double() * float(cell_area)).contiguous()
        cap = (self.tables["st_sum"] * float(cell_area)).contiguous()
        for k in ("rainv", "spillv", "v", "pctv"):
            res[k] = torch.empty((ne, n), dtype=torch.float64, device=dev)
        if ne:
            self._call("ms_rain_events_dev", n, _p(parent), _p(area), _p(cap), ne, _lib.ptr(mm),
                       _network.SUM_MODE if sum_mode is None else sum_mode, _p(res["rainv"]), _p(res["spillv"]),
                       _p(res["v"]), _p(res["pctv"]), None, st)
        return res

    # ---- water levels and depth rasters after the rain events (csrc/flood.cu) -------------------------------------
    _FLOOD_LOCAL = 1 << 30          # this rank's library call or allocation failed (not a data error)

    def _flood_phase(self, name, *args):
        """One phase's library call; a failure on this rank becomes a flag, so that no rank is left waiting in the
        collective that follows.  Returns _FLOOD_LOCAL or 0."""
        try:
            self._call(name, *args)
            return 0
        except (RuntimeError, ValueError, IndexError) as e:
            self._flood_error = e
            return self._FLOOD_LOCAL

    def _flood_flags(self, flags):
        """Combine the error flags of a flood phase over all ranks; every rank raises."""
        bits = (self._FLOOD_LOCAL, _lib.MS_FLOOD_LABEL, _lib.MS_FLOOD_CAPACITY, _lib.MS_FLOOD_UNIFORM,
                _lib.MS_FLOOD_VOLUME, _lib.MS_FLOOD_SIZE)
        got = self.comm.all_reduce(torch.tensor([1 if flags & b else 0 for b in bits], dtype=torch.int32,
                                                device=self.device), "max").tolist()
        if got[0]:
            if flags & self._FLOOD_LOCAL:
                raise self._flood_error
            raise RuntimeError("flood: the phase failed on another band")
        if got[1]:
            raise IndexError("flood: a label outside [0, %d] or outside its band's range" % self.nlabels)
        if got[2]:
            raise ValueError("flood: a band holds more labels of lower bands than its first and last rows can carry "
                             "(labels must be the connected bluespot labels of this run)")
        if got[3]:
            raise ValueError("flood: the fill is not uniform over a label (labels must be bluespots of this fill)")
        if got[4]:
            raise ValueError("flood: a negative volume")
        if got[5]:
            raise ValueError("flood: the bluespots owned by one band hold 2^31 cells or more")

    def flood(self, net, cell_area):
        """RasterPipeline.flood for a banded run: every rank returns the complete `level` float64 and `wet` int64
        [n_events, nlabels+1], bitwise what RasterPipeline.flood gives on the whole raster with the same st_sum and v.
        The band that numbered a label owns it; every other band sends it its cells' z keys (keys travel only
        towards lower ranks), the owner solves its labels, and the owned column ranges are gathered."""
        comm, dev, st, n = self.comm, self.device, self._stream(), self.nlabels + 1
        v = net["v"].contiguous()
        if v.dim() != 2 or v.shape[1] != n or v.dtype != torch.float64 or v.device != self.device:
            raise ValueError("flood: net['v'] must be a float64 tensor [n_events, %d] on %s" % (n, self.device))
        ca = float(cell_area)
        if not (ca > 0.0 and np.isfinite(ca)):
            raise ValueError("flood: cell_area must be > 0 (%g)" % ca)
        ne = int(v.shape[0])
        level = torch.full((ne, n), float("nan"), dtype=torch.float64, device=dev)
        wet = torch.zeros((ne, n), dtype=torch.int64, device=dev)
        if ne == 0 or self.nlabels == 0:
            return {"level": level, "wet": wet}
        lo, cnt_g = self.label_ranges[comm.rank]
        hi = lo + cnt_g
        i64, cint = ctypes.c_int64, ctypes.c_int
        rasters = (_p(self.dem), _p(self.out["filled"]), _p(self.out["labels"]), self.rows, self.cols, self.nlabels,
                   lo, hi)
        cnt = torch.empty(n + 1, dtype=torch.int32, device=dev)
        off = torch.empty(n + 1, dtype=torch.int32, device=dev)
        lkey = torch.empty(n, dtype=torch.int32, device=dev)
        # a foreign label reaches the band's first or last row, where at most cols / 2 labels fit in each
        cap = 2 * self.cols
        foreign = torch.empty((cap, 3), dtype=torch.int32, device=dev)
        nf, nsend, flags = i64(0), i64(0), cint(0)
        err = self._flood_phase("ms_band_flood_count_dev", *rasters, _p(cnt), _p(lkey), _p(off), _p(foreign), cap,
                                ctypes.byref(nf), ctypes.byref(nsend), ctypes.byref(flags), st)
        self._flood_flags(flags.value | err)
        # every foreign run to its owner: the list is in label order, so each owner's part is contiguous
        foreign = foreign[: nf.value]
        starts = torch.tensor([o for o, _ in self.label_ranges], dtype=torch.int64, device=dev)
        dest = label_owner(foreign[:, 0].long(), starts)
        runs = torch.bincount(dest, minlength=comm.size).tolist()
        keys = torch.zeros(comm.size, dtype=torch.int64, device=dev).index_add_(0, dest, foreign[:, 1].long()).tolist()
        recv = torch.cat(comm.all_to_all_var(list(foreign.split(runs)))).contiguous()
        recv_pos = torch.empty(recv.shape[0], dtype=torch.int32, device=dev)
        ncells = i64(0)
        err = self._flood_phase("ms_band_flood_layout_dev", self.nlabels, lo, hi, _p(cnt), _p(lkey), _p(off), _p(recv),
                                recv.shape[0], _p(recv_pos), ctypes.byref(ncells), ctypes.byref(flags), st)
        self._flood_flags(flags.value | err)
        self.stats.update(flood_keys_sent=nsend.value, flood_crossing_labels=int(torch.unique(recv[:, 0]).numel()))
        try:
            seg = torch.empty(ncells.value, dtype=torch.int32, device=dev)
            send = torch.empty(nsend.value, dtype=torch.int32, device=dev)
        except RuntimeError as e:                       # out of device memory on this rank
            self._flood_error, seg, send = e, None, None
        err = self._FLOOD_LOCAL if seg is None else self._flood_phase(
            "ms_band_flood_scatter_dev", *rasters, _p(cnt), _p(lkey), _p(off), _p(seg), _p(send), ctypes.byref(flags), st)
        self._flood_flags(flags.value | err)
        recv_keys = torch.cat(comm.all_to_all_var(list(send.split(keys)))).contiguous()
        err = self._flood_phase("ms_band_flood_solve_dev", self.nlabels, lo, hi, _p(off), _p(lkey), _p(seg), _p(recv),
                                recv.shape[0], _p(recv_pos), _p(recv_keys), recv_keys.numel(),
                                _p(self.tables["st_sum"]), ca, ne, _p(v), _p(level), _p(wet), ctypes.byref(flags), st)
        self._flood_flags(flags.value | err)
        own = torch.cat([level[:, lo + 1:hi + 1].T, wet[:, lo + 1:hi + 1].T.view(torch.float64)], 1).contiguous()
        got = torch.cat(comm.all_gather_var(own)).T
        level[:, 1:] = got[:ne]
        wet[:, 1:] = got[ne:].contiguous().view(torch.int64)
        return {"level": level, "wet": wet}

    def water_depth(self, level_row, out=None):
        """RasterPipeline.water_depth for the band's rows: level_row is one row of flood()'s `level`."""
        n = self.nlabels + 1
        level_row = level_row.contiguous()
        if level_row.shape != (n,) or level_row.dtype != torch.float64 or level_row.device != self.device:
            raise ValueError("water_depth: level_row must be a float64 tensor [%d] on %s" % (n, self.device))
        if out is None:
            out = torch.empty((self.rows, self.cols), dtype=torch.float32, device=self.device)
        elif (out.shape != (self.rows, self.cols) or out.dtype != torch.float32 or not out.is_contiguous()
              or out.device != self.device):
            raise ValueError("water_depth: out must be a contiguous float32 tensor of the band's shape on %s"
                             % self.device)
        self._call("ms_water_depth_dev", _p(self.dem), _p(self.out["filled"]), _p(self.out["labels"]), self.rows,
                   self.cols, self.nlabels, _p(level_row), _p(out), self._stream())
        return out

    # ---- host-buffer front end (bench `e2e`): H2D of the band's DEM rows, the run, D2H of every raster + table
    def host_buffers(self):
        if getattr(self, "_host", None) is None:
            h = {"dem": torch.empty((self.rows, self.cols), dtype=torch.float32).pin_memory()}
            for name, t in self.out.items():
                if name != "fnf":      # an intermediate of the reference's tools (dem.py:80-86): stays in HBM
                    h[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
            self._host = h
        return self._host

    def run_host(self, dem_host=None):
        """Pinned host DEM rows -> H2D -> the staged run -> D2H.  Every rank brings back its own rows of the rasters,
        each over a copy stream as soon as the stage that produces it is done (so the copies overlap the later stages,
        as in RasterPipeline.run_host); the per-label tables are replicated on every rank, so rank 0 alone ships
        them, into pinned buffers.  Returns the dict of pinned host tensors (`tables` only on rank 0)."""
        h = self.host_buffers()
        if dem_host is not None:
            h["dem"].copy_(torch.from_numpy(dem_host) if isinstance(dem_host, np.ndarray) else dem_host)
        self.dem.copy_(h["dem"], non_blocking=True)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        side, cur = self._copy_stream, torch.cuda.current_stream(self.device)

        def ship(names):
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for name in names:
                    if name in h:
                        # in pieces of ~32 MB: the stages that follow read counters back every round, and such a
                        # read-back queues behind whatever the copy engine is busy with (csrc/pipeline.cu ship())
                        dst, src = h[name], self.out[name]
                        step = max(1, (32 << 20) // max(1, src[0].numel() * src.element_size()))
                        for a in range(0, src.shape[0], step):
                            dst[a:a + step].copy_(src[a:a + step], non_blocking=True)

        self.run(ship=ship)
        tabs = {}
        if self.comm.rank == 0:
            m = self.nlabels + 1
            pinned = getattr(self, "_host_tabs", None)
            if pinned is None:
                pinned = self._host_tabs = {}
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for k, v in self.tables.items():
                    buf = pinned.get(k)
                    if buf is None or buf.numel() < m or buf.dtype != v.dtype:
                        buf = pinned[k] = torch.empty(m + m // 4 + 1, dtype=v.dtype).pin_memory()
                    buf[:m].copy_(v[:m], non_blocking=True)
                    tabs[k] = buf[:m]
        side.synchronize()
        cur.synchronize()
        h["tables"] = tabs
        return h

    def bytes_h2d(self):
        return self.rows * self.cols * 4

    def bytes_d2h(self):
        """Per rank: its rows of the rasters; rank 0 also ships the (replicated) tables."""
        per_cell = sum(t.element_size() for k, t in self.out.items() if k != "fnf")
        per_label = sum(t.element_size() for t in self.tables.values()) if self.comm.rank == 0 else 0
        return self.rows * self.cols * per_cell + (self.nlabels + 1) * per_label


def run_threaded(dem, nbands, device=0, after=None, eps=None):
    """One process, one GPU, `nbands` bands as threads (the decomposition without NCCL): returns the BandPipelines
    after the run.  `dem`: cuda float32 tensor [rows, cols].  `after(pipeline)`, if given, runs in every band's
    thread after the run (for calls that communicate, like `network`); its result is kept in `p.after_result`."""
    rows, cols = dem.shape
    grp = ThreadGroup(nbands)
    pipes, errs = [None] * nbands, []

    def work(rank):
        try:
            torch.cuda.set_device(device)
            p = BandPipeline(rows, cols, ThreadComm(grp, rank), device=device, eps=eps)
            pipes[rank] = p
            p.dem.copy_(dem[p.r0:p.r1])
            p.run()
            if after is not None:
                p.after_result = after(p)
        except BaseException as e:      # noqa: BLE001 - report and release the other threads
            errs.append(e)
            grp.barrier.abort()

    ts = [threading.Thread(target=work, args=(r,)) for r in range(nbands)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errs:
        real = [e for e in errs if not isinstance(e, threading.BrokenBarrierError)]
        raise (real or errs)[0]
    torch.cuda.synchronize()
    return pipes
