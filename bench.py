#!/usr/bin/env python
"""bench.py — DEM cells/s end-to-end (fill -> D8 -> accum -> bluespot / watershed labels) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--size S] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the whole raster hot path over ONE S x S synthetic fractal DEM (default S = 32768,
BASELINE.json configs[2], the largest single-GPU configuration):
  N = 1   the whole raster on one B200 (malstroem_b200.pipeline.RasterPipeline -> ms_pipeline_dev);
  N > 1   (torchrun, one rank per GPU) THE SAME raster as N row bands (malstroem_b200.bands.BandPipeline over NCCL /
          NVLink peer memory, SURVEY.md 8(e)) — total work is fixed, so the scaling is strong.
`value` is timed with the DEM already resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` is
the same path through the host-buffer front end (pinned host DEM -> H2D -> all stages -> D2H of every raster the
reference's tools write and of every table).  After the timed region (outside it) every rank certifies its rasters and
tables (tools/big_check.py, SURVEY.md A.5) and, for N > 1, the banded result is compared with a single-GPU run of the
same raster on rank 0 (`parity` in the JSON line).  Sub-records on the same line: `config2` = BASELINE configs[1]
(8192^2 on one GPU), `same_config` = the window the reference arm times (so one same-config ratio exists), and at
N = 8 `config4` = BASELINE configs[3] (65536^2 as 8 bands, certified).
`--impl reference` times the reference's own stock CPU implementation (baseline/_ref: malstroem.algorithms with its
own speedups.enable(), i.e. its Cython path, scipy labelling, pure-Python label_max_index) on the host, one core
(the reference has no parallel path), on a bounded window of the same DEM.
"""
import argparse
import importlib.util
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "DEM cells/sec end-to-end (fill->D8->accum->bluespot/watershed labels)"
UNIT = "Mcells/s"
BYTES_PER_CELL = 79.0     # SURVEY.md 8(d): compulsory traffic of the eight stages
# algorithmic bytes per cell of the stage each raster-wide kernel belongs to (SURVEY.md 8(d) / DESIGN.md 4)
STAGE_BYTES = {
    "k_descent_tile": 12, "k_forest_jump_list": 12, "k_ws_tile<L>": 9, "k_forest_jump": 12, "k_rootflag": 12, "k_catchment_ids": 12, "k_minedge<false>": 12, "k_minedge_first4": 12, "k_minedge<true>": 12,
    "k_fill_final": 12, "k_scan_reduce<SELF>": 8, "k_scan_final<SELF>": 8,
    "k_nf_init": 12, "k_nf_seedcand": 12, "k_nf_solve<true>": 12, "k_nf_solve<false>": 12, "k_nf_solve_ir": 12, "k_nf_finish_ir": 12, "k_nf_init_tile": 12, "k_nf_verify": 12,
    "k_flowdir": 9, "k_acc_tile_a": 9, "k_acc_tile_c": 9, "k_acc_tile_c<false>": 9, "k_acc_tile_c<true>": 9, "k_minedge_band<false>": 12, "k_minedge_band<true>": 12, "k_acc_links": 9, "k_acc_node_trace": 9,
    "k_cc_tile<T>": 8, "k_cc_border": 8, "k_cc_flatten": 8, "k_cc_number": 8,
    "k_label_stats<T>": 8, "k_ws_ptr<L>": 9, "k_ws_assign<L>": 9, "k_label_count": 9,
    "k_extreme_key<true>": 12, "k_extreme_key<false>": 12, "k_extreme_index": 12, "k_minmax": 4,
    "k_tables_a<true>": 28, "k_tables_a<false>": 20, "k_tables_a2<true>": 28, "k_tables_a2<false>": 20, "k_tables_b<true>": 20, "k_tables_b<false>": 12,
}
WORKLOAD = ("synthetic fractal DEM %dx%d float32 (seed 1, 1 mm quantised): fill+depths, no-flats fill, D8, accum, "
            "bluespot labels, stats, watersheds, pour points")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def ref_window(steps, warmup):
    """Window edge both arms use for the same-config comparison: the largest of 512 / 1024 / 2048 the reference's CPU
    path finishes `warmup + steps` times in ~200 s (measured in the build container: 1.2 / 4.5 / 18 s per pass)."""
    n = max(1, steps + warmup)
    for s, sec in ((2048, 18.0), (1024, 4.5)):
        if n * sec <= 200.0:
            return s
    return 512


def load_big_check():
    spec = importlib.util.spec_from_file_location("big_check", os.path.join(ROOT, "tools", "big_check.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


# ------------------------------------------------------------------------------------ reference arm
def stock_reference():
    """The installed, unmodified reference package (baseline/_ref, see baseline/install_ref.py) with its own
    speedups.enable(): exactly the functions DemTool.process / BluespotTool.process call."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "malstroem")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        from malstroem.algorithms import fill, flow, label, speedups
        speedups.enable()
        if not speedups.enabled:
            return None
        return fill, flow, label
    except Exception:       # noqa: BLE001 - the port takes over
        return None


def reference_stages(mods, dem):
    """dem.py:67-91 and bluespots.py:158-206 on the reference's own functions (stock path)."""
    fill, flow, label = mods
    t0 = time.perf_counter()
    filled = fill.fill_terrain(dem)
    depths = filled - dem
    short, diag = fill.minimum_safe_short_and_diag(dem)
    fnf = fill.fill_terrain_no_flats(dem, short, diag)
    fd = flow.terrain_flowdirection(fnf, edges_flow_outward=True)
    acc = flow.accumulated_flow(fd)
    lab, n = label.connected_components(depths)
    label.label_stats(depths, lab)
    ws = lab.copy()
    flow.watersheds_from_labels(fd, ws, unassigned=0)
    label.label_count(ws)
    label.label_min_index(fnf, lab, n)
    label.label_max_index(acc, lab, n)       # pure Python in the reference (label.py:135-166)
    return time.perf_counter() - t0


def port_stages(dem):
    from oracle import port
    t0 = time.perf_counter()
    filled = port.fill_terrain(dem)
    depths = filled - dem
    short, diag = port.minimum_safe_short_and_diag(dem)
    fnf = port.fill_terrain_no_flats(dem, short, diag)
    fd = port.terrain_flowdirection(fnf, True)
    acc = port.accumulated_flow(fd)
    lab, n = port.connected_components(depths)
    port.label_stats(depths, lab)
    ws = lab.copy()
    port.watersheds_from_labels(fd, ws, 0)
    port.label_count(ws)
    port.label_min_index(fnf, lab, n)
    port.label_max_index(acc, lab, n)
    return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from malstroem_b200 import synth
    s = args.ref_size or ref_window(args.steps, args.warmup)
    dem = synth.fractal_dem(s, s, seed=1)
    mods = stock_reference()
    kind = "reference" if mods is not None else "port"
    times = []
    for i in range(args.warmup + args.steps):
        t = reference_stages(mods, dem) if mods is not None else port_stages(dem)
        if i >= args.warmup:
            times.append(t)
    tot = sum(times)
    val = s * s * len(times) / tot / 1e6
    sample = ("%dx%d window (origin 0,0) of the seed-1 fractal DEM per step, every stage through the stock "
              "malstroem.algorithms functions of baseline/_ref (Cython path, pure-Python label_max_index); the "
              "reference is single-threaded" % (s, s)) if kind == "reference" else \
             "%dx%d window of the seed-1 fractal DEM per step, C port of the reference (oracle/ms_oracle.c)" % (s, s)
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * tot / len(times), 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD % (args.size, args.size), "sample": sample, "window": s,
                       "same_config_as": "the `same_config` record of the GPU arm (same window, same DEM)"},
            "cpu_baseline": {"value": round(val, 4), "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
            "e2e": {"value": round(val, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "host": {"cpus_available": len(os.sched_getaffinity(0))}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """SM clock and throttle reasons DURING the timed region, sampled through NVML from a background thread
    (an `nvidia-smi -lms` child process contends for the driver lock with the path's many small syncs and
    slowed the step several-fold; NVML reads are the same counters without that cost)."""

    def __init__(self, index, period=0.1):
        import threading
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.mode = os.environ.get("BENCH_CLOCKS", "nvml")
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        if self.mode == "off":
            return
        self.period = period
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()

    def _sample(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                          ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80)):
            if r & bit:
                self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "source": "nvml thread, 100 ms"}
        if self.nv is None:
            out["source"] = "unavailable"
            return out
        if self._t is not None:
            self._stop.set()
            self._t.join(timeout=2)
        else:
            try:
                self._sample()
            except Exception:
                pass
        if self.samples:
            out["sm_mhz"] = float(np.median(self.samples))
            out["samples"] = len(self.samples)
        out["reasons"] = sorted(self.reasons)
        return out


# ---------------------------------------------------------------------------------------- our arm
def profile_report(lib):
    import ctypes
    buf = ctypes.create_string_buffer(1 << 16)
    lib.ms_profile_report(buf, len(buf))
    rows = {}
    for line in buf.value.decode().splitlines():
        name, n, ms, units = line.rsplit(" ", 3)
        rows[name] = (int(n), float(ms), int(units))
    return rows


class Job(object):
    """Rank / device / process group of this bench process."""

    def __init__(self):
        import torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (malstroem_b200 has no CPU fallback)")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        import torch
        torch.cuda.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        import torch
        t = torch.tensor(values, dtype=torch.float64, device="cuda")
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]


def make_pipe(job, rows, cols, banded):
    from malstroem_b200.pipeline import RasterPipeline, synth_fractal
    if banded:
        from malstroem_b200 import bands
        pipe = bands.BandPipeline(rows, cols, bands.DistComm(), device=job.local)
        synth_fractal(pipe.rows, cols, seed=1, row0=pipe.r0, col0=0, device=job.local, out=pipe.dem)
    else:
        pipe = RasterPipeline(rows, cols, device=job.local, with_accum=True)
        synth_fractal(rows, cols, seed=1, device=job.local, out=pipe.dem)
    return pipe


def timed_steps(job, lib, pipe, steps, warmup, profile=True, sampler=None):
    """`warmup` untimed passes, then exactly `steps` passes between CUDA events on the launching stream, a barrier and
    a device synchronisation on both sides; returns (ms over all steps [max over ranks], launches, per-kernel rows)."""
    import torch
    lib.ms_kernel_launches(1)
    for _ in range(warmup):
        pipe.run()
    job.barrier()
    per_step = int(lib.ms_kernel_launches(1)) // max(warmup, 1)
    if profile:       # event pairs are created before the clock starts; the per-kernel events stay on inside the timed
        lib.ms_profile(max(2, int(per_step * steps * 1.5)))      # region (they are what `roofline.achieved` is read from)
    lib.ms_kernel_launches(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    job.barrier()
    if sampler is not None:
        sampler = sampler()
    e0.record()
    for _ in range(steps):
        pipe.run()
    e1.record()
    job.barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler is not None else None
    launches = int(lib.ms_kernel_launches(1))
    prof = profile_report(lib) if profile else {}
    lib.ms_profile(0)
    return job.max_over_ranks([ms])[0], launches, prof, clocks


# --dump-outputs: a fixed, seeded sample of what RasterPipeline.run hands its caller, so that two builds can be compared
# output for output.  2^19 cells of each raster and 2^18 entries of each table stay under 64 MB in float64.
DUMP_CELLS, DUMP_LABELS, DUMP_SEED = 1 << 19, 1 << 18, 20240601


def sample_index(n, k, seed):
    """`min(n, k)` distinct indices of [0, n), ascending; the same for the same (n, k, seed)."""
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False)).astype(np.int64)


def dump_outputs(pipe, out_dir):
    """Every raster and per-label table of the pipeline's last run at the sampled positions as `<out_dir>/<name>.npy`:
    float32 for the float32 and uint8 rasters, float64 (exact) for the rest.  `cell_index` / `label_index` hold the
    sampled flat cell positions and label ids; `nlabels`, `short_eps` and `diag_eps` are the run's scalars."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cells = sample_index(pipe.rows * pipe.cols, DUMP_CELLS, DUMP_SEED)
    labels = sample_index(pipe.nlabels + 1, DUMP_LABELS, DUMP_SEED + 1)
    arrays = {"cell_index": cells.astype(np.float64), "label_index": labels.astype(np.float64),
              "nlabels": np.array([pipe.nlabels], np.float64), "short_eps": np.array([pipe.short], np.float64),
              "diag_eps": np.array([pipe.diag], np.float64)}
    for index, source in ((cells, {k: t.view(-1) for k, t in pipe.out.items()}), (labels, pipe.tables)):
        idx = torch.from_numpy(index).to(pipe.device)
        for name, t in source.items():
            v = t.index_select(0, idx).cpu().numpy()
            exact32 = v.dtype == np.float32 or v.dtype == np.uint8
            arrays[name] = v.astype(np.float32 if exact32 else np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sum(a.nbytes for a in arrays.values())


def timed_e2e(job, pipe, steps):
    """Host buffers in, host buffers out: H2D of the DEM and D2H of every raster + table inside the timed region."""
    import torch
    host = pipe.host_buffers()
    host["dem"].copy_(pipe.dem)
    torch.cuda.synchronize()
    pipe.run_host()
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        pipe.run_host()
    job.barrier()
    return job.max_over_ranks([(time.perf_counter() - t0) * 1e3])[0]


def parity_record(job, pipe, banded, rows, cols, bc, single_compare=True):
    """Outside the timed region: the A.5 certificates on every rank's rasters and tables and, for a banded run, the
    comparison with the single-GPU path on rank 0 (additive position-weighted checksums of every raster, exact
    comparison of every table)."""
    import torch
    world, rank = job.world, job.rank
    t0 = time.perf_counter()
    if banded:
        import torch.distributed as dist
        ops = {"min": dist.ReduceOp.MIN, "max": dist.ReduceOp.MAX, "sum": dist.ReduceOp.SUM}

        def reduce(t, op):
            dist.all_reduce(t, op=ops[op])
        st, sb = (1 if rank > 0 else 0), (1 if rank + 1 < world else 0)
        fill_bad, acc_bad, ws_bad, _ = bc.certify(pipe, CH=1024, skip_top=st, skip_bottom=sb)
        more = bc.certify_more(pipe, pipe.short, pipe.diag, CH=1024, skip_top=st, skip_bottom=sb, row_offset=pipe.r0,
                               total_rows=rows, reduce=reduce, tables=pipe.tables, nlabels=pipe.nlabels)
        acc = pipe.out["accum"]
        bsum = acc[:, 0].sum() + acc[:, -1].sum()
        if rank == 0:
            bsum = bsum + acc[0, 1:-1].sum()
        if rank + 1 == world:
            bsum = bsum + acc[-1, 1:-1].sum()
        v = torch.tensor([fill_bad, acc_bad, ws_bad, more["noflats"], more["d8"], more["cc_adjacent"],
                          more["cc_foreground"], more["label_range"]], dtype=torch.float64, device="cuda")
        v = torch.cat([v, bsum.double().view(1)])
        dist.all_reduce(v)
        fill_bad, acc_bad, ws_bad = int(v[0]), int(v[1]), int(v[2])
        more.update(noflats=int(v[3]), d8=int(v[4]), cc_adjacent=int(v[5]), cc_foreground=int(v[6]), label_range=int(v[7]))
        term = float(v[8])
        note = "per band; the first / last row of a band (neighbours in another band) is covered by vs_single_gpu"
    else:
        fill_bad, acc_bad, ws_bad, term = bc.certify(pipe, CH=1024)
        more = bc.certify_more(pipe, pipe.short, pipe.diag, CH=1024)
        note = "whole raster"
    tables_bad = more.pop("tables")
    cert = {"fill": fill_bad, "noflats": more["noflats"], "d8": more["d8"], "accum": acc_bad,
            "accum_border_sum_minus_cells": term - float(rows) * float(cols), "watersheds": ws_bad,
            "cc": {k: more[k] for k in ("cc_adjacent", "cc_foreground", "label_range", "cc_unused_labels", "cc_order")},
            "tables": tables_bad}
    flat = [fill_bad, more["noflats"], more["d8"], acc_bad, ws_bad, cert["accum_border_sum_minus_cells"]] + \
        list(cert["cc"].values()) + list(tables_bad.values())
    rec = {"certificates": cert, "certificates_ok": all(x == 0 for x in flat), "scope": note,
           "nlabels": int(pipe.nlabels)}
    if banded and single_compare:
        import torch.distributed as dist
        from malstroem_b200.pipeline import RasterPipeline, synth_fractal
        sums = bc.raster_checksums(pipe, row_offset=pipe.r0)
        names = sorted(sums)
        v = torch.stack([sums[k] for k in names])
        dist.all_reduce(v)
        verdict = None
        if rank == 0:
            ref = RasterPipeline(rows, cols, device=job.local)
            synth_fractal(rows, cols, seed=1, device=job.local, out=ref.dem)
            ref.run()
            want = bc.raster_checksums(ref)
            diff = [k for i, k in enumerate(names) if int(v[i]) != int(want[k])]
            m = ref.nlabels + 1
            if ref.nlabels != pipe.nlabels:
                diff.append("nlabels")
            else:
                for k in pipe.tables:
                    a, b = pipe.tables[k][:m], ref.tables[k][:m]
                    if k == "st_sum":
                        same = bool(((a - b).abs() <= 1e-6 * b.abs().clamp(min=1e-300)).all())
                    else:
                        same = bool(torch.equal(a, b))
                    if not same:
                        diff.append(k)
            verdict = "equal" if not diff else "differs: " + ",".join(diff)
            del ref
            torch.cuda.empty_cache()
        rec["vs_single_gpu"] = verdict
        rec["vs_single_gpu_how"] = ("rank 0 runs the single-GPU path on the same %dx%d raster; every raster by "
                                    "position-weighted 64-bit checksums summed over the bands, every table "
                                    "element-wise (st_sum to 1e-6)" % (rows, cols))
    rec["seconds"] = round(time.perf_counter() - t0, 1)
    return rec


def plugin_sequence(mods, dem):
    """The calls DemTool.process (dem.py:67-91) and BluespotTool.process (bluespots.py:158-206) make, in their order and
    on their operands (numpy arrays in, numpy arrays out; the arithmetic the tools do in between included), with the
    accumulation as pour-point source AND the no-flats pour points of the default path."""
    fill, flow, label = mods
    filled = fill.fill_terrain(dem)
    depths = filled - dem
    del filled
    short, diag = fill.minimum_safe_short_and_diag(dem)
    fnf = fill.fill_terrain_no_flats(dem, short=short, diag=diag)
    flowdir = flow.terrain_flowdirection(fnf, edges_flow_outward=True)
    del fnf
    accum = flow.accumulated_flow(flowdir)
    raw, _ = label.connected_components(depths)
    raw_stats = label.label_stats(depths, raw)
    keepers = (raw_stats["max"] > 0.05).tolist()
    comps = label.keep_labels(raw, keepers)
    del raw
    lab, n = label.connected_components(comps)
    label.label_stats(depths, lab)
    ws = np.copy(lab)
    flow.watersheds_from_labels(flowdir, ws, unassigned=0)
    label.label_count(ws)
    label.label_max_index(accum, lab, n)
    short, diag = fill.minimum_safe_short_and_diag(dem)
    fnf = fill.fill_terrain_no_flats(dem, short, diag)
    label.label_min_index(fnf, lab, n)
    return n


def plugin_record(size, reps=3):
    """`e2e_plugin`: the same path through the seam `malstroem complete` uses - the reference's own modules
    (baseline/_ref) with malstroem_b200.speedups.enable(), i.e. the twelve rebound functions called one by one on host
    numpy arrays (pageable memory), each with its own H2D / D2H; device twins of the arrays are kept between the calls
    (csrc/cache.cu) and dropped before every pass, so a pass starts cold like a single run of the tools."""
    import malstroem_b200.speedups as sp
    from malstroem_b200 import _lib, synth
    from malstroem_b200.pipeline import synth_fractal
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    via = "malstroem_b200.algorithms (baseline/_ref not installed)"
    mods = None
    if os.path.isdir(os.path.join(ref_dir, "malstroem")):
        if ref_dir not in sys.path:
            sys.path.insert(0, ref_dir)
        try:
            import malstroem.algorithms as alg
            from malstroem.algorithms import fill, flow, label      # noqa: F401
            sp.enable(alg)
            mods = (alg.fill, alg.flow, alg.label)
            via = "malstroem.algorithms of baseline/_ref after malstroem_b200.speedups.enable()"
        except Exception:       # noqa: BLE001
            mods = None
    if mods is None:
        from malstroem_b200.algorithms import fill, flow, label
        mods = (fill, flow, label)
    dem = synth_fractal(size, size, seed=1).cpu().numpy()
    plugin_sequence(mods, dem)          # warm-up: context, scratch arena
    times = []
    for _ in range(reps):
        _lib.cache_clear()
        t0 = time.perf_counter()
        n = plugin_sequence(mods, dem)
        times.append(time.perf_counter() - t0)
    st = _lib.cache_stats()
    sp.disable()
    _lib.cache_clear()
    t = min(times)
    return {"value": round(size * size / t / 1e6, 2), "unit": UNIT, "ms_per_pass": round(t * 1e3, 2),
            "ms_per_pass_all": [round(x * 1e3, 2) for x in times], "via": via, "calls": 16, "nlabels_filtered": int(n),
            "host_memory": "pageable numpy arrays (what the tools hold)", "cache": st}


def config5_record(job, lib, bc, size, banded):
    """BASELINE configs[4]: the pathological DEM (5 m plateaus = large exact flats, nested square craters centred on
    the k * rows / 8 band edges, a raster-wide flat strip) through the whole path, whole on one GPU or as row bands,
    certified, then the bluespot network and the 10 / 30 / 100 mm rain events on the device (SURVEY.md 8(f1, f2))."""
    import torch
    spec = importlib.util.spec_from_file_location("c5_check", os.path.join(ROOT, "tools", "c5_check.py"))
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    c5 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(c5)
    if banded:
        from malstroem_b200 import bands
        pipe = bands.BandPipeline(size, size, bands.DistComm(), device=job.local)
        pipe.dem.copy_(c5.pathological_dem_device(size, row0=pipe.r0, nrows=pipe.rows, device=job.local))
    else:
        from malstroem_b200.pipeline import RasterPipeline
        pipe = RasterPipeline(size, size, device=job.local, with_accum=True)
        pipe.dem.copy_(c5.pathological_dem_device(size, device=job.local))
    torch.cuda.synchronize()
    ms, _, _, _ = timed_steps(job, lib, pipe, 2, 3, profile=False)
    par = parity_record(job, pipe, banded, size, size, bc, single_compare=False)
    events = [10.0, 30.0, 100.0]
    pipe.network(cell_area=0.16, events_mm=events)       # warm-up
    job.barrier()
    t0 = time.perf_counter()
    net = pipe.network(cell_area=0.16, events_mm=events)
    job.barrier()
    net_ms = job.max_over_ranks([(time.perf_counter() - t0) * 1e3])[0]
    tabs = pipe.tables if banded else {k: pipe.table(k) for k in pipe.tables}
    cap = tabs["st_sum"] * 0.16
    roots = net["parent"] < 0
    rain = []
    for e, mm_ in enumerate(events):
        r, sp, v = net["rainv"][e], net["spillv"][e], net["v"][e]
        lhs, rhs = float(r.sum()), float(v.sum() + sp[roots].sum())
        rain.append({"mm": mm_, "conservation_rel_error": abs(lhs - rhs) / max(lhs, 1e-300),
                     "bound_violations": int(((v < 0) | (v > cap) | (sp < 0) | ((sp > 0) & (v < cap))).sum()),
                     "full_bluespots": int(((v >= cap) & (cap > 0)).sum())})
    rec = {"workload": "pathological DEM %dx%d float32 (5 m plateaus, nested craters on the k*rows/8 band edges, a "
                       "raster-wide flat) + bluespot network + rain events 10/30/100 mm" % (size, size),
           "baseline_config": "BASELINE.json configs[4]",
           "parallelism": ("%d row bands, one per GPU" % job.world) if banded else "1 GPU",
           "ms_per_step": round(ms / 2, 3), "value": round(size * size * 2 / (ms * 1e-3) / 1e6, 2), "unit": UNIT,
           "network_and_rain_ms": round(net_ms, 2), "nodes": int(net["parent"].numel()), "roots": int(roots.sum()),
           "rain_events": rain, "parity": par, "stats": dict(pipe.stats)}
    if banded:
        pipe.close()
    del pipe, net
    torch.cuda.empty_cache()
    return rec


def sub_record(job, lib, size, steps, warmup, e2e_steps=2):
    """One more single-GPU size on the same line (rank 0's GPU): device-resident value and e2e."""
    import torch
    pipe = make_pipe(job, size, size, False)
    ms, _, _, _ = timed_steps(job, lib, pipe, steps, warmup, profile=False)
    e2e_ms = timed_e2e(job, pipe, e2e_steps)
    n = size * size
    rec = {"workload": WORKLOAD % (size, size), "ms_per_step": round(ms / steps, 3),
           "value": round(n * steps / (ms * 1e-3) / 1e6, 2), "unit": UNIT, "steps": steps, "warmup": warmup,
           "e2e": {"value": round(n * e2e_steps / (e2e_ms * 1e-3) / 1e6, 2), "unit": UNIT,
                   "ms_per_step": round(e2e_ms / e2e_steps, 3), "h2d_bytes_per_step": pipe.bytes_h2d(),
                   "d2h_bytes_per_step": pipe.bytes_d2h()},
           "nlabels": pipe.nlabels}
    del pipe
    torch.cuda.empty_cache()
    return rec


def run_ours(args):
    import torch
    from malstroem_b200 import _lib

    job = Job()
    world, rank = job.world, job.rank
    lib = _lib.lib()
    bc = load_big_check()
    S = args.size
    n = S * S
    banded = world > 1
    pipe = make_pipe(job, S, S, banded)
    torch.cuda.synchronize()
    ms, launches, prof, clocks = timed_steps(job, lib, pipe, args.steps, args.warmup, profile=True,
                                             sampler=(lambda: ClockSampler(job.local)) if rank == 0 else None)
    if args.dump_outputs:
        dumped = dump_outputs(pipe, args.dump_outputs)
    # ---- e2e: host buffers in, host buffers out
    e2e_steps = max(1, min(args.steps, 2))
    e2e_ms = timed_e2e(job, pipe, e2e_steps)
    h2d, d2h = pipe.bytes_h2d(), pipe.bytes_d2h()
    if banded:
        tot = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
        import torch.distributed as dist
        dist.all_reduce(tot)
        h2d, d2h = int(tot[0]), int(tot[1])
    if hasattr(pipe, "_host"):
        pipe._host = None            # pinned buffers are not needed any more
    parity = None if args.no_parity else parity_record(job, pipe, banded, S, S, bc)
    nlabels, stats = pipe.nlabels, dict(pipe.stats)
    if banded:
        pipe.close()
    del pipe
    torch.cuda.empty_cache()
    sub = {}
    if not args.no_sub:
        if world == 1:
            if S != 8192:
                sub["config2"] = sub_record(job, lib, 8192, max(3, args.steps), 3)
                sub["config2"]["baseline_config"] = "BASELINE.json configs[1]"
                sub["config2"]["e2e_plugin"] = plugin_record(8192)
            w = ref_window(args.steps, args.warmup)
            sub["same_config"] = sub_record(job, lib, w, max(5, args.steps), 3)
            sub["same_config"]["note"] = ("the window `bench.py --impl reference --steps %d --warmup %d` times "
                                          "(%dx%d): GPU arm on the same DEM window" % (args.steps, args.warmup, w, w))
        if not args.no_config5 and (world == 1 or world == 8 or args.config5_size):
            sub["config5"] = config5_record(job, lib, bc, args.config5_size or S, banded)
        big = args.config4_size or (65536 if world == 8 and not args.no_config4 else 0)
        if big and world > 1:
            p4 = make_pipe(job, big, big, True)
            ms4, _, _, _ = timed_steps(job, lib, p4, 2, 2, profile=False)
            par4 = parity_record(job, p4, True, big, big, bc, single_compare=False)
            sub["config4"] = {"workload": WORKLOAD % (big, big), "baseline_config": "BASELINE.json configs[3]",
                              "parallelism": "%d row bands of %d rows, one per GPU" % (world, p4.rows),
                              "ms_per_step": round(ms4 / 2, 3), "steps": 2, "warmup": 2,
                              "value": round(big * big * 2 / (ms4 * 1e-3) / 1e6, 2), "unit": UNIT,
                              "pipeline_frac": None, "nlabels": p4.nlabels, "parity": par4,
                              "e2e": "not measured: the 107 GB of output rasters do not fit the host's pinned memory"}
            peak, _ = peaks()
            sub["config4"]["pipeline_frac"] = round(sub["config4"]["value"] * 1e6 * BYTES_PER_CELL / (world * peak * 1e9), 5)
            p4.close()
            del p4
            torch.cuda.empty_cache()
    if rank == 0:
        peak, peak_kind = peaks()
        value = n * args.steps / (ms * 1e-3) / 1e6
        e2e = n * e2e_steps / (e2e_ms * 1e-3) / 1e6
        # dominant kernel: largest share of the kernel time inside the timed region (rank 0's kernels)
        tot_ms = sum(v[1] for v in prof.values())
        dname, (dn, dms, dunits) = max(prof.items(), key=lambda kv: kv[1][1])
        cells_rank = n // world
        units = dunits if dunits else dn * cells_rank
        bpc = STAGE_BYTES.get(dname, 8)
        achieved = bpc * units / (dms * 1e-3) / 1e9
        traffic = None
        try:        # per-launch DRAM bytes of this kernel at this size from the committed ncu capture, if there is one
            with open(os.path.join(ROOT, "profiles", "top_kernel_traffic.json")) as f:
                ent = json.load(f).get(dname, {}).get(str(S) if world == 1 else "%d/%d" % (S, world))
            if ent:
                traffic = {"dram_bytes_per_launch": ent["dram_bytes_per_launch"],
                           "vs_algorithmic": round(ent["dram_bytes_per_launch"] / (bpc * units / max(dn, 1)), 3),
                           "source": ent["source"]}
        except (OSError, ValueError):
            pass
        kernels = {k: {"launches": v[0], "ms_per_step": round(v[1] / args.steps, 3),
                       "share": round(v[1] / tot_ms, 4)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
        line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
                "config": {"workload": WORKLOAD % (S, S),
                           "baseline_config": "BASELINE.json configs[2]" if S == 32768 else "--size %d" % S,
                           "parallelism": "1 GPU" if world == 1 else
                           "%d row bands of %d rows of the SAME %dx%d raster, one band per GPU, exchanges over NCCL / "
                           "NVLink peer memory" % (world, -(-S // world), S, S),
                           "l2": "inputs (%.1f GB DEM, %.1f GB working set) exceed the 126 MB L2; no flush" %
                                 (n * 4 / 1e9, n * 37 / 1e9),
                           "timed_region": "per-kernel CUDA event pairs are recorded inside the timed region (they are "
                                           "the source of `kernels` and `roofline`)",
                           "e2e_d2h": "filled f32, depths f32, flowdir u8, accum f64, bluespot labels i32, watersheds i32 "
                                      "(what DemTool / BluespotTool write, dem.py:67-93, bluespots.py:169,189) + all "
                                      "per-label tables; the float64 no-flats surface is an intermediate and stays in HBM",
                           "nlabels": nlabels, "stats": stats},
                "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_ms / e2e_steps, 3), "steps": e2e_steps},
                "gpu_launches": launches,
                "roofline": {"bound": "hbm", "kernel": dname, "achieved": round(achieved, 2), "peak": peak,
                             "peak_kind": peak_kind, "unit": "GB/s", "frac": round(achieved / peak, 4),
                             "traffic": traffic, "bytes_per_unit": bpc, "units_per_launch": units // max(dn, 1),
                             "launch_ms": round(dms / max(dn, 1), 4), "share_of_kernel_time": round(dms / tot_ms, 4),
                             "kernel_ms_per_step_rank0": round(tot_ms / args.steps, 3),
                             "pipeline_frac": round(value * 1e6 * BYTES_PER_CELL / (world * peak * 1e9), 5)},
                "parity": parity, "kernels": kernels, "clocks": clocks}
        if args.dump_outputs:
            line["dump_outputs"] = {"dir": args.dump_outputs, "bytes": dumped,
                                    "sample": "%d cells, %d labels, seed %d" % (DUMP_CELLS, DUMP_LABELS, DUMP_SEED)}
        line.update(sub)
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def cpu_baseline(args):
    from malstroem_b200 import synth
    s = args.ref_size_baseline
    dem = synth.fractal_dem(s, s, seed=1)
    mods = stock_reference()
    if mods is not None:
        t = reference_stages(mods, dem)
        kind = "reference"
    else:
        t = port_stages(dem)
        kind = "port"
    return {"value": round(s * s / t / 1e6, 4), "unit": UNIT, "cores": 1, "kind": kind,
            "sample": "%dx%d window (origin 0,0) of the same seed-1 fractal DEM, all stages once through the stock "
                      "functions of baseline/_ref (%.1f s)" % (s, s, t),
            "host_cpus_available": len(os.sched_getaffinity(0))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=32768, help="edge of the ONE raster every configuration of N works on")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--ref-size", type=int, default=0, help="window edge per step of --impl reference (0: from K + W)")
    ap.add_argument("--ref-size-baseline", type=int, default=2048, help="window edge of the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the certificates / single-GPU comparison")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records (config2, same_config, config4)")
    ap.add_argument("--no-config4", action="store_true", help="N = 8: skip the 65536^2 sub-record")
    ap.add_argument("--no-config5", action="store_true", help="skip the pathological-DEM sub-record (N = 1 and N = 8)")
    ap.add_argument("--config5-size", type=int, default=0, help="edge of the `config5` sub-record (default: --size)")
    ap.add_argument("--config4-size", type=int, default=0, help="N > 1: edge of the `config4` sub-record (default: 65536 at N = 8, none otherwise)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of every raster and table of the last step as "
                         "DIR/<name>.npy (one GPU, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs a single-GPU run of --impl ours")
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    # exactly one JSON line on stdout: libraries that write to fd 1 (NCCL's version banner) go to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
