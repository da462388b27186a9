"""Water levels and depth rasters across row bands (BandPipeline.flood / water_depth), one band per GPU, run under
torch.distributed.run (NCCL).  Workloads: the S^2 fractal DEM (seed 1) and the S^2 pathological DEM (BASELINE
configs[4], tools/c5_check.py) with the 10 / 30 / 100 mm bluespot network, S = 32768 by default; 65536^2 only runs in
bands (a device holds at most 2^30 cells).  Per workload: `flood` for 3 events (CUDA events between two barriers, the
maximum over the ranks, median after a warm-up), one `water_depth`, the z keys sent between bands and the labels that
cross a band edge.  Certificates as tools/flood_bench.py, per band with index_add_ and an all-reduce: per bluespot
sum(d) * ca == v to 1e-6 relative plus the float64 rounding of the level, no wet cell outside a bluespot, d <= depths.
Below 2^31 cells rank 0 also runs the single-GPU flood on the whole raster with the band run's st_sum and v and checks
that levels and wet counts are bitwise equal.
usage: python -m torch.distributed.run --nproc-per-node N tools/band_flood_bench.py [--size 32768] [--reps 5]
       [--no-c5] [--no-fractal]
   or: python tools/band_flood_bench.py --threads N ...   (N bands as threads of one process on one GPU: the bands'
       phases run one after another on the device, so the times are those of all bands together)"""
import argparse
import ctypes
import importlib.util
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from malstroem_b200 import _lib, bands  # noqa: E402
from malstroem_b200.pipeline import synth_fractal  # noqa: E402

CA, MM = 0.16, [10.0, 30.0, 100.0]


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                            text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return "%s, power limit %s" % (name, pl or "unknown")


def say(comm, *a):
    if comm.rank == 0:
        print(*a)
        sys.stdout.flush()


def barrier(comm, dev):
    comm.all_reduce(torch.zeros(1, dtype=torch.int32, device=dev), "sum")
    torch.cuda.synchronize(dev)


def timed(comm, dev, fn, reps):
    """median / min / max over reps (after one warm-up) of the maximum over the ranks, CUDA events between barriers"""
    fn()
    ts = []
    for _ in range(reps):
        barrier(comm, dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        ts.append(float(comm.all_reduce(t, "max").item()))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def total(comm, dev, x):
    return int(comm.all_reduce(torch.tensor([x], dtype=torch.int64, device=dev), "sum").item())


def single_gpu_equal(p, net, fl):
    """Rank 0: ms_flood_levels_dev on the whole raster (gathered) with the band run's st_sum and v."""
    comm, dev, n = p.comm, p.device, p.nlabels + 1
    rasters = (p.dem, p.out["filled"], p.out["labels"])
    if isinstance(comm, bands.ThreadComm):        # one device: rank 0 reads the other bands' rows in place
        parts = [comm._swap(t) for t in rasters]
        whole = [torch.cat(x) for x in parts] if comm.rank == 0 else None
        comm._swap(None)                          # the other bands keep their rows until rank 0 has copied them
    else:                                         # rank 0 receives every band's rows; the others only send
        whole = None
        if comm.rank == 0:
            rows = bands.band_rows(p.R, comm.size)
            whole = [torch.empty((p.R, p.cols), dtype=t.dtype, device=dev) for t in rasters]
            for w, t in zip(whole, rasters):
                w[: p.rows].copy_(t)
                for g in range(1, comm.size):
                    dist.recv(w[rows[g][0]:rows[g][1]], src=g, group=comm.group)
        else:
            for t in rasters:
                dist.send(t.contiguous(), dst=0, group=comm.group)
    if comm.rank != 0:
        del whole
        return True
    ne = len(MM)
    level = torch.empty((ne, n), dtype=torch.float64, device=dev)
    wet = torch.empty((ne, n), dtype=torch.int64, device=dev)
    v = net["v"].contiguous()

    def one():
        with _lib.lock:
            _lib.check(_lib.lib().ms_flood_levels_dev(
                whole[0].data_ptr(), whole[1].data_ptr(), whole[2].data_ptr(), p.R, p.cols, p.nlabels,
                p.tables["st_sum"].data_ptr(), CA, ne, v.data_ptr(), level.data_ptr(), wet.data_ptr(),
                ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "ms_flood_levels_dev")
    one()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    one()
    b.record()
    b.synchronize()
    print("   single-GPU flood of the whole raster (3 events, one run after a warm-up): %.2f ms" % a.elapsed_time(b))
    del whole
    return bool(torch.equal(level.view(torch.int64), fl["level"].view(torch.int64)) and torch.equal(wet, fl["wet"]))


def workload(name, p, reps, ran=False):
    comm, dev = p.comm, p.device
    n = p.R * p.cols
    if not ran:
        p.run()
    net = p.network(cell_area=CA, events_mm=MM)
    fl = p.flood(net, CA)
    t_fl = timed(comm, dev, lambda: p.flood(net, CA), reps)
    out = torch.empty((p.rows, p.cols), dtype=torch.float32, device=dev)
    t_d = timed(comm, dev, lambda: p.water_depth(fl["level"][1], out=out), reps)
    keys = total(comm, dev, p.stats["flood_keys_sent"])
    crossing = total(comm, dev, p.stats["flood_crossing_labels"])
    wet_cells = int(p.tables["st_count"][1:].sum())
    say(comm, "== %s in %d bands: %d labels, %d bluespot cells (%.1f %%)"
        % (name, comm.size, p.nlabels, wet_cells, 100.0 * wet_cells / n))
    say(comm, "   labels crossing a band edge: %d; z keys sent between bands: %d (%.2f %% of the bluespot cells)"
        % (crossing, keys, 100.0 * keys / max(wet_cells, 1)))
    say(comm, "   wet cells after 10/30/100 mm: %s" % [int(fl["wet"][e].sum()) for e in range(len(MM))])
    say(comm, "   flood levels (3 events): median %.2f ms (min %.2f, max %.2f), max over ranks" % t_fl)
    say(comm, "   water_depth (1 event):   median %.2f ms (min %.2f, max %.2f), max over ranks" % t_d)
    # certificates, per band and all-reduced
    lab = p.out["labels"].reshape(-1).long()
    depths = p.out["depths"].reshape(-1)
    count = p.tables["st_count"].double()
    L = torch.zeros(p.nlabels + 1, dtype=torch.float64, device=dev)
    L[lab] = p.out["filled"].reshape(-1).double().abs()
    comm.all_reduce(L, "max")                  # |F| of every label (0 in the bands that lack it)
    ok_all = True
    for e in range(len(MM)):
        d = p.water_depth(fl["level"][e], out=out).view(-1)
        vol = torch.zeros(p.nlabels + 1, dtype=torch.float64, device=dev)
        vol.index_add_(0, lab, d.double())
        comm.all_reduce(vol, "sum")
        vol *= CA
        v = net["v"][e]
        ok = ~torch.isnan(v)
        ok[0] = False
        err = (vol - v).abs()
        rel = (err / v.abs().clamp_min(1e-300))[ok & (v > 0)]
        tol = 1e-6 * v.abs() + 4 * 2.0 ** -52 * L.abs() * count * CA
        within = bool((err[ok] <= tol[ok]).all())
        zero_ok = bool((vol[ok & (v == 0)] == 0).all())
        outside = total(comm, dev, int(((d > 0) & (lab == 0)).sum()))
        above = total(comm, dev, int((d > depths).sum()))
        worst = float(rel.max()) if rel.numel() else 0.0
        good = within and zero_ok and outside == 0 and above == 0
        say(comm, "   certificate %g mm: max rel |sum(d)*ca - v| = %.3e (all within 1e-6 rel + float64 level rounding: "
            "%s), v = 0 -> no water: %s, wet cells outside bluespots: %d, cells with d > depths: %d -> %s"
            % (MM[e], worst, within, zero_ok, outside, above, "ok" if good else "FAIL"))
        ok_all = ok_all and good
    del lab, depths, out
    if n < (1 << 31):
        eq = single_gpu_equal(p, net, fl)
        eq = bool(comm.all_reduce(torch.tensor([0 if eq else 1], dtype=torch.int32, device=dev), "max").item() == 0)
        say(comm, "   levels and wet counts bitwise equal to the single-GPU flood: %s" % eq)
        ok_all = ok_all and eq
    torch.cuda.empty_cache()
    return ok_all


def threaded(args):
    """--threads N: the same workloads with N bands as threads on GPU 0 (bands.run_threaded)."""
    S, ok = args.size, True
    print("cards: ['%s']  (%d bands as threads on one GPU)" % (card(), args.threads))
    sys.stdout.flush()
    loads = []
    if not args.no_fractal:
        loads.append(("fractal %dx%d" % (S, S), synth_fractal(S, S, seed=1)))
    if not args.no_c5:
        spec = importlib.util.spec_from_file_location("c5_check", os.path.join(ROOT, "tools", "c5_check.py"))
        c5 = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(c5)
        loads.append(("pathological %dx%d (config 5)" % (S, S), None))
    for name, dem in loads:
        if dem is None:
            dem = c5.pathological_dem_device(S)
        pipes = bands.run_threaded(dem, args.threads, after=lambda p: workload(name, p, args.reps, ran=True))
        ok = all(p.after_result for p in pipes) and ok
        for p in pipes:
            p.close()
        del pipes, dem
        torch.cuda.empty_cache()
    print("RESULT OK" if ok else "RESULT FAIL")
    if not ok:
        raise SystemExit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--no-fractal", action="store_true")
    ap.add_argument("--threads", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("band_flood_bench needs CUDA devices")
    if args.threads:
        return threaded(args)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    comm = bands.DistComm()
    dev = torch.device("cuda", local)
    names = comm.all_gather_var(torch.tensor(list(card().encode()), dtype=torch.uint8, device=dev))
    say(comm, "cards: %s" % sorted(set(bytes(x.cpu().tolist()).decode() for x in names)))
    S, ok = args.size, True
    try:
        if not args.no_fractal:
            p = bands.BandPipeline(S, S, comm, device=local)
            synth_fractal(p.rows, S, seed=1, row0=p.r0, out=p.dem)
            ok = workload("fractal %dx%d" % (S, S), p, args.reps) and ok
            p.close()
            del p
            torch.cuda.empty_cache()
        if not args.no_c5:
            spec = importlib.util.spec_from_file_location("c5_check", os.path.join(ROOT, "tools", "c5_check.py"))
            c5 = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(c5)
            p = bands.BandPipeline(S, S, comm, device=local)
            p.dem.copy_(c5.pathological_dem_device(S, row0=p.r0, nrows=p.rows, device=local))
            ok = workload("pathological %dx%d (config 5)" % (S, S), p, args.reps) and ok
            p.close()
        say(comm, "RESULT OK" if ok else "RESULT FAIL")
    finally:
        dist.destroy_process_group()
    if not ok:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
