"""Water levels and water-depth rasters (csrc/flood.cu) timed on device-resident pipeline runs.

Workloads: the 8192^2 and 32768^2 fractal DEMs (seed 1) and the 32768^2 pathological DEM (BASELINE configs[4], see
tools/c5_check.py), each with the 10 / 30 / 100 mm bluespot network.  Times `RasterPipeline.flood` (3 events) and one
`water_depth` with CUDA events (warm-up, then the median of the repetitions), next to the network + rain events on the
same raster.  At 32768^2 it checks conservation with torch scatter reductions: per bluespot sum(d) * ca == v to 1e-6
relative, every wet cell in a bluespot, d <= depths.
usage: python tools/flood_bench.py [--reps 10] [--sizes 8192,32768] [--no-c5]"""
import argparse
import importlib.util
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from malstroem_b200 import _lib  # noqa: E402
from malstroem_b200.pipeline import RasterPipeline, synth_fractal  # noqa: E402

PEAK_GBS = 6556.5          # measured HBM copy bandwidth of the B200 (DESIGN.md)
CA, MM = 0.16, [10.0, 30.0, 100.0]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return "%s, power limit %s" % (name, pl or "unknown")


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def segment_classes(pipe):
    cnt = pipe.table("st_count")[1:]
    out = []
    for lo, hi in ((1, 512), (513, 8192), (8193, 1 << 40)):
        m = (cnt >= lo) & (cnt <= hi)
        out.append("%d..%s cells: %d labels, %d cells" % (lo, hi if hi < 1 << 40 else "", int(m.sum()),
                                                        int(cnt[m].sum())))
    return "; ".join(out)


def workload(name, pipe, reps, certify):
    n = pipe.rows * pipe.cols
    pipe.run()
    torch.cuda.synchronize()
    net = pipe.network(cell_area=CA, events_mm=MM)
    t_net = timed(lambda: pipe.network(cell_area=CA, events_mm=MM), reps)
    fl = pipe.flood(net, CA)
    t_fl = timed(lambda: pipe.flood(net, CA), reps)
    wet_cells = int(pipe.table("st_count")[1:].sum())
    out = torch.empty((pipe.rows, pipe.cols), dtype=torch.float32, device=pipe.device)
    t_d = timed(lambda: pipe.water_depth(fl["level"][1], out=out), reps)
    print("== %s: %d labels, %d bluespot cells (%.1f %%)" % (name, pipe.nlabels, wet_cells, 100.0 * wet_cells / n))
    print("   segments: %s" % segment_classes(pipe))
    print("   wet cells after 10/30/100 mm: %s" % [int(fl["wet"][e].sum()) for e in range(len(MM))])
    print("   network + rain events (3): median %.2f ms (min %.2f, max %.2f)" % t_net)
    # bytes the algorithm has to move: labels + F (count pass), labels + F + dem (scatter pass), the 4 B key of every
    # bluespot cell written once and read once by the sort / scan
    fb = 20.0 * n + 8.0 * wet_cells
    print("   flood levels (3 events):    median %.2f ms (min %.2f, max %.2f); %.1f B/cell -> %.0f GB/s = %.1f %% of %.1f"
          % (t_fl + (fb / n, fb / (t_fl[0] * 1e-3) / 1e9, 100.0 * fb / (t_fl[0] * 1e-3) / 1e9 / PEAK_GBS, PEAK_GBS)))
    gbs = 16.0 * n / (t_d[0] * 1e-3) / 1e9
    print("   water_depth (1 event):      median %.2f ms (min %.2f, max %.2f); 16 B/cell -> %.0f GB/s = %.1f %% of %.1f"
          % (t_d + (gbs, 100.0 * gbs / PEAK_GBS, PEAK_GBS)))
    with _lib.lock:
        _lib.check(_lib.lib().ms_profile(1), "ms_profile")
    pipe.flood(net, CA)
    torch.cuda.synchronize()
    import ctypes
    buf = ctypes.create_string_buffer(1 << 16)
    with _lib.lock:
        _lib.check(_lib.lib().ms_profile_report(buf, len(buf)), "ms_profile_report")
        _lib.check(_lib.lib().ms_profile(0), "ms_profile")
    print("   per-kernel (one profiled flood call):")
    for line in buf.value.decode().splitlines():
        print("     " + line)
    ok_all = True
    if certify:
        lab = pipe.out["labels"].view(-1).long()
        depths = pipe.out["depths"].view(-1)
        count = pipe.table("st_count").double()
        L = torch.zeros(pipe.nlabels + 1, dtype=torch.float64, device=pipe.device)
        L[lab] = pipe.out["filled"].view(-1).double()
        for e in range(len(MM)):
            d = pipe.water_depth(fl["level"][e], out=out).view(-1)
            vol = torch.zeros(pipe.nlabels + 1, dtype=torch.float64, device=pipe.device)
            vol.index_add_(0, lab, d.double())
            vol *= CA
            v = net["v"][e]
            ok = ~torch.isnan(v)
            ok[0] = False
            err = (vol - v).abs()
            rel = (err / v.abs().clamp_min(1e-300))[ok & (v > 0)]
            # 1e-6 relative, plus the float64 rounding of the level itself (a few ulp of |L|, over every cell)
            tol = 1e-6 * v.abs() + 4 * 2.0 ** -52 * L.abs() * count * CA
            within = bool((err[ok] <= tol[ok]).all())
            zero_ok = bool((vol[ok & (v == 0)] == 0).all())
            outside = int(((d > 0) & (lab == 0)).sum())
            above = int((d > depths).sum())
            worst = float(rel.max()) if rel.numel() else 0.0
            good = within and zero_ok and outside == 0 and above == 0
            print("   certificate %g mm: max rel |sum(d)*ca - v| = %.3e (all within 1e-6 rel + float64 level rounding: "
                  "%s), v = 0 -> no water: %s, wet cells outside bluespots: %d, cells with d > depths: %d -> %s"
                  % (MM[e], worst, within, zero_ok, outside, above, "ok" if good else "FAIL"))
            ok_all = ok_all and good
        del lab, depths, L
    sys.stdout.flush()
    return ok_all


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sizes", default="8192,32768")
    ap.add_argument("--no-c5", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flood_bench needs a CUDA device")
    print("card: %s" % card())
    ok = True
    for s in [int(x) for x in args.sizes.split(",")]:
        pipe = RasterPipeline(s, s)
        synth_fractal(s, s, seed=1, out=pipe.dem)
        ok = workload("fractal %dx%d" % (s, s), pipe, args.reps, s >= 32768) and ok
        del pipe
        torch.cuda.empty_cache()
    if not args.no_c5:
        spec = importlib.util.spec_from_file_location("c5_check", os.path.join(ROOT, "tools", "c5_check.py"))
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        c5 = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(c5)
        s = 32768
        pipe = RasterPipeline(s, s)
        pipe.dem.copy_(c5.pathological_dem_device(s, device=0))
        ok = workload("pathological %dx%d (config 5)" % (s, s), pipe, args.reps, True) and ok
    if not ok:
        raise SystemExit("flood_bench: a certificate failed")


if __name__ == "__main__":
    main()
