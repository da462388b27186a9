"""The bluespot filter (csrc/bfilter.cu) timed and certified on device-resident pipeline runs.

Workloads: the fractal DEM (seed 1) and the pathological DEM (BASELINE configs[4], tools/c5_check.py) at S x S, with
`-filter 'maxdepth > 0.05'` and the cell area 0.16.  `RasterPipeline.run()` and `run(bluespot_filter=...)` are timed
alternately with CUDA events (warm-up, then the median of the repetitions); one profiled run of each (ms_profile)
splits the added time into raw stats, keep + LUT and relabel (per-kernel totals, filtered minus unfiltered); the
network + 3 rain events + flood are timed on both.  Certificates: the unfiltered run's tables, evaluated with plain
torch ops (FilterProgram.evaluate) and ranked with torch.cumsum, must give the filtered labels bitwise; the watershed
recurrence and the table certificates of tools/big_check.py must hold on the filtered rasters.  Then one line per
row-band run (bands as threads on one GPU, N = 2 / 4): wall time with and without the filter, labels equal to the
single-GPU filtered run.
usage: python tools/filter_bench.py [S] [--reps 5] [--no-c5] [--no-bands]"""
import argparse
import ctypes
import importlib.util
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from malstroem_b200 import _lib, bands  # noqa: E402
from malstroem_b200 import bluespot_filter as bf  # noqa: E402
from malstroem_b200.pipeline import RasterPipeline, synth_fractal  # noqa: E402
import big_check  # noqa: E402
from flood_bench import card  # noqa: E402

FILTER, CA, MM = "maxdepth > 0.05", 0.16, [10.0, 30.0, 100.0]
STAGES = (("raw stats", ("k_stats_init", "k_label_stats", "k_stats_finish")),
          ("keep + LUT", ("k_bluespot_keep", "k_scan_reduce", "k_scan_bsums", "k_scan_final", "k_keep_lut")),
          ("relabel", ("k_relabel",)))


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def median(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2], ts[0], ts[-1]


def profile(fn):
    """ms_profile per-kernel totals {name: (launches, ms)} of one call of fn."""
    with _lib.lock:
        _lib.check(_lib.lib().ms_profile(1), "ms_profile")
    fn()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    with _lib.lock:
        _lib.check(_lib.lib().ms_profile_report(buf, len(buf)), "ms_profile_report")
        _lib.check(_lib.lib().ms_profile(0), "ms_profile")
    out = {}
    for line in buf.value.decode().splitlines():
        f = line.split()
        if len(f) >= 3:
            name = f[0].split("<")[0].split("::")[-1]
            n, ms = out.get(name, (0, 0.0))
            out[name] = (n + int(f[1]), ms + float(f[2]))
    return out


def workload(name, pipe, reps):
    kw = dict(bluespot_filter=FILTER, cell_area=CA)
    pipe.run()
    pipe.run(**kw)
    torch.cuda.synchronize()
    t_plain, t_filt = [], []
    for _ in range(reps):
        t_plain.append(event_ms(lambda: pipe.run()))
        t_filt.append(event_ms(lambda: pipe.run(**kw)))
    raw, kept = pipe.stats["bluespots_raw"], pipe.nlabels
    print("== %s: %d raw bluespots, %d kept by %r (cell area %g)" % (name, raw, kept, FILTER, CA))
    mp, mf = median(t_plain), median(t_filt)
    print("   pipeline run(), alternating, %d reps: unfiltered median %.2f ms (min %.2f, max %.2f); filtered median "
          "%.2f ms (min %.2f, max %.2f); added %.2f ms" % ((reps,) + mp + mf + (mf[0] - mp[0],)))
    pp, pf = profile(lambda: pipe.run()), profile(lambda: pipe.run(**kw))
    total = 0.0
    for stage, kernels in STAGES:
        ms = sum(pf.get(k, (0, 0.0))[1] - pp.get(k, (0, 0.0))[1] for k in kernels)
        total += ms
        print("   added kernels, %-10s %7.2f ms  (%s)" % (stage + ":", ms, ", ".join(
            "%s %d x %.2f ms" % (k, pf[k][0] - pp.get(k, (0, 0))[0], pf[k][1] - pp.get(k, (0, 0.0))[1])
            for k in kernels if k in pf and pf[k][0] > pp.get(k, (0, 0))[0])))
    print("   added kernels, total:     %7.2f ms" % total)
    for k in ("k_tables_a2", "k_tables_b"):
        if k in pp:
            print("   for comparison, %s: %.2f ms unfiltered, %.2f ms filtered" % (k, pp[k][1], pf.get(k, (0, 0.0))[1]))
    for label, args in (("unfiltered", {}), ("filtered", kw)):
        pipe.run(**args)
        net = pipe.network(cell_area=CA, events_mm=MM)
        pipe.flood(net, CA)
        t_net = median([event_ms(lambda: pipe.network(cell_area=CA, events_mm=MM)) for _ in range(reps)])
        t_fl = median([event_ms(lambda: pipe.flood(net, CA)) for _ in range(reps)])
        print("   %-10s %8d bluespots: network + rain events (3) median %.2f ms, flood (3 events) median %.2f ms"
              % (label, pipe.nlabels, t_net[0], t_fl[0]))
    # certificates
    pipe.run()
    raw_lab = pipe.out["labels"].clone()
    m = pipe.nlabels + 1
    prog = bf.compile_filter(FILTER)
    keep = prog.evaluate(pipe.table("st_count").double() * CA, pipe.table("st_max"), pipe.table("st_sum") * CA)
    keep[0] = False
    lut = (torch.cumsum(keep.to(torch.int64), 0) * keep).to(torch.int32)
    pipe.run(**kw)
    same = bool(torch.equal(pipe.out["labels"], lut[raw_lab.long()]))
    del raw_lab
    ok_n = pipe.nlabels == int(keep.sum()) and pipe.stats["bluespots_raw"] == m - 1
    bad_fill, bad_acc, bad_ws, _ = big_check.certify(pipe)
    more = big_check.certify_more(pipe, pipe.short, pipe.diag)
    bad_tab = sum(more["tables"].values())
    bad_num = more["cc_unused_labels"] + more["cc_order"]
    good = same and ok_n and bad_ws == 0 and bad_fill == 0 and bad_acc == 0 and bad_tab == 0 and bad_num == 0
    print("   certificate: filtered labels == torch lut[raw labels] bitwise: %s; kept count matches: %s; watershed "
          "recurrence violations: %d; fill / accumulation violations: %d / %d; table violations: %d %s; labels "
          "unused or out of first-cell order: %d -> %s"
          % (same, ok_n, bad_ws, bad_fill, bad_acc, bad_tab, more["tables"], bad_num, "ok" if good else "FAIL"))
    sys.stdout.flush()
    return good


def band_lines(dem, want_labels, want_n, counts):
    ok = True
    for nb in counts:
        ts = {}
        for label, kw in (("unfiltered", {}), ("filtered", dict(bluespot_filter=FILTER, cell_area=CA))):
            pipes = bands.run_threaded(dem, nb, **kw)          # warm-up
            for p in pipes:
                p.close()
            del pipes
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipes = bands.run_threaded(dem, nb, **kw)
            ts[label] = (time.perf_counter() - t0) * 1e3
            if kw:
                got = torch.cat([p.out["labels"] for p in pipes])
                same = bool(torch.equal(got, want_labels)) and all(p.nlabels == want_n for p in pipes)
                del got
            for p in pipes:
                p.close()
            del pipes
            torch.cuda.empty_cache()
        ok = ok and same
        print("   bands as threads, N = %d: run %.1f ms unfiltered, %.1f ms filtered (wall clock, one run after a "
              "warm-up); labels and counts equal to the single-GPU filtered run: %s"
              % (nb, ts["unfiltered"], ts["filtered"], same))
        sys.stdout.flush()
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("size", type=int, nargs="?", default=32768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--no-bands", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("filter_bench needs a CUDA device")
    print("card: %s" % card())
    s = args.size
    pipe = RasterPipeline(s, s)
    synth_fractal(s, s, seed=1, out=pipe.dem)
    ok = workload("fractal %dx%d (seed 1)" % (s, s), pipe, args.reps)
    if not args.no_bands:
        dem = pipe.dem.clone()
        want, n = pipe.out["labels"].clone(), pipe.nlabels          # the filtered run is the last one
        del pipe
        torch.cuda.empty_cache()
        ok = band_lines(dem, want, n, (2, 4)) and ok
        del dem, want
    else:
        del pipe
    torch.cuda.empty_cache()
    if not args.no_c5:
        spec = importlib.util.spec_from_file_location("c5_check", os.path.join(ROOT, "tools", "c5_check.py"))
        c5 = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(c5)
        pipe = RasterPipeline(s, s)
        pipe.dem.copy_(c5.pathological_dem_device(s, device=0))
        ok = workload("pathological %dx%d (config 5)" % (s, s), pipe, args.reps) and ok
    print("RESULT %s" % ("OK" if ok else "FAIL"))
    if not ok:
        raise SystemExit("filter_bench: a certificate failed")


if __name__ == "__main__":
    main()
