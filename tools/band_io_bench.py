"""GeoTIFF files in and out of a banded run: the S^2 fractal DEM (seed 1) is synthesized band by band, written as one
file by every band (RasterWriter.write_band), read back band by band into BandPipeline.dem (RasterReader.read_rows)
and checked; the pipeline runs; the six rasters the host front end ships (filled, depths, flowdir, accum, labels,
wsheds) are written the same way, and every file is read back band by band and compared with torch.equal.  Where the
raster fits one device (<= 2^30 cells) rank 0 also runs RasterPipeline + RasterWriter.write on the same DEM and
compares the files' bytes (sha256).
Per raster: encode + pack time on the device (max over ranks), bytes exchanged across band edges (all ranks), file
size against raw size, write and read wall time (between barriers) and the aggregate rate (raw bytes / wall time).
Files go to a scratch directory (--dir, default the system's temporary directory), each is deleted after its check,
and a raster is skipped, with the reason printed, when the file system has too little free space for it.
usage: python -m torch.distributed.run --nproc-per-node N tools/band_io_bench.py [--size 32768] [--dir D]
   or: python tools/band_io_bench.py --threads N ...   (N bands as threads of one process on one GPU)"""
import argparse
import hashlib
import os
import shutil
import sys
import tempfile
import threading
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from malstroem_b200 import bands, io as mio  # noqa: E402
from malstroem_b200.pipeline import RasterPipeline, synth_fractal  # noqa: E402
from band_flood_bench import card  # noqa: E402

TRANSFORM = (720000.0, 0.4, 0.0, 6193000.0, 0.0, -0.4)
NAMES = ("filled", "depths", "flowdir", "accum", "labels", "wsheds")
SINGLE_GPU_CELLS = 1 << 30        # rows * cols <= 2^30 on one device (DESIGN §3)

_print_lock = threading.Lock()


def say(comm, *a):
    if comm.rank == 0:
        with _print_lock:
            print(*a)
            sys.stdout.flush()


def agree(comm, dev, x, op):
    return comm.all_reduce(torch.tensor([x], dtype=torch.float64, device=dev), op).item()


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 24), b""):
            h.update(b)
    return h.hexdigest()


def enough_space(comm, dev, d, raw):
    """rank 0 decides for everyone: the file (deflate output is at most ~1.15x raw) plus 1 GB must fit"""
    free = shutil.disk_usage(d).free if comm.rank == 0 else 0
    need = int(raw * 1.15) + (1 << 30)
    ok = agree(comm, dev, 1.0 if comm.rank != 0 or free >= need else 0.0, "min") > 0
    return ok, free, need


def one_raster(comm, dev, p, name, t, d, hashes, into=None):
    """write_band `t` (this band's rows) to d/name.tif, read it back band by band, check; returns ok"""
    path = os.path.join(d, name + ".tif")
    raw = p.R * p.cols * t.element_size()
    ok_space, free, need = enough_space(comm, dev, d, raw)
    if not ok_space:
        say(comm, "%-8s skipped: %.1f GB free in %s, %.1f GB needed" % (name, free / 1e9, d, need / 1e9))
        return True
    w = mio.RasterWriter(path, TRANSFORM, "EPSG:25832")
    agree(comm, dev, 0.0, "sum")
    torch.cuda.synchronize(dev)
    a = time.perf_counter()
    w.write_band(comm, t, p.r0, p.R, device=dev)
    t_w = agree(comm, dev, time.perf_counter() - a, "max")
    enc = agree(comm, dev, w.stats["encode_ms"], "max")
    exch = agree(comm, dev, w.stats["exchanged_bytes"], "sum")
    r = mio.RasterReader(path)
    back = into if into is not None else torch.empty_like(t)
    agree(comm, dev, 0.0, "sum")
    torch.cuda.synchronize(dev)
    a = time.perf_counter()
    r.read_rows(p.r0, p.r1, device=dev, out=back)
    torch.cuda.synchronize(dev)
    t_r = agree(comm, dev, time.perf_counter() - a, "max")
    same = agree(comm, dev, 1.0 if torch.equal(back, t) else 0.0, "min") > 0
    fb = w.stats["file_bytes"]
    say(comm, "%-8s %-8s %9.1f %9.1f %6.2f %9.2f %12d %9.1f %9.1f %6.2f/%5.2f  read back equal: %s"
        % (name, str(t.dtype).replace("torch.", ""), raw / 1e6, fb / 1e6, raw / fb, enc, int(exch), t_w * 1e3,
           t_r * 1e3, raw / t_w / 1e9, raw / t_r / 1e9, same))
    if comm.rank == 0:
        if hashes is not None:
            hashes[name] = sha256(path)
        os.remove(path)
    return same


def work(comm, dev, S, base):
    # one scratch directory for all ranks: rank 0 makes it, everyone learns its name
    name = tempfile.mkdtemp(prefix="band_io_", dir=base) if comm.rank == 0 else ""
    got = comm.all_gather_var(torch.tensor(list(name.encode()) or [0], dtype=torch.uint8, device=dev))
    d = bytes(got[0].cpu().tolist()).decode()
    try:
        return _work(comm, dev, S, d)
    finally:
        agree(comm, dev, 0.0, "sum")
        if comm.rank == 0:
            shutil.rmtree(d, ignore_errors=True)


def _work(comm, dev, S, d):
    single = S * S <= SINGLE_GPU_CELLS
    hashes = {} if single and comm.rank == 0 else None
    p = bands.BandPipeline(S, S, comm, device=dev)
    say(comm, "== %dx%d fractal DEM (seed 1) in %d bands, files in %s" % (S, S, comm.size, d))
    say(comm, "band rows: %s" % bands.band_rows(S, comm.size))
    crossing = sum(1 for x in mio.band_tile_plan(bands.band_rows(S, comm.size), S) if x["cross"] is not None)
    say(comm, "tile rows that cross a band edge: %d" % crossing)
    say(comm, "%-8s %-8s %9s %9s %6s %9s %12s %9s %9s %12s" % ("raster", "dtype", "raw MB", "file MB", "ratio",
                                                             "encode ms", "edge bytes", "write ms", "read ms",
                                                             "GB/s w/r"))
    want = synth_fractal(p.rows, S, seed=1, row0=p.r0, device=dev.index)
    ok = one_raster(comm, dev, p, "dem", want, d, hashes, into=p.dem)
    del want
    torch.cuda.empty_cache()
    p.run()
    for name in NAMES:
        ok = one_raster(comm, dev, p, name, p.out[name], d, hashes) and ok
    p.close()
    del p
    torch.cuda.empty_cache()
    if single:
        ident = True
        if comm.rank == 0:
            q = RasterPipeline(S, S, device=dev)
            synth_fractal(S, S, seed=1, device=dev.index, out=q.dem)
            q.run()
            for name in ("dem",) + NAMES:
                if name not in hashes:
                    continue
                path = os.path.join(d, "whole_" + name + ".tif")
                torch.cuda.synchronize(dev)
                a = time.perf_counter()
                mio.RasterWriter(path, TRANSFORM, "EPSG:25832").write(q.dem if name == "dem" else q.out[name],
                                                                       device=dev.index)
                t_w = time.perf_counter() - a
                same = sha256(path) == hashes[name]
                os.remove(path)
                print("%-8s file byte-identical to RasterPipeline + RasterWriter.write: %s  (that write: %.1f ms)"
                      % (name, same, t_w * 1e3))
                ident = ident and same
            del q
            torch.cuda.empty_cache()
        ident = agree(comm, dev, 1.0 if ident else 0.0, "min") > 0
        say(comm, "all files byte-identical to the single-GPU writer: %s" % ident)
        ok = ok and ident
    else:
        say(comm, "single-GPU comparison: not run (%d cells is more than one device holds)" % (S * S))
    return ok


def threaded(args):
    print("cards: ['%s']  (%d bands as threads on one GPU)" % (card(), args.threads))
    grp = bands.ThreadGroup(args.threads)
    res, errs = [None] * args.threads, []

    def run(rank):
        try:
            torch.cuda.set_device(0)
            res[rank] = work(bands.ThreadComm(grp, rank), torch.device("cuda", 0), args.size, args.dir)
        except BaseException as e:      # noqa: BLE001 - report and release the other threads
            errs.append(e)
            grp.barrier.abort()

    ts = [threading.Thread(target=run, args=(r,)) for r in range(args.threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errs:
        raise [e for e in errs if not isinstance(e, threading.BrokenBarrierError)][0]
    return all(res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--dir", default=None, help="scratch directory for the files (default: the temporary directory)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("band_io_bench needs CUDA devices")
    if args.threads:
        ok = threaded(args)
        print("RESULT OK" if ok else "RESULT FAIL")
    else:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        comm = bands.DistComm()
        dev = torch.device("cuda", local)
        try:
            names = comm.all_gather_var(torch.tensor(list(card().encode()), dtype=torch.uint8, device=dev))
            say(comm, "cards: %s" % sorted(set(bytes(x.cpu().tolist()).decode() for x in names)))
            ok = work(comm, dev, args.size, args.dir)
            say(comm, "RESULT OK" if ok else "RESULT FAIL")
        finally:
            dist.destroy_process_group()
    if not ok:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
