"""Label polygonisation on row bands (vector.polygonize_band) against one GPU (vector.polygonize_labels_device):
bluespot and watershed labels of the S^2 fractal DEM (seed 1).  Per band count: wall time of the collective (device
synchronised at both ends), rings, vertices and boundary edges, the bytes each exchange moves (summed over ranks) and
whether the concatenated polygons equal the single-GPU ones exactly.  Where the raster does not fit one device
(> 2^30 cells) there is no single-GPU run: the property checks of test_pipeline_labels_2048_properties are reported
instead (ring areas: exteriors > 0, holes < 0, their sum = the cell count; axis-parallel closed rings).
usage: python tools/band_poly_bench.py --threads 2,4,8 [--size 32768]      (bands as threads on one GPU)
   or: python -m torch.distributed.run --nproc-per-node N tools/band_poly_bench.py [--size S]"""
import argparse
import os
import sys
import threading
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from malstroem_b200 import bands, vector  # noqa: E402
from malstroem_b200.pipeline import RasterPipeline, synth_fractal  # noqa: E402
from band_flood_bench import card  # noqa: E402

SINGLE_GPU_CELLS = 1 << 30


def flat(rings):
    """(per polygon: value, region, ring count), ring order, as arrays, for an exact comparison."""
    polys = rings.polygons()
    order = np.array([k for _, ks in polys for k in ks], dtype=np.int64)
    head = np.array([[v, int(rings.region[ks[0]]), len(ks)] for v, ks in polys], dtype=np.int64).reshape(-1, 3)
    a, b = rings.offset[order], rings.offset[order + 1]
    n = b - a
    idx = np.repeat(a - np.concatenate([[0], np.cumsum(n)[:-1]]), n) + np.arange(int(n.sum()))
    return {"head": head, "ring": np.stack([rings.value[order], rings.hole[order], n]).T if len(order) else
            np.zeros((0, 3), dtype=np.int64), "v": np.stack([rings.vrow[idx], rings.vcol[idx]])}


def equal(one, parts):
    f1, fp = flat(one), [flat(r) for r in parts]
    return all(np.array_equal(f1[k], np.concatenate([f[k] for f in fp], axis=-1 if k == "v" else 0)) for k in f1)


def properties(rings):
    """(sum of region areas, ok) of one rank's rings"""
    r, c = rings.vrow.astype(np.int64), rings.vcol.astype(np.int64)
    if len(r) == 0:
        return 0, True
    nxt = np.arange(len(r)) + 1
    nxt[rings.offset[1:] - 1] = rings.offset[:-1]
    area2 = np.add.reduceat(c * r[nxt] - c[nxt] * r, rings.offset[:-1])
    ext = rings.hole == 0
    ok = bool(np.all(area2[ext] > 0) and np.all(area2[~ext] < 0) and np.all((r != r[nxt]) ^ (c != c[nxt])))
    ok = ok and rings.nedges == int(np.abs(r - r[nxt]).sum() + np.abs(c - c[nxt]).sum())
    return int(area2.sum() // 2), ok


def summary(parts):
    ex = {}
    for r in parts:
        for k, v in r.band_stats["exchange_bytes"].items():
            ex[k] = ex.get(k, 0) + v
    return (sum(len(r) for r in parts), sum(len(r.vrow) for r in parts), sum(r.nedges for r in parts),
            sum(r.band_stats["segments"] for r in parts) // len(parts), ex)


def run_threads(lab, n):
    rows = lab.shape[0]
    bounds = bands.band_rows(rows, n)
    grp = bands.ThreadGroup(n)
    out, errs = [None] * n, []

    def work(rank):
        try:
            torch.cuda.set_device(0)
            r0, r1 = bounds[rank]
            out[rank] = vector.polygonize_band(bands.ThreadComm(grp, rank), lab[r0:r1], r0, rows)
        except BaseException as e:      # noqa: BLE001
            errs.append(e)
            grp.barrier.abort()

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ts = [threading.Thread(target=work, args=(r,)) for r in range(n)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    torch.cuda.synchronize()
    if errs:
        raise errs[0]
    return out, (time.perf_counter() - t0) * 1e3


def threads_main(S, counts):
    print("card: %s" % card())
    p = RasterPipeline(S, S)
    synth_fractal(S, S, seed=1, out=p.dem)
    p.run()
    ok_all = True
    for which in ("labels", "wsheds"):
        lab = p.out[which]
        vector.polygonize_labels_device(lab)                 # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        one = vector.polygonize_labels_device(lab)
        torch.cuda.synchronize()
        t1 = (time.perf_counter() - t0) * 1e3
        print("%s %d^2 one GPU: %.1f ms, %d rings, %d vertices, %d edges" % (which, S, t1, len(one), len(one.vrow),
                                                                             one.nedges))
        for n in counts:
            run_threads(lab, n)                              # warm-up
            parts, ms = run_threads(lab, n)
            eq = equal(one, parts)
            ok_all &= eq
            nr, nv, ne, nseg, ex = summary(parts)
            print("%s %d^2 %d bands as threads: %.1f ms, %d rings, %d vertices, %d edges, %d segments, exchange bytes "
                  "%s, equal to one GPU: %s" % (which, S, n, ms, nr, nv, ne, nseg, ex, eq))
    print("RESULT %s" % ("OK" if ok_all else "MISMATCH"))


def dist_main(S):
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    comm = bands.DistComm()
    dev = torch.device("cuda", local)
    p = bands.BandPipeline(S, S, comm, device=dev)
    synth_fractal(p.rows, S, seed=1, row0=p.r0, device=local, out=p.dem)
    p.run()
    ok_all = True
    if comm.rank == 0:
        print("card: %s; %d ranks" % (card(), comm.size))
    for which in ("labels", "wsheds"):
        lab = p.out[which]
        vector.polygonize_band(comm, lab, p.r0, S)           # warm-up
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        rings = vector.polygonize_band(comm, lab, p.r0, S)
        torch.cuda.synchronize()
        dist.barrier()
        ms = (time.perf_counter() - t0) * 1e3
        area, ok = properties(rings)
        got = [None] * comm.size
        small = S * S <= SINGLE_GPU_CELLS and S <= 8192
        dist.all_gather_object(got, rings if small else (area, ok, len(rings), len(rings.vrow), rings.nedges,
                                                         rings.band_stats))
        if comm.rank == 0:
            if small:
                whole = torch.cat([x.to(dev) for x in _gather_rows(comm, lab)])
                one = vector.polygonize_labels_device(whole)
                eq = equal(one, got)
                ok_all &= eq
                nr, nv, ne, nseg, ex = summary(got)
                print("%s %d^2 on %d GPUs: %.1f ms, %d rings, %d vertices, %d edges, exchange bytes %s, equal to one "
                      "GPU: %s" % (which, S, comm.size, ms, nr, nv, ne, ex, eq))
            else:
                areas = sum(x[0] for x in got)
                props = all(x[1] for x in got) and areas == S * S
                ok_all &= props
                print("%s %d^2 on %d GPUs: %.1f ms, %d rings, %d vertices, %d edges, properties hold: %s"
                      % (which, S, comm.size, ms, sum(x[2] for x in got), sum(x[3] for x in got),
                         sum(x[4] for x in got), props))
        elif S * S <= SINGLE_GPU_CELLS and S <= 8192:
            _gather_rows(comm, lab)
    if comm.rank == 0:
        print("RESULT %s" % ("OK" if ok_all else "MISMATCH"))
    p.close()
    dist.destroy_process_group()


def _gather_rows(comm, lab):
    return [x.cpu() for x in comm.all_gather_var(lab.contiguous())]


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--threads", default=None, help="band counts, e.g. 2,4,8 (bands as threads of one process)")
    a = ap.parse_args()
    if a.threads:
        threads_main(a.size, [int(x) for x in a.threads.split(",")])
    else:
        dist_main(a.size)
