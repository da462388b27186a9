"""Under torchrun (one rank per GPU, NCCL): the row-band run of one raster against the single-GPU run on rank 0.

    band_check_dist.py [rows [cols [kind]]]

kind: fractal (default, generated on the device) or one of the numpy builders of malstroem_b200.synth in KINDS."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from malstroem_b200 import bands, synth
from malstroem_b200.pipeline import RasterPipeline, synth_fractal

KINDS = {
    "noise": lambda R, C: np.random.default_rng(2).random((R, C), dtype=np.float32) * np.float32(100.0),
    "serpentine": lambda R, C: synth.serpentine_dem(R, C, 4),
    "serpentine_pit": lambda R, C: synth.serpentine_dem(R, C, 4, pit=True),
    "comb": lambda R, C: synth.mask_dem(synth.comb_mask(R, C)),
    "speckle": lambda R, C: synth.mask_dem(synth.speckle_mask(R, C)),
    "pit_chain": lambda R, C: synth.pit_chain_dem(R, C),
    "sea_bowl": lambda R, C: synth.sea_bowl_dem(R, C),
}

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
R = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
C = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
kind = sys.argv[3] if len(sys.argv) > 3 else "fractal"
if kind != "fractal" and kind not in KINDS:
    raise SystemExit("unknown raster kind %r (fractal, %s)" % (kind, ", ".join(KINDS)))
p = bands.BandPipeline(R, C, bands.DistComm(), device=local)
dem = None if kind == "fractal" else torch.from_numpy(KINDS[kind](R, C))
if dem is None:
    synth_fractal(p.rows, C, seed=1, row0=p.r0, col0=0, device=local, out=p.dem)
else:
    p.dem.copy_(dem[p.r0:p.r1])
p.run()
torch.cuda.synchronize()
ok = True
if rank == 0:
    ref = RasterPipeline(R, C, device=local)
    if dem is None:
        synth_fractal(R, C, seed=1, device=local, out=ref.dem)
    else:
        ref.dem.copy_(dem)
    ref.run()
for name in ("filled", "depths", "fnf", "flowdir", "accum", "labels", "wsheds"):
    t = p.out[name].contiguous()
    parts = bands.DistComm().all_gather_var(t)
    if rank == 0:
        got = torch.cat(parts)
        same = torch.equal(got, ref.out[name])
        ok &= same
        print(name, "OK" if same else "MISMATCH (%d cells)" % int((got != ref.out[name]).sum()))
if rank == 0:
    m = ref.nlabels + 1
    print("nlabels", p.nlabels, ref.nlabels)
    ok &= p.nlabels == ref.nlabels
    for name in ("st_min", "st_max", "st_count", "ws_count", "ppmin_row", "ppmin_col", "ppmax_row", "ppmax_col"):
        same = torch.equal(p.tables[name][:m], ref.tables[name][:m])
        ok &= same
        print("table", name, "OK" if same else "MISMATCH")
    print("stats", p.stats)
    print("RESULT", "OK" if ok else "FAIL")
dist.destroy_process_group()
