"""The multi-GPU data plane under test on REAL GPUs (needs >= 2; skipped on a one-GPU box): one process per GPU over
NCCL, the no-flats solver kernels of all bands running at once and exchanging edge rows / tile activations over NVLink
peer memory (CUDA IPC mailboxes, system-scope atomics, distributed termination count).  The banded run must equal the
single-GPU run of the same raster bit for bit - every raster, every exact table (tools/band_check_dist.py) - and where
a lake crosses the band edge it must have gone through the peer path (noflat_ir == 1).  Besides the fractal DEM: white
noise, a serpentine channel that carries most of the raster across the band edge many times, and a comb of bluespots
joined only in the last band's rows, whose flat lake spans the raster."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _check_dist(shape, kind, lake):
    if _ngpus() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tools", "band_check_dist.py"), str(shape[0]),
           str(shape[1]), kind]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "RESULT OK" in r.stdout, r.stdout[-3000:]
    if lake:
        assert "'noflat_ir': 1" in r.stdout, r.stdout[-3000:]
    assert "MISMATCH" not in r.stdout


@pytest.mark.parametrize("shape", [(4096, 4096), (2048, 6000)])
def test_two_gpu_bands_equal_single_gpu(shape):
    _check_dist(shape, "fractal", True)


@pytest.mark.parametrize("kind,shape,lake", [("noise", (2048, 2051), True), ("serpentine", (2048, 1024), False),
                                             ("comb", (2048, 2051), True)])
def test_two_gpu_stress_rasters(kind, shape, lake):
    """lake: the raster has a lake across the band edge (noise: many; comb: one flat at 10 over the whole raster);
    the serpentine drains without one."""
    _check_dist(shape, kind, lake)
