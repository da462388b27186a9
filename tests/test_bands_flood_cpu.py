"""CPU tests of the host side of the banded flood (BandPipeline.flood): the variable all-to-all of the exchange layer
under ThreadComm and under gloo with world_size 2, and the label -> owner routing.  The band phases themselves are
CUDA (tests/test_bands_flood_gpu.py)."""
import os
import socket
import threading

import numpy as np
import pytest
import torch

from malstroem_b200 import _lib, bands


def _chunks(rank, size):
    """What rank `rank` sends: to rank j, (rank + 2 j) % 3 rows of [k, 3] int32 (some empty) tagged with both ranks."""
    out = []
    for j in range(size):
        k = (rank + 2 * j) % 3
        out.append(torch.arange(3 * k, dtype=torch.int32).view(k, 3) + 1000 * rank + 100 * j)
    return out


def _check_received(got, rank, size):
    assert len(got) == size
    for j in range(size):
        want = _chunks(j, size)[rank]
        assert got[j].dtype == want.dtype and got[j].shape == want.shape
        assert torch.equal(got[j], want)


def test_all_to_all_var_threadcomm():
    size = 4
    grp = bands.ThreadGroup(size)
    errs = []

    def work(rank):
        try:
            comm = bands.ThreadComm(grp, rank)
            _check_received(comm.all_to_all_var(_chunks(rank, size)), rank, size)
            got = comm.all_to_all_var([torch.zeros(0, dtype=torch.int32)] * size)        # nothing at all
            assert [g.numel() for g in got] == [0] * size
            flat = comm.all_to_all_var([torch.full((rank + j,), rank, dtype=torch.int64) for j in range(size)])
            assert [g.tolist() for g in flat] == [[j] * (j + rank) for j in range(size)]
        except BaseException as e:      # noqa: BLE001 - reported below
            errs.append(e)
            grp.barrier.abort()

    ts = [threading.Thread(target=work, args=(r,)) for r in range(size)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port_no, result_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        comm = bands.DistComm()
        _check_received(comm.all_to_all_var(_chunks(rank, world)), rank, world)
        got = comm.all_to_all_var([torch.zeros((0, 3), dtype=torch.int32)] * world)
        assert [tuple(g.shape) for g in got] == [(0, 3)] * world
        # uneven 1-D chunks, one of them empty
        flat = comm.all_to_all_var([torch.full((rank * 3 + j,), 7 * rank + j, dtype=torch.int64) for j in range(world)])
        assert [g.tolist() for g in flat] == [[7 * j + rank] * (j * 3 + rank) for j in range(world)]
        open(os.path.join(result_dir, "ok%d" % rank), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_all_to_all_var_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(os.path.join(str(tmp_path), "ok%d" % r)) for r in range(world))


@pytest.mark.parametrize("counts", [[5, 0, 4, 3], [0, 0, 7], [1], [3, 0, 0, 2, 0], [0, 6, 0]])
def test_label_owner_matches_ranges(counts):
    offsets = np.concatenate([[0], np.cumsum(counts)[:-1]])
    labels = np.arange(1, sum(counts) + 1)
    want = [next(g for g, (o, c) in enumerate(zip(offsets, counts)) if o < l <= o + c) for l in labels]
    got = bands.label_owner(torch.from_numpy(labels), torch.from_numpy(offsets))
    assert got.tolist() == want


def test_flood_flag_bits_match_the_header():
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "malstroem_b200.h")).read()
    for name in ("LABEL", "UNIFORM", "VOLUME", "SIZE", "CAPACITY"):
        line = next(ln for ln in src.splitlines() if ln.startswith("#define MS_FLOOD_%s " % name))
        assert int(line.split()[2]) == getattr(_lib, "MS_FLOOD_" + name)
