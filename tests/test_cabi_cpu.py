"""CPU-side checks (no GPU needed): the C-ABI library loads and exports every symbol the header declares,
the plug-in switch rebinds / restores the reference's names, argument validation mirrors the reference's error
behaviour, and the synthetic DEM generator is window-consistent."""
import os
import re
import sys
import types

import numpy as np
import pytest

from malstroem_b200 import _lib, speedups, synth
from malstroem_b200.algorithms import fill, flow, label

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "malstroem_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ms_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    names = header_symbols()
    assert len(names) >= 36
    for n in names:
        assert hasattr(L, n), "libmalstroem_b200.so does not export %s" % n
        assert n in _lib.SIGNATURES, "%s has no ctypes signature" % n
    assert sorted(_lib.SIGNATURES) == names
    assert L.ms_version() >= 100
    assert isinstance(L.ms_device_count(), int)


def test_no_cpu_fallback():
    if _lib.lib().ms_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fill.fill_terrain(np.zeros((8, 8), np.float32))
    with pytest.raises(RuntimeError):
        label.connected_components(np.ones((4, 4), np.float32))


def test_argument_validation_before_any_device_work():
    with pytest.raises(ValueError, match="dtype mismatch"):
        fill.fill_terrain(np.zeros((8, 8), np.float64))              # _fill.pyx:30 typed buffer
    with pytest.raises(ValueError, match="processing area is zero"):
        fill.fill_terrain(np.zeros((3, 9), np.float32))              # _fill.pyx:31-32
    with pytest.raises(ValueError):
        fill.fill_terrain_no_flats(np.zeros((9, 9), np.int32))
    with pytest.raises(ValueError, match="dtype mismatch"):
        flow.terrain_flowdirection(np.zeros((8, 8), np.float32))     # _flow.pyx:99 double[:, :]
    with pytest.raises(ValueError, match="dtype mismatch"):
        flow.accumulated_flow(np.zeros((8, 8), np.int64))            # _flow.pyx:257 uint8[:, :]
    with pytest.raises(ValueError):
        flow.watersheds_from_labels(np.zeros((8, 8), np.uint8), np.zeros((8, 9), np.int32), 0)
    with pytest.raises(ValueError):
        label.label_stats(np.zeros((4, 4)), np.zeros((4, 5), np.int32))
    with pytest.raises(ValueError):
        label.connected_components(np.zeros((0, 4)))


def _fake_reference():
    pkg = types.ModuleType("fake_malstroem_algorithms")
    for modname, names in speedups.REBOUND.items():
        m = types.ModuleType(modname)
        for n in names:
            setattr(m, n, (lambda tag: (lambda *a, **k: tag))("orig:" + n))
        setattr(pkg, modname, m)
    pkg.speedups = types.ModuleType("speedups")
    pkg.speedups.enabled = False
    return pkg


def test_enable_disable_rebinds_the_twelve_names():
    pkg = _fake_reference()
    assert sum(len(v) for v in speedups.REBOUND.values()) == 12
    speedups.enable(pkg)
    try:
        assert speedups.enabled and pkg.speedups.enabled is True
        assert pkg.fill.fill_terrain is fill.fill_terrain
        assert pkg.fill.fill_terrain_no_flats is fill.fill_terrain_no_flats
        assert pkg.fill.minimum_safe_short_and_diag is fill.minimum_safe_short_and_diag
        assert pkg.flow.terrain_flowdirection is flow.terrain_flowdirection
        assert pkg.flow.accumulated_flow is flow.accumulated_flow
        assert pkg.flow.watersheds_from_labels is flow.watersheds_from_labels
        for n in speedups.REBOUND["label"]:
            assert getattr(pkg.label, n) is getattr(label, n)
        speedups.enable(pkg)            # idempotent, like speedups/__init__.py:44-45
    finally:
        speedups.disable()
    assert not speedups.enabled and pkg.speedups.enabled is False
    assert pkg.fill.fill_terrain() == "orig:fill_terrain" and pkg.label.label_count() == "orig:label_count"


# A stand-in with the module layout of the reference package and the binding styles its tool layer relies on: modules
# that bind `fill` / `flow` / `label` / `net` by module and resolve the functions at call time (dem.py:67, streams.py:72),
# a `Network` class with its own `rain_event` (network.py:113), and a module that binds vectorize_labels_file by name at
# import (bluespots.py:17).  Function bodies are irrelevant: the tests check which object each name resolves to.
REFERENCE_LAYOUT = {
    "malstroem/__init__.py": "",
    "malstroem/algorithms/__init__.py": "from . import speedups\n",
    "malstroem/algorithms/speedups/__init__.py": "enabled = False\n",
    "malstroem/algorithms/fill.py": "def fill_terrain(dtm): pass\ndef fill_terrain_no_flats(dtm, short, diag): pass\n"
                                    "def minimum_safe_short_and_diag(dtm): pass\n",
    "malstroem/algorithms/flow.py": "def terrain_flowdirection(t, edges_flow_outward=True): pass\n"
                                    "def accumulated_flow(fd): pass\ndef watersheds_from_labels(fd, lab, unassigned=0): pass\n",
    "malstroem/algorithms/label.py": "".join("def %s(*a, **k): pass\n" % n for n in (
        "connected_components", "label_stats", "keep_labels", "label_min_index", "label_max_index", "label_count")),
    "malstroem/algorithms/net.py": "def next_downstream_label(*a, **k): pass\ndef pourpoint_network(*a, **k): pass\n"
                                   "def geometric_pourpoint_network(*a, **k): pass\n",
    "malstroem/network.py": "class Network(object):\n    def rain_event(self, mmrain): pass\n",
    "malstroem/vector.py": "def vectorize_labels_file(*a, **k): pass\n",
    "malstroem/bluespots.py": "from malstroem.vector import vectorize_labels_file\n",
    "malstroem/dem.py": "from malstroem.algorithms import fill, flow\n",
    "malstroem/streams.py": "from malstroem.algorithms import net\n",
}


@pytest.fixture
def reference_layout(tmp_path):
    for rel, src in REFERENCE_LAYOUT.items():
        p = tmp_path / rel
        p.parent.mkdir(parents=True, exist_ok=True)
        p.write_text(src)
    sys.path.insert(0, str(tmp_path))
    for k in [k for k in sys.modules if k == "malstroem" or k.startswith("malstroem.")]:
        del sys.modules[k]
    try:
        yield
    finally:
        speedups.disable()
        sys.path.remove(str(tmp_path))
        for k in [k for k in sys.modules if k == "malstroem" or k.startswith("malstroem.")]:
            del sys.modules[k]


def test_enable_on_a_package_with_the_reference_layout(reference_layout):
    import malstroem.algorithms as alg
    from malstroem.algorithms import fill as rfill, flow as rflow, label as rlabel
    orig = rfill.fill_terrain
    speedups.enable()
    assert alg.speedups.enabled and rfill.fill_terrain is fill.fill_terrain
    assert rflow.watersheds_from_labels is flow.watersheds_from_labels
    assert rlabel.label_max_index is label.label_max_index
    # the tool layer resolves through the module at call time (malstroem/dem.py:67)
    from malstroem import dem as rdem
    assert rdem.fill.fill_terrain is fill.fill_terrain
    # BluespotTool's import-time binding is replaced as well (bluespots.py:17)
    from malstroem import bluespots as rbluespots
    from malstroem_b200 import vector
    assert rbluespots.vectorize_labels_file is vector.vectorize_labels_file
    speedups.disable()
    assert rfill.fill_terrain is orig and not alg.speedups.enabled


def test_minimum_safe_short_and_diag_scalar_part():
    # non-float32 input takes the numpy path (no device): fill.py:246-249 examples of SURVEY.md A.3
    for m, e in ((51.46, -37), (100.0, -36), (200.0, -35), (999.0, -33)):
        short, diag = fill.minimum_safe_short_and_diag(np.array([[0.0, m], [-1.0, 3.0]]))
        assert short == 2.0 ** e and diag == short * 2 ** 0.5
        assert diag / short - 2 ** 0.5 < 0.0001        # tests/test_raster_fill.py:70-72


def test_synth_is_window_consistent_and_quantised():
    full = synth.fractal_dem(96, 160, seed=5)
    part = synth.fractal_dem(40, 70, seed=5, row0=30, col0=50)
    assert np.array_equal(full[30:70, 50:120], part)
    mm = synth.fractal_mm(96, 160, seed=5)
    assert mm.min() >= 0 and mm.max() <= synth.RELIEF_MM
    assert np.array_equal(full, mm.astype(np.float32) * np.float32(0.001))
    assert not np.array_equal(full, synth.fractal_dem(96, 160, seed=6))
    p = synth.pathological_dem(128, 128)
    assert p.dtype == np.float32 and (p[128 // 3] == np.float32(100000) * np.float32(0.001)).all()


# ------------------------------------------------------------------------------------------ SURVEY 8(f) rows
def test_net_argument_validation_before_any_device_work():
    from malstroem_b200.algorithms import net
    fd = np.zeros((5, 6), np.uint8)
    lab = np.zeros((5, 6), np.int32)
    with pytest.raises(ValueError):
        net.pourpoint_network(fd.astype(np.int32), lab, [(1, 1)], 0)          # flowdir must be uint8
    with pytest.raises(ValueError):
        net.pourpoint_network(fd, lab.astype(np.float32), [(1, 1)], 0)        # labels must be integers
    with pytest.raises(ValueError):
        net.pourpoint_network(fd, lab[:4], [(1, 1)], 0)                       # same shape
    with pytest.raises(IndexError):
        net.next_downstream_label(fd, lab, (5, 0), 0)                         # labeled[cell] would raise (net.py:163)
    # json-type pour points and plain pairs enumerate alike (net.py:21-40)
    feats = [dict(properties=dict(bspot_id=7, cell_row=1, cell_col=2)), (3, 4)]
    assert list(net._pourpoint_enumerator(feats)) == [(7, (1, 2)), (1, (3, 4))]


def test_network_class_bookkeeping_matches_reference_contract():
    from malstroem_b200 import network
    nw = network.Network()
    nodes = [dict(nodeid=5, dstrnodeid=2, wshed_area=10.0, bspot_vol=1.0),
             dict(nodeid=2, dstrnodeid=None, wshed_area=20.0, bspot_vol=0.0),
             dict(nodeid=9, dstrnodeid=77, wshed_area=5.0, bspot_vol=2.0)]
    nw.add_nodes(nodes)                                   # network.py:43-71
    assert nw.nodes == nodes and nw.root_nodes == [2]
    assert nw.nodes_index[5] is nodes[0] and dict(nw.upstream_tree) == {2: [5], None: [2], 77: [9]}
    parent, area, cap = nw._arrays()
    assert parent.tolist() == [1, -1, -2] and area.tolist() == [10.0, 20.0, 5.0] and cap.tolist() == [1.0, 0.0, 2.0]
    nw.add_node(dict(nodeid=5, dstrnodeid=None, wshed_area=1.0, bspot_vol=1.0))
    with pytest.raises(ValueError):
        nw._arrays()                                      # duplicate ids cannot be indexed
    if _lib.lib().ms_device_count() == 0:                 # no CPU fallback for the §8(f) rows either
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            network.rain_events_arrays([-1], [1.0], [1.0], [10.0])
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            from malstroem_b200.algorithms import net
            net.pourpoint_network(np.zeros((4, 4), np.uint8), np.zeros((4, 4), np.int32), [(1, 1)], 0)


def test_enable_rebinds_net_and_network_on_the_reference_layout(reference_layout):
    from malstroem.algorithms import fill as rfill, flow as rflow, label as rlabel      # noqa: F401
    from malstroem.algorithms import net as rnet
    from malstroem import network as rnetwork, streams as rstreams
    from malstroem_b200.algorithms import net
    orig_pp, orig_rain = rnet.pourpoint_network, rnetwork.Network.rain_event
    speedups.enable()
    assert rnet.pourpoint_network is net.pourpoint_network
    assert rnet.next_downstream_label is net.next_downstream_label
    assert rnet.geometric_pourpoint_network is net.geometric_pourpoint_network
    assert rstreams.net.pourpoint_network is net.pourpoint_network      # StreamTool resolves at call time
    assert rnetwork.Network.rain_event is not orig_rain
    speedups.disable()
    assert rnet.pourpoint_network is orig_pp and rnetwork.Network.rain_event is orig_rain
