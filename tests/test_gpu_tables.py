"""The per-label tables of the device-resident pipeline (csrc/labels.cu: k_tables_a2 / k_tables_b, and the one-table
kernels the pipeline falls back to) against the CPU oracle, on inputs built to reach every path of those kernels.

The fused passes are driven directly through the band entry points (`ms_band_tables_a_dev` / `ms_band_tables_b_dev`
run exactly k_tables_a2<true> / k_tables_b<true>) on arbitrary numpy rasters: whole, and cut into row pieces that are
combined the way BandPipeline._tables combines the bands.  The families fill the 256-slot per-tile tables, exhaust a
probe chain, put run ends on the 4-cell vector and 16-cell thread-segment boundaries, force the scalar loads, and plant
tied extremes, NaN, infinities, denormals and the largest finite values.  Then the pipeline without accumulation
(k_tables_a2<false>), and the pipeline's non-fused path (label_stats / label_count / label_min_index kernels).

Counts, rows and columns must be equal; minima, maxima and arg-extreme values equal bit for bit after `+ 0.0` (the sign
of zero is not kept, DESIGN.md §2); st_sum within 1e-6 of the sum of |x| of the label, against math.fsum."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch

import band_cases as bc
from malstroem_b200 import _lib, synth
from malstroem_b200.pipeline import TABLES, RasterPipeline
from oracle import port

pytestmark = pytest.mark.gpu
TILE, SLOTS, PROBES = 64, 256, 32
F32_MAX = float(np.finfo(np.float32).max)
NONE = np.iinfo(np.int64).max


def slot(lbl):
    """The first slot of `lbl` in a tile table: slot_of in csrc/labels.cu (k_tables_a2)."""
    return ((np.asarray(lbl, np.uint64) * np.uint64(2654435761)) % np.uint64(1 << 32)) >> np.uint64(24)


# ------------------------------------------------------------------------------------------- the fused passes
def fused_tables(c, cuts):
    """k_tables_a2 / k_tables_b on the row pieces [cuts[k], cuts[k + 1]) of case `c`: min / max / sum reductions of
    phase A across the pieces, phase B with the global extremes, then a min over the global indices."""
    L, dev = _lib.lib(), torch.device("cuda", 0)
    rows, cols = c["labels"].shape
    m = c["nlabels"] + 1
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    f64, i64 = torch.float64, torch.int64
    pieces = []
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        pieces.append((r0, {k: torch.from_numpy(np.ascontiguousarray(c[k][r0:r1])).to(dev)
                            for k in ("depths", "labels", "wsheds", "fnf", "accum")}))
    part = []
    for r0, t in pieces:
        o = {k: torch.empty(m, dtype=f64 if k in ("st_min", "st_max", "st_sum", "vmin", "vmax") else i64, device=dev)
             for k in ("st_min", "st_max", "st_sum", "st_count", "ws_count", "vmin", "vmax")}
        with _lib.lock:
            _lib.check(L.ms_band_tables_a_dev(*(t[k].data_ptr() for k in ("depths", "labels", "fnf", "accum", "wsheds")),
                                              t["labels"].numel(), cols, c["nlabels"],
                                              *(o[k].data_ptr() for k in ("st_min", "st_max", "st_sum", "st_count",
                                                                          "ws_count", "vmin", "vmax")), stream),
                       "ms_band_tables_a_dev")
        part.append(o)
    g = {}
    for k, red in (("st_min", torch.minimum), ("vmin", torch.minimum), ("st_max", torch.maximum),
                   ("vmax", torch.maximum)):
        g[k] = part[0][k]
        for o in part[1:]:
            g[k] = red(g[k], o[k])
    for k in ("st_sum", "st_count", "ws_count"):
        g[k] = sum(o[k] for o in part)
    idx = torch.full((2, m), NONE, dtype=i64, device=dev)
    for r0, t in pieces:
        ib = torch.empty((2, m), dtype=i64, device=dev)
        with _lib.lock:
            _lib.check(L.ms_band_tables_b_dev(t["labels"].data_ptr(), t["fnf"].data_ptr(), t["accum"].data_ptr(),
                                              t["labels"].numel(), c["nlabels"], g["vmin"].data_ptr(),
                                              g["vmax"].data_ptr(), r0 * cols, ib[0].data_ptr(), ib[1].data_ptr(),
                                              stream), "ms_band_tables_b_dev")
        idx = torch.minimum(idx, ib)
    out = {k: v.cpu().numpy() for k, v in g.items()}
    idx = idx.cpu().numpy()
    for k, key, val in ((0, "ppmin", "vmin"), (1, "ppmax", "vmax")):
        none = idx[k] == NONE
        out[key + "_value"] = out[val]
        out[key + "_row"] = np.where(none, -1, idx[k] // cols)
        out[key + "_col"] = np.where(none, -1, idx[k] % cols)
    return out


def same_bits(a, b):
    """Equal bit for bit after + 0.0 (so -0.0 == +0.0), NaN against NaN of any payload."""
    a = np.asarray(a, np.float64) + 0.0
    b = np.asarray(b, np.float64) + 0.0
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    ok = ~np.isnan(a)
    return np.array_equal(a[ok].view(np.int64), b[ok].view(np.int64))


def oracle(c):
    lab, n = c["labels"], c["nlabels"]
    return dict(stats=port.label_stats(c["depths"], lab, n), count=port.label_count(c["wsheds"]),
                ppmin=port.label_min_index(c["fnf"], lab, n), ppmax=port.label_max_index(c["accum"], lab, n))


def check_sum(got, depths, labels, m, want):
    """st_sum against math.fsum of every label's values (the oracle's sum where a label holds NaN or an infinity:
    NaN, or the infinity, in any order), within 1e-6 of the label's sum of |x|."""
    d = depths.ravel().astype(np.float64)
    order = np.argsort(labels.ravel(), kind="stable")
    v = d[order]
    b = np.searchsorted(labels.ravel()[order], np.arange(m + 1))
    for lbl in range(m):
        x = v[b[lbl]:b[lbl + 1]]
        if not np.isfinite(x).all():
            assert same_bits(got[lbl], want[lbl]), (lbl, got[lbl], want[lbl])
            continue
        ref = math.fsum(x.tolist())
        assert abs(got[lbl] - ref) <= 1e-6 * math.fsum(np.abs(x).tolist()), (lbl, got[lbl], ref)


def check_tables(t, c, want, skip=()):
    """Every table of `t` but those in `skip` against the oracle's (`want`: stats, count, ppmin, ppmax)."""
    m = c["nlabels"] + 1
    st = want["stats"]
    assert same_bits(t["st_min"][:m], st["min"]) and same_bits(t["st_max"][:m], st["max"])
    assert np.array_equal(t["st_count"][:m], st["count"])
    check_sum(t["st_sum"][:m], c["depths"], c["labels"], m, st["sum"])
    if "ws_count" not in skip:
        k = len(want["count"])
        assert np.array_equal(t["ws_count"][:k], want["count"]) and not t["ws_count"][k:m].any()
    for key in ("ppmin", "ppmax"):
        if key + "_row" in skip:
            continue
        assert np.array_equal(t[key + "_row"][:m], want[key]["row"]), key + "_row"
        assert np.array_equal(t[key + "_col"][:m], want[key]["col"]), key + "_col"
        assert same_bits(t[key + "_value"][:m], want[key]["value"]), key + "_value"


def piece_cuts(rows):
    """Whole, and 2 - 4 row pieces cut at rows that are not multiples of 64."""
    out = [[0, rows]]
    if rows >= 2:
        k = min(2 + rows % 3, rows)
        cuts = sorted({max(1, min(rows - 1, (rows * j) // k)) for j in range(1, k)})
        cuts = [x + 1 if x % TILE == 0 and x + 1 < rows else x for x in cuts]
        out.append([0] + sorted(set(cuts)) + [rows])
    for cu in out[1:]:
        assert all(x % TILE for x in cu[1:-1])
    return out


# --------------------------------------------------------------------------------------------- the families
def tied_values(rng, shape):
    """depths: signed (sums cancel), fnf / accum: a few levels each, so that every label meets ties of its extreme."""
    return dict(depths=(rng.standard_normal(shape) * 4).astype(np.float32),
                fnf=rng.integers(0, 12, shape) * 0.5, accum=rng.integers(1, 16, shape).astype(np.float64))


def fam_lattice(rows, cols, seed):
    """One-cell labels on a 2-cell lattice: 1024 bluespot labels in a full tile, and as many watershed labels on the
    other lattice, numbered in a seeded order."""
    rng = np.random.default_rng(seed)
    lab = np.zeros((rows, cols), np.int32)
    a = lab[0::2, 0::2]
    a[...] = np.arange(1, a.size + 1).reshape(a.shape)
    ws = np.zeros((rows, cols), np.int32)
    b = ws[1::2, 1::2]
    b[...] = rng.permutation(b.size).reshape(b.shape) + 1
    c = dict(labels=lab, wsheds=ws, nlabels=int(max(lab.max(), ws.max())), **tied_values(rng, (rows, cols)))
    assert bc.labels_per_tile(lab).max() > SLOTS and bc.labels_per_tile(ws).max() > SLOTS
    return c


def fam_probe(rows, cols, seed):
    """48 labels that all start at the same slot of the tile tables, in runs of 1 - 5 cells in the first tile (bluespot
    and watershed labels in different places) and scattered over the rest of the raster: 16 of them find no slot after
    32 probes."""
    rng = np.random.default_rng(seed)
    cand = np.arange(1, 40000)
    same = cand[slot(cand) == 77][:48]
    assert same.size == 48

    def place():
        out = rng.choice(same, (rows, cols)).astype(np.int32)
        out[rng.random((rows, cols)) < 0.3] = 0
        t = out[:TILE, :TILE]
        pos = 0
        for lbl in rng.permutation(same):
            n = int(rng.integers(1, 6))
            r, c0 = divmod(pos, t.shape[1])
            if r >= t.shape[0]:
                break
            t[r, c0:c0 + n] = lbl
            pos += n + 1
        return out

    lab, ws = place(), place()
    c = dict(labels=lab, wsheds=ws, nlabels=int(same.max()) + 5, **tied_values(rng, (rows, cols)))
    for x in (lab, ws):
        t = np.unique(x[:TILE, :TILE])
        assert (slot(t[t > 0]) == 77).sum() > PROBES
    return c


def fam_runs(rows, cols, seed):
    """Row patterns, chosen per row and per 64-column block: a label change at every cell; runs of 4 and of 16 cells
    aligned with the vector loads and the thread segments; one label over the whole block (a run over a whole tile row,
    one label in many tiles); seeded runs of 1 - 19 cells; background.  Label 0 only in the tiles of even
    (tile row + tile column)."""
    rng = np.random.default_rng(seed)
    R, C = np.mgrid[0:rows, 0:cols]

    def pattern(shift):
        k = (R + C // TILE + shift) % 6
        ends = np.cumsum(rng.integers(1, 20, (rows, cols)), axis=1)
        pick = rng.integers(0, 32, (rows, cols))
        rand = np.take_along_axis(pick, np.stack([np.searchsorted(e, np.arange(cols), side="right") for e in ends]), 1)
        out = np.select([k == 0, k == 1, k == 2, k == 3, k == 4],
                        [1 + (C + R) % 7, 8 + (C // 4 + R) % 5, 13 + (C // 16 + R) % 3, np.full_like(C, 20), rand], 0)
        out[(out == 0) & ((R // TILE + C // TILE) % 2 == 1)] = 31
        return out.astype(np.int32)

    lab, ws = pattern(0), pattern(3)
    c = dict(labels=lab, wsheds=ws, nlabels=40, **tied_values(rng, (rows, cols)))
    assert c["nlabels"] > max(lab.max(), ws.max())                 # empty labels at the end keep the defaults
    w = min(cols, TILE)
    assert (np.diff(lab[:, :w], axis=1) != 0).all(1).any()          # a change at every cell
    for run in (4, 16):
        if cols > run and (rows >= 6 or cols >= 2 * TILE):
            assert aligned_run(lab, run), run
    if cols >= TILE and (rows >= 6 or cols >= 4 * TILE):
        assert (lab[:, :TILE * (cols // TILE)].reshape(rows, -1, TILE) == 20).all(2).any()   # a whole tile row
    nt = bc.labels_per_tile(lab).size
    if nt >= 2 and rows >= 6:
        assert (bc.labels_per_tile(lab == 20) > 0).sum() >= max(1, nt // 2)     # one label over many tiles
        z = bc.labels_per_tile(lab == 0)
        assert z.max() > 0 and z.min() == 0                         # label 0 in some tiles and not in others
    return c


def aligned_run(lab, run):
    """Whether some row has a run of exactly `run` cells that starts on a multiple of `run`."""
    cols = lab.shape[1]
    for s in range(0, cols - run + 1, run):
        seg = lab[:, s:s + run]
        ok = (seg == seg[:, :1]).all(1)
        if s > 0:
            ok &= lab[:, s - 1] != lab[:, s]
        if s + run < cols:
            ok &= lab[:, s + run] != lab[:, s]
        if ok.any():
            return True
    return False


def block_labels(rows, cols, bh, bw):
    lab = (1 + (np.arange(rows)[:, None] // bh) * (-(-cols // bw)) + np.arange(cols)[None, :] // bw).astype(np.int32)
    lab[:, ::7] = 0
    return lab


def fam_ties(rows, cols, seed, cuts):
    """Blocks of 100 x 90 cells (each over several tiles and pieces); each label's smallest fnf and largest accum are
    held by a pair in one 4-cell vector, a cell 16 columns on (another thread), and cells in other rows (other tiles,
    other pieces): the smallest flat index must win."""
    rng = np.random.default_rng(seed)
    lab = block_labels(rows, cols, 100, 90)
    c = dict(labels=lab, wsheds=np.ascontiguousarray(lab[::-1]), nlabels=int(lab.max()), **tied_values(rng, lab.shape))
    c["fnf"] += 10.0
    for lbl in range(1, c["nlabels"] + 1):
        r, cc = np.nonzero(lab == lbl)
        if r.size == 0:
            continue
        r0, c0 = r.min(), cc.min()
        c4 = c0 + (-c0) % 4 + 4
        holders = [(r0 + 1, c4 + 1), (r0 + 1, c4 + 2), (r0 + 1, c4 + 17)]
        holders += list(zip(rng.choice(r, 5), rng.choice(cc, 5)))
        holders = [(y, x) for y, x in holders if y < rows and x < cols and lab[y, x] == lbl]
        hr, hc = np.array(holders).T
        c["fnf"][hr, hc] = -0.5 * (lbl % 3)
        c["accum"][hr, hc] = 100.0 + lbl % 4
    band = np.searchsorted(np.array(cuts[1:-1]), np.arange(rows), side="right")
    reach = dict(vector=False, thread=False, tile=False, piece=False)
    for key, ext in (("fnf", np.min), ("accum", np.max)):
        for lbl in range(1, c["nlabels"] + 1):
            r, cc = np.nonzero((lab == lbl) & (c[key] == ext(c[key][lab == lbl])))
            if r.size < 2:
                continue
            reach["vector"] |= any(((r == r[i]) & (cc // 4 == cc[i] // 4)).sum() >= 2 for i in range(r.size))
            reach["thread"] |= any(((r == r[i]) & (cc // 16 != cc[i] // 16) & (cc // TILE == cc[i] // TILE)).any()
                                   for i in range(r.size))
            reach["tile"] |= np.unique((r // TILE) * 1000 + cc // TILE).size >= 2
            reach["piece"] |= np.unique(band[r]).size >= 2
    assert all(reach.values()), reach
    return c


def fam_special(rows, cols, seed):
    """NaN in each raster (never an extreme, a NaN sum); labels whose only values are NaN (depths, fnf, accum), +inf
    (fnf) or -inf (accum): no extreme, (+-inf, -1, -1); infinities, denormals (no flush to zero) and the largest
    finite values as extremes; -0.0 against +0.0."""
    rng = np.random.default_rng(seed)
    lab = block_labels(rows, cols, 40, 30)
    n = int(lab.max())
    c = dict(labels=lab, wsheds=np.ascontiguousarray(lab[:, ::-1]), nlabels=n + 3, **tied_values(rng, lab.shape))
    d, f, a = c["depths"], c["fnf"], c["accum"]
    for x in (d, f, a):
        x[rng.random(x.shape) < 0.03] = np.nan
    plan = {1: "nan", 2: "inf", 3: "denormal", 4: "huge", 5: "zeros", 6: "minus_inf", 7: "nan", 8: "inf"}
    for lbl, what in plan.items():
        m = lab == lbl
        assert m.sum() >= 8
        i = np.flatnonzero(m)
        if what == "nan":
            for x in (d, f, a):
                x[m] = np.nan
        elif what == "inf":
            d[m] = np.inf
            f[m] = np.inf
            a[m] = -np.inf
        elif what == "minus_inf":
            d.flat[i[3]] = -np.inf
            d.flat[i[5]] = np.inf
            f.flat[i[2]] = -np.inf
            a.flat[i[4]] = np.inf
        elif what == "denormal":
            d[m] = np.abs(d[m]) + 1.0
            d.flat[i[1]] = np.float32(1e-45)
            d.flat[i[6]] = -np.float32(1e-45)
            f[m] = np.abs(f[m]) + 1.0
            f.flat[i[2]] = 5e-324
            f.flat[i[3]] = 5e-324
            a[m] = -np.abs(a[m])
            a.flat[i[4]] = -5e-324
        elif what == "huge":
            d.flat[i[0]] = F32_MAX
            d.flat[i[1]] = -F32_MAX
            f.flat[i[2]] = -np.finfo(np.float64).max
            a.flat[i[3]] = np.finfo(np.float64).max
            a.flat[i[7]] = np.finfo(np.float64).max
        elif what == "zeros":
            d[m] = np.where(rng.random(m.sum()) < 0.5, np.float32(-0.0), np.float32(0.0))
            f[m] = np.where(rng.random(m.sum()) < 0.5, -0.0, 0.0)
            a[m] = np.where(rng.random(m.sum()) < 0.5, -0.0, 0.0)
    for x in (d, f, a):
        assert np.isnan(x).any() and np.isnan(x[lab == 1]).all()
    assert np.isposinf(f[lab == 2]).all() and np.isneginf(a[lab == 2]).all()
    assert (d[lab == 3] == np.float32(-1e-45)).any() and (f[lab == 3] == 5e-324).any()
    assert (d == F32_MAX).any() and np.signbit(f[lab == 5]).any() and (f[lab == 6] == -np.inf).any()
    return c


SHAPES = [(70, 5), (67, 13), (130, 63), (129, 65), (100, 130), (131, 68), (65, 100), (200, 132), (1, 300), (1, 5),
          (192, 256)]
CASES = ([("lattice", s, lambda s=s, k=k: fam_lattice(*s, k)) for k, s in enumerate([(130, 256), (131, 130)])]
         + [("probe", s, lambda s=s, k=k: fam_probe(*s, k)) for k, s in enumerate([(100, 132), (70, 65)])]
         + [("runs", s, lambda s=s, k=k: fam_runs(*s, k)) for k, s in enumerate(SHAPES)]
         + [("ties", s, lambda s=s, k=k: fam_ties(*s, k, piece_cuts(s[0])[-1])) for k, s in
            enumerate([(300, 257), (257, 300), (200, 132)])]
         + [("special", s, lambda s=s, k=k: fam_special(*s, k)) for k, s in enumerate([(200, 257), (129, 300)])])


@pytest.mark.parametrize("family,shape,build", CASES, ids=["%s-%dx%d" % (f, *s) for f, s, _ in CASES])
def test_fused_tables(family, shape, build):
    c = build()
    want = oracle(c)
    for cuts in piece_cuts(shape[0]):
        check_tables(fused_tables(c, cuts), c, want)


# -------------------------------------------------------------------------------- the pipeline's table paths
PIPELINE_DEMS = {"fractal": lambda: synth.fractal_dem(300, 515, seed=12),
                 "serpentine": lambda: synth.serpentine_dem(300, 260, 4, pit=True),
                 "pit_lattice": lambda: bc.case("pit_lattice")[0]}


@functools.lru_cache(maxsize=None)
def pipeline_case(name):
    """The DEM, the oracle's results on it, and the case record check_tables reads."""
    dem, want = bc.case(name) if name == "pit_lattice" else (None, None)
    if dem is None:
        dem = PIPELINE_DEMS[name]()
        want = bc.oracle_all(dem)
    return dem, want, dict(nlabels=want["n"], depths=want["depths"], labels=want["labels"])


def host_tables(p, h):
    return {k: h[k].numpy()[: p.nlabels + 1] for k in p.tables}


def check_same_tables(a, b, names):
    for k in names:
        if k == "st_sum":
            np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=0)
        elif a[k].dtype == np.float64:
            assert same_bits(a[k], b[k]), k
        else:
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", list(PIPELINE_DEMS))
def test_pipeline_without_accum(name):
    """k_tables_a2<false> / k_tables_b<false>: every table of a run without accumulation equals the oracle's and the
    run with accumulation's; the network on the fnf pour points works, the accum pour points are refused."""
    dem, want, c = pipeline_case(name)
    assert want["n"] >= 1
    if name == "pit_lattice":
        assert bc.labels_per_tile(want["labels"]).max() > SLOTS
    p0, p1 = RasterPipeline(*dem.shape, with_accum=False), RasterPipeline(*dem.shape)
    h0, h1 = p0.run_host(dem), p1.run_host(dem)
    assert "accum" not in p0.out and not any(k.startswith("ppmax") for k in p0.tables)
    for k in ("flowdir", "labels", "wsheds"):
        assert np.array_equal(h0[k].numpy(), want[k]), k
    t0, t1 = host_tables(p0, h0), host_tables(p1, h1)
    assert p0.nlabels == p1.nlabels == want["n"]
    check_tables(t0, c, want, skip=("ppmax_row",))
    check_same_tables(t0, t1, t0)
    with pytest.raises(ValueError, match="not part of the run"):
        p0.network(use_accum_pourpoints=True)
    n0, n1 = p0.network(events_mm=[20.0]), p1.network(events_mm=[20.0])
    for k in n1:
        torch.testing.assert_close(n0[k], n1[k], rtol=0, atol=0, equal_nan=True)


@pytest.mark.parametrize("dropped", [("ws_count",), ("ppmin_value", "ppmin_row", "ppmin_col")])
@pytest.mark.parametrize("name", ["fractal", "pit_lattice"])
def test_pipeline_unfused_tables(name, dropped):
    """Without one of the tables the pipeline takes the one-table kernels (label_stats, label_count, label_min_index,
    label_max_index): the tables it still produces equal the fused run's and the oracle's."""
    dem, want, c = pipeline_case(name)
    pf, p = RasterPipeline(*dem.shape), RasterPipeline(*dem.shape)
    for k in dropped:
        setattr(p.io, k, None)
    tf, t = host_tables(pf, pf.run_host(dem)), host_tables(p, p.run_host(dem))
    assert p.nlabels == pf.nlabels == want["n"]
    check_tables(t, c, want, skip=dropped)
    check_same_tables(t, tf, [k for k, _ in TABLES if k not in dropped])
