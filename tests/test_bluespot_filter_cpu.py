"""The bluespot filter compiler (malstroem_b200/bluespot_filter.py) without a GPU: its programs, run by the element-wise
interpreter that restates the device's operations, decide like the CLI's `-filter` lambda (tests/toolchain.py
parse_filter, scripts/_utils.py:29-40) evaluated the reference's way on numpy scalars; rejections name the offending
node; and the label ranges of the row bands follow a filter."""
import os
import re

import numpy as np
import pytest
import torch

from malstroem_b200 import bluespot_filter as bf
from toolchain import parse_filter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CELL_AREA = 16 * 15 / 0.94

FILTERS = [
    "area > 20.5 and maxdepth > 0.5 or volume > 2.5",
    "maxdepth > 0.05",
    "0.1 < maxdepth < 2",
    "0.1 < maxdepth <= area < 40 != volume",
    "not maxdepth > 1 and area >= 3",
    "not (area > 2 or volume <= 1)",
    "maxdepth * 2 - 1 > -volume / 3",
    "area - maxdepth * 3 + volume / 2 > 1 or maxdepth == 0.5",
    "area != 4 and maxdepth == maxdepth",
    "maxdepth",
    "not volume",
    "maxdepth and area or not volume",
    "-maxdepth < -0.5 or +area > 10",
    "1 + 2 * 3 < area",
    "area / 0 > 1 or volume / maxdepth < 2",
    "True and maxdepth > 0",
    "1 < 2 < 3 and maxdepth > 0.5",
    "maxdepth > 0.5 and 2 > 3",
    "maxdepth > 0.5 or 2 > 3",
    "0.1 + 0.2 + maxdepth > 0.8",
    "area > 9007199254740992",
    "maxdepth < 1e308 * 10",
    "volume >= -0.0 and maxdepth <= 0",
    "(area > 20.5) and (maxdepth > 0.5 or volume > 2.5)",
    "1",
    "0 and area",
    "- - maxdepth > 0.5 - 1 / 4",
]


def header_enum():
    src = open(os.path.join(ROOT, "include", "malstroem_b200.h")).read()
    body = re.search(r"enum \{(.*?)\};", src[src.index("MS_BF_MAX_STACK"):], re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"MS_BF_([A-Z]+)", body)
    assert re.search(r"MS_BF_AREA\s*=\s*1\b", body)
    return {n: k + 1 for k, n in enumerate(names)}


def test_op_codes_match_the_header():
    enum = header_enum()
    assert len(enum) == 18
    for name, code in enum.items():
        assert getattr(bf, name) == code, name
    src = open(os.path.join(ROOT, "include", "malstroem_b200.h")).read()
    assert "#define MS_BF_MAX_OPS %d" % bf.MAX_OPS in src and "#define MS_BF_MAX_STACK %d" % bf.MAX_STACK in src


def stats_cases(cell_area, seed):
    """Raw label stats: random ones plus values exactly at the thresholds above, +-0, +-inf and NaN."""
    rng = np.random.default_rng(seed)
    n = 400
    count = rng.integers(0, 60, n).astype(np.int64)
    vmax = rng.uniform(-0.2, 3.0, n)
    vsum = rng.uniform(-1.0, 5.0, n)
    special = np.array([0.0, -0.0, 0.05, 0.1, 0.5, 1.0, 2.0, 2.5, 0.25, -0.5, np.inf, -np.inf, np.nan,
                        np.nextafter(0.05, 1), np.nextafter(0.05, -1), np.nextafter(0.5, 1), 0.1 + 0.2])
    k = len(special)
    vmax[:k] = special
    vmax[k:2 * k] = special[::-1]
    vsum[:k] = special[::-1] / cell_area
    vsum[2 * k:3 * k] = special
    vsum[3 * k:4 * k] = 2.5 / cell_area
    count[:12] = [0, 1, 2, 3, 4, 5, 7, 8, 20, 21, 40, 41]
    if cell_area == 0.5:
        count[12:14] = [41, 80]             # area exactly 20.5 and 40
    return count, vmax, vsum


def reference_decisions(text, count, vmax, vsum, cell_area):
    fn = parse_filter(text)
    out = []
    with np.errstate(all="ignore"):
        for c, m, s in zip(count, vmax, vsum):
            stats = {"area": np.int64(c) * cell_area, "max": np.float64(m), "volume": np.float64(s) * cell_area}
            out.append(bool(fn(stats)))
    return np.array(out)


@pytest.mark.parametrize("cell_area", [1.0, 0.5, CELL_AREA])
@pytest.mark.parametrize("text", FILTERS)
def test_program_decides_like_the_cli_lambda(text, cell_area):
    prog = bf.compile_filter(text)
    assert 1 <= len(prog.code) <= bf.MAX_OPS and prog.max_stack <= bf.MAX_STACK
    count, vmax, vsum = stats_cases(cell_area, seed=len(text))
    want = reference_decisions(text, count, vmax, vsum, cell_area)
    area, volume = count.astype(np.float64) * cell_area, vsum * cell_area
    got = prog.evaluate(area, vmax, volume)
    assert got.dtype == np.bool_ and got.shape == want.shape
    assert np.array_equal(got, want), np.nonzero(got != want)[0][:10]
    # the same program on torch tensors (what tools/filter_bench.py certifies the device with)
    t = prog.evaluate(torch.from_numpy(area), torch.from_numpy(vmax), torch.from_numpy(volume))
    assert np.array_equal(t.numpy(), want)


def test_constant_folding_and_program_shape():
    assert bf.compile_filter(None) is None and bf.compile_filter("") is None
    p = bf.compile_filter("maxdepth > 0.05")
    assert p.code == ((bf.MAXDEPTH, 0.0), (bf.CONST, 0.05), (bf.GT, 0.0)) and p.reads == {bf.MAXDEPTH}
    assert bf.compile_filter("1 + 2 * 3 < area").code == ((bf.CONST, 7.0), (bf.AREA, 0.0), (bf.LT, 0.0))
    assert bf.compile_filter("area > 7 / 2").code[1] == (bf.CONST, 3.5)
    assert bf.compile_filter("1 < 2 < 3").code == ((bf.CONST, 1.0),)
    assert bf.compile_filter("not 1 or 0").code == ((bf.CONST, 0.0),)
    neg0 = bf.compile_filter("maxdepth > -0.0").code[1][1]
    assert neg0 == 0.0 and np.signbit(neg0)
    assert not np.signbit(bf.compile_filter("maxdepth > -0").code[1][1])      # int -0 is 0
    assert bf.compile_filter("area > 1").reads == {bf.AREA}
    p = bf.compile_filter("area > 20.5 and maxdepth > 0.5 or volume > 2.5")
    assert p.reads == {bf.AREA, bf.MAXDEPTH, bf.VOLUME}
    assert [op for op, _ in p.code][-1] == bf.OR


@pytest.mark.parametrize("text,match", [
    ("area ** 2 > 1", r"\*\*"),
    ("area % 2 > 1", "%"),
    ("area // 2 > 1", "//"),
    ("abs(area) > 1", "Call"),
    ("stats.area > 1", "Attribute"),
    ("area[0] > 1", "Subscript"),
    ("depth > 1", "unknown name 'depth'"),
    ("max > 1", "unknown name 'max'"),
    ("1 / 0 > area", "division by zero"),
    ("area > 1 / (2 - 2)", "division by zero"),
    ("(area > 1) + 1", "boolean context"),
    ("-(area > 2)", "boolean context"),
    ("area > (maxdepth > 1)", "boolean context"),
    ("(area > 1 and volume) * 2 > 1", "'and' / 'or'"),
    ("not area + (not volume)", "'not' is allowed only"),
    ("'a' > area", "unsupported constant"),
    ("None", "unsupported constant"),
    ("9007199254740993 < area", r"2\*\*53"),
    ("area > 4503599627370496 * 4", r"2\*\*53"),
    ("area is None", "is"),
    ("area in (1, 2)", "in"),
    ("~area", "~"),
    ("lambda: 1", "Lambda"),
    ("area if volume else maxdepth", "IfExp"),
    ("area >", "syntax error"),
    ("   ", "syntax error"),
])
def test_rejections_name_the_node(text, match):
    with pytest.raises(ValueError, match=match):
        bf.compile_filter(text)


def test_program_size_limits():
    flat = " + ".join(["area"] * 33) + " > 1"           # 33 pushes, 32 adds, const, compare: 67 operations
    with pytest.raises(ValueError, match="exceed"):
        bf.compile_filter(flat)
    deep = "(" * 16 + "area" + "".join(" + (volume" for _ in range(16)) + ")" * 32 + " > 1"
    with pytest.raises(ValueError, match="exceed"):
        bf.compile_filter(deep)
    ok = bf.compile_filter(" + ".join(["area"] * 31) + " > 1")
    assert len(ok.code) == 63 and ok.max_stack == 2


def test_struct_carries_program_and_cell_area():
    p = bf.compile_filter("area > 20.5 and maxdepth > 0.5 or volume > 2.5")
    s = p.struct(CELL_AREA)
    assert s.n_ops == len(p.code) and s.cell_area == CELL_AREA
    assert [(s.op[k], s.imm[k]) for k in range(s.n_ops)] == list(p.code)
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="cell_area"):
            p.struct(bad)


def test_golden_raw_stats_keep_counts(dtm188):
    """dtm188's raw bluespots: the reference CLI's filter keeps 486 of 523, and relabelling the kept raw labels by
    rank is what the second connected_components gives."""
    cnt, mx, sm = dtm188["raw_stats_count"], dtm188["raw_stats_max"], dtm188["raw_stats_sum"]
    assert int(dtm188["raw_nlabels"]) == 523
    for text, nkeep in (("area > 20.5 and maxdepth > 0.5 or volume > 2.5", 486), ("maxdepth > 0.05", 382)):
        keep = bf.compile_filter(text).evaluate(cnt.astype(np.float64) * CELL_AREA, mx, sm * CELL_AREA)
        keep[0] = False
        assert np.array_equal(keep[1:], reference_decisions(text, cnt, mx, sm, CELL_AREA)[1:])
        assert int(keep.sum()) == nkeep
    # a filter that keeps exactly the golden bluespots: the rank table reproduces the golden labelled raster
    raw, lab = dtm188["raw_labels"], dtm188["labelled"]
    keep = np.zeros(cnt.size, bool)
    keep[np.unique(raw[lab > 0])] = True
    lut = np.cumsum(keep) * keep
    assert np.array_equal(lut[raw], lab) and int(keep.sum()) == int(lab.max()) == 104


def test_label_ranges_after_filter():
    # three bands numbering 4, 0 and 5 raw labels (1..4, -, 5..9)
    ranges = [(0, 4), (4, 0), (4, 5)]
    keep = np.array([True, True, False, True, False, False, True, True, False, True])
    assert bf.label_ranges_after_filter(ranges, keep) == [(0, 2), (2, 0), (2, 3)]
    assert bf.label_ranges_after_filter(ranges, np.ones(10, bool)) == ranges            # keep-all: unchanged
    assert bf.label_ranges_after_filter(ranges, np.zeros(10, bool)) == [(0, 0), (0, 0), (0, 0)]
    # every kept label stays with the band that numbered it
    rng = np.random.default_rng(3)
    for _ in range(20):
        counts = rng.integers(0, 6, rng.integers(1, 6))
        ranges = [(int(counts[:g].sum()), int(c)) for g, c in enumerate(counts)]
        keep = rng.random(int(counts.sum()) + 1) < 0.5
        lut = np.cumsum(keep * (np.arange(keep.size) > 0)) * keep
        lut[0] = 0
        out = bf.label_ranges_after_filter(ranges, keep)
        assert sum(c for _, c in out) == int(keep[1:].sum())
        for (o, c), (o2, c2) in zip(ranges, out):
            mine = lut[o + 1:o + c + 1]
            mine = mine[mine > 0]
            assert c2 == mine.size and (c2 == 0 or (mine.min() == o2 + 1 and mine.max() == o2 + c2))
