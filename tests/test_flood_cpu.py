"""Bluespot water levels without a GPU: the numpy oracle (oracle/flood.py) against an exact brute-force solution of the
level-pool equation, the uniform fill over bluespots the contract relies on, and argument validation of
malstroem_b200.flood before any device work."""
from fractions import Fraction

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from malstroem_b200 import _lib, flood
from oracle import flood as oflood
from oracle import port


def brute_level(z, T, L):
    """The level h >= min z with sum max(0, h - z) = T, solved exactly (Fractions), capped at L; and #{z < h}."""
    zs = sorted(Fraction(float(x)) for x in z)
    if T == 0:
        h = zs[0]
    else:
        S = Fraction(0)
        for j, x in enumerate(zs, 1):
            S += x
            hj = (T + S) / j
            if hj > x and (j == len(zs) or hj <= zs[j]):
                h = hj
                break
    h = min(h, Fraction(float(L)))
    return h, sum(1 for x in zs if x < h)


def _bluespots(dem):
    filled = port.fill_terrain(dem)
    lab, n = port.connected_components(filled - dem)
    st_sum = port.label_stats(filled - dem, lab, n)["sum"]
    return filled, lab, n, st_sum


@settings(max_examples=60, deadline=None)
@given(rows=st.integers(3, 9), cols=st.integers(3, 9), seed=st.integers(0, 2 ** 31 - 1), integer=st.booleans())
def test_oracle_matches_exact_level(rows, cols, seed, integer):
    rng = np.random.default_rng(seed)
    dem = (rng.integers(0, 6, (rows, cols)) if integer else rng.random((rows, cols)) * 5).astype(np.float32)
    filled, lab, n, st_sum = _bluespots(dem)
    if n == 0:
        return
    cap = st_sum * 1.0
    fr = rng.random((4, n + 1))
    v = np.floor(fr * cap) if integer else fr * cap
    v[1] = cap                                      # full
    v[2] = 0.0
    v[3, rng.random(n + 1) < 0.3] = np.nan
    got = oflood.water_levels(dem, filled, lab, v, 1.0, st_sum)
    assert np.isnan(got["level"][:, 0]).all() and (got["wet"][:, 0] == 0).all()
    for l in range(1, n + 1):
        m = lab == l
        L = float(filled[m][0])
        for e in range(4):
            if np.isnan(v[e, l]):
                assert np.isnan(got["level"][e, l]) and got["wet"][e, l] == 0
                continue
            if v[e, l] >= cap[l]:
                assert got["level"][e, l] == L and got["wet"][e, l] == m.sum()
                continue
            h, w = brute_level(dem[m], Fraction(float(v[e, l])), L)
            if integer:
                assert got["level"][e, l] == float(h) and got["wet"][e, l] == w
            else:
                assert abs(got["level"][e, l] - float(h)) <= 1e-12 * max(1.0, abs(float(h)))


def _check_uniform(dem, filled):
    lab, n = port.connected_components(filled - dem)
    for l in range(1, n + 1):
        assert np.unique(filled[lab == l]).size == 1


def test_fill_is_uniform_over_bluespots(small_cases, fractal256):
    # the fixed point of the fill (the pure-Python reference's and this library's); on one small case the Cython
    # sweep stops one cell short of it, which is why the library checks the property instead of assuming it
    cases, _ = small_cases
    for c in cases:
        _check_uniform(c["dem"], c["filled_py"])
    _check_uniform(fractal256["dem"], fractal256["filled_cy"])


def test_oracle_rejects_non_bluespot_labels():
    dem = np.array([[3, 3, 3, 3], [3, 1, 2, 3], [3, 3, 3, 3]], np.float32)
    filled = dem.copy()
    filled[1, 1] = 2.5
    lab = np.array([[0, 0, 0, 0], [0, 1, 1, 0], [0, 0, 0, 0]], np.int32)
    with pytest.raises(ValueError):
        oflood.water_levels(dem, filled, lab, [np.nan, 0.5], 1.0, [0.0, 1.0])


def test_argument_validation_before_any_device_work():
    dem = np.zeros((4, 5), np.float32)
    lab = np.zeros((4, 5), np.int32)
    v = np.zeros(3)
    with pytest.raises(ValueError):
        flood.water_levels(dem.astype(np.float64), dem, lab, v, 1.0, np.zeros(3))
    with pytest.raises(ValueError):
        flood.water_levels(dem, dem[:, :4], lab, v, 1.0, np.zeros(3))
    with pytest.raises(ValueError):
        flood.water_levels(dem, dem, lab.astype(np.float32), v, 1.0, np.zeros(3))
    with pytest.raises(ValueError):
        flood.water_levels(dem, dem, lab, v, 1.0, np.zeros(4))                 # v of the wrong length
    with pytest.raises(ValueError):
        flood.water_levels(dem, dem, lab, np.zeros((2, 2, 3)), 1.0, np.zeros(3))
    for ca in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            flood.water_levels(dem, dem, lab, v, ca, np.zeros(3))
    with pytest.raises(ValueError):
        flood.water_depth(dem, dem, lab[:3], np.zeros(3))
    with pytest.raises(ValueError):
        flood.water_depth(dem, dem, lab, np.zeros((2, 3)))


def test_no_cpu_fallback():
    if _lib.lib().ms_device_count() > 0:
        pytest.skip("a CUDA device is present")
    dem = np.zeros((4, 5), np.float32)
    lab = np.zeros((4, 5), np.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        flood.water_levels(dem, dem, lab, np.zeros(3), 1.0, np.zeros(3))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        flood.water_depth(dem, dem, lab, np.zeros(3))
