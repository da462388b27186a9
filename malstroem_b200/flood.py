"""Bluespot water levels and water-depth rasters after rain events (csrc/flood.cu, DESIGN.md §4, "water levels").

Given the stored volume `v` of every bluespot per rain event (the `v` of `network.rain_events_arrays` or of
`RasterPipeline.network`), `water_levels` gives the water level and the number of wet cells of each bluespot, and
`water_depth` the water depth raster of one event.

Level-pool approximation: the water of a bluespot is taken as one flat surface at level h holding
cell_area * sum max(0, h - z) over the bluespot's cells.  This ignores that separate sub-pits of one bluespot may fill
one after another.  A full bluespot (v >= capacity) stands at its fill level, and its depths are the fill's `depths`.
"""
import numpy as np

from . import _lib
from .algorithms.label import _labels32, label_stats


def _rasters(dem, filled, labels, what):
    dem, filled = np.asarray(dem), np.asarray(filled)
    if dem.dtype != np.float32 or filled.dtype != np.float32:
        raise ValueError("%s: dem and filled must be float32" % what)
    lab = _labels32(labels, what)
    if dem.ndim != 2 or dem.size == 0 or filled.shape != dem.shape or lab.shape != dem.shape:
        raise ValueError("%s: dem, filled and labels must be 2-D with the same non-empty shape" % what)
    return np.ascontiguousarray(dem), np.ascontiguousarray(filled), lab


def water_levels(dem, filled, labels, v, cell_area, st_sum=None):
    """Water level and wet-cell count of every bluespot after each rain event.

    dem, filled: float32 rasters (the DEM and its plain fill); labels: the bluespot labels (0 = none) of `filled - dem`;
    v: stored volume per bluespot, [nlabels+1] or [n_events, nlabels+1] (m^3; NaN for nodes the network never
    reaches); cell_area > 0; st_sum: per-label sum of `filled - dem` (label_stats(...)['sum']), computed when None.
    Returns {'level': float64 [n_events, nlabels+1], 'wet': int64 [n_events, nlabels+1]}.  Label 0, NaN volumes and
    bluespots without cells get NaN / 0.  Raises ValueError for bad arguments, for labels over which `filled` is not
    uniform (not bluespots of this fill) and for negative volumes, IndexError for a label above nlabels."""
    dem, filled, lab = _rasters(dem, filled, labels, "water_levels")
    v = np.asarray(v, dtype=np.float64)
    if v.ndim not in (1, 2) or v.shape[-1] < 1:
        raise ValueError("water_levels: v must be [nlabels+1] or [n_events, nlabels+1]")
    v = np.ascontiguousarray(np.atleast_2d(v))
    ne, nl1 = v.shape
    cell_area = float(cell_area)
    if not (cell_area > 0.0 and np.isfinite(cell_area)):
        raise ValueError("water_levels: cell_area must be > 0, got %r" % cell_area)
    if st_sum is None:
        st_sum = label_stats(filled - dem, lab, nl1 - 1)["sum"] if nl1 > 1 else np.zeros(1)
    st_sum = np.ascontiguousarray(st_sum, dtype=np.float64)
    if st_sum.shape != (nl1,):
        raise ValueError("water_levels: st_sum must have nlabels+1 = %d entries, got shape %s" % (nl1, st_sum.shape))
    level = np.empty((ne, nl1), np.float64)
    wet = np.empty((ne, nl1), np.int64)
    with _lib.lock:
        _lib.check(_lib.lib().ms_flood_levels(_lib.ptr(dem), _lib.ptr(filled), _lib.ptr(lab), dem.shape[0],
                                              dem.shape[1], nl1 - 1, _lib.ptr(st_sum), cell_area, ne, _lib.ptr(v),
                                              _lib.ptr(level), _lib.ptr(wet)), "water_levels")
    _lib.track(dem, filled, lab)
    return {"level": level, "wet": wet}


def water_depth(dem, filled, labels, level):
    """Water depth raster (float32) of one event from its levels (one row of water_levels' `level`, nlabels+1
    entries): filled - dem where the bluespot is full (bitwise the fill's depths), level - z (float64, rounded once)
    where z < level, 0 elsewhere and outside bluespots."""
    dem, filled, lab = _rasters(dem, filled, labels, "water_depth")
    level = np.asarray(level, dtype=np.float64)
    if level.ndim != 1 or level.size < 1:
        raise ValueError("water_depth: level must be one event's levels, [nlabels+1]")
    level = np.ascontiguousarray(level)
    out = _lib.result_array(dem.shape, np.float32)
    with _lib.lock:
        _lib.check(_lib.lib().ms_water_depth(_lib.ptr(dem), _lib.ptr(filled), _lib.ptr(lab), dem.shape[0],
                                             dem.shape[1], level.size - 1, _lib.ptr(level), _lib.ptr(out)),
                   "water_depth")
    _lib.track(dem, filled, lab, out)
    return out
