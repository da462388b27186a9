"""Plain numpy restatement of the bluespot water levels and water-depth rasters (csrc/flood.cu's contract), used only
by the tests: per label np.sort, a sequential np.cumsum in float64 and a linear search for the last breakpoint."""
import numpy as np


def water_levels(dem, filled, labels, v, cell_area, st_sum):
    z = np.asarray(dem, np.float32).astype(np.float64).ravel()
    F = np.asarray(filled, np.float32).ravel()
    lab = np.asarray(labels).ravel().astype(np.int64)
    v = np.atleast_2d(np.asarray(v, np.float64))
    ne, nl1 = v.shape
    if lab.size and (lab.min() < 0 or lab.max() >= nl1):
        raise IndexError("label outside [0, nlabels]")
    level = np.full((ne, nl1), np.nan)
    wet = np.zeros((ne, nl1), np.int64)
    order = np.argsort(lab, kind="stable")
    bounds = np.searchsorted(lab[order], np.arange(nl1 + 1))
    for l in range(1, nl1):
        cells = order[bounds[l]:bounds[l + 1]]
        n = cells.size
        if n == 0:
            continue
        Fl = np.unique(F[cells])
        if Fl.size != 1:
            raise ValueError("the fill is not uniform over label %d" % l)
        L = float(Fl[0])
        cap = float(st_sum[l]) * cell_area
        zs = np.sort(z[cells])
        S = np.cumsum(zs)
        g = np.arange(1, n + 1, dtype=np.float64) * zs - S
        for e in range(ne):
            x = float(v[e, l])
            if np.isnan(x):
                continue
            if x < 0:
                raise ValueError("negative volume")
            if x >= cap:
                level[e, l], wet[e, l] = L, n
                continue
            T = x / cell_area
            k = int(np.nonzero(g <= T)[0][-1]) + 1
            h = min(L, (T + S[k - 1]) / k)
            level[e, l], wet[e, l] = h, int(np.count_nonzero(zs < h))
    return {"level": level, "wet": wet}


def water_depth(dem, filled, labels, level):
    dem = np.asarray(dem, np.float32)
    F = np.asarray(filled, np.float32)
    lab = np.asarray(labels)
    h = np.asarray(level, np.float64)[lab]
    h[lab == 0] = np.nan
    z = dem.astype(np.float64)
    with np.errstate(invalid="ignore"):
        full = h == F.astype(np.float64)
        part = ~full & (z < h)
    out = np.zeros(dem.shape, np.float32)
    out[full] = (F - dem)[full]
    out[part] = (h - z)[part].astype(np.float32)
    return out
