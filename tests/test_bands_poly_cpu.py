"""bands.ring_segments (the rings that cross band edges, linked from their segments) against a brute-force walk of
random rings: random edge numbers, random sides (corners where the side changes), cut into segments where the band
changes along the ring.  Cases include rings that touch three or more bands, leaders inside a middle segment and
segments of length 1."""
import numpy as np
import pytest
import torch

from malstroem_b200 import bands


def make_rings(rng, nrings, nbands, maxlen):
    """Rings as lists of (edge number, side, band); every ring touches at least two bands."""
    rings = []
    for _ in range(nrings):
        L = int(rng.integers(4, maxlen + 1))
        cuts = np.sort(rng.choice(np.arange(1, L), size=int(rng.integers(1, min(L - 1, 6) + 1)), replace=False))
        runs = np.split(np.arange(L), cuts)
        band = []
        prev = -1
        for run in runs:
            b = int(rng.integers(0, nbands))
            while b == prev:
                b = int(rng.integers(0, nbands))
            band += [b] * len(run)
            prev = b
        if band[0] == band[-1]:          # the ring must leave its first band: rotate so it starts at a change
            k = next(i for i in range(1, L) if band[i] != band[0])
            band = band[k:] + band[:k]
        sides = rng.integers(0, 4, size=L).tolist()
        rings.append((band, sides))
    # edge numbers: band-major (lower bands first), random within the band
    per_band = [sum(b.count(g) for b, _ in rings) for g in range(nbands)]
    base = np.concatenate([[0], np.cumsum(per_band)])
    pools = [list(rng.permutation(per_band[g]) + base[g]) for g in range(nbands)]
    out = []
    for band, sides in rings:
        out.append([(int(pools[b].pop()), s, b) for b, s in zip(band, sides)])
    return out


def brute(rings):
    """Per ring: leader, L, V and for every edge its position and (if a corner) vertex index."""
    res = []
    for ring in rings:
        L = len(ring)
        k0 = min(range(L), key=lambda i: ring[i][0])
        walk = ring[k0:] + ring[:k0]
        corner = [walk[i][1] != walk[i - 1][1] for i in range(L)]
        vidx = np.cumsum([0] + corner[:-1])
        res.append({"leader": walk[0][0], "L": L, "V": int(sum(corner)),
                    "pos": {e: i for i, (e, _, _) in enumerate(walk)},
                    "vert": {walk[i][0]: int(vidx[i]) for i in range(L) if corner[i]}})
    return res


def segments(rings):
    """Segment records (as the bands build them) and each segment's edges in order."""
    recs, edges = [], []
    for ring in rings:
        L = len(ring)
        starts = [i for i in range(L) if ring[i][2] != ring[i - 1][2]]
        for j, a in enumerate(starts):
            b = starts[(j + 1) % len(starts)]
            run = [ring[(a + t) % L] for t in range((b - a) % L or L)]
            nxt = ring[b % L]
            ids = [e for e, _, _ in run]
            tmin = int(np.argmin(ids))
            c = [0] + [int(run[t][1] != run[t - 1][1]) for t in range(1, len(run))]
            recs.append([ids[0], nxt[0], len(run), ids[tmin], tmin, sum(c), sum(c[:tmin]), int(nxt[1] != run[-1][1])])
            edges.append(run)
    return recs, edges


@pytest.mark.parametrize("seed", range(12))
@pytest.mark.parametrize("nbands", [2, 3, 8])
def test_ring_segments_equal_a_walk(seed, nbands):
    rng = np.random.default_rng(seed * 31 + nbands)
    rings = make_rings(rng, int(rng.integers(1, 40)), nbands, int(rng.choice([5, 12, 60])))
    recs, edges = segments(rings)
    perm = rng.permutation(len(recs))             # the gathered order carries no meaning
    recs = [recs[i] for i in perm]
    edges = [edges[i] for i in perm]
    t = torch.tensor(recs, dtype=torch.int64)
    sol = bands.ring_segments(*[t[:, k].contiguous() for k in range(8)])
    want = brute(rings)
    by_leader = {w["leader"]: w for w in want}
    assert sol["leader"].tolist() == sorted(by_leader)
    for k, ld in enumerate(sol["leader"].tolist()):
        assert int(sol["L"][k]) == by_leader[ld]["L"] and int(sol["V"][k]) == by_leader[ld]["V"]
    seen_len1 = seen_mid = False
    for s, run in enumerate(edges):
        w = by_leader[int(sol["leader"][sol["ring"][s]])]
        L, V = w["L"], max(w["V"], 1)
        eoff, voff, ce = int(sol["eoff"][s]), int(sol["voff"][s]), int(sol["centry"][s])
        u = 0
        for t, (e, _, _) in enumerate(run):
            assert (eoff + t) % L == w["pos"][e]
            if t == 0:
                assert ce == (e in w["vert"])
                if ce:
                    assert voff % V == w["vert"][e]
            elif e in w["vert"]:
                assert (voff + ce + u) % V == w["vert"][e]
                u += 1
        seen_len1 |= len(run) == 1
        seen_mid |= 0 < [e for e, _, _ in run].index(min(e for e, _, _ in run)) < len(run) - 1
    if seed == 0:
        assert seen_len1 or seen_mid or len(edges) < 4


def test_ring_through_every_band_with_leader_mid_segment():
    # one ring visiting bands 0, 1, 2, 3, 2, 1 with its smallest edge in the middle of the band-1 run
    band = [0, 0, 1, 1, 1, 2, 3, 3, 2, 1]
    ids = [5, 6, 12, 2, 13, 20, 30, 31, 21, 14]
    sides = [0, 0, 1, 1, 2, 2, 3, 0, 0, 1]
    rings = [[(e, s, b) for e, s, b in zip(ids, sides, band)]]
    recs, edges = segments(rings)
    assert any(len(r) == 1 for r in edges)
    t = torch.tensor(recs, dtype=torch.int64)
    sol = bands.ring_segments(*[t[:, k].contiguous() for k in range(8)])
    w = brute(rings)[0]
    assert sol["leader"].tolist() == [2] and int(sol["L"][0]) == 10 and int(sol["V"][0]) == w["V"]
    for s, run in enumerate(edges):
        for tt, (e, _, _) in enumerate(run):
            assert (int(sol["eoff"][s]) + tt) % 10 == w["pos"][e]


def test_ring_segments_reject_a_broken_link():
    t = torch.tensor([[0, 7, 2, 0, 0, 0, 0, 0], [3, 0, 2, 3, 0, 0, 0, 0]], dtype=torch.int64)
    with pytest.raises(ValueError):
        bands.ring_segments(*[t[:, k].contiguous() for k in range(8)])


def test_no_segments():
    e = torch.zeros(0, dtype=torch.int64)
    sol = bands.ring_segments(*([e] * 8))
    assert sol["leader"].numel() == 0 and sol["eoff"].numel() == 0
