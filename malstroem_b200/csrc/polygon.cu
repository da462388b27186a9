// polygon.cu — SURVEY.md §8(f4): label polygonisation.
//
// Replaces vector.py:42-87 (`vectorize_labels_file`): `gdal.Polygonize(band, band.GetMaskBand(), layer, 0,
// ['8CONNECTED=8'])` — one polygon (an exterior ring and its holes) per 8-connected region of equal cell value; cells
// equal to the band's nodata value (if it has one) belong to no polygon.  GDAL walks the raster two rows at a time on
// one core and stitches edge strings; here every step is a data-parallel pass over cells or over boundary edges:
//
//   1. k_poly_count / scan      per cell: which of its 4 sides face another value (or the raster's edge) -> the cell's
//                               first edge number.  A boundary edge is DIRECTED: a cell's sides are walked clockwise on
//                               the screen (top: east, right: south, bottom: west, left: north), so the cell's region
//                               lies on the right-hand side of every edge.
//   2. k_poly_edges             the successor of every edge, decided at its end vertex from the two cells ahead:
//                               8-connected: ahead-left cell in the region -> turn left (the ring crosses over to the
//                               diagonal neighbour), else ahead-right in the region -> straight on, else turn right
//                               around the cell's corner; 4-connected: the mirror rule.  Every edge has exactly one
//                               successor and one predecessor: the edges fall into disjoint cycles, the rings.
//   3. k_poly_minjump           pointer doubling with a running minimum: every edge learns the lowest edge number of
//                               its ring (the ring's leader).  Synchronous rounds on a ping-pong pair of (leader, jump)
//                               words; a round that changes no leader is the last (proof in DESIGN.md §4 f4).
//   4. k_poly_rankjump          the same doubling with distances: steps from every edge to its ring's leader = its
//                               position in the ring.
//   5. scans + k_poly_place     rings numbered by leader, edges placed at (ring start + position); an edge whose
//                               predecessor runs in another direction starts at a corner: the corners, scanned, are the
//                               ring's vertices in order (k_poly_emit).
//   6. k_poly_union / k_poly_ring   which region a ring belongs to: union-find over the cells (equal value, 4 / 8
//                               neighbours), roots = the region's first cell in raster order.  A ring is an exterior
//                               ring iff its leader is a TOP side (the first cell of the region in raster order), a hole
//                               iff it is a BOTTOM side (the cells above the hole's first row) — no area sums needed.
// The result (ring table + vertex rows / columns as lattice corners) stays on the device until ms_polygonize_fetch
// copies it out; the host side (malstroem_b200/vector.py) groups rings into features and applies the geotransform.
#include <string.h>

#include "common.cuh"

namespace ms {

struct PolyHold {
    int64_t nrings = 0, nverts = 0, nedges = 0;
    int64_t *voff = nullptr;      // nrings + 1
    int32_t *value = nullptr;     // nrings
    int64_t *cell = nullptr;      // nrings: the leader's cell
    int64_t *region = nullptr;    // nrings: first cell of the ring's region
    uint8_t *hole = nullptr;      // nrings
    int32_t *vrow = nullptr, *vcol = nullptr;      // nverts
};
static PolyHold g_poly;

void poly_release() {
    cudaFree(g_poly.voff); cudaFree(g_poly.value); cudaFree(g_poly.cell); cudaFree(g_poly.region);
    cudaFree(g_poly.hole); cudaFree(g_poly.vrow); cudaFree(g_poly.vcol);
    g_poly = PolyHold();
}

// The kernels walk rows [0, rows) of `lab`; rows [r_lo, r_hi) may be read as neighbours.  One GPU: r_lo = 0,
// r_hi = rows.  A row band: r_lo = -1 / r_hi = rows + 1 where the neighbouring band's edge row is present as a halo row
// (lab - cols, lab + rows * cols), so that masks and successors on the band's first and last rows are the raster's.
struct PolyGrid {
    const int32_t *lab;
    int rows, cols;
    int connect8, has_nodata;
    int32_t nodata;
    int r_lo, r_hi;
};

__device__ inline bool poly_same(const PolyGrid &g, int r, int c, int32_t v) {
    return r >= g.r_lo && r < g.r_hi && c >= 0 && c < g.cols && g.lab[(int64_t)r * g.cols + c] == v;
}

// sides of the cell that are boundary edges: bit 0 top, 1 right, 2 bottom, 3 left
__device__ inline int poly_mask(const PolyGrid &g, int r, int c, int32_t v) {
    if (g.has_nodata && v == g.nodata) return 0;
    return (poly_same(g, r - 1, c, v) ? 0 : 1) | (poly_same(g, r, c + 1, v) ? 0 : 2) | (poly_same(g, r + 1, c, v) ? 0 : 4) |
           (poly_same(g, r, c - 1, v) ? 0 : 8);
}

__global__ void __launch_bounds__(256) k_poly_count(PolyGrid g, int *cnt) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)g.rows * g.cols) return;
    int r = (int)(i / g.cols), c = (int)(i - (int64_t)r * g.cols);
    cnt[i] = __popc(poly_mask(g, r, c, g.lab[i]));
}

// heading of side s: 0 east, 1 south, 2 west, 3 north; forward and right-hand vectors as (dr, dc)
__device__ __constant__ const int kFR[4] = {0, 1, 0, -1}, kFC[4] = {1, 0, -1, 0};
__device__ __constant__ const int kRR[4] = {1, 0, -1, 0}, kRC[4] = {0, -1, 0, 1};

// A row band's view of its neighbours (all null on one GPU, where no successor leaves the raster's rows).  A successor
// on a halo row is an EXIT: it gets the slot (row above: 2 c + {top 0, left 1}, row below: 2 cols + 2 c + {right 0,
// bottom 1}) as its ring key, points at itself and leaves its global successor in the slot; every other edge's key is
// its number with bit 31 set, so that pointer doubling gives a chain's edges the slot of their exit and a closed ring's
// edges (bit 31 set) their leader.
struct PolyHalo {
    const int64_t *eoff;          // [2][cols]: global first edge number of the halo cells (above, below)
    const uint8_t *mask;          // [2][cols]: their side masks
    int32_t *exit_edge;           // [4 cols]: local edge number in the slot (-1: none)
    int64_t *exit_next;           // [4 cols]: global number of its successor
    uint8_t *exit_corner;         // [4 cols]: 1 if that successor starts at a corner
};
constexpr unsigned kPolyChainBit = 0x80000000u;

__global__ void __launch_bounds__(256) k_poly_edges(PolyGrid g, const int *__restrict__ eoff, uint32_t *ecell,
                                                    int *succ, unsigned long long *state, PolyHalo hb) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)g.rows * g.cols) return;
    int r = (int)(i / g.cols), c = (int)(i - (int64_t)r * g.cols);
    const int32_t v = g.lab[i];
    const int mask = poly_mask(g, r, c, v);
    if (!mask) return;
    int e = eoff[i];
    for (int s = 0; s < 4; s++) {
        if (!(mask & (1 << s))) continue;
        // the cells ahead of the end vertex: ahead-right continues on the region's side, ahead-left on the other
        const int arr = r + kFR[s], arc = c + kFC[s];
        const int alr = arr - kRR[s], alc = arc - kRC[s];
        const bool in_ar = poly_same(g, arr, arc, v), in_al = poly_same(g, alr, alc, v);
        int nr, nc, ns;
        bool left, straight;
        if (g.connect8) { left = in_al; straight = !left && in_ar; }
        else { left = in_ar && in_al; straight = in_ar && !in_al; }
        if (left) { nr = alr; nc = alc; ns = (s + 3) & 3; }
        else if (straight) { nr = arr; nc = arc; ns = s; }
        else { nr = r; nc = c; ns = (s + 1) & 3; }
        ecell[e] = (uint32_t)((i << 2) | s);
        if (nr < 0 || nr >= g.rows) {         // only on a band with a halo row
            const int h = nr < 0 ? 0 : 1;
            const int slot = 2 * h * g.cols + 2 * c + ((s == 0 || s == 1) ? 0 : 1);
            hb.exit_edge[slot] = e;
            hb.exit_next[slot] = hb.eoff[h * g.cols + nc] + __popc(hb.mask[h * g.cols + nc] & ((1 << ns) - 1));
            hb.exit_corner[slot] = ns != s;
            succ[e] = e;
            state[e] = ((unsigned long long)(unsigned)slot << 32) | (unsigned)e;
            e++;
            continue;
        }
        const int64_t j = (int64_t)nr * g.cols + nc;
        const int nmask = (nr == r && nc == c) ? mask : poly_mask(g, nr, nc, v);
        const int q = eoff[j] + __popc(nmask & ((1 << ns) - 1));
        succ[e] = q;
        const unsigned key = hb.exit_edge ? ((unsigned)e | kPolyChainBit) : (unsigned)e;
        state[e] = ((unsigned long long)key << 32) | (unsigned)q;      // (leader so far, jump)
        e++;
    }
}

// hi word: lowest edge number among the 2^k edges from here on; lo word: the edge 2^k steps ahead
__global__ void __launch_bounds__(256) k_poly_minjump(const unsigned long long *__restrict__ a, unsigned long long *b,
                                                      int n, int *changed) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned long long x = a[e];
    const unsigned long long y = a[(unsigned)x];
    const unsigned lx = (unsigned)(x >> 32), ly = (unsigned)(y >> 32);
    const unsigned l = lx < ly ? lx : ly;
    b[e] = ((unsigned long long)l << 32) | (unsigned)y;
    if (l != lx) *changed = 1;
}

// hi word: steps from here to the jump target; lo word: the jump target (the leader points at itself, 0 steps; on a
// band an exit too, which ends its chain; key_bit: kPolyChainBit on a band, else 0)
__global__ void __launch_bounds__(256) k_poly_rankinit(const unsigned long long *__restrict__ lead_state,
                                                       const int *__restrict__ succ, unsigned long long *c, int n,
                                                       unsigned key_bit) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned lead = (unsigned)(lead_state[e] >> 32);
    const int q = succ[e];
    c[e] = (lead == ((unsigned)e | key_bit) || q == e) ? (unsigned long long)(unsigned)e : ((1ull << 32) | (unsigned)q);
}

__global__ void __launch_bounds__(256) k_poly_rankjump(const unsigned long long *__restrict__ a, unsigned long long *b,
                                                       int n, int *changed) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned long long x = a[e];
    const unsigned long long y = a[(unsigned)x];
    b[e] = (((x >> 32) + (y >> 32)) << 32) | (unsigned)y;
    if ((unsigned)y != (unsigned)x) *changed = 1;
}

// leaders: flag + ring length (scanned into ring number / ring start)
__global__ void __launch_bounds__(256) k_poly_leaders(const unsigned long long *__restrict__ lead_state,
                                                      const unsigned long long *__restrict__ rank,
                                                      const int *__restrict__ succ, int *isleader, int *ringlen, int n) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const bool ld = (unsigned)(lead_state[e] >> 32) == (unsigned)e;
    isleader[e] = ld;
    ringlen[e] = ld ? (int)(rank[succ[e]] >> 32) + 1 : 0;
}

// every edge goes to (start of its ring + position in the ring); it tells its successor's slot whether that one
// starts at a corner
__global__ void __launch_bounds__(256) k_poly_place(const unsigned long long *__restrict__ lead_state,
                                                    const unsigned long long *__restrict__ rank,
                                                    const int *__restrict__ succ, const uint32_t *__restrict__ ecell,
                                                    const int *__restrict__ rstart, const int *__restrict__ ringlen,
                                                    uint32_t *placed, int *corner, int n) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned lead = (unsigned)(lead_state[e] >> 32);
    const int L = ringlen[lead], base = rstart[lead];
    const int d = (int)(rank[e] >> 32);
    const int pos = d == 0 ? 0 : L - d;
    placed[base + pos] = ecell[e];
    const int q = succ[e];
    corner[base + (pos + 1 == L ? 0 : pos + 1)] = (ecell[q] & 3u) != (ecell[e] & 3u);
}

__global__ void __launch_bounds__(256) k_poly_emit(const uint32_t *__restrict__ placed, const int *__restrict__ corner,
                                                   const int *__restrict__ vidx, int cols, int row0, int32_t *vrow,
                                                   int32_t *vcol, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || !corner[k]) return;
    const uint32_t ec = placed[k];
    const int s = (int)(ec & 3u);
    const int64_t i = (int64_t)(ec >> 2);
    const int r = (int)(i / cols), c = (int)(i - (int64_t)r * cols);
    // start vertex of the side: top (r, c), right (r, c + 1), bottom (r + 1, c + 1), left (r + 1, c)
    const int v = vidx[k];
    vrow[v] = row0 + r + (s >= 2 ? 1 : 0);
    vcol[v] = c + ((s == 1 || s == 2) ? 1 : 0);
}

// ---- regions: union-find over the cells, roots = lowest cell index (every write is an atomicMin towards an ancestor)
__device__ inline int poly_root(int *par, int x) {
    for (;;) {
        int p = *(volatile int *)(par + x);
        if (p == x) return x;
        int gp = *(volatile int *)(par + p);
        if (gp != p) atomicMin(par + x, gp);
        x = p;
    }
}

__device__ inline void poly_unite(int *par, int a, int b) {
    for (;;) {
        a = poly_root(par, a);
        b = poly_root(par, b);
        if (a == b) return;
        const int hi = a > b ? a : b, lo = a > b ? b : a;
        const int old = atomicMin(par + hi, lo);
        if (old == hi) return;
        a = old;
        b = lo;
    }
}

__global__ void __launch_bounds__(256) k_poly_parinit(int *par, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) par[i] = (int)i;
}

// the cells of rows [0, rows) only: a band joins its regions to its neighbours' afterwards (ms_cc_boundary_merge_values)
__global__ void __launch_bounds__(256) k_poly_union(PolyGrid g, int *par) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)g.rows * g.cols) return;
    g.r_lo = 0;
    g.r_hi = g.rows;
    int r = (int)(i / g.cols), c = (int)(i - (int64_t)r * g.cols);
    const int32_t v = g.lab[i];
    if (g.has_nodata && v == g.nodata) return;
    if (poly_same(g, r, c - 1, v)) poly_unite(par, (int)i, (int)i - 1);
    if (poly_same(g, r - 1, c, v)) poly_unite(par, (int)i, (int)i - g.cols);
    if (g.connect8) {
        // a diagonal neighbour only matters when neither cell between the two joins them already
        if (poly_same(g, r - 1, c - 1, v) && !poly_same(g, r - 1, c, v) && !poly_same(g, r, c - 1, v))
            poly_unite(par, (int)i, (int)i - g.cols - 1);
        if (poly_same(g, r - 1, c + 1, v) && !poly_same(g, r - 1, c, v)) poly_unite(par, (int)i, (int)i - g.cols + 1);
    }
}

__global__ void __launch_bounds__(256) k_poly_ring(PolyGrid g, const int *__restrict__ isleader,
                                                   const int *__restrict__ ridx, const int *__restrict__ rstart,
                                                   const int *__restrict__ vidx, const uint32_t *__restrict__ ecell,
                                                   int *par, int64_t *voff, int32_t *value, int64_t *cell, int64_t *region,
                                                   uint8_t *hole, int n, int64_t nrings, int64_t nverts) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e == 0) voff[nrings] = nverts;
    if (e >= n || !isleader[e]) return;
    const int k = ridx[e];
    const uint32_t ec = ecell[e];
    const int64_t i = (int64_t)(ec >> 2);
    voff[k] = vidx[rstart[e]];
    value[k] = g.lab[i];
    cell[k] = i;
    region[k] = poly_root(par, (int)i);
    hole[k] = (ec & 3u) != 0u;        // exterior rings start with a top side, holes with a bottom side
}

// synchronous doubling rounds on a ping-pong pair; *a holds the result
static int jump_rounds(bool rank, unsigned long long **a, unsigned long long **b, int n, cudaStream_t s) {
    DevBuf<int> flag;
    MS_TRY(flag.alloc(1, s));
    int64_t *h = host_flags().h;
    for (int round = 0;; round++) {
        if (round > 40) { set_error("polygonize: ring %s did not converge", rank ? "positions" : "leaders"); return MS_ERR_NOCONV; }
        MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
        if (rank) MS_LAUNCH(k_poly_rankjump, cdiv(n, 256), 256, 0, s, (const unsigned long long *)*a, *b, n, flag.p);
        else MS_LAUNCH(k_poly_minjump, cdiv(n, 256), 256, 0, s, (const unsigned long long *)*a, *b, n, flag.p);
        MS_TRY(ms::readback(h, flag.p, sizeof(int), s));
        MS_TRY(stream_sync(s));
        unsigned long long *t = *a; *a = *b; *b = t;
        if (*(int *)h == 0) return MS_OK;
    }
}

template <class T>
static int hold_alloc(T **p, size_t count) {
    if (cudaMalloc((void **)p, (count ? count : 1) * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        set_error("polygonize: cudaMalloc of %zu bytes failed", count * sizeof(T));
        return MS_ERR_CUDA;
    }
    return MS_OK;
}

int polygonize_dev_impl(const int32_t *labels, int64_t rows, int64_t cols, int connect8, int has_nodata, int32_t nodata,
                        int64_t *counts3, cudaStream_t s) {
    if (!labels || !counts3 || rows < 1 || cols < 1 || rows * cols > (1ll << 30)) {
        set_error("polygonize: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_ARG;
    }
    poly_release();
    const int64_t n = rows * cols;
    PolyGrid g{labels, (int)rows, (int)cols, connect8 ? 1 : 0, has_nodata ? 1 : 0, nodata, 0, (int)rows};
    int64_t *h = host_flags().h;
    DevBuf<int> eoff;
    DevBuf<int64_t> total;
    MS_TRY(eoff.alloc((size_t)n, s));
    MS_TRY(total.alloc(1, s));
    MS_LAUNCH(k_poly_count, cdiv(n, 256), 256, 0, s, g, eoff.p);
    {
        // the scan's block sums are int32: the edge count has to fit
        MS_TRY(exclusive_scan_i32(eoff.p, eoff.p, n, total.p, s));
        MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
        MS_TRY(stream_sync(s));
    }
    const int64_t E = h[0];
    if (E < 0 || E >= (1ll << 31) - 1024) { set_error("polygonize: %lld boundary edges do not fit", (long long)E); return MS_ERR_ARG; }
    counts3[0] = counts3[1] = 0;
    counts3[2] = E;
    if (E == 0) {        // everything is nodata
        MS_TRY(hold_alloc(&g_poly.voff, 1));
        MS_CUDA(cudaMemsetAsync(g_poly.voff, 0, sizeof(int64_t), s));
        MS_TRY(stream_sync(s));
        return MS_OK;
    }
    const int ne = (int)E;
    DevBuf<uint32_t> ecell, placed;
    DevBuf<int> succ, isleader, ringlen, par;
    DevBuf<unsigned long long> sa, sb, ra, rb;
    MS_TRY(ecell.alloc((size_t)ne, s));
    MS_TRY(succ.alloc((size_t)ne, s));
    MS_TRY(sa.alloc((size_t)ne, s));
    MS_TRY(sb.alloc((size_t)ne, s));
    MS_LAUNCH(k_poly_edges, cdiv(n, 256), 256, 0, s, g, (const int *)eoff.p, ecell.p, succ.p, sa.p, PolyHalo{});
    unsigned long long *a = sa.p, *b = sb.p;
    MS_TRY(jump_rounds(false, &a, &b, ne, s));
    unsigned long long *lead_state = a;       // hi word = the ring's leader; the other buffer is free again
    MS_TRY(ra.alloc((size_t)ne, s));
    MS_LAUNCH(k_poly_rankinit, cdiv(ne, 256), 256, 0, s, (const unsigned long long *)lead_state, (const int *)succ.p, ra.p, ne,
              0u);
    unsigned long long *c = ra.p, *d = b;
    MS_TRY(jump_rounds(true, &c, &d, ne, s));
    unsigned long long *rank = c;
    // the regions (independent of the rings; the ring table needs their roots)
    MS_TRY(par.alloc((size_t)n, s));
    MS_LAUNCH(k_poly_parinit, cdiv(n, 256), 256, 0, s, par.p, n);
    MS_LAUNCH(k_poly_union, cdiv(n, 256), 256, 0, s, g, par.p);
    // ring numbers and ring starts
    MS_TRY(isleader.alloc((size_t)ne, s));
    MS_TRY(ringlen.alloc((size_t)ne, s));
    MS_LAUNCH(k_poly_leaders, cdiv(ne, 256), 256, 0, s, (const unsigned long long *)lead_state, (const unsigned long long *)rank,
              (const int *)succ.p, isleader.p, ringlen.p, ne);
    DevBuf<int> ridx, rstart, corner, vidx;
    MS_TRY(ridx.alloc((size_t)ne, s));
    MS_TRY(rstart.alloc((size_t)ne, s));
    MS_TRY(exclusive_scan_i32(isleader.p, ridx.p, ne, total.p, s));
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(stream_sync(s));
    const int64_t nrings = h[0];
    MS_TRY(exclusive_scan_i32(ringlen.p, rstart.p, ne, total.p, s));
    MS_TRY(placed.alloc((size_t)ne, s));
    MS_TRY(corner.alloc((size_t)ne, s));
    MS_TRY(vidx.alloc((size_t)ne, s));
    MS_LAUNCH(k_poly_place, cdiv(ne, 256), 256, 0, s, (const unsigned long long *)lead_state, (const unsigned long long *)rank,
              (const int *)succ.p, (const uint32_t *)ecell.p, (const int *)rstart.p, (const int *)ringlen.p, placed.p, corner.p, ne);
    MS_TRY(exclusive_scan_i32(corner.p, vidx.p, ne, total.p, s));
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(stream_sync(s));
    const int64_t nverts = h[0];
    MS_TRY(hold_alloc(&g_poly.voff, (size_t)nrings + 1));
    MS_TRY(hold_alloc(&g_poly.value, (size_t)nrings));
    MS_TRY(hold_alloc(&g_poly.cell, (size_t)nrings));
    MS_TRY(hold_alloc(&g_poly.region, (size_t)nrings));
    MS_TRY(hold_alloc(&g_poly.hole, (size_t)nrings));
    MS_TRY(hold_alloc(&g_poly.vrow, (size_t)nverts));
    MS_TRY(hold_alloc(&g_poly.vcol, (size_t)nverts));
    MS_LAUNCH(k_poly_emit, cdiv(ne, 256), 256, 0, s, (const uint32_t *)placed.p, (const int *)corner.p, (const int *)vidx.p,
              (int)cols, 0, g_poly.vrow, g_poly.vcol, ne);
    MS_LAUNCH(k_poly_ring, cdiv(ne, 256), 256, 0, s, g, (const int *)isleader.p, (const int *)ridx.p, (const int *)rstart.p,
              (const int *)vidx.p, (const uint32_t *)ecell.p, par.p, g_poly.voff, g_poly.value, g_poly.cell, g_poly.region,
              g_poly.hole, ne, nrings, nverts);
    MS_TRY(stream_sync(s));
    g_poly.nrings = nrings;
    g_poly.nverts = nverts;
    g_poly.nedges = E;
    counts3[0] = nrings;
    counts3[1] = nverts;
    return MS_OK;
}


// ---- row bands (DESIGN.md §8(f4), malstroem_b200/vector.py polygonize_band) -------------------------------------------
// Every buffer that lives from one phase to the next belongs to the caller: the bands of one process run these calls
// from several threads.  Edge numbers are the band's own (0 .. n_edges - 1); the band's first edge has global number
// base = the edge counts of the lower bands, so local order is global order.  After the doubling an edge's ring key
// says what it is: bit 31 set -> a closed ring of the band (key - bit 31 = its leader), else the slot of the exit that
// ends its chain.  A chain starts at an ENTRY (an edge whose predecessor lies in another band) and runs to its exit: a
// SEGMENT.  Units = closed rings and segments, numbered by their head (the leader, the entry) in edge order; every
// edge is placed at (unit start + position), the leader / the entry at position 0.

static inline PolyGrid poly_band_grid(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8,
                                          int has_nodata, int32_t nodata) {
    return PolyGrid{lab, (int)rows, (int)cols, connect8 ? 1 : 0, has_nodata ? 1 : 0, nodata, (halo & 1) ? -1 : 0,
                    (int)rows + ((halo & 2) ? 1 : 0)};
}

// local first edge number and side mask of the band's first and last row (for the neighbours' halo)
__global__ void __launch_bounds__(256) k_poly_band_rows(PolyGrid g, const int *__restrict__ eoff, int32_t *row_eoff,
                                                        uint8_t *row_mask) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= 2 * g.cols) return;
    const int r = k < g.cols ? 0 : g.rows - 1, c = k < g.cols ? k : k - g.cols;
    const int64_t i = (int64_t)r * g.cols + c;
    row_eoff[k] = eoff[i];
    row_mask[k] = (uint8_t)poly_mask(g, r, c, g.lab[i]);
}

// predecessor flags; the smallest edge of every segment (by its exit's slot)
__global__ void __launch_bounds__(256) k_poly_band_pred(const unsigned long long *__restrict__ lead_state,
                                                        const int *__restrict__ succ, int *haspred, int *seg_min, int n) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int q = succ[e];
    if (q != e) haspred[q] = 1;
    const unsigned key = (unsigned)(lead_state[e] >> 32);
    if (!(key & kPolyChainBit)) atomicMin((unsigned *)seg_min + key, (unsigned)e);
}

// unit heads and lengths (scanned into unit number / unit start); a segment's entry registers in its exit's slot
__global__ void __launch_bounds__(256) k_poly_band_heads(const unsigned long long *__restrict__ lead_state,
                                                         const unsigned long long *__restrict__ rank,
                                                         const int *__restrict__ succ, const int *__restrict__ haspred,
                                                         int *ishead, int *ulen, int *seg_entry, int n) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned key = (unsigned)(lead_state[e] >> 32);
    bool h;
    int len = 0;
    if (key & kPolyChainBit) {
        h = key == ((unsigned)e | kPolyChainBit);
        if (h) len = (int)(rank[succ[e]] >> 32) + 1;
    } else {
        h = !haspred[e];
        if (h) { len = (int)(rank[e] >> 32) + 1; seg_entry[key] = e; }
    }
    ishead[e] = h;
    ulen[e] = len;
}

// as k_poly_place, for closed rings (position from the leader) and segments (position from the entry: length - 1 -
// steps to the exit); a segment's first slot stays 0 here (its corner flag depends on the band before it)
__global__ void __launch_bounds__(256) k_poly_band_place(const unsigned long long *__restrict__ lead_state,
                                                         const unsigned long long *__restrict__ rank,
                                                         const int *__restrict__ succ, const uint32_t *__restrict__ ecell,
                                                         const int *__restrict__ ustart, const int *__restrict__ ulen,
                                                         const int *__restrict__ seg_entry,
                                                         const int *__restrict__ seg_min, uint32_t *placed, int *corner,
                                                         int *seg_tmin, int n) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const unsigned key = (unsigned)(lead_state[e] >> 32);
    const int d = (int)(rank[e] >> 32);
    const int q = succ[e];
    const bool ring = key & kPolyChainBit;
    const int head = ring ? (int)(key & ~kPolyChainBit) : seg_entry[key];
    const int L = ulen[head], base = ustart[head];
    const int pos = ring ? (d == 0 ? 0 : L - d) : L - 1 - d;
    placed[base + pos] = ecell[e];
    if (ring) corner[base + (pos + 1 == L ? 0 : pos + 1)] = (ecell[q] & 3u) != (ecell[e] & 3u);
    else {
        if (q != e) corner[base + pos + 1] = (ecell[q] & 3u) != (ecell[e] & 3u);
        if ((unsigned)seg_min[key] == (unsigned)e) seg_tmin[key] = pos;
    }
}

// the unit table: head edge, length, first vertex, vertex count, value, region root (global cell index of the band's
// local root), exit slot (-1: a closed ring)
__global__ void __launch_bounds__(256) k_poly_band_units(PolyGrid g, const unsigned long long *__restrict__ lead_state,
                                                         const int *__restrict__ ishead, const int *__restrict__ uidx,
                                                         const int *__restrict__ ustart, const int *__restrict__ ulen,
                                                         const int *__restrict__ vidx, const uint32_t *__restrict__ ecell,
                                                         int *par, int64_t cell0, int n, int nverts, int32_t *u_head,
                                                         int32_t *u_len, int32_t *u_vstart, int32_t *u_vcount,
                                                         int32_t *u_value, int64_t *u_root, int32_t *u_slot) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n || !ishead[e]) return;
    const int k = uidx[e];
    const int a = ustart[e], L = ulen[e];
    const int v0 = vidx[a];
    const unsigned key = (unsigned)(lead_state[e] >> 32);
    const int i = (int)(ecell[e] >> 2);
    u_head[k] = e;
    u_len[k] = L;
    u_vstart[k] = v0;
    u_vcount[k] = (a + L < n ? vidx[a + L] : nverts) - v0;
    u_value[k] = g.lab[i];
    u_root[k] = cell0 + poly_root(par, i);
    u_slot[k] = (key & kPolyChainBit) ? -1 : (int)key;
}

// region roots (global cell index, -1 for nodata) of the band's first and last row
__global__ void __launch_bounds__(256) k_poly_band_rowroots(PolyGrid g, int *par, int64_t cell0, int64_t *root_rows) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= 2 * g.cols) return;
    const int r = k < g.cols ? 0 : g.rows - 1, c = k < g.cols ? k : k - g.cols;
    const int i = r * g.cols + c;
    root_rows[k] = (g.has_nodata && g.lab[i] == g.nodata) ? -1 : cell0 + poly_root(par, i);
}

static int band_poly_args(const int32_t *lab, int64_t rows, int64_t cols, int halo) {
    if (!lab || rows < 1 || cols < 1 || rows * cols > (1ll << 30) || (halo & ~3)) {
        set_error("band polygonize: unsupported band %lld x %lld (halo %d)", (long long)rows, (long long)cols, halo);
        return MS_ERR_ARG;
    }
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_polygonize_dev(const int32_t *labels, int64_t rows, int64_t cols, int connect8, int has_nodata, int32_t nodata,
                      int64_t *counts3, void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::polygonize_dev_impl(labels, rows, cols, connect8, has_nodata, nodata, counts3, (cudaStream_t)stream);
}

int ms_polygonize(const int32_t *labels, int64_t rows, int64_t cols, int connect8, int has_nodata, int32_t nodata,
                  int64_t *counts3) {
    MS_TRY(ms::ensure_init());
    if (!labels || !counts3 || rows < 1 || cols < 1) { ms::set_error("polygonize: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    ms::HostCall hc;
    int32_t *l = nullptr;
    MS_TRY(hc.in(labels, (size_t)(rows * cols), s, &l));
    return ms::polygonize_dev_impl(l, rows, cols, connect8, has_nodata, nodata, counts3, s);
}

int ms_band_poly_count_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                           int32_t nodata, int32_t *eoff, int64_t *n_edges, int32_t *row_eoff, uint8_t *row_mask,
                           void *stream) {
    MS_TRY(ms::ensure_init());
    MS_TRY(ms::band_poly_args(lab, rows, cols, halo));
    if (!eoff || !n_edges || !row_eoff || !row_mask) { ms::set_error("band_poly_count: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = rows * cols;
    ms::PolyGrid g = ms::poly_band_grid(lab, rows, cols, halo, connect8, has_nodata, nodata);
    ms::DevBuf<int64_t> total;
    MS_TRY(total.alloc(1, s));
    MS_LAUNCH(ms::k_poly_count, ms::cdiv(n, 256), 256, 0, s, g, eoff);
    MS_TRY(ms::exclusive_scan_i32(eoff, eoff, n, total.p, s));
    MS_LAUNCH(ms::k_poly_band_rows, ms::cdiv(2 * cols, 256), 256, 0, s, g, (const int *)eoff, row_eoff, row_mask);
    int64_t *h = ms::host_flags().h;
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    *n_edges = h[0];
    if (h[0] < 0 || h[0] >= (1ll << 31) - 1024) {
        ms::set_error("band polygonize: %lld boundary edges in one band do not fit", (long long)h[0]);
        return MS_ERR_ARG;
    }
    return MS_OK;
}

int ms_band_poly_edges_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                           int32_t nodata, const int32_t *eoff, int64_t n_edges, const int64_t *halo_eoff,
                           const uint8_t *halo_mask, uint32_t *ecell, int32_t *succ, uint64_t *lead, uint64_t *rank,
                           int32_t *exit_edge, int64_t *exit_next, uint8_t *exit_corner, void *stream) {
    MS_TRY(ms::ensure_init());
    MS_TRY(ms::band_poly_args(lab, rows, cols, halo));
    if (n_edges < 1 || n_edges >= (1ll << 31) - 1024 || !eoff || !halo_eoff || !halo_mask || !ecell || !succ || !lead ||
        !rank || !exit_edge || !exit_next || !exit_corner) {
        ms::set_error("band_poly_edges: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = rows * cols;
    const int ne = (int)n_edges;
    ms::PolyGrid g = ms::poly_band_grid(lab, rows, cols, halo, connect8, has_nodata, nodata);
    MS_CUDA(cudaMemsetAsync(exit_edge, 0xff, (size_t)4 * cols * sizeof(int32_t), s));
    ms::PolyHalo hb{halo_eoff, halo_mask, exit_edge, exit_next, exit_corner};
    unsigned long long *sa = (unsigned long long *)lead, *sr = (unsigned long long *)rank;
    MS_LAUNCH(ms::k_poly_edges, ms::cdiv(n, 256), 256, 0, s, g, eoff, ecell, succ, sa, hb);
    ms::DevBuf<unsigned long long> tmp;
    MS_TRY(tmp.alloc((size_t)ne, s));
    unsigned long long *a = sa, *b = tmp.p;
    MS_TRY(ms::jump_rounds(false, &a, &b, ne, s));
    if (a != sa) MS_CUDA(cudaMemcpyAsync(sa, a, (size_t)ne * 8, cudaMemcpyDeviceToDevice, s));
    MS_LAUNCH(ms::k_poly_rankinit, ms::cdiv(ne, 256), 256, 0, s, (const unsigned long long *)sa, (const int *)succ, sr, ne,
              ms::kPolyChainBit);
    a = sr;
    b = tmp.p;
    MS_TRY(ms::jump_rounds(true, &a, &b, ne, s));
    if (a != sr) MS_CUDA(cudaMemcpyAsync(sr, a, (size_t)ne * 8, cudaMemcpyDeviceToDevice, s));
    return ms::stream_sync(s);
}

int ms_band_poly_place_dev(int64_t cols, int64_t n_edges, const uint32_t *ecell, const int32_t *succ,
                           const uint64_t *lead, const uint64_t *rank, int32_t *ishead, int32_t *uidx, int32_t *ulen,
                           int32_t *ustart, uint32_t *placed, int32_t *corner, int32_t *vidx, int32_t *seg_entry,
                           int32_t *seg_min, int32_t *seg_tmin, int64_t *counts2, void *stream) {
    MS_TRY(ms::ensure_init());
    if (cols < 1 || n_edges < 1 || n_edges >= (1ll << 31) - 1024 || !ecell || !succ || !lead || !rank || !ishead ||
        !uidx || !ulen || !ustart || !placed || !corner || !vidx || !seg_entry || !seg_min || !seg_tmin || !counts2) {
        ms::set_error("band_poly_place: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int ne = (int)n_edges;
    const unsigned long long *ls = (const unsigned long long *)lead, *rk = (const unsigned long long *)rank;
    MS_CUDA(cudaMemsetAsync(corner, 0, (size_t)ne * sizeof(int), s));       // first the predecessor flags
    MS_CUDA(cudaMemsetAsync(seg_min, 0xff, (size_t)4 * cols * sizeof(int), s));        // compared as unsigned
    MS_LAUNCH(ms::k_poly_band_pred, ms::cdiv(ne, 256), 256, 0, s, ls, (const int *)succ, corner, seg_min, ne);
    MS_LAUNCH(ms::k_poly_band_heads, ms::cdiv(ne, 256), 256, 0, s, ls, rk, (const int *)succ, (const int *)corner, ishead,
              ulen, seg_entry, ne);
    ms::DevBuf<int64_t> total;
    MS_TRY(total.alloc(1, s));
    int64_t *h = ms::host_flags().h;
    MS_TRY(ms::exclusive_scan_i32(ishead, uidx, ne, total.p, s));
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    counts2[0] = h[0];
    MS_TRY(ms::exclusive_scan_i32(ulen, ustart, ne, total.p, s));
    MS_CUDA(cudaMemsetAsync(corner, 0, (size_t)ne * sizeof(int), s));
    MS_LAUNCH(ms::k_poly_band_place, ms::cdiv(ne, 256), 256, 0, s, ls, rk, (const int *)succ, ecell, (const int *)ustart,
              (const int *)ulen, (const int *)seg_entry, (const int *)seg_min, placed, corner, seg_tmin, ne);
    MS_TRY(ms::exclusive_scan_i32(corner, vidx, ne, total.p, s));
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    counts2[1] = h[0];
    return MS_OK;
}

int ms_band_poly_emit_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                          int32_t nodata, int64_t row0, int64_t n_edges, const uint32_t *ecell, const uint64_t *lead,
                          const int32_t *ishead, const int32_t *uidx, const int32_t *ulen, const int32_t *ustart,
                          const uint32_t *placed, const int32_t *corner, const int32_t *vidx, int64_t nverts,
                          int32_t *vrow, int32_t *vcol, int32_t *u_head, int32_t *u_len, int32_t *u_vstart,
                          int32_t *u_vcount, int32_t *u_value, int64_t *u_root, int32_t *u_slot, int64_t *root_rows,
                          void *stream) {
    MS_TRY(ms::ensure_init());
    MS_TRY(ms::band_poly_args(lab, rows, cols, halo));
    if (n_edges < 1 || n_edges >= (1ll << 31) - 1024 || nverts < 0 || nverts > n_edges || !ecell || !lead || !ishead ||
        !uidx || !ulen || !ustart || !placed || !corner || !vidx || !vrow || !vcol || !u_head || !u_len || !u_vstart ||
        !u_vcount || !u_value || !u_root || !u_slot || !root_rows) {
        ms::set_error("band_poly_emit: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = rows * cols, cell0 = row0 * cols;
    const int ne = (int)n_edges;
    ms::PolyGrid g = ms::poly_band_grid(lab, rows, cols, halo, connect8, has_nodata, nodata);
    MS_LAUNCH(ms::k_poly_emit, ms::cdiv(ne, 256), 256, 0, s, placed, corner, vidx, (int)cols, (int)row0, vrow, vcol, ne);
    ms::DevBuf<int> par;
    MS_TRY(par.alloc((size_t)n, s));
    MS_LAUNCH(ms::k_poly_parinit, ms::cdiv(n, 256), 256, 0, s, par.p, n);
    MS_LAUNCH(ms::k_poly_union, ms::cdiv(n, 256), 256, 0, s, g, par.p);
    MS_LAUNCH(ms::k_poly_band_units, ms::cdiv(ne, 256), 256, 0, s, g, (const unsigned long long *)lead, ishead, uidx,
              ustart, ulen, vidx, ecell, par.p, cell0, ne, (int)nverts, u_head, u_len, u_vstart, u_vcount, u_value,
              u_root, u_slot);
    MS_LAUNCH(ms::k_poly_band_rowroots, ms::cdiv(2 * cols, 256), 256, 0, s, g, par.p, cell0, root_rows);
    return ms::stream_sync(s);
}

/* copies the rings of the last ms_polygonize* call to host arrays (sizes from its counts) and releases them */
int ms_polygonize_fetch(int64_t *ring_vertex_offset, int32_t *ring_value, int64_t *ring_cell, int64_t *ring_region,
                        uint8_t *ring_hole, int32_t *vertex_row, int32_t *vertex_col) {
    MS_TRY(ms::ensure_init());
    ms::PolyHold &p = ms::g_poly;
    if (!p.voff) { ms::set_error("polygonize_fetch: no result is held (ms_polygonize first)"); return MS_ERR_ARG; }
    if (!ring_vertex_offset || (p.nrings && (!ring_value || !ring_cell || !ring_region || !ring_hole)) ||
        (p.nverts && (!vertex_row || !vertex_col))) {
        ms::set_error("polygonize_fetch: null pointer");
        return MS_ERR_ARG;
    }
    cudaStream_t s = nullptr;
    MS_CUDA(cudaMemcpyAsync(ring_vertex_offset, p.voff, (size_t)(p.nrings + 1) * 8, cudaMemcpyDeviceToHost, s));
    if (p.nrings) {
        MS_CUDA(cudaMemcpyAsync(ring_value, p.value, (size_t)p.nrings * 4, cudaMemcpyDeviceToHost, s));
        MS_CUDA(cudaMemcpyAsync(ring_cell, p.cell, (size_t)p.nrings * 8, cudaMemcpyDeviceToHost, s));
        MS_CUDA(cudaMemcpyAsync(ring_region, p.region, (size_t)p.nrings * 8, cudaMemcpyDeviceToHost, s));
        MS_CUDA(cudaMemcpyAsync(ring_hole, p.hole, (size_t)p.nrings, cudaMemcpyDeviceToHost, s));
    }
    if (p.nverts) {
        MS_CUDA(cudaMemcpyAsync(vertex_row, p.vrow, (size_t)p.nverts * 4, cudaMemcpyDeviceToHost, s));
        MS_CUDA(cudaMemcpyAsync(vertex_col, p.vcol, (size_t)p.nverts * 4, cudaMemcpyDeviceToHost, s));
    }
    MS_TRY(ms::stream_sync(s));
    ms::poly_release();
    return MS_OK;
}

}  // extern "C"
