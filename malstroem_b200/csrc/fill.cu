// fill.cu — K0 (min/max) and K1: plain depression fill as a catchment graph + Boruvka contraction.
//
// Replaces fill.fill_terrain (malstroem/algorithms/fill.py:112-171; sweeps speedups/_fill.pyx:28-70),
// whose result is the greatest fixed point of W = max(z, min over the 8 neighbours of W) with W = z on
// the raster border, i.e. W(c) = the lowest "highest cell" over all paths from c to the border.  Only
// min/max of input values are involved, so any algorithm that reaches the fixed point is bit-exact.
//
//   1. k_descent_tile every interior cell points at the smallest cell of its 3x3 window in the strict
//                     total order (z, flat index); border cells drain to "outside" (id 0); the local minima
//                     ("catchments") get dense ids in tile order (a decoupled look-back over the per-tile counts);
//                     in-tile paths are compressed in shared memory
//   2. forest_resolve_ids  pointer jumping for the cells whose path leaves their tile -> every cell holds the id of
//                     the catchment it drains to
//   3. Boruvka on the catchment graph (edge weight = max(z_a, z_b) over adjacent cells of two catchments).
//                     One CTA per tile (k_tile_edges) writes the catchment-pair edge list, aggregated per tile, and
//                     finds every catchment's lowest edge (64-bit atomicMin of (weight, list position)).  Each
//                     round every live component hooks across its lowest edge and records that weight (wk); the
//                     roots that have not reached "outside" get dense new ids, and the edges are relabelled, those
//                     inside one component dropped, the rest compacted and searched for the next round's lowest
//                     edges.  After the last round E = max of wk over the levels of the
//                     catchment's component until it reaches outside (k_spill_down, top level first).
//                     Claim (DESIGN.md §K1): E is the catchment's spill elevation.
//   4. k_fill_final   filled = max(z, E[catchment]), depths = filled - z
#include <string.h>

#include "common.cuh"
#include "tma.cuh"

namespace ms {

constexpr unsigned long long KEY_NONE = ~0ull;
constexpr unsigned long long HASH_EMPTY = ~0ull;

// ---- K0 -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_minmax(const float *z, int64_t n, uint32_t *keys, int vec) {
    uint32_t lo = 0xffffffffu, hi = 0u;
    int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    for (; i < n; i += stride) {
        if (vec && i + 4 <= n) {
            float4 v = *reinterpret_cast<const float4 *>(z + i);
            uint32_t a = okey32(v.x), b = okey32(v.y), c = okey32(v.z), d = okey32(v.w);
            lo = min(lo, min(min(a, b), min(c, d)));
            hi = max(hi, max(max(a, b), max(c, d)));
        } else {
            for (int64_t j = i; j < n && j < i + 4; j++) {
                uint32_t a = okey32(z[j]);
                lo = min(lo, a);
                hi = max(hi, a);
            }
        }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    __shared__ uint32_t slo[8], shi[8];
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { slo[w] = lo; shi[w] = hi; }
    __syncthreads();
    if (w == 0) {
        lo = lane < 8 ? slo[lane] : 0xffffffffu;
        hi = lane < 8 ? shi[lane] : 0u;
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (lane == 0) {
            atomicMin(&keys[0], lo);
            atomicMax(&keys[1], hi);
        }
    }
}

__global__ void k_minmax_finish(const uint32_t *keys, float *out) {
    out[0] = okey32_inv(keys[0]);
    out[1] = okey32_inv(keys[1]);
}

int minmax_dev(const float *z, int64_t n, float *out2, cudaStream_t s) {
    DevBuf<uint32_t> keys;
    MS_TRY(keys.alloc(2, s));
    static const uint32_t init[2] = {0xffffffffu, 0u};
    MS_CUDA(cudaMemcpyAsync(keys.p, init, sizeof(init), cudaMemcpyHostToDevice, s));
    int64_t want = (n / 4 + 255) / 256;
    int blocks = (int)(want < 1 ? 1 : (want > 148 * 16 ? 148 * 16 : want));
    // 128-bit loads need a 16-byte aligned base (a band's first own row need not be)
    MS_LAUNCH(k_minmax, blocks, 256, 0, s, z, n, keys.p, (int)(((uintptr_t)z & 15) == 0));
    MS_LAUNCH(k_minmax_finish, 1, 1, 0, s, keys.p, out2);
    return MS_OK;
}

// ---- K1 -------------------------------------------------------------------------------------------
// Catchment numbering in tile order: the local minima of tile T get the ids base(T) + 1 .. base(T) + count(T), where
// base(T) is the number of local minima in the tiles before T (0 = "outside").  base comes from a single-pass
// decoupled look-back over one status word per tile: flag in the high half, catchment count in the low half, so that
// one load reads both.  TS_AGG: the tile's own count; TS_INCL: the count of the tile and every tile before it.
constexpr unsigned long long TS_AGG = 1ull << 32, TS_INCL = 2ull << 32;

__device__ __forceinline__ void st_release_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.gpu.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// one full warp: catchments of the tiles before `tile`.  Every tile before it has taken its ticket (so it runs) and
// publishes its TS_AGG word before it waits for anything, so the wait ends.
__device__ int tile_lookback(const unsigned long long *status, int tile) {
    const int lane = threadIdx.x & 31;
    int excl = 0;
    for (int end = tile - 1; end >= 0; end -= 32) {
        const int j = end - lane;
        unsigned long long st;
        for (;;) {
            st = j >= 0 ? ld_acquire_u64(status + j) : TS_INCL;
            if (__all_sync(0xffffffffu, (st >> 32) != 0)) break;
        }
        const unsigned incl = __ballot_sync(0xffffffffu, (st >> 32) == 2);
        // the nearest inclusive word ends the look-back: add it and the aggregates after it
        int v = (int)(unsigned)st;
        if (incl && lane > __ffs(incl) - 1) v = 0;
        excl += __reduce_add_sync(0xffffffffu, v);
        if (incl) break;
    }
    return excl;
}

// `open` (row bands): bit 0 / 1 = the first / last row is not the raster border but continues in another band; its
// cells are ordinary cells whose window is clipped to the band (a catchment never crosses a band edge).
// Descent pointers + most of the pointer jumping: a CTA holds a 64x64 tile of z (+ apron) in shared memory, finds
// every cell's pointer, numbers the tile's local minima, compresses the in-tile paths by pointer doubling, and writes
// for every cell what its tile-local root stands for: the catchment id of a local minimum, 0 (raster border =
// "outside"), or - when the root's lowest neighbour lies in another tile - -(1 + that neighbour's index).  Only cells
// of the last kind still need global pointer jumping (forest_resolve_ids); they are appended to `list` (catchments
// are ~50 cells, so that is a small fraction).  The tile index comes from a ticket (`ticket`, zeroed), not from
// blockIdx, so that every tile before it has started: the look-back waits for them.
// mm_keys (optional, {okey32 max, 0} on entry): K0's min / max keys of the raster, reduced from the z tile.
// TMA = true: the tile + apron comes in with ONE cp.async.bulk.tensor.2d issued by thread 0 - a 66 x 72 box starting at
// column c0 - 4 (the innermost box coordinate and width must be multiples of 16 bytes: measured with tools/tma_probe.cu,
// a start at c0 - 1 raises an illegal-instruction fault); cells outside the raster arrive as NaN, which no comparison
// below selects - the same effect as the +inf the LDG -> STS form stores for them.
constexpr int DT_LD_TMA = FT + 8, DT_X0_TMA = 4;
template <bool TMA>
__global__ void __launch_bounds__(256) k_descent_tile(const float *__restrict__ z, int *__restrict__ lab, int rows,
                                                      int cols, int tiles_x, int open, int *list, int *n_list,
                                                      unsigned long long *status, int *ticket, uint32_t *mm_keys,
                                                      const __grid_constant__ CUtensorMap zmap) {
    constexpr int LD = TMA ? DT_LD_TMA : FT + 2;
    constexpr int X0 = TMA ? DT_X0_TMA : 1;          // shared column of the tile's first cell
    __shared__ __align__(128) float sz[(FT + 2) * LD];
    __shared__ unsigned short sp[FT * FT];
    __shared__ int tgt[FT * FT];          // per tile-local root: > 0 catchment rank in the tile, 0 outside, < 0: -(1 + cell in another tile)
    __shared__ uint64_t bar;
    __shared__ int tile_s, base_s, wcnt[8];
    __shared__ uint32_t wlo[8], whi[8];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) {
        tile_s = atomicAdd(ticket, 1);
        if (TMA) mbar_init(&bar, 1);
    }
    __syncthreads();
    const int tile = tile_s;
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int r0 = ty * FT, c0 = tx * FT;
    if (TMA) {
        if (tid == 0) {
            mbar_expect_tx(&bar, (unsigned)sizeof(sz));
            tma_load_2d(sz, &zmap, &bar, c0 - DT_X0_TMA, r0 - 1);
        }
        mbar_wait(&bar, 0);
    } else {
        for (int k = tid; k < (FT + 2) * (FT + 2); k += 256) {
            int lr = k / (FT + 2), lc = k - lr * (FT + 2);
            int r = r0 + lr - 1, c = c0 + lc - 1;
            sz[k] = (r >= 0 && r < rows && c >= 0 && c < cols) ? z[(size_t)r * cols + c] : INFINITY;
        }
        __syncthreads();
    }
    unsigned minbits = 0;                 // which of this thread's cells are local minima
    uint32_t klo = 0xffffffffu, khi = 0u;
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        unsigned short p = (unsigned short)k;
        int t = 0;
        if (r < rows && c < cols) {
            int i = r * cols + c;
            float bz = sz[(lr + 1) * LD + lc + X0];
            uint32_t key = okey32(bz);
            klo = min(klo, key);
            khi = max(khi, key);
            if ((r == 0 && !(open & 1)) || c == 0 || (r == rows - 1 && !(open & 2)) || c == cols - 1) {
                t = 0;                                   // raster border: "outside"
            } else {
                int bi = i, bdr = 0, bdc = 0;
#pragma unroll
                for (int dr = -1; dr <= 1; dr++)
#pragma unroll
                    for (int dc = -1; dc <= 1; dc++) {
                        if (dr == 0 && dc == 0) continue;
                        if (r + dr < 0 || r + dr >= rows) continue;
                        int j = i + dr * cols + dc;
                        float zj = sz[(lr + 1 + dr) * LD + lc + X0 + dc];
                        if (zj < bz || (zj == bz && j < bi)) { bz = zj; bi = j; bdr = dr; bdc = dc; }
                    }
                int tr = lr + bdr, tc = lc + bdc;
                if (bi == i) minbits |= 1u << u;                              // local minimum (ranked below)
                else if (tr >= 0 && tr < FT && tc >= 0 && tc < FT) p = (unsigned short)(tr * FT + tc);
                else t = -(1 + bi);                                           // lowest neighbour is in another tile
            }
        }
        sp[k] = p;
        tgt[k] = t;
    }
    // rank of the tile's local minima: (warp, lane, cell) order
    const int cnt = __popc(minbits);
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (mm_keys) {
        klo = __reduce_min_sync(0xffffffffu, klo);
        khi = __reduce_max_sync(0xffffffffu, khi);
        if (lane == 0) { wlo[w] = klo; whi[w] = khi; }
    }
    if (lane == 31) wcnt[w] = inc;
    __syncthreads();
    int rank = inc - cnt, total = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        rank += k < w ? wcnt[k] : 0;
        total += wcnt[k];
    }
    if (tid == 0) {
        st_release_u64(status + tile, (tile ? TS_AGG : TS_INCL) | (unsigned)total);
        if (mm_keys) {
            uint32_t lo = wlo[0], hi = whi[0];
            for (int k = 1; k < 8; k++) { lo = min(lo, wlo[k]); hi = max(hi, whi[k]); }
            // a stale (larger / smaller) value only costs an atomic that changes nothing
            if (lo < mm_keys[0]) atomicMin(&mm_keys[0], lo);
            if (hi > mm_keys[1]) atomicMax(&mm_keys[1], hi);
        }
    }
    for (unsigned b = minbits; b; b &= b - 1) tgt[tid + 256 * (__ffs(b) - 1)] = ++rank;
    tile_pointer_double(sp);
    if (w == 0) {
        int excl = tile_lookback(status, tile);
        if (tid == 0) {
            base_s = excl;
            if (tile) st_release_u64(status + tile, TS_INCL | (unsigned)(excl + total));
        }
    }
    __syncthreads();
    const int base = base_s;
    int mine[16], nl = 0;
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        mine[u] = -1;
        if (r < rows && c < cols) {
            int t = tgt[sp[k]];
            int i = r * cols + c;
            if (t > 0) t += base;
            else if (t < 0) { mine[u] = i; nl++; }
            lab[i] = t;
        }
    }
    int pos = block_append_pos(nl, n_list);
#pragma unroll 4
    for (int u = 0; u < 16; u++)
        if (mine[u] >= 0) list[pos++] = mine[u];
}

__global__ void __launch_bounds__(256) k_boruvka_init(int *comp, uint32_t *E, int nC) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < nC) {
        comp[l] = l;
        E[l] = okey32(-INFINITY);
    }
}

// Row-band fill: lowest outgoing edge of every component that has not reached "outside" (component 0) yet.
// An edge into a halo row (the neighbouring band) is "foreign": its key carries FOREIGN_BIT, which also
// sorts it behind every local edge of the same weight; a component whose lowest edge is foreign freezes (k_hook).
constexpr unsigned FOREIGN_BIT = 0x80000000u;

constexpr int ME_PER_THREAD = 4;      // cells per thread: one list append (atomic) per 1024 cells

// FIRST: round 1, where every catchment is its own component (comp[l] == l) and nothing is frozen yet — the component
// lookups (a gather per neighbour across a catchment boundary) are skipped.
// r: the cell's row, or for a cell given by its index alone (the list rounds) 0 / 1 / rows - 1 for first / any other /
// last row - only "does the neighbour row exist" is asked; c < 0: the column is worked out if a foreign edge needs it
template <bool FIRST>
__device__ inline bool minedge_cell(const float *__restrict__ z, const int *__restrict__ lab,
                                    const int *__restrict__ comp, const uint8_t *__restrict__ frozen,
                                    unsigned long long *best, int rows, int cols, int i, int r, int c) {
    int l = lab[i];
    int cc = FIRST ? l : (l ? comp[l] : 0);
    if (cc == 0) return false;
    // a cell of a FROZEN component no longer searches, but stays listed while a neighbour lies in another component -
    // the boundary graph of the frozen components is built from the last list (k_band_edges)
    const bool fz = !FIRST && frozen[cc];
    bool other = false;
    float zc = z[i];
    unsigned long long bk = KEY_NONE;
    // interior cell (label != 0 implies not on the border): all 8 neighbours are in the raster, or in a halo row
#pragma unroll
    for (int dr = -1; dr <= 1; dr++)
#pragma unroll
        for (int dc = -1; dc <= 1; dc++) {
            if (dr == 0 && dc == 0) continue;
            int j = i + dr * cols + dc;
            if (r + dr < 0 || r + dr >= rows) {
                if (fz) { other = true; continue; }
                float w = fmaxf(zc, __ldg(z + j));
                if (c < 0) c = i % cols;
                unsigned long long key = ((unsigned long long)okey32(w) << 32) | FOREIGN_BIT | (unsigned)c;
                bk = key < bk ? key : bk;
                continue;
            }
            int lj = __ldg(lab + j);
            if (lj == l) continue;
            if (!FIRST && __ldg(comp + lj) == cc) continue;
            if (fz) { other = true; continue; }
            float w = fmaxf(zc, __ldg(z + j));
            // symmetric edge id: lower cell index and the direction to the higher one (E, SW, S, SE)
            int lo = j < i ? j : i;
            int code = (dr == 0) ? 0 : ((dr * dc == -1) ? 1 : (dc == 0 ? 2 : 3));
            unsigned long long key = ((unsigned long long)okey32(w) << 32) | (unsigned)(((unsigned)lo << 2) | code);
            bk = key < bk ? key : bk;
        }
    if (fz) return other;
    if (bk == KEY_NONE) return false;
    if (bk < best[cc]) atomicMin(&best[cc], bk);
    return true;
}

// LIST = false: a CTA covers 16 rows x 64 columns of the raster (round 1).  LIST = true: 1024 entries of list_in.
// Either way the cells that still have a neighbour in another component are appended to list_out: a cell inside its
// component never has an outgoing edge again, and components grow every round, so the later rounds touch ever
// fewer cells.
// append the survivors: block-wide exclusive scan of the per-thread counts, one atomic per CTA
__device__ __forceinline__ void minedge_append(unsigned keepbits, const int (&cell)[ME_PER_THREAD], int *list_out, int *n_out) {
    __shared__ int wsum[8];
    __shared__ int base_s;
    int cnt = __popc(keepbits), lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int k = 0; k < 8; k++) { int t = wsum[k]; wsum[k] = tot; tot += t; }
        base_s = tot ? atomicAdd(n_out, tot) : 0;
    }
    __syncthreads();
    int pos = base_s + wsum[w] + inc - cnt;
#pragma unroll
    for (int u = 0; u < ME_PER_THREAD; u++)
        if (keepbits & (1u << u)) list_out[pos++] = cell[u];
}

template <bool LIST>
__global__ void __launch_bounds__(256) k_minedge_band(const float *__restrict__ z, const int *__restrict__ lab,
                                                      const int *__restrict__ comp, const uint8_t *__restrict__ frozen,
                                                      unsigned long long *best, int rows, int cols,
                                                      const int *__restrict__ list_in, int n_in, int *list_out, int *n_out) {
    int cell[ME_PER_THREAD];
    unsigned keepbits = 0;
#pragma unroll
    for (int u = 0; u < ME_PER_THREAD; u++) {
        int i = -1, r = 0, c = 0;
        if (LIST) {
            int k = (blockIdx.x * ME_PER_THREAD + u) * 256 + threadIdx.x;
            if (k < n_in) {
                i = list_in[k];
                // no division per entry: only the first and the last row have a neighbour row missing
                r = i < cols ? 0 : (i >= (rows - 1) * cols ? rows - 1 : 1);
                c = -1;
            }
        } else {
            c = blockIdx.x * 64 + (threadIdx.x & 63);
            r = (blockIdx.y * ME_PER_THREAD + u) * 4 + (threadIdx.x >> 6);
            if (r < rows && c < cols) i = r * cols + c;
        }
        cell[u] = i;
        if (i >= 0 && minedge_cell<!LIST>(z, lab, comp, frozen, best, rows, cols, i, r, c)) keepbits |= 1u << u;
    }
    minedge_append(keepbits, cell, list_out, n_out);
}

__device__ inline int edge_other(int lo, int code, int cols) {
    return lo + (code == 0 ? 1 : (code == 1 ? cols - 1 : (code == 2 ? cols : cols + 1)));
}

// every live component hooks to the component across its lowest edge; mutual pairs keep the smaller id
__global__ void __launch_bounds__(256) k_hook(const unsigned long long *__restrict__ best,
                                              const int *__restrict__ comp, const int *__restrict__ lab,
                                              int *parent, uint32_t *wk, uint8_t *frozen, int nC, int cols) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nC) return;
    parent[k] = k;
    wk[k] = okey32(-INFINITY);
    if (k == 0 || comp[k] != k) return;
    unsigned long long b = best[k];
    if (b == KEY_NONE) return;
    unsigned id = (unsigned)(b & 0xffffffffu);
    if (frozen && (id & FOREIGN_BIT)) {
        // lowest way out leads into another band: the component waits for the boundary graph (fill_band_*)
        frozen[k] = 1;
        return;
    }
    int lo = (int)(id >> 2), code = (int)(id & 3u);
    int hi = edge_other(lo, code, cols);
    int ca = comp[lab[lo]], cb = comp[lab[hi]];
    int t = (ca == k) ? cb : ca;
    wk[k] = (uint32_t)(b >> 32);
    if (t != 0 && best[t] == b && k < t) t = k;
    parent[k] = t;
}

__device__ inline int uf_find(int *parent, int k) {
    int p = parent[k];
    for (;;) {
        int g = parent[p];
        if (g == p) return p;
        parent[k] = g;
        k = p;
        p = g;
    }
}

// E = max(E, weight of the edge the catchment's component left through); component := merged root
__global__ void __launch_bounds__(256) k_boruvka_update(int *comp, uint32_t *E, int *parent,
                                                        const uint32_t *__restrict__ wk,
                                                        const uint8_t *__restrict__ frozen, int nC,
                                                        unsigned long long *best, int *remaining) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    int live = 0;
    if (l < nC) {
        best[l] = KEY_NONE;
        int k = comp[l];
        if (k != 0) {
            uint32_t e = E[l], w = wk[k];
            if (w > e) E[l] = w;
            int r = uf_find(parent, k);
            comp[l] = r;
            live = (r == l) && !(frozen && frozen[r]);      // still searching: neither at 0 nor frozen
        }
    }
    int cnt = __syncthreads_count(live);
    if (threadIdx.x == 0 && cnt) atomicAdd(remaining, cnt);
}

__global__ void __launch_bounds__(256) k_fill_final(const float *__restrict__ z, const int *__restrict__ lab,
                                                    const uint32_t *__restrict__ E, float *__restrict__ filled,
                                                    float *__restrict__ depths, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float zc = z[i];
    float w = fmaxf(zc, okey32_inv(__ldg(E + lab[i])));
    filled[i] = w;
    if (depths) depths[i] = __fsub_rn(w, zc);
}

// every cell -> the id of the catchment it drains to (0 = outside), tile-local compression, then pointer jumping over
// the cells whose path leaves their tile.  `scratch` (n ints) holds that list.  *nC: catchments + 1 (for "outside").
static int descent_resolve(const float *dem, int *lab, int *scratch, int64_t rows, int64_t cols, int open,
                           uint32_t *mm_keys, int *nC, int64_t *rounds_out, cudaStream_t s) {
    int tiles_x = (int)cdiv(cols, FT), tiles = tiles_x * (int)cdiv(rows, FT);
    // the tiles' status words, then {ticket, list length}
    DevBuf<unsigned long long> st;
    MS_TRY(st.alloc((size_t)tiles + 1, s));
    MS_CUDA(cudaMemsetAsync(st.p, 0, ((size_t)tiles + 1) * sizeof(unsigned long long), s));
    int *ctl = (int *)(st.p + tiles);
    prof_units(rows * cols);
    CUtensorMap zmap;
    memset(&zmap, 0, sizeof(zmap));
    // (a band's rows sit inside a raster with halo rows: it keeps the LDG -> STS form)
    if (!open && tma_map_2d(&zmap, dem, rows, cols, FT + 2, DT_LD_TMA, true, true))
        MS_LAUNCH(k_descent_tile<true>, tiles, 256, 0, s, dem, lab, (int)rows, (int)cols, tiles_x, open, scratch, ctl + 1,
                  st.p, ctl, mm_keys, zmap);
    else
        MS_LAUNCH(k_descent_tile<false>, tiles, 256, 0, s, dem, lab, (int)rows, (int)cols, tiles_x, open, scratch, ctl + 1,
                  st.p, ctl, mm_keys, zmap);
    int64_t *h = host_flags().h;
    MS_TRY(ms::readback(h, st.p + tiles - 1, 2 * sizeof(unsigned long long), s));
    MS_TRY(ms::stream_sync(s));
    *nC = 1 + (int)(unsigned)h[0];
    return forest_resolve_ids(lab, scratch, ((int *)(h + 1))[1], rounds_out, s);
}

// The Boruvka rounds of the row-band fill, on the band's cells.  comp / E initialised by k_boruvka_init, `frozen`
// zeroed.  The last work list goes to B (BB_BLIST) for the boundary graph.
static int boruvka_rounds_band(const float *dem, const int *lab, int *comp, uint32_t *E, uint8_t *frozen, int nC,
                               int64_t rows, int64_t cols, cudaStream_t s, ms_band *B) {
    int64_t n = rows * cols;
    DevBuf<int> parent, counters, listA, listB;
    DevBuf<uint32_t> wk;
    DevBuf<unsigned long long> best;
    MS_TRY(parent.alloc(nC, s));
    MS_TRY(wk.alloc(nC, s));
    MS_TRY(best.alloc(nC, s));
    MS_TRY(counters.alloc(2, s));
    MS_TRY(listA.alloc((size_t)n, s));
    unsigned gc = cdiv(nC, 256);
    int64_t *h = host_flags().h;
    MS_CUDA(cudaMemsetAsync(best.p, 0xff, (size_t)nC * sizeof(unsigned long long), s));
    int rounds = 0;
    int64_t live = nC - 1;       // live components; each round every one of them merges with another (or freezes)
    int n_list = 0;
    int *lin = nullptr, *lout = listA.p;
    while (live > 0) {
        MS_CUDA(cudaMemsetAsync(counters.p, 0, 2 * sizeof(int), s));
        if (rounds == 0) {
            prof_units(n);
            dim3 g2m(cdiv(cols, 64), cdiv(rows, 4 * ME_PER_THREAD));
            MS_LAUNCH(k_minedge_band<false>, g2m, 256, 0, s, dem, lab, (const int *)comp, (const uint8_t *)frozen, best.p,
                      (int)rows, (int)cols, (const int *)nullptr, 0, lout, counters.p + 1);
        } else {
            prof_units(n_list);
            MS_LAUNCH(k_minedge_band<true>, cdiv(n_list, 256 * ME_PER_THREAD), 256, 0, s, dem, lab, (const int *)comp,
                      (const uint8_t *)frozen, best.p, (int)rows, (int)cols, (const int *)lin, n_list, lout, counters.p + 1);
        }
        MS_LAUNCH(k_hook, gc, 256, 0, s, best.p, comp, lab, parent.p, wk.p, frozen, nC, (int)cols);
        MS_LAUNCH(k_boruvka_update, gc, 256, 0, s, comp, E, parent.p, wk.p, (const uint8_t *)frozen, nC, best.p,
                  counters.p);
        MS_TRY(ms::readback(h, counters.p, 2 * sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        int64_t now = ((int *)h)[0];
        n_list = ((int *)h)[1];
        rounds++;
        if (now >= live || rounds > 64) {
            set_error("band fill: Boruvka contraction stalled (%lld -> %lld live components, round %d)",
                      (long long)live, (long long)now, rounds);
            return MS_ERR_NOCONV;
        }
        live = now;
        if (live > 0 && n_list == 0) {
            set_error("band fill: live components without an outgoing edge");
            return MS_ERR_NOCONV;
        }
        // the survivors of this round are the next round's work; the second list is sized by the first's count
        if (rounds == 1 && live > 0) MS_TRY(listB.alloc((size_t)n_list, s));
        lin = lout;
        lout = (lout == listA.p) ? listB.p : listA.p;
    }
    // the last list: every cell that had a neighbour in another component in the last round (components only
    // merge, so it is a superset of the cells on the borders between the frozen components)
    B->n_blist = 0;
    if (rounds > 0 && n_list > 0) {
        int *dst = (int *)band_buf(B, BB_BLIST, (size_t)n_list * sizeof(int));
        if (!dst) return MS_ERR_CUDA;
        MS_CUDA(cudaMemcpyAsync(dst, lin, (size_t)n_list * sizeof(int), cudaMemcpyDeviceToDevice, s));
        MS_TRY(ms::stream_sync(s));      // the list buffers go back to the arena when this function returns
        B->n_blist = n_list;
    }
    return MS_OK;
}

// ---- single GPU: Boruvka on an explicit catchment edge list -------------------------------------------------------
// The tile pass collects, per 64x64 tile, the lowest cell-pair edge between every pair of
// catchments that touch inside it (or across its right / lower edge); later rounds work on that list only.  At
// 32768^2 (fractal DEM) it holds 68.8 M entries for 20.3 M catchments, where the cell-list rounds visited ~650 M
// boundary cells in round 2 alone; the list and the vertex arrays shrink every round (DESIGN.md §K1).
constexpr int TE_SLOTS = 512;        // shared hash slots per tile: a tile of a DEM holds ~80 catchments, white noise ~450
constexpr int TE_PROBES = 32;        // a candidate that finds no slot within this many goes straight to the global list

// list entry `pos` = edge (a < b, ordered weight w); Boruvka's key of the entry for both endpoints is (w, pos), a strict
// total order over the list, so the same pair listed by two tiles cannot form a hook cycle.  Vertex 0 ("outside")
// does not search.
__device__ __forceinline__ void edge_put(int *ea, int *eb, uint32_t *ew, unsigned long long *best, int pos, int a, int b,
                                         uint32_t w) {
    ea[pos] = a;
    eb[pos] = b;
    ew[pos] = w;
    unsigned long long key = ((unsigned long long)w << 32) | (unsigned)pos;
    if (a && key < best[a]) atomicMin(&best[a], key);
    if (key < best[b]) atomicMin(&best[b], key);
}

__device__ __forceinline__ void tile_edge_insert(unsigned long long *hk, uint32_t *hw, int a, int b, uint32_t w,
                                                 int *ea, int *eb, uint32_t *ew, int cap, int *n_edges,
                                                 unsigned long long *best) {
    unsigned long long key = ((unsigned long long)(unsigned)a << 32) | (unsigned)b;
    unsigned h = (unsigned)((key * 0x9E3779B97F4A7C15ull) >> 32) & (TE_SLOTS - 1);
    for (int p = 0; p < TE_PROBES; p++) {
        unsigned long long cur = hk[h];
        if (cur == HASH_EMPTY) {
            unsigned long long old = atomicCAS(hk + h, HASH_EMPTY, key);
            cur = (old == HASH_EMPTY) ? key : old;
        }
        if (cur == key) {
            atomicMin(hw + h, w);
            return;
        }
        h = (h + 1) & (TE_SLOTS - 1);
    }
    int pos = atomicAdd(n_edges, 1);      // table full: unaggregated (counted even past the capacity)
    if (pos < cap) edge_put(ea, eb, ew, best, pos, a, b, w);
}

// One CTA per 64x64 tile (the tiling of k_descent_tile, and its TMA box of z): every cell pair is looked at from its
// lower cell (directions E, SW, S, SE); a pair of different catchments a < b is an edge of weight max(z_i, z_j) (a = 0:
// an edge to "outside"), aggregated per pair in shared memory (minimum weight), then appended to the list with one
// atomic per CTA, which also does round 1's lowest-edge search.  Past `cap` the entries are counted but not written
// (the caller re-runs the pass with the counted size).
// TMA = true: the catchment ids of rows r0 .. r0 + 64, columns c0 - 1 .. c0 + 64 come in as a second box (65 x 72 from
// column c0 - 4, like z's), cells outside the raster as 0; no pair with such a cell is looked at.
template <bool TMA>
__global__ void __launch_bounds__(256) k_tile_edges(const float *__restrict__ z, const int *__restrict__ lab, int rows,
                                                    int cols, int tiles_x, int *ea, int *eb, uint32_t *ew, int cap,
                                                    int *n_edges, unsigned long long *best,
                                                    const __grid_constant__ CUtensorMap zmap,
                                                    const __grid_constant__ CUtensorMap lmap) {
    constexpr int LD = TMA ? DT_LD_TMA : FT + 2;
    constexpr int X0 = TMA ? DT_X0_TMA : 1;
    __shared__ __align__(128) float sz[(FT + 2) * LD];
    __shared__ __align__(128) int sl[(FT + 1) * LD];
    __shared__ unsigned long long hk[TE_SLOTS];
    __shared__ uint32_t hw[TE_SLOTS];
    __shared__ uint64_t bar;
    int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    int r0 = ty * FT, c0 = tx * FT, tid = threadIdx.x;
    if (TMA) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            mbar_expect_tx(&bar, (unsigned)(sizeof(sz) + sizeof(sl)));
            tma_load_2d(sz, &zmap, &bar, c0 - DT_X0_TMA, r0 - 1);
            tma_load_2d(sl, &lmap, &bar, c0 - DT_X0_TMA, r0);
        }
    } else {
        for (int k = tid; k < (FT + 2) * (FT + 2); k += 256) {
            int lr = k / (FT + 2), lc = k - lr * (FT + 2);
            int r = r0 + lr - 1, c = c0 + lc - 1;
            sz[k] = (r >= 0 && r < rows && c >= 0 && c < cols) ? z[(size_t)r * cols + c] : INFINITY;
        }
        for (int k = tid; k < (FT + 1) * (FT + 2); k += 256) {
            int lr = k / (FT + 2), lc = k - lr * (FT + 2);
            int r = r0 + lr, c = c0 + lc - 1;
            sl[k] = (r < rows && c >= 0 && c < cols) ? lab[(size_t)r * cols + c] : 0;
        }
    }
    for (int k = tid; k < TE_SLOTS; k += 256) { hk[k] = HASH_EMPTY; hw[k] = 0xffffffffu; }
    __syncthreads();
    if (TMA) mbar_wait(&bar, 0);
    // a thread walks 16 cells down one column: the pairs of a catchment border repeat along it, so consecutive
    // candidates of the same pair are merged in registers before they reach the table
    const int lc = tid & 63, lr0 = (tid >> 6) * 16, c = c0 + lc;
    int pa = -1, pb = -1;
    uint32_t pw = 0;
    if (c < cols) {
        for (int u = 0; u < 16; u++) {
            const int lr = lr0 + u, r = r0 + lr;
            if (r >= rows) break;
            const int l = sl[lr * LD + lc + X0];
            const float zc = sz[(lr + 1) * LD + lc + X0];
#pragma unroll
            for (int d = 0; d < 4; d++) {
                const int dr = d == 0 ? 0 : 1, dc = d == 0 ? 1 : d - 2;
                if (r + dr >= rows || c + dc < 0 || c + dc >= cols) continue;
                const int m = sl[(lr + dr) * LD + lc + X0 + dc];
                if (m == l) continue;
                const uint32_t w = okey32(fmaxf(zc, sz[(lr + 1 + dr) * LD + lc + X0 + dc]));
                const int a = min(l, m), b = max(l, m);
                if (a == pa && b == pb) { pw = min(pw, w); continue; }
                if (pa >= 0) tile_edge_insert(hk, hw, pa, pb, pw, ea, eb, ew, cap, n_edges, best);
                pa = a; pb = b; pw = w;
            }
        }
    }
    if (pa >= 0) tile_edge_insert(hk, hw, pa, pb, pw, ea, eb, ew, cap, n_edges, best);
    __syncthreads();
    int cnt = 0;
#pragma unroll
    for (int k = tid; k < TE_SLOTS; k += 256) cnt += hk[k] != HASH_EMPTY;
    int pos = block_append_pos(cnt, n_edges);
#pragma unroll
    for (int k = tid; k < TE_SLOTS; k += 256) {
        unsigned long long key = hk[k];
        if (key == HASH_EMPTY) continue;
        if (pos < cap) edge_put(ea, eb, ew, best, pos, (int)(key >> 32), (int)(key & 0xffffffffu), hw[k]);
        pos++;
    }
}

// every live vertex v != 0 hooks across its lowest edge (mutual pairs keep the smaller id); wk = that edge's weight,
// flag = 1 for the roots of the new components that have not reached outside
__global__ void __launch_bounds__(256) k_hook_edges(const unsigned long long *__restrict__ best,
                                                    const int *__restrict__ ea, const int *__restrict__ eb,
                                                    int *parent, uint32_t *wk, int *flag, int V) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    int p = v;
    uint32_t w = okey32(-INFINITY);
    unsigned long long b = v ? best[v] : KEY_NONE;
    if (b != KEY_NONE) {
        unsigned e = (unsigned)(b & 0xffffffffu);
        int x = ea[e], y = eb[e];
        int t = (x == v) ? y : x;
        w = (uint32_t)(b >> 32);
        if (t != 0 && best[t] == b && v < t) t = v;
        p = t;
    }
    parent[v] = p;
    wk[v] = w;
    flag[v] = (v != 0 && p == v) ? 1 : 0;
}

// the next level's id of v's component (0 = outside); nid = exclusive scan of the live-root flags.  The root is
// looked up, not stored over parent: another thread's path halving may still overwrite parent[v] with an ancestor.
__global__ void __launch_bounds__(256) k_level_map(int *parent, const int *__restrict__ nid, int *map, int V) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    int r = uf_find(parent, v);
    map[v] = r ? nid[r] + 1 : 0;
}

// endpoints -> next level's ids; an edge inside one component (or between two that reached outside) goes; the rest
// is compacted and searched for the next round's lowest edges
__global__ void __launch_bounds__(256) k_edges_relabel(const int *__restrict__ ia, const int *__restrict__ ib,
                                                       const uint32_t *__restrict__ iw, int m,
                                                       const int *__restrict__ map, int *oa, int *ob, uint32_t *ow,
                                                       int *n_out, unsigned long long *best) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    int a = 0, b = 0;
    uint32_t w = 0;
    if (e < m) {
        a = __ldg(map + ia[e]);
        b = __ldg(map + ib[e]);
        w = iw[e];
        if (a > b) { int t = a; a = b; b = t; }
    }
    int keep = a != b;
    int pos = block_append_pos(keep, n_out);
    if (keep) edge_put(oa, ob, ow, best, pos, a, b, w);
}

// spill elevations, top level down: X_t[v] = max(wk_t[v], X_{t+1}[map_t(v)]) unless map_t(v) = 0 (written over wk_t)
__global__ void __launch_bounds__(256) k_spill_down(uint32_t *wk, const int *__restrict__ map,
                                                    const uint32_t *__restrict__ x_up, int V) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    int u = map[v];
    if (u) {
        uint32_t x = x_up[u];
        if (x > wk[v]) wk[v] = x;
    }
}

int fill_terrain_dev_impl(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols,
                          int64_t *stats, cudaStream_t s, float *minmax_out) {
    if (!dtm || !filled) { set_error("fill_terrain: null pointer"); return MS_ERR_ARG; }
    if (rows < 3 || cols < 3 || rows * cols > (1ll << 30)) {
        set_error("fill_terrain: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    int64_t n = rows * cols;
    DevBuf<int64_t> ctr;
    DevBuf<uint32_t> mm_keys;
    DevBuf<int> lab, list;
    MS_TRY(ctr.alloc(2, s));
    if (minmax_out) {
        MS_TRY(mm_keys.alloc(2, s));
        MS_CUDA(cudaMemsetAsync(mm_keys.p, 0xff, sizeof(uint32_t), s));
        MS_CUDA(cudaMemsetAsync(mm_keys.p + 1, 0, sizeof(uint32_t), s));
    }
    MS_TRY(lab.alloc((size_t)n, s));
    MS_TRY(list.alloc((size_t)n, s));
    int64_t *h = host_flags().h;

    int64_t jump_rounds = 0;
    int nC = 0;
    MS_TRY(descent_resolve(dtm, lab.p, list.p, rows, cols, 0, mm_keys.p, &nC, &jump_rounds, s));
    list.release();
    if (minmax_out) MS_LAUNCH(k_minmax_finish, 1, 1, 0, s, mm_keys.p, minmax_out);

    // per vertex: the lowest edge and the parent / flags of the current level; wk and map of every level (the live
    // vertices at least halve per round, so all levels together hold < 2 nC + rounds)
    const int64_t lv_cap = 2 * (int64_t)nC + 64;
    DevBuf<unsigned long long> best;
    DevBuf<int> parent, nid, map_all;
    DevBuf<uint32_t> wk_all;
    MS_TRY(best.alloc(nC, s));
    MS_TRY(parent.alloc(nC, s));
    MS_TRY(nid.alloc(nC, s));
    MS_TRY(map_all.alloc((size_t)lv_cap, s));
    MS_TRY(wk_all.alloc((size_t)lv_cap, s));

    // the edge list takes half of what the arena has left from earlier calls (the other half is for the compacted
    // copy); when that is too small the pass has counted every edge and runs once more with the counted size plus a
    // quarter (a tile whose table fills lists some pairs more than once, and how often depends on the timing)
    const int64_t cap_max = n * 4 < 0x7fffffffll ? n * 4 : 0x7fffffffll;
    int64_t cap = (int64_t)(arena_room() / (2 * (2 * sizeof(int) + sizeof(uint32_t))));
    if (cap < n / 16 + 4096) cap = n / 16 + 4096;
    if (cap > cap_max) cap = cap_max;
    DevBuf<int> ea[2], eb[2];
    DevBuf<uint32_t> ew[2];
    CUtensorMap zmap, lmap;
    memset(&zmap, 0, sizeof(zmap));
    memset(&lmap, 0, sizeof(lmap));
    const bool tma = tma_map_2d(&zmap, dtm, rows, cols, FT + 2, DT_LD_TMA, true, true) &&
                     tma_map_2d(&lmap, lab.p, rows, cols, FT + 1, DT_LD_TMA, false, false);
    const int tiles_x = (int)cdiv(cols, FT), tiles = tiles_x * (int)cdiv(rows, FT);
    int64_t m = 0;
    for (int attempt = 0;; attempt++) {
        MS_TRY(ea[0].alloc((size_t)cap, s));
        MS_TRY(eb[0].alloc((size_t)cap, s));
        MS_TRY(ew[0].alloc((size_t)cap, s));
        MS_CUDA(cudaMemsetAsync(best.p, 0xff, (size_t)nC * sizeof(unsigned long long), s));
        MS_CUDA(cudaMemsetAsync(ctr.p + 1, 0, sizeof(int64_t), s));
        prof_units(n);
        if (tma)
            MS_LAUNCH(k_tile_edges<true>, tiles, 256, 0, s, dtm, (const int *)lab.p, (int)rows, (int)cols, tiles_x, ea[0].p,
                      eb[0].p, ew[0].p, (int)cap, (int *)(ctr.p + 1), best.p, zmap, lmap);
        else
            MS_LAUNCH(k_tile_edges<false>, tiles, 256, 0, s, dtm, (const int *)lab.p, (int)rows, (int)cols, tiles_x, ea[0].p,
                      eb[0].p, ew[0].p, (int)cap, (int *)(ctr.p + 1), best.p, zmap, lmap);
        MS_TRY(ms::readback(h, ctr.p + 1, sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        m = (int64_t)(unsigned)((int *)h)[0];
        if (m <= cap) break;
        if (attempt > 0 || cap == cap_max) {
            set_error("fill_terrain: %lld catchment edges do not fit the list (%lld)", (long long)m, (long long)cap);
            return MS_ERR_NOCONV;
        }
        ew[0].release();
        eb[0].release();
        ea[0].release();
        cap = m + m / 4 < cap_max ? m + m / 4 : cap_max;
    }
    MS_TRY(ea[1].alloc((size_t)m, s));
    MS_TRY(eb[1].alloc((size_t)m, s));
    MS_TRY(ew[1].alloc((size_t)m, s));

    // Boruvka rounds on the list; level t has V vertices (0 = outside), its wk / map at lv_off[t]
    int64_t lv_off[66];
    int64_t V = nC, live = nC - 1;
    int rounds = 0, cur = 0;
    lv_off[0] = 0;
    if (live == 0) MS_LAUNCH(k_hook_edges, 1, 256, 0, s, best.p, ea[0].p, eb[0].p, parent.p, wk_all.p, nid.p, (int)V);
    while (live > 0) {
        uint32_t *wk = wk_all.p + lv_off[rounds];
        int *map = map_all.p + lv_off[rounds];
        unsigned gv = cdiv(V, 256);
        MS_LAUNCH(k_hook_edges, gv, 256, 0, s, best.p, ea[cur].p, eb[cur].p, parent.p, wk, nid.p, (int)V);
        MS_TRY(exclusive_scan_i32(nid.p, nid.p, V, ctr.p, s));
        MS_LAUNCH(k_level_map, gv, 256, 0, s, parent.p, nid.p, map, (int)V);
        MS_CUDA(cudaMemsetAsync(best.p, 0xff, (size_t)V * sizeof(unsigned long long), s));
        MS_CUDA(cudaMemsetAsync(ctr.p + 1, 0, sizeof(int64_t), s));
        prof_units(m);
        if (m > 0)
            MS_LAUNCH(k_edges_relabel, cdiv(m, 256), 256, 0, s, ea[cur].p, eb[cur].p, ew[cur].p, (int)m, map, ea[1 - cur].p,
                      eb[1 - cur].p, ew[1 - cur].p, (int *)(ctr.p + 1), best.p);
        MS_TRY(ms::readback(h, ctr.p, 2 * sizeof(int64_t), s));
        MS_TRY(ms::stream_sync(s));
        int64_t now = h[0];
        m = (int64_t)((int *)(h + 1))[0];
        rounds++;
        lv_off[rounds] = lv_off[rounds - 1] + V;
        if (now >= live || rounds > 64 || lv_off[rounds] + now + 1 > lv_cap) {
            set_error("fill_terrain: Boruvka contraction stalled (%lld -> %lld live components, round %d)",
                      (long long)live, (long long)now, rounds);
            return MS_ERR_NOCONV;
        }
        live = now;
        if (live > 0 && m == 0) {
            set_error("fill_terrain: live components without an outgoing edge");
            return MS_ERR_NOCONV;
        }
        V = live + 1;
        cur = 1 - cur;
    }
    // the last level's components all reached outside: X = wk there; E = X_0
    for (int t = rounds - 2; t >= 0; t--) {
        int64_t Vt = lv_off[t + 1] - lv_off[t];
        MS_LAUNCH(k_spill_down, cdiv(Vt, 256), 256, 0, s, wk_all.p + lv_off[t], (const int *)map_all.p + lv_off[t],
                  (const uint32_t *)wk_all.p + lv_off[t + 1], (int)Vt);
    }
    MS_LAUNCH(k_fill_final, cdiv(n, 256), 256, 0, s, dtm, lab.p, wk_all.p, filled, depths, n);
    if (stats) { stats[0] = rounds; stats[1] = nC; stats[5] = jump_rounds; }
    return MS_OK;
}


// =====================================================================================================
// Row-band fill (SURVEY.md §8(e), K1).  The band runs the same Boruvka contraction on its own rows; a component
// whose lowest outgoing edge leads into a neighbouring band cannot decide locally and freezes (every hook made
// before that is a hook the global algorithm makes too, because a component that hooks knows all its edges).
// What is left is a small graph: frozen components of all bands + "outside", joined by the lowest cell-pair edge
// between each pair (inside a band and across band edges).  By the same claim as in the single-GPU case the spill
// elevation of a catchment is max(E collected so far, minimax height from its frozen component to "outside" in
// that graph).  Phases: fill_band_local -> (all-gather of counts) -> fill_band_edge_ids -> (halo exchange of ids)
// -> fill_band_edges -> (all-gather of edge lists) -> graph_minimax (every rank, same result) -> fill_band_finish.
// =====================================================================================================
__global__ void __launch_bounds__(256) k_frozen_flags(const int *comp, const uint8_t *frozen, int *flag, int nC) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nC) flag[k] = (k != 0 && comp[k] == k && frozen[k]) ? 1 : 0;
}

__device__ inline int band_gid(int K, const int *frank, int base) { return K ? 1 + base + frank[K] : 0; }

__global__ void __launch_bounds__(256) k_band_edge_ids(const int *__restrict__ lab, const int *__restrict__ comp,
                                                       const int *__restrict__ frank, int base, int rows, int cols,
                                                       int32_t *top, int32_t *bot) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    top[c] = band_gid(comp[lab[c]], frank, base);
    bot[c] = band_gid(comp[lab[(size_t)(rows - 1) * cols + c]], frank, base);
}

__device__ inline void edge_insert(unsigned long long *hk, uint32_t *hv, unsigned H, int ga, int gb, uint32_t w,
                                   int *overflow) {
    int a = ga < gb ? ga : gb, b = ga < gb ? gb : ga;
    unsigned long long key = ((unsigned long long)(unsigned)a << 32) | (unsigned)b;
    unsigned long long x = key * 0x9E3779B97F4A7C15ull;
    unsigned h = (unsigned)(x >> 32) & (H - 1);
    for (unsigned probes = 0; probes < H; probes++) {
        unsigned long long cur = hk[h];
        if (cur == HASH_EMPTY) {
            unsigned long long old = atomicCAS(hk + h, HASH_EMPTY, key);
            cur = (old == HASH_EMPTY) ? key : old;
        }
        if (cur == key) {
            if (w < hv[h]) atomicMin(hv + h, w);
            return;
        }
        h = (h + 1) & (H - 1);
    }
    *overflow = 1;
}

// lowest cell-pair edge between every frozen component of the band and each different neighbour (another frozen
// component, "outside" incl. the components that reached it, or a component of the neighbouring band)
__global__ void __launch_bounds__(256) k_band_edges(const float *__restrict__ z, const int *__restrict__ lab,
                                                    const int *__restrict__ comp, const int *__restrict__ frank,
                                                    int base, const int32_t *__restrict__ halo_top,
                                                    const int32_t *__restrict__ halo_bot, int rows, int cols,
                                                    unsigned long long *hk, uint32_t *hv, unsigned H, int *overflow,
                                                    const int *__restrict__ list, int n_list) {
    // over the last list of the Boruvka rounds (round 2; a pass over the whole band before: 4.7 of 37 ms of the fill
    // of a 16384 x 32768 band, spent on a label read and a component gather per cell to find the few frozen ones)
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_list) return;
    int i = list[k];
    int r = i / cols, c = i - r * cols;
    int l = lab[i];
    if (l == 0) return;
    int K = comp[l];
    if (K == 0) return;
    int ga = band_gid(K, frank, base);
    float zc = z[i];
    int last_gb = -1;
    uint32_t last_w = 0;
#pragma unroll
    for (int dr = -1; dr <= 1; dr++)
#pragma unroll
        for (int dc = -1; dc <= 1; dc++) {
            if (dr == 0 && dc == 0) continue;
            int j = i + dr * cols + dc;
            int gb;
            if (r + dr < 0) gb = halo_top[c + dc];
            else if (r + dr >= rows) gb = halo_bot[c + dc];
            else {
                int lj = __ldg(lab + j);
                if (lj == l) continue;
                int Kj = lj ? __ldg(comp + lj) : 0;
                if (Kj == K) continue;
                gb = band_gid(Kj, frank, base);
            }
            uint32_t w = okey32(fmaxf(zc, __ldg(z + j)));
            if (gb == last_gb && w >= last_w) continue;      // same neighbour component again, no better
            last_gb = gb;
            last_w = w;
            edge_insert(hk, hv, H, ga, gb, w, overflow);
        }
}

__global__ void __launch_bounds__(256) k_band_edges_compact(const unsigned long long *hk, const uint32_t *hv,
                                                            unsigned H, int32_t *ea, int32_t *eb, float *ew,
                                                            int64_t cap, int *count) {
    unsigned h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= H) return;
    unsigned long long key = hk[h];
    if (key == HASH_EMPTY) return;
    int k = atomicAdd(count, 1);
    if (k < cap) {
        ea[k] = (int32_t)(key >> 32);
        eb[k] = (int32_t)(key & 0xffffffffu);
        ew[k] = okey32_inv(hv[h]);
    }
}

// minimax height to node 0 on a small undirected graph: Bellman-Ford with (max, min), one CTA
__global__ void __launch_bounds__(1024) k_graph_minimax(int nn, const int32_t *__restrict__ ea,
                                                        const int32_t *__restrict__ eb, const float *__restrict__ ew,
                                                        int ne, uint32_t *X, float *out, int *iters) {
    for (int k = threadIdx.x; k < nn; k += blockDim.x) X[k] = k ? 0xffffffffu : okey32(-INFINITY);
    __syncthreads();
    int it = 0;
    for (;; it++) {
        int changed = 0;
        for (int e = threadIdx.x; e < ne; e += blockDim.x) {
            int a = ea[e], b = eb[e];
            uint32_t w = okey32(ew[e]);
            uint32_t xa = *(volatile uint32_t *)(X + a), xb = *(volatile uint32_t *)(X + b);
            uint32_t ca = w > xb ? w : xb, cb = w > xa ? w : xa;
            if (ca < xa) { atomicMin(X + a, ca); changed = 1; }
            if (cb < xb) { atomicMin(X + b, cb); changed = 1; }
        }
        if (!__syncthreads_or(changed)) break;
    }
    for (int k = threadIdx.x; k < nn; k += blockDim.x) out[k] = okey32_inv(X[k]);
    if (threadIdx.x == 0 && iters) *iters = it;
}

__global__ void __launch_bounds__(256) k_band_raise(uint32_t *E, const int *__restrict__ comp,
                                                    const int *__restrict__ frank, int base,
                                                    const float *__restrict__ X, int nC) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nC || l == 0) return;
    int K = comp[l];
    if (K == 0) return;
    uint32_t x = okey32(X[band_gid(K, frank, base)]);
    if (x > E[l]) E[l] = x;
}

int fill_band_local(ms_band *B, const float *dem, int64_t *n_frozen, cudaStream_t s) {
    int64_t rows = B->rows, cols = B->cols, n = rows * cols;
    int *lab = (int *)band_buf(B, BB_LAB, (size_t)n * sizeof(int));
    if (!lab) return MS_ERR_CUDA;
    DevBuf<int64_t> total;
    DevBuf<int> tmp;
    MS_TRY(total.alloc(1, s));
    MS_TRY(tmp.alloc((size_t)n, s));
    int64_t *h = host_flags().h;
    int nC = 0;
    MS_TRY(descent_resolve(dem, lab, tmp.p, rows, cols, B->open, nullptr, &nC, nullptr, s));
    tmp.release();
    B->nC = nC;
    int *comp = (int *)band_buf(B, BB_COMP, (size_t)nC * sizeof(int));
    uint32_t *E = (uint32_t *)band_buf(B, BB_E, (size_t)nC * sizeof(uint32_t));
    uint8_t *frozen = (uint8_t *)band_buf(B, BB_FROZEN, (size_t)nC);
    int *frank = (int *)band_buf(B, BB_FRANK, (size_t)nC * sizeof(int));
    if (!comp || !E || !frozen || !frank) return MS_ERR_CUDA;
    unsigned gc = cdiv(nC, 256);
    MS_LAUNCH(k_boruvka_init, gc, 256, 0, s, comp, E, nC);
    MS_CUDA(cudaMemsetAsync(frozen, 0, (size_t)nC, s));
    MS_TRY(boruvka_rounds_band(dem, lab, comp, E, frozen, nC, rows, cols, s, B));
    // dense ranks of the frozen component roots
    MS_LAUNCH(k_frozen_flags, gc, 256, 0, s, comp, frozen, frank, nC);
    MS_TRY(exclusive_scan_i32(frank, frank, nC, total.p, s));
    MS_TRY(ms::readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    B->nF = (int)h[0];
    if (n_frozen) *n_frozen = B->nF;
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_band_fill_local_dev(ms_band *B, const float *dem, int64_t *n_frozen, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!B || !dem) { ms::set_error("band fill: null pointer"); return MS_ERR_ARG; }
    return ms::fill_band_local(B, dem, n_frozen, (cudaStream_t)stream);
}

int ms_band_fill_edge_ids_dev(ms_band *B, int64_t gid_base, int32_t *gid_top, int32_t *gid_bot, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !gid_top || !gid_bot || !B->buf[BB_LAB]) { set_error("band fill: edge ids before the local phase"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    B->gid_base = (int)gid_base;
    MS_LAUNCH(k_band_edge_ids, cdiv(B->cols, 256), 256, 0, s, (const int *)B->buf[BB_LAB], (const int *)B->buf[BB_COMP],
              (const int *)B->buf[BB_FRANK], B->gid_base, (int)B->rows, (int)B->cols, gid_top, gid_bot);
    return MS_OK;
}

int ms_band_fill_edges_dev(ms_band *B, const float *dem, const int32_t *halo_gid_top, const int32_t *halo_gid_bot,
                           int32_t *edge_a, int32_t *edge_b, float *edge_w, int64_t capacity, int64_t *n_edges,
                           void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !edge_a || !edge_b || !edge_w || !n_edges) { set_error("band fill: null pointer"); return MS_ERR_ARG; }
    if (((B->open & 1) && !halo_gid_top) || ((B->open & 2) && !halo_gid_bot)) {
        set_error("band fill: halo component ids missing for an open band edge");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t *h = host_flags().h;
    unsigned H = 4096;
    while ((int64_t)H < 16ll * ((int64_t)B->nF + B->cols)) H <<= 1;
    for (int attempt = 0; attempt < 6; attempt++, H <<= 1) {
        unsigned long long *hk = (unsigned long long *)band_buf(B, BB_HASHK, (size_t)H * 8);
        uint32_t *hv = (uint32_t *)band_buf(B, BB_HASHV, (size_t)H * 4);
        int *cnt = (int *)band_buf(B, BB_MISC, 64);
        if (!hk || !hv || !cnt) return MS_ERR_CUDA;
        MS_CUDA(cudaMemsetAsync(hk, 0xff, (size_t)H * 8, s));
        MS_CUDA(cudaMemsetAsync(hv, 0xff, (size_t)H * 4, s));
        MS_CUDA(cudaMemsetAsync(cnt, 0, 64, s));
        if (B->n_blist > 0)
            MS_LAUNCH(k_band_edges, cdiv(B->n_blist, 256), 256, 0, s, dem, (const int *)B->buf[BB_LAB], (const int *)B->buf[BB_COMP],
                      (const int *)B->buf[BB_FRANK], B->gid_base, halo_gid_top, halo_gid_bot, (int)B->rows, (int)B->cols, hk,
                      hv, H, cnt + 1, (const int *)B->buf[BB_BLIST], B->n_blist);
        MS_LAUNCH(k_band_edges_compact, cdiv(H, 256), 256, 0, s, hk, hv, H, edge_a, edge_b, edge_w, capacity, cnt);
        MS_TRY(ms::readback(h, cnt, 2 * sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        int ne = ((int *)h)[0], overflow = ((int *)h)[1];
        if (overflow) continue;      // table too small: double it
        if (ne > capacity) {
            set_error("band fill: %d boundary-graph edges do not fit the caller's capacity %lld", ne, (long long)capacity);
            *n_edges = ne;
            return MS_ERR_ARG;
        }
        *n_edges = ne;
        return MS_OK;
    }
    set_error("band fill: boundary-graph edge table overflow");
    return MS_ERR_NOCONV;
}

int ms_graph_minimax_dev(int64_t n_nodes, const int32_t *edge_a, const int32_t *edge_b, const float *edge_w,
                         int64_t n_edges, float *out_x, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (n_nodes < 1 || n_edges < 0 || !out_x || (n_edges && (!edge_a || !edge_b || !edge_w))) {
        set_error("graph_minimax: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    DevBuf<uint32_t> X;
    MS_TRY(X.alloc((size_t)n_nodes, s));
    MS_LAUNCH(k_graph_minimax, 1, 1024, 0, s, (int)n_nodes, edge_a, edge_b, edge_w, (int)n_edges, X.p, out_x,
              (int *)nullptr);
    return MS_OK;
}

int ms_band_fill_finish_dev(ms_band *B, const float *dem, const float *graph_x, float *filled, float *depths,
                            void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !filled || !B->buf[BB_LAB] || (B->nF && !graph_x)) { set_error("band fill: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t n = B->rows * B->cols;
    if (B->nF)
        MS_LAUNCH(k_band_raise, cdiv(B->nC, 256), 256, 0, s, (uint32_t *)B->buf[BB_E], (const int *)B->buf[BB_COMP],
                  (const int *)B->buf[BB_FRANK], B->gid_base, graph_x, B->nC);
    MS_LAUNCH(k_fill_final, cdiv(n, 256), 256, 0, s, dem, (const int *)B->buf[BB_LAB], (const uint32_t *)B->buf[BB_E],
              filled, depths, n);
    return MS_OK;
}

int ms_minmax_f32_dev(const float *dem, int64_t n, float *out_minmax_dev2, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!dem || !out_minmax_dev2 || n <= 0) { ms::set_error("minmax: bad argument"); return MS_ERR_ARG; }
    return ms::minmax_dev(dem, n, out_minmax_dev2, (cudaStream_t)stream);
}

int ms_minmax_f32(const float *dem, int64_t n, float *out_min, float *out_max) {
    MS_TRY(ms::ensure_init());
    if (!dem || n <= 0) { ms::set_error("minmax: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    ms::HostCall hc;
    float *d = nullptr;
    ms::DevBuf<float> o;
    MS_TRY(hc.in(dem, (size_t)n, s, &d));
    MS_TRY(o.alloc(2, s));
    MS_TRY(ms::minmax_dev(d, n, o.p, s));
    float r[2];
    MS_CUDA(cudaMemcpyAsync(r, o.p, sizeof(r), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    *out_min = r[0];
    *out_max = r[1];
    return MS_OK;
}

int ms_fill_terrain_dev(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols,
                        void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::fill_terrain_dev_impl(dtm, filled, depths, rows, cols, nullptr, (cudaStream_t)stream);
}

int ms_fill_terrain(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols) {
    MS_TRY(ms::ensure_init());
    if (!dtm || !filled) { ms::set_error("fill_terrain: null pointer"); return MS_ERR_ARG; }
    if (rows < 3 || cols < 3 || rows * cols > (1ll << 30)) {
        ms::set_error("fill_terrain: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    float *d = nullptr;
    MS_TRY(hc.in(dtm, n, s, &d));
    // the plain fill (and the depths) of this DEM may still be on the device (an earlier call on the same array)
    float *f = (float *)ms::cache_find_derived(d, ms::CK_FILLED, 0, 0);
    float *dp = (float *)ms::cache_find_derived(d, ms::CK_DEPTHS, 0, 0);
    if (!f || (depths && !dp)) {
        MS_TRY(hc.out(n, &f));
        MS_TRY(hc.out(n, &dp));
        MS_TRY(ms::fill_terrain_dev_impl(d, f, dp, rows, cols, nullptr, s));
        ms::cache_bind_derived(f, d, ms::CK_FILLED, 0, 0);
        ms::cache_bind_derived(dp, d, ms::CK_DEPTHS, 0, 0);
    }
    MS_CUDA(cudaMemcpyAsync(filled, f, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (depths) MS_CUDA(cudaMemcpyAsync(depths, dp, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(f, filled, n * sizeof(float));
    if (depths) ms::cache_bind_host(dp, depths, n * sizeof(float));
    return MS_OK;
}

}  // extern "C"
