// labels.cu — K5/K6 connected components in scipy's numbering, K8 per-label statistics, K8'/K8'' per-label
// arg-min / arg-max with raster-order tie-break, K9 keep-LUT gather, K10 label histogram.
#include <math.h>

#include "common.cuh"

namespace ms {

// ------------------------------------------------------------------------------------------------
// K5/K6.  label.connected_components (label.py:19-40 -> scipy.ndimage.label, full 3x3 structure):
// foreground = value != 0 (NaN and denormals are foreground, -0.0 is not), 8-connectivity, int32 labels
// numbered 1..n by each component's first cell in row-major order.  Union-find over cell indices where a
// union always hangs the larger root under the smaller, so every component's root is its minimum index;
// an exclusive scan of the root flags in raster order then gives scipy's numbering.
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ inline bool is_fg(T v) { return v != (T)0; }

__device__ inline int cc_find(const int *parent, int x) {
    int p = __ldcg(parent + x);
    while (p != x) { x = p; p = __ldcg(parent + x); }
    return x;
}

__device__ inline void cc_union(int *parent, int a, int b) {
    for (;;) {
        a = cc_find(parent, a);
        b = cc_find(parent, b);
        if (a == b) return;
        if (a > b) { int t = a; a = b; b = t; }
        int old = atomicMin(parent + b, a);      // b was a root: hang it under the smaller root a
        if (old == b) return;
        b = old;                                  // somebody re-parented b meanwhile: retry from there
    }
}

// Tile-local phase: one CTA labels a 64x64 tile in shared memory with the same union-find (row runs pre-linked,
// atomicMin hooking, smaller index wins), then writes each cell's tile-local root as a GLOBAL cell index.  Only the
// cells on tile edges are merged through global memory afterwards (k_cc_border): 3 % of the raster instead of all.
constexpr int CT = 64;

// Shared-memory layout of the tile forest: one pad word per 16 cells.  A thread owns 16 consecutive cells, so with
// the plain layout the lanes of a warp would sit 16 words apart (2 banks in use, 16-way conflicts on every access);
// with the pad lane t's cells start at word 17 t and the 32 lanes hit 32 different banks.
__device__ inline int cpad(int i) { return i + (i >> 4); }

__device__ inline int cc_find_s(const int *p, int x) {
    int q = p[cpad(x)];
    while (q != x) { x = q; q = p[cpad(x)]; }
    return x;
}

__device__ inline void cc_union_s(int *p, int a, int b) {
    for (;;) {
        a = cc_find_s(p, a);
        b = cc_find_s(p, b);
        if (a == b) return;
        if (a > b) { int t = a; a = b; b = t; }
        int old = atomicMin(p + cpad(b), a);
        if (old == b) return;
        b = old;
    }
}

template <typename T>
__global__ void __launch_bounds__(256) k_cc_tile(const T *__restrict__ data, int *__restrict__ parent, int rows, int cols,
                                                 int tiles_x) {
    __shared__ int sp[CT * CT + CT * CT / 16];
    int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    int r0 = ty * CT, c0 = tx * CT, tid = threadIdx.x;
    // Coalesced load of the tile's foreground bits: a warp reads half a row per instruction and votes it into one word
    // of the row masks.  Then a thread owns 16 consecutive cells of one row (runs are linked while its cells are set up).
    __shared__ unsigned rowmask[CT * 2];
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int rr = r0 + (k >> 6), cc = c0 + (k & 63);
        bool f = rr < rows && cc < cols && is_fg(data[(size_t)rr * cols + cc]);
        unsigned b = __ballot_sync(0xffffffffu, f);
        if ((tid & 31) == 0) rowmask[k >> 5] = b;
    }
    __syncthreads();
    // Round 2: everything from here on works on the 64-bit foreground masks of the thread's row and of the row above.
    // A thread owns 16 consecutive cells of one row.  Runs are whole-row runs (the start of a cell's run comes from a
    // count of the set bits below it), so there is nothing to join between the 16-cell segments; the links to the row
    // above are one union per pair of touching runs, found as bit events (a run starts under / next to a run above, or
    // a run above starts beside the cell), and a root is looked up once per run, not once per cell.  (Round 1 walked the
    // 16 cells three times under divergent branches: ncu 15 of 32 lanes active, 10.5 stall cycles per issue at barriers.)
    const int lr = tid >> 2, cb = (tid & 3) * 16;
    const unsigned long long M = ((unsigned long long)rowmask[lr * 2 + 1] << 32) | rowmask[lr * 2];
    const unsigned long long U = lr > 0 ? (((unsigned long long)rowmask[lr * 2 - 1] << 32) | rowmask[lr * 2 - 2]) : 0ull;
    const unsigned fg = (unsigned)(M >> cb) & 0xffffu;
    auto run_start = [&](int x) {          // first column of the run that holds column x (bit x of M is set)
        const unsigned long long z = ~M & ((1ull << x) - 1ull);
        return z ? 64 - __clzll((long long)z) : 0;
    };
    {
        int run = -1;
        if (cb > 0 && (fg & 1u) && ((M >> (cb - 1)) & 1ull)) run = lr * CT + run_start(cb);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            int idx = lr * CT + cb + k;
            if (fg & (1u << k)) { if (run < 0) run = idx; sp[cpad(idx)] = run; }
            else { sp[cpad(idx)] = -1; run = -1; }
        }
    }
    __syncthreads();
    if (lr > 0 && fg) {
        const unsigned long long seg = 0xffffull << cb;
        const unsigned long long start = M & ~(M << 1);
        unsigned long long e_n = start & U & seg;                          // a run starts under a cell of the row above
        unsigned long long e_nw = start & ~U & (U << 1) & seg;             // ... or right of the end of a run above
        unsigned long long e_ne = M & ~U & (U >> 1) & seg;                 // a run above starts right of this cell
        while (e_n) { int x = __ffsll((long long)e_n) - 1; e_n &= e_n - 1; cc_union_s(sp, lr * CT + x, (lr - 1) * CT + x); }
        while (e_nw) { int x = __ffsll((long long)e_nw) - 1; e_nw &= e_nw - 1; cc_union_s(sp, lr * CT + x, (lr - 1) * CT + x - 1); }
        while (e_ne) { int x = __ffsll((long long)e_ne) - 1; e_ne &= e_ne - 1; cc_union_s(sp, lr * CT + x, (lr - 1) * CT + x + 1); }
    }
    __syncthreads();
    // every cell's tile-local root as a GLOBAL cell index: found with the forest intact (once per run), then staged in
    // shared memory so that the raster is written with full rows of the tile per instruction
    int vout[16];
    {
        int v = -1;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            if (fg & (1u << k)) {
                if (k == 0 || !(fg & (1u << (k - 1)))) {
                    int root = cc_find_s(sp, lr * CT + cb + k);
                    v = (r0 + (root >> 6)) * cols + c0 + (root & 63);
                }
                vout[k] = v;
            } else vout[k] = -1;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; k++) sp[cpad(lr * CT + cb + k)] = vout[k];
    __syncthreads();
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int rr = r0 + (k >> 6), cc = c0 + (k & 63);
        if (rr < rows && cc < cols) parent[(size_t)rr * cols + cc] = sp[cpad(k)];
    }
}

// merges across tile edges: cells of a tile's first row look up (3 neighbours), cells of its first column look left.
// One CTA of 128 threads per tile: threads 0..63 are the tile's first row, 64..127 its first column (the raster is not
// swept for the 3 % of cells that have something to do).
__global__ void __launch_bounds__(128) k_cc_border(int *parent, int rows, int cols, int tiles_x) {
    int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    int t = threadIdx.x & 63;
    bool top = threadIdx.x < 64;
    int r = ty * CT + (top ? 0 : t), c = tx * CT + (top ? t : 0);
    if (r >= rows || c >= cols) return;
    int i = r * cols + c;
    if (parent[i] < 0) return;
    if (top) {
        if (r == 0) return;
        int up = i - cols;
        if (c > 0 && parent[up - 1] >= 0) cc_union(parent, i, up - 1);
        if (parent[up] >= 0) cc_union(parent, i, up);
        if (c < cols - 1 && parent[up + 1] >= 0) cc_union(parent, i, up + 1);
    } else {
        if (c == 0) return;
        if (r > 0 && parent[i - cols - 1] >= 0) cc_union(parent, i, i - cols - 1);
        if (parent[i - 1] >= 0) cc_union(parent, i, i - 1);
        if (r < rows - 1 && parent[i + cols - 1] >= 0) cc_union(parent, i, i + cols - 1);
    }
}

__global__ void __launch_bounds__(256) k_cc_flatten(int *parent, int *flag, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = parent[i];
    int f = 0;
    if (p >= 0) {
        int root = cc_find(parent, (int)i);
        if (root != p) parent[i] = root;
        f = (root == (int)i);
    }
    if (flag) flag[i] = f;
}

__global__ void __launch_bounds__(256) k_cc_number(const int *__restrict__ parent, const int *__restrict__ rank,
                                                   int32_t *__restrict__ labels, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = parent[i];
    labels[i] = p < 0 ? 0 : rank[cc_find(parent, p)] + 1;
}

template <typename T>
int cc_dev_t(const T *data, int32_t *labels, int64_t rows, int64_t cols, int64_t *nlabels_dev, cudaStream_t s) {
    int64_t n = rows * cols;
    DevBuf<int> parent, flag;
    MS_TRY(parent.alloc((size_t)n, s));
    MS_TRY(flag.alloc((size_t)n, s));
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    unsigned g1 = cdiv(n, 256);
    int tiles_x = (int)cdiv(cols, CT), tiles_y = (int)cdiv(rows, CT);
    prof_units(n);
    MS_LAUNCH(k_cc_tile<T>, tiles_x * tiles_y, 256, 0, s, data, parent.p, (int)rows, (int)cols, tiles_x);
    MS_LAUNCH(k_cc_border, tiles_x * tiles_y, 128, 0, s, parent.p, (int)rows, (int)cols, tiles_x);
    // roots are the cells that point at themselves, flattened or not: number them in raster order, then every cell
    // walks its (2-4 hop) chain once and takes its root's number — no separate flattening pass
    MS_TRY(exclusive_scan_selfptr(parent.p, flag.p, n, nlabels_dev, s));
    MS_LAUNCH(k_cc_number, g1, 256, 0, s, parent.p, flag.p, labels, n);
    return MS_OK;
}

int cc_dev_impl(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols, int64_t *nlabels_dev,
                cudaStream_t s) {
    if (!data || !labels) { set_error("connected_components: null pointer"); return MS_ERR_ARG; }
    if (rows < 1 || cols < 1 || rows * cols > (1ll << 30)) {
        set_error("connected_components: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    switch (dtype) {
        case MS_F32: return cc_dev_t<float>((const float *)data, labels, rows, cols, nlabels_dev, s);
        case MS_F64: return cc_dev_t<double>((const double *)data, labels, rows, cols, nlabels_dev, s);
        case MS_U8: return cc_dev_t<uint8_t>((const uint8_t *)data, labels, rows, cols, nlabels_dev, s);
        case MS_I32: return cc_dev_t<int32_t>((const int32_t *)data, labels, rows, cols, nlabels_dev, s);
        case MS_I64: return cc_dev_t<int64_t>((const int64_t *)data, labels, rows, cols, nlabels_dev, s);
    }
    set_error("connected_components: unsupported dtype code %d", dtype);
    return MS_ERR_ARG;
}


// ------------------------------------------------------------------------------------------------
// Row-band connected components (SURVEY.md §8(e), K5/K6).  Phase 1: union-find on the band's own rows; the roots
// of the first / last row go to the host side as global cell indices.  The host merges components that touch
// across band edges (ms_cc_boundary_merge, CPU, a few thousand cells) — a component keeps the smallest global
// root.  Phase 2: roots that lost their rank to a root of another band (or of this band, through another band)
// are taken out of the numbering, every band counts its surviving roots, the counts are scanned across bands
// (host side) and the labels are written with the band's offset; the few re-rooted components get the label
// their new root received from its owner.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cc_edge_roots(const int *__restrict__ parent, int64_t cell_offset, int rows,
                                                       int cols, int64_t *top, int64_t *bot) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    int a = parent[c], b = parent[(size_t)(rows - 1) * cols + c];
    top[c] = a < 0 ? -1 : cell_offset + a;
    bot[c] = b < 0 ? -1 : cell_offset + b;
}

__global__ void __launch_bounds__(256) k_scatter_i32(int *dst, const int32_t *__restrict__ idx,
                                                     const int32_t *__restrict__ val, int constant, int64_t offset,
                                                     int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) dst[idx[k]] = val ? (int)(val[k] - offset - 1) : constant;
}

__global__ void __launch_bounds__(256) k_gather_labels(const int *__restrict__ rank, const int32_t *__restrict__ idx,
                                                       int64_t offset, int32_t *out, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = (int32_t)(rank[idx[k]] + offset + 1);
}

__global__ void __launch_bounds__(256) k_cc_number_off(const int *__restrict__ parent, const int *__restrict__ rank,
                                                       int64_t offset, int32_t *__restrict__ labels, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = parent[i];
    labels[i] = p < 0 ? 0 : (int32_t)(rank[p] + offset + 1);
}

template <typename T>
int cc_band_local_t(ms_band *B, const T *data, int64_t cell_offset, int64_t *root_top, int64_t *root_bot,
                    cudaStream_t s) {
    int64_t rows = B->rows, cols = B->cols, n = rows * cols;
    int *parent = (int *)band_buf(B, BB_CC_PARENT, (size_t)n * sizeof(int));
    int *rank = (int *)band_buf(B, BB_CC_RANK, (size_t)n * sizeof(int));
    if (!parent || !rank) return MS_ERR_CUDA;
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    int tiles_x = (int)cdiv(cols, CT), tiles_y = (int)cdiv(rows, CT);
    MS_LAUNCH(k_cc_tile<T>, tiles_x * tiles_y, 256, 0, s, data, parent, (int)rows, (int)cols, tiles_x);
    MS_LAUNCH(k_cc_border, tiles_x * tiles_y, 128, 0, s, parent, (int)rows, (int)cols, tiles_x);
    MS_LAUNCH(k_cc_flatten, cdiv(n, 256), 256, 0, s, parent, rank, n);
    MS_LAUNCH(k_cc_edge_roots, cdiv(cols, 256), 256, 0, s, parent, cell_offset, (int)rows, (int)cols, root_top, root_bot);
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_band_cc_local_dev(ms_band *B, const void *data, int dtype, int64_t cell_offset, int64_t *root_top,
                         int64_t *root_bot, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !data || !root_top || !root_bot) { set_error("band connected_components: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    switch (dtype) {
        case MS_F32: return cc_band_local_t<float>(B, (const float *)data, cell_offset, root_top, root_bot, s);
        case MS_F64: return cc_band_local_t<double>(B, (const double *)data, cell_offset, root_top, root_bot, s);
        case MS_U8: return cc_band_local_t<uint8_t>(B, (const uint8_t *)data, cell_offset, root_top, root_bot, s);
        case MS_I32: return cc_band_local_t<int32_t>(B, (const int32_t *)data, cell_offset, root_top, root_bot, s);
        case MS_I64: return cc_band_local_t<int64_t>(B, (const int64_t *)data, cell_offset, root_top, root_bot, s);
    }
    set_error("band connected_components: unsupported dtype code %d", dtype);
    return MS_ERR_ARG;
}

/* `rerooted` (device, int32 local cell indices, n_rerooted of them): roots of this band that are not the smallest
 * cell of their (cross-band) component.  Returns the number of components this band numbers. */
int ms_band_cc_count_dev(ms_band *B, const int32_t *rerooted, int64_t n_rerooted, int64_t *count, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !count || !B->buf[BB_CC_RANK] || (n_rerooted && !rerooted)) { set_error("band connected_components: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t n = B->rows * B->cols;
    int *rank = (int *)B->buf[BB_CC_RANK];
    if (n_rerooted)
        MS_LAUNCH(k_scatter_i32, cdiv(n_rerooted, 256), 256, 0, s, rank, rerooted, (const int32_t *)nullptr, 0, (int64_t)0,
                  (int)n_rerooted);
    DevBuf<int64_t> tot;
    MS_TRY(tot.alloc(1, s));
    MS_TRY(exclusive_scan_i32(rank, rank, n, tot.p, s));
    int64_t *h = host_flags().h;
    MS_TRY(ms::readback(h, tot.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    *count = h[0];
    return MS_OK;
}

/* labels (offset + rank + 1) of the given root cells of this band */
int ms_band_cc_root_labels_dev(ms_band *B, const int32_t *roots, int64_t n_roots, int64_t label_offset,
                               int32_t *labels_out, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->buf[BB_CC_RANK] || (n_roots && (!roots || !labels_out))) { set_error("band connected_components: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    if (n_roots)
        MS_LAUNCH(k_gather_labels, cdiv(n_roots, 256), 256, 0, s, (const int *)B->buf[BB_CC_RANK], roots, label_offset,
                  labels_out, (int)n_roots);
    return MS_OK;
}

int ms_band_cc_finish_dev(ms_band *B, const int32_t *rerooted, const int32_t *rerooted_label, int64_t n_rerooted,
                          int64_t label_offset, int32_t *labels, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !labels || !B->buf[BB_CC_RANK] || (n_rerooted && (!rerooted || !rerooted_label))) {
        set_error("band connected_components: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t n = B->rows * B->cols;
    int *rank = (int *)B->buf[BB_CC_RANK];
    if (n_rerooted)
        MS_LAUNCH(k_scatter_i32, cdiv(n_rerooted, 256), 256, 0, s, rank, rerooted, rerooted_label, 0, label_offset,
                  (int)n_rerooted);
    MS_LAUNCH(k_cc_number_off, cdiv(n, 256), 256, 0, s, (const int *)B->buf[BB_CC_PARENT], (const int *)rank, label_offset,
              labels, n);
    return MS_OK;
}

}  // extern "C"

namespace ms {

// ------------------------------------------------------------------------------------------------
// label range (the `nlabels = np.max(labelled)` default, label.py:57,116,150)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_label_range(const int32_t *__restrict__ lab, int64_t n, int32_t *out) {
    int lo = INT32_MAX, hi = INT32_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int v = lab[i];
        lo = min(lo, v);
        hi = max(hi, v);
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0) {
        atomicMin(out, lo);
        atomicMax(out + 1, hi);
    }
}

int label_range_dev_impl(const int32_t *lab, int64_t n, int32_t *out2, cudaStream_t s) {
    static const int32_t init[2] = {INT32_MAX, INT32_MIN};
    MS_CUDA(cudaMemcpyAsync(out2, init, sizeof(init), cudaMemcpyHostToDevice, s));
    int64_t want = (n + 1023) / 1024;
    int blocks = (int)(want < 1 ? 1 : (want > 148 * 8 ? 148 * 8 : want));
    MS_LAUNCH(k_label_range, blocks, 256, 0, s, lab, n, out2);
    return MS_OK;
}

// ------------------------------------------------------------------------------------------------
// K8.  label.label_stats (label.py:43-75; speedups/_label.pyx:31-97): per label min, max, sum (float64),
// count.  Labels are spatially coherent, so lanes of a warp that hold the same label are combined first
// (match.any + redux for the ordered min/max keys, a lane-ordered shuffle sum) and one lane issues the
// atomics; label 0 (the background, most of the raster) is kept in registers and reduced per CTA.
// min / max / count are exact; sum is float64 in a different association than the reference's raster
// order (within 1e-6 relative, north_star).
// ------------------------------------------------------------------------------------------------
template <typename T> struct KeyOf;
template <> struct KeyOf<float> {
    typedef uint32_t K;
    static __device__ K key(float v) { return okey32(v); }
    static __device__ double inv(K k) { return (double)okey32_inv(k); }
    static constexpr K kMax = 0xffffffffu;
};
template <> struct KeyOf<double> {
    typedef unsigned long long K;
    static __device__ K key(double v) { return okey64(v); }
    static __device__ double inv(K k) { return okey64_inv(k); }
    static constexpr K kMax = ~0ull;
};

__device__ inline uint32_t grp_min(unsigned m, uint32_t v) { return __reduce_min_sync(m, v); }
__device__ inline uint32_t grp_max(unsigned m, uint32_t v) { return __reduce_max_sync(m, v); }
__device__ inline unsigned long long grp_min(unsigned m, unsigned long long v) {
    // 64-bit: high word first, then the low word among the lanes that hold the winning high word
    uint32_t hi = (uint32_t)(v >> 32);
    uint32_t bh = __reduce_min_sync(m, hi);
    uint32_t lo = (hi == bh) ? (uint32_t)v : 0xffffffffu;
    return ((unsigned long long)bh << 32) | __reduce_min_sync(m, lo);
}
__device__ inline unsigned long long grp_max(unsigned m, unsigned long long v) {
    uint32_t hi = (uint32_t)(v >> 32);
    uint32_t bh = __reduce_max_sync(m, hi);
    uint32_t lo = (hi == bh) ? (uint32_t)v : 0u;
    return ((unsigned long long)bh << 32) | __reduce_max_sync(m, lo);
}

__device__ inline double grp_sum(unsigned m, double v) {
    if (m == 0xffffffffu) {              // the whole warp holds one label (inside a bluespot): butterfly
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }
    double s = 0.0;
    unsigned rest = m;
    while (rest) {                       // lane order = raster order inside the group
        int src = __ffs(rest) - 1;
        rest &= rest - 1;
        s += __shfl_sync(m, v, src);
    }
    return s;
}

template <typename T>
__global__ void __launch_bounds__(256) k_label_stats(const T *__restrict__ data, const int32_t *__restrict__ lab,
                                                     int64_t n, int64_t nlabels, typename KeyOf<T>::K *tmin,
                                                     typename KeyOf<T>::K *tmax, double *tsum,
                                                     unsigned long long *tcnt, int *err) {
    typedef typename KeyOf<T>::K K;
    K bmin = KeyOf<T>::kMax, bmax = 0;
    double bsum = 0.0;
    unsigned long long bcnt = 0;
    bool nan_in_bg = false;
    int64_t span = (int64_t)gridDim.x * blockDim.x;
    int64_t nround = (n + span - 1) / span;
    for (int64_t it = 0; it < nround; it++) {
        int64_t i = it * span + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        int lbl = -1;
        T v = 0;
        if (i < n) {
            lbl = lab[i];
            v = data[i];
            if (lbl < 0 || lbl > nlabels) { *err = 1; lbl = -1; }
        }
        if (lbl == 0) {
            K k = KeyOf<T>::key(v);
            if (v == v) { bmin = k < bmin ? k : bmin; bmax = k > bmax ? k : bmax; } else nan_in_bg = true;
            bsum += (double)v;
            bcnt++;
        }
        unsigned act = __ballot_sync(0xffffffffu, lbl > 0);
        if (lbl > 0) {
            unsigned g = __match_any_sync(act, lbl);
            bool ok = (v == v);                  // NaN never wins a strict comparison (label.py:70-73)
            K k = KeyOf<T>::key(ok ? v : (T)0);
            K kmn = grp_min(g, ok ? k : KeyOf<T>::kMax);
            K kmx = grp_max(g, ok ? k : (K)0);
            double sm = grp_sum(g, (double)v);
            if ((int)(__ffs(g) - 1) == (int)(threadIdx.x & 31)) {
                if (kmn < tmin[lbl]) atomicMin(tmin + lbl, kmn);
                if (kmx > tmax[lbl]) atomicMax(tmax + lbl, kmx);
                atomicAdd(tsum + lbl, sm);
                atomicAdd(tcnt + lbl, (unsigned long long)__popc(g));
            }
        }
    }
    (void)nan_in_bg;
    // CTA reduction of the background accumulators
    unsigned full = 0xffffffffu;
    K wmin = grp_min(full, bmin), wmax = grp_max(full, bmax);
    double wsum = bsum;
    unsigned long long wcnt = bcnt;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        wsum += __shfl_xor_sync(full, wsum, o);
        wcnt += __shfl_xor_sync(full, wcnt, o);
    }
    __shared__ K smin[8], smax[8];
    __shared__ double ssum[8];
    __shared__ unsigned long long scnt[8];
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { smin[w] = wmin; smax[w] = wmax; ssum[w] = wsum; scnt[w] = wcnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; k++) {
            wmin = smin[k] < wmin ? smin[k] : wmin;
            wmax = smax[k] > wmax ? smax[k] : wmax;
            wsum += ssum[k];
            wcnt += scnt[k];
        }
        if (wcnt) {
            atomicMin(tmin, wmin);
            atomicMax(tmax, wmax);
            atomicAdd(tsum, wsum);
            atomicAdd(tcnt, wcnt);
        }
    }
}

template <typename K>
__global__ void __launch_bounds__(256) k_stats_init(K *tmin, K *tmax, double *tsum, unsigned long long *tcnt,
                                                    int64_t m, K kmax) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l < m) { tmin[l] = kmax; tmax[l] = 0; tsum[l] = 0.0; tcnt[l] = 0; }
}

template <typename T>
__global__ void __launch_bounds__(256) k_stats_finish(const typename KeyOf<T>::K *tmin,
                                                      const typename KeyOf<T>::K *tmax, const unsigned long long *tcnt,
                                                      double *omin, double *omax, int64_t *ocnt, int64_t m) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= m) return;
    typedef typename KeyOf<T>::K K;
    K a = tmin[l], b = tmax[l];
    omin[l] = (a == KeyOf<T>::kMax) ? (double)INFINITY : KeyOf<T>::inv(a);     // label.py:61-62 defaults
    omax[l] = (b == (K)0) ? (double)-INFINITY : KeyOf<T>::inv(b);
    ocnt[l] = (int64_t)tcnt[l];
}

template <typename T>
int label_stats_dev_t(const T *data, const int32_t *lab, int64_t n, int64_t nlabels, double *omin, double *omax,
                      double *osum, int64_t *ocnt, int *err_dev, cudaStream_t s) {
    typedef typename KeyOf<T>::K K;
    int64_t m = nlabels + 1;
    DevBuf<K> tmin, tmax;
    DevBuf<unsigned long long> tcnt;
    MS_TRY(tmin.alloc((size_t)m, s));
    MS_TRY(tmax.alloc((size_t)m, s));
    MS_TRY(tcnt.alloc((size_t)m, s));
    unsigned gm = cdiv(m, 256);
    MS_LAUNCH(k_stats_init<K>, gm, 256, 0, s, tmin.p, tmax.p, osum, tcnt.p, m, KeyOf<T>::kMax);
    int64_t want = (n + 255) / 256;
    int blocks = (int)(want > 148 * 16 ? 148 * 16 : want);
    MS_LAUNCH(k_label_stats<T>, blocks, 256, 0, s, data, lab, n, nlabels, tmin.p, tmax.p, osum, tcnt.p, err_dev);
    MS_LAUNCH(k_stats_finish<T>, gm, 256, 0, s, tmin.p, tmax.p, tcnt.p, omin, omax, ocnt, m);
    return MS_OK;
}

int label_stats_dev_impl(const void *data, int dtype, const int32_t *lab, int64_t n, int64_t nlabels, double *omin,
                         double *omax, double *osum, int64_t *ocnt, int *err_dev, cudaStream_t s) {
    if (!data || !lab || !omin || !omax || !osum || !ocnt || n < 1 || nlabels < 0) {
        set_error("label_stats: bad argument");
        return MS_ERR_ARG;
    }
    if (dtype == MS_F32) return label_stats_dev_t<float>((const float *)data, lab, n, nlabels, omin, omax, osum, ocnt, err_dev, s);
    if (dtype == MS_F64) return label_stats_dev_t<double>((const double *)data, lab, n, nlabels, omin, omax, osum, ocnt, err_dev, s);
    set_error("label_stats: data dtype must be MS_F32 or MS_F64");
    return MS_ERR_ARG;
}

// ------------------------------------------------------------------------------------------------
// K8' / K8''.  label.label_min_index / label_max_index (label.py:101-166; speedups/_label.pyx:99-128):
// strict comparison while scanning in raster order, so among equal extreme values the smallest flat
// index wins; NaN never wins; labels never seen keep (+-inf, -1, -1).  Two passes: the extreme ordered
// key per label, then the smallest index among the cells that hold it.  (-0.0 and +0.0 share a key, as
// they compare equal; the reported value is read back from the winning cell.)
// ------------------------------------------------------------------------------------------------
template <bool MAX>
__global__ void __launch_bounds__(256) k_extreme_key(const double *__restrict__ data, const int32_t *__restrict__ lab,
                                                     int64_t n, int64_t nlabels, unsigned long long *tkey, int *err) {
    unsigned long long bg = MAX ? 0ull : ~0ull;
    int64_t span = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += span) {
        int lbl = lab[i];
        double v = data[i];
        if (lbl < 0 || lbl > nlabels) { *err = 1; continue; }
        if (v != v) continue;
        unsigned long long k = okey64(v);
        if (lbl == 0) {
            bg = MAX ? (k > bg ? k : bg) : (k < bg ? k : bg);
        } else if (MAX) {
            if (k > tkey[lbl]) atomicMax(tkey + lbl, k);
        } else {
            if (k < tkey[lbl]) atomicMin(tkey + lbl, k);
        }
    }
    bg = MAX ? grp_max(0xffffffffu, bg) : grp_min(0xffffffffu, bg);
    if ((threadIdx.x & 31) == 0) {
        if (MAX) { if (bg > tkey[0]) atomicMax(tkey, bg); }
        else     { if (bg < tkey[0]) atomicMin(tkey, bg); }
    }
}

__global__ void __launch_bounds__(256) k_extreme_index(const double *__restrict__ data, const int32_t *__restrict__ lab,
                                                       int64_t n, int64_t nlabels,
                                                       const unsigned long long *__restrict__ tkey, int *tidx) {
    int64_t span = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += span) {
        int lbl = lab[i];
        if (lbl < 0 || lbl > nlabels) continue;
        double v = data[i];
        if (v != v) continue;
        if (okey64(v) != tkey[lbl]) continue;
        if ((int)i < tidx[lbl]) atomicMin(tidx + lbl, (int)i);
    }
}

__global__ void __launch_bounds__(256) k_extreme_finish(const double *__restrict__ data, const int *__restrict__ tidx,
                                                        int64_t m, int cols, int want_max, double *oval, int64_t *orow,
                                                        int64_t *ocol) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= m) return;
    int i = tidx[l];
    if (i == INT32_MAX) {
        oval[l] = want_max ? (double)-INFINITY : (double)INFINITY;
        orow[l] = -1;
        ocol[l] = -1;
    } else {
        oval[l] = data[i];
        orow[l] = i / cols;
        ocol[l] = i % cols;
    }
}

__global__ void __launch_bounds__(256) k_fill_u64(unsigned long long *p, unsigned long long v, int *q, int w, int64_t m) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l < m) { p[l] = v; q[l] = w; }
}

int label_extreme_dev_impl(const double *data, const int32_t *lab, int64_t rows, int64_t cols, int64_t nlabels,
                           int want_max, double *oval, int64_t *orow, int64_t *ocol, int *err_dev, cudaStream_t s) {
    if (!data || !lab || !oval || !orow || !ocol || rows < 1 || cols < 1 || nlabels < 0 || rows * cols > (1ll << 30)) {
        set_error("label_min/max_index: bad argument");
        return MS_ERR_ARG;
    }
    int64_t n = rows * cols, m = nlabels + 1;
    DevBuf<unsigned long long> tkey;
    DevBuf<int> tidx;
    MS_TRY(tkey.alloc((size_t)m, s));
    MS_TRY(tidx.alloc((size_t)m, s));
    unsigned gm = cdiv(m, 256);
    MS_LAUNCH(k_fill_u64, gm, 256, 0, s, tkey.p, want_max ? 0ull : ~0ull, tidx.p, INT32_MAX, m);
    int64_t want = (n + 255) / 256;
    int blocks = (int)(want > 148 * 16 ? 148 * 16 : want);
    if (want_max) MS_LAUNCH(k_extreme_key<true>, blocks, 256, 0, s, data, lab, n, nlabels, tkey.p, err_dev);
    else MS_LAUNCH(k_extreme_key<false>, blocks, 256, 0, s, data, lab, n, nlabels, tkey.p, err_dev);
    MS_LAUNCH(k_extreme_index, blocks, 256, 0, s, data, lab, n, nlabels, tkey.p, tidx.p);
    MS_LAUNCH(k_extreme_finish, gm, 256, 0, s, data, tidx.p, m, (int)cols, want_max, oval, orow, ocol);
    return MS_OK;
}


// ------------------------------------------------------------------------------------------------
// The per-label tables of the whole path in two passes (device-resident pipeline only; the numpy-level functions
// keep their one-table kernels above).  BluespotTool asks for label_stats(depths, labels), label_count(wsheds),
// label_min_index(fnf, labels) and label_max_index(accum, labels) (bluespots.py:160-205): five rasters, the labels
// read four times.  Pass A (k_tables_a2) reads every raster once — depth min / max / sum / count, the extreme keys of
// the no-flats surface and of the accumulation per bluespot and the watershed histogram.  Pass B (k_tables_b) finds
// the smallest flat index holding each extreme (raster-order tie-break, label.py:101-166) for both tables at once.
// 28 + 20 B/cell instead of 8 + 4 + 12 + 12 + 12 + 12.
// ------------------------------------------------------------------------------------------------
// Pass A: one CTA per 64 x 64 tile, a thread walks 16 consecutive cells of a tile row.  Bluespots and watersheds are
// blobs, so a thread sees runs of one label: it keeps the run's partial results in registers and folds a finished run
// into a small shared-memory table keyed by label (open addressing, 256 slots; a tile holds a few dozen labels), and
// the table goes to the global per-label tables with one set of atomics per label and tile - instead of one
// warp-aggregated set per label and 32 cells (measured: 21.6 ms at 32768^2, 54 % issue-bound on the match /
// group-reduction instructions).  Label 0 stays in registers.
constexpr int TA_SLOTS = 256;
template <bool ACC>
__global__ void __launch_bounds__(256) k_tables_a2(const float *__restrict__ depths, const int32_t *__restrict__ lab,
                                                   const double *__restrict__ fnf, const double *__restrict__ accum,
                                                   const int32_t *__restrict__ ws, int rows, int cols, int tiles_x,
                                                   int64_t nlabels, uint32_t *tmin, uint32_t *tmax, double *tsum,
                                                   unsigned long long *tcnt, unsigned long long *kmin,
                                                   unsigned long long *kmax, unsigned long long *wcnt, int *err) {
    __shared__ int s_key[TA_SLOTS], s_wkey[TA_SLOTS];
    __shared__ uint32_t s_min[TA_SLOTS], s_max[TA_SLOTS], s_cnt[TA_SLOTS], s_wcnt[TA_SLOTS];
    __shared__ double s_sum[TA_SLOTS];
    __shared__ unsigned long long s_kmin[TA_SLOTS], s_kmax[TA_SLOTS];
    const unsigned full = 0xffffffffu;
    const int tid = threadIdx.x;
    {
        s_key[tid] = 0; s_wkey[tid] = 0; s_min[tid] = 0xffffffffu; s_max[tid] = 0; s_cnt[tid] = 0; s_wcnt[tid] = 0;
        s_sum[tid] = 0.0; s_kmin[tid] = ~0ull; s_kmax[tid] = 0ull;
    }
    __syncthreads();
    const int tile = blockIdx.x, ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int r = ty * 64 + (tid >> 2), c0 = tx * 64 + (tid & 3) * 16;
    // label-0 accumulators (registers, reduced over the CTA at the end)
    uint32_t bmin = 0xffffffffu, bmax = 0;
    double bsum = 0.0;
    unsigned long long bcnt = 0, bwz = 0, bkmin = ~0ull, bkmax = 0ull;
    // the current run of one bluespot label, and of one watershed label
    int cur = -1, wcur = -1;
    uint32_t rmin = 0xffffffffu, rmax = 0, rcnt = 0, wn = 0;
    double rsum = 0.0;
    unsigned long long rkmin = ~0ull, rkmax = 0ull;
    auto slot_of = [&](int *keys, int lbl) {
        unsigned h = ((unsigned)lbl * 2654435761u) >> 24;
        for (int probe = 0; probe < 32; probe++) {
            int old = atomicCAS(keys + h, 0, lbl);
            if (old == 0 || old == lbl) return (int)h;
            h = (h + 1) & (TA_SLOTS - 1);
        }
        return -1;
    };
    auto flush_run = [&]() {
        if (cur == 0) {
            bmin = rmin < bmin ? rmin : bmin; bmax = rmax > bmax ? rmax : bmax;
            bsum += rsum; bcnt += rcnt;
            bkmin = rkmin < bkmin ? rkmin : bkmin;
            if (ACC) bkmax = rkmax > bkmax ? rkmax : bkmax;
        } else if (cur > 0) {
            int h = slot_of(s_key, cur);
            if (h >= 0) {
                atomicMin(s_min + h, rmin); atomicMax(s_max + h, rmax);
                atomicAdd(s_sum + h, rsum); atomicAdd(s_cnt + h, rcnt);
                atomicMin(s_kmin + h, rkmin);
                if (ACC) atomicMax(s_kmax + h, rkmax);
            } else {            // table full: straight to the global tables
                atomicMin(tmin + cur, rmin); atomicMax(tmax + cur, rmax);
                atomicAdd(tsum + cur, rsum); atomicAdd(tcnt + cur, (unsigned long long)rcnt);
                atomicMin(kmin + cur, rkmin);
                if (ACC) atomicMax(kmax + cur, rkmax);
            }
        }
        rmin = 0xffffffffu; rmax = 0; rcnt = 0; rsum = 0.0; rkmin = ~0ull; rkmax = 0ull;
    };
    auto flush_w = [&]() {
        if (wcur == 0) bwz += wn;
        else if (wcur > 0) {
            int h = slot_of(s_wkey, wcur);
            if (h >= 0) atomicAdd(s_wcnt + h, wn);
            else atomicAdd(wcnt + wcur, (unsigned long long)wn);
        }
        wn = 0;
    };
    if (r < rows) {
        const size_t base = (size_t)r * cols + c0;
        const bool vec = ((cols & 3) == 0) && (c0 + 16 <= cols);
#pragma unroll 1
        for (int sub = 0; sub < 4; sub++) {
            int lv[4], wv[4];
            float dv[4];
            double fv[4], av[4];
            const size_t i0 = base + sub * 4;
            if (vec) {
                const int4 l4 = __ldg(reinterpret_cast<const int4 *>(lab + i0)), w4 = __ldg(reinterpret_cast<const int4 *>(ws + i0));
                const float4 d4 = __ldg(reinterpret_cast<const float4 *>(depths + i0));
                const double2 f0 = __ldg(reinterpret_cast<const double2 *>(fnf + i0)), f1 = __ldg(reinterpret_cast<const double2 *>(fnf + i0 + 2));
                lv[0] = l4.x; lv[1] = l4.y; lv[2] = l4.z; lv[3] = l4.w;
                wv[0] = w4.x; wv[1] = w4.y; wv[2] = w4.z; wv[3] = w4.w;
                dv[0] = d4.x; dv[1] = d4.y; dv[2] = d4.z; dv[3] = d4.w;
                fv[0] = f0.x; fv[1] = f0.y; fv[2] = f1.x; fv[3] = f1.y;
                if (ACC) {
                    const double2 a0 = __ldg(reinterpret_cast<const double2 *>(accum + i0)), a1 = __ldg(reinterpret_cast<const double2 *>(accum + i0 + 2));
                    av[0] = a0.x; av[1] = a0.y; av[2] = a1.x; av[3] = a1.y;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const bool in = c0 + sub * 4 + j < cols;
                    lv[j] = in ? lab[i0 + j] : -2;
                    wv[j] = in ? ws[i0 + j] : -2;
                    dv[j] = in ? depths[i0 + j] : 0.f;
                    fv[j] = in ? fnf[i0 + j] : 0.0;
                    av[j] = (ACC && in) ? accum[i0 + j] : 0.0;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                int lbl = lv[j], w = wv[j];
                if (lbl == -2) continue;                       // beyond the raster
                if (lbl < 0 || lbl > nlabels) { *err = 1; lbl = -1; }
                if (w < 0 || w > nlabels) { *err = 1; w = -1; }
                if (lbl != cur) { flush_run(); cur = lbl; }
                if (w != wcur) { flush_w(); wcur = w; }
                wn++;
                const float v = dv[j];
                const double f = fv[j], a = ACC ? av[j] : 0.0;
                const bool vok = (v == v);
                const uint32_t k = okey32(vok ? v : 0.f);
                if (vok) { rmin = k < rmin ? k : rmin; rmax = k > rmax ? k : rmax; }
                rsum += (double)v;
                rcnt++;
                const unsigned long long fk = (f == f) ? okey64(f) : ~0ull;
                rkmin = fk < rkmin ? fk : rkmin;
                if (ACC) {
                    const unsigned long long ak = (a == a) ? okey64(a) : 0ull;
                    rkmax = ak > rkmax ? ak : rkmax;
                }
            }
        }
        flush_run();
        flush_w();
    }
    __syncthreads();
    // the tile's tables -> the global tables
    {
        const int lbl = s_key[tid];
        if (lbl > 0) {
            if (s_min[tid] < tmin[lbl]) atomicMin(tmin + lbl, s_min[tid]);
            if (s_max[tid] > tmax[lbl]) atomicMax(tmax + lbl, s_max[tid]);
            atomicAdd(tsum + lbl, s_sum[tid]);
            atomicAdd(tcnt + lbl, (unsigned long long)s_cnt[tid]);
            if (s_kmin[tid] < kmin[lbl]) atomicMin(kmin + lbl, s_kmin[tid]);
            if (ACC && s_kmax[tid] > kmax[lbl]) atomicMax(kmax + lbl, s_kmax[tid]);
        }
        const int w = s_wkey[tid];
        if (w > 0) atomicAdd(wcnt + w, (unsigned long long)s_wcnt[tid]);
    }
    // CTA reduction of the label-0 accumulators
    uint32_t wmin = grp_min(full, bmin), wmax = grp_max(full, bmax);
    unsigned long long wkmin = grp_min(full, bkmin), wkmax = grp_max(full, bkmax);
    double wsum = bsum;
    unsigned long long wc = bcnt, wz = bwz;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        wsum += __shfl_xor_sync(full, wsum, o);
        wc += __shfl_xor_sync(full, wc, o);
        wz += __shfl_xor_sync(full, wz, o);
    }
    __shared__ uint32_t smin[8], smax[8];
    __shared__ double ssum[8];
    __shared__ unsigned long long scnt[8], swz[8], skmin[8], skmax[8];
    int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    if (lane == 0) { smin[wp] = wmin; smax[wp] = wmax; ssum[wp] = wsum; scnt[wp] = wc; swz[wp] = wz; skmin[wp] = wkmin; skmax[wp] = wkmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; k++) {
            wmin = smin[k] < wmin ? smin[k] : wmin;
            wmax = smax[k] > wmax ? smax[k] : wmax;
            wsum += ssum[k];
            wc += scnt[k];
            wz += swz[k];
            wkmin = skmin[k] < wkmin ? skmin[k] : wkmin;
            wkmax = skmax[k] > wkmax ? skmax[k] : wkmax;
        }
        if (wc) {
            atomicMin(tmin, wmin);
            atomicMax(tmax, wmax);
            atomicAdd(tsum, wsum);
            atomicAdd(tcnt, wc);
            atomicMin(kmin, wkmin);
            if (ACC) atomicMax(kmax, wkmax);
        }
        if (wz) atomicAdd(wcnt, wz);
    }
}

template <bool ACC>
__global__ void __launch_bounds__(256) k_tables_b(const int32_t *__restrict__ lab, const double *__restrict__ fnf,
                                                  const double *__restrict__ accum, int64_t n, int64_t nlabels,
                                                  const unsigned long long *__restrict__ kmin,
                                                  const unsigned long long *__restrict__ kmax, int *imin, int *imax) {
    int64_t span = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += span) {
        int lbl = lab[i];
        if (lbl < 0 || lbl > nlabels) continue;
        double f = fnf[i];
        if (f == f && okey64(f) == kmin[lbl] && (int)i < imin[lbl]) atomicMin(imin + lbl, (int)i);
        if (ACC) {
            double a = accum[i];
            if (a == a && okey64(a) == kmax[lbl] && (int)i < imax[lbl]) atomicMin(imax + lbl, (int)i);
        }
    }
}

// io: the pipeline's rasters and tables (see ms_rasters); all tables are written for labels 0..nlabels
int pipeline_tables_dev_impl(const float *depths, const int32_t *lab, const double *fnf, const double *accum,
                             const int32_t *ws, int64_t rows, int64_t cols, int64_t nlabels, double *st_min,
                             double *st_max, double *st_sum, int64_t *st_count, int64_t *ws_count, double *pmin_v,
                             int64_t *pmin_r, int64_t *pmin_c, double *pmax_v, int64_t *pmax_r, int64_t *pmax_c,
                             int *err_dev, cudaStream_t s) {
    int64_t n = rows * cols, m = nlabels + 1;
    const bool acc = accum && pmax_v;
    DevBuf<uint32_t> tmin, tmax;
    DevBuf<unsigned long long> tcnt, kmin, kmax;
    DevBuf<int> imin, imax;
    MS_TRY(tmin.alloc((size_t)m, s));
    MS_TRY(tmax.alloc((size_t)m, s));
    MS_TRY(tcnt.alloc((size_t)m, s));
    MS_TRY(kmin.alloc((size_t)m, s));
    MS_TRY(kmax.alloc((size_t)m, s));
    MS_TRY(imin.alloc((size_t)m, s));
    MS_TRY(imax.alloc((size_t)m, s));
    unsigned gm = cdiv(m, 256);
    MS_LAUNCH(k_stats_init<uint32_t>, gm, 256, 0, s, tmin.p, tmax.p, st_sum, tcnt.p, m, 0xffffffffu);
    MS_LAUNCH(k_fill_u64, gm, 256, 0, s, kmin.p, ~0ull, imin.p, INT32_MAX, m);
    MS_LAUNCH(k_fill_u64, gm, 256, 0, s, kmax.p, 0ull, imax.p, INT32_MAX, m);
    MS_CUDA(cudaMemsetAsync(ws_count, 0, (size_t)m * sizeof(int64_t), s));
    int64_t want = (n + 255) / 256;
    int blocks = (int)(want > 148 * 16 ? 148 * 16 : want);
    prof_units(n);
    const int tiles_x = (int)cdiv(cols, 64), ntiles = tiles_x * (int)cdiv(rows, 64);
    if (acc) MS_LAUNCH(k_tables_a2<true>, ntiles, 256, 0, s, depths, lab, fnf, accum, ws, (int)rows, (int)cols, tiles_x, nlabels,
                       tmin.p, tmax.p, st_sum, tcnt.p, kmin.p, kmax.p, (unsigned long long *)ws_count, err_dev);
    else MS_LAUNCH(k_tables_a2<false>, ntiles, 256, 0, s, depths, lab, fnf, accum, ws, (int)rows, (int)cols, tiles_x, nlabels,
                   tmin.p, tmax.p, st_sum, tcnt.p, kmin.p, kmax.p, (unsigned long long *)ws_count, err_dev);
    MS_LAUNCH(k_stats_finish<float>, gm, 256, 0, s, tmin.p, tmax.p, tcnt.p, st_min, st_max, st_count, m);
    prof_units(n);
    if (acc) MS_LAUNCH(k_tables_b<true>, blocks, 256, 0, s, lab, fnf, accum, n, nlabels, kmin.p, kmax.p, imin.p, imax.p);
    else MS_LAUNCH(k_tables_b<false>, blocks, 256, 0, s, lab, fnf, accum, n, nlabels, kmin.p, kmax.p, imin.p, imax.p);
    MS_LAUNCH(k_extreme_finish, gm, 256, 0, s, fnf, imin.p, m, (int)cols, 0, pmin_v, pmin_r, pmin_c);
    if (acc) MS_LAUNCH(k_extreme_finish, gm, 256, 0, s, accum, imax.p, m, (int)cols, 1, pmax_v, pmax_r, pmax_c);
    return MS_OK;
}


// Row-band arg-min / arg-max (K8', K8''): phase 1 = the band's extreme value per label (as float64, so the bands'
// tables combine with an ordinary min / max all-reduce); phase 2 = with the global extreme per label, the
// smallest GLOBAL flat index among the band's cells that hold it (combined with a min all-reduce).
__global__ void __launch_bounds__(256) k_key_to_val(const unsigned long long *__restrict__ tkey, double *val, int64_t m,
                                                    int want_max) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= m) return;
    unsigned long long k = tkey[l];
    if (want_max) val[l] = (k == 0ull) ? (double)-INFINITY : okey64_inv(k);
    else val[l] = (k == ~0ull) ? (double)INFINITY : okey64_inv(k);
}

__global__ void __launch_bounds__(256) k_val_to_key(const double *__restrict__ val, unsigned long long *tkey, int *tidx,
                                                    int64_t m) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= m) return;
    tkey[l] = okey64(val[l]);
    tidx[l] = INT32_MAX;
}

__global__ void __launch_bounds__(256) k_idx_global(const int *__restrict__ tidx, int64_t cell_offset, int64_t *idx,
                                                    int64_t m) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l < m) idx[l] = tidx[l] == INT32_MAX ? INT64_MAX : cell_offset + tidx[l];
}

}  // namespace ms

extern "C" {

/* The per-label tables of a band in two fused passes (k_tables_a2 / k_tables_b; see pipeline_tables_dev_impl).
 * Phase A: the band's partial stats, watershed histogram and extreme values (float64, +-inf where the band does not see a
 * label) — combine across bands with min / max / sum all-reduces.  Phase B: with the GLOBAL extremes, the smallest
 * global flat index holding each (INT64_MAX: not in this band) — combine with a min all-reduce. */
int ms_band_tables_a_dev(const float *depths, const int32_t *labels, const double *fnf, const double *accum,
                         const int32_t *wsheds, int64_t n, int64_t cols, int64_t nlabels, double *st_min, double *st_max,
                         double *st_sum, int64_t *st_count, int64_t *ws_count, double *vmin, double *vmax,
                         void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!depths || !labels || !fnf || !accum || !wsheds || !st_min || !st_max || !st_sum || !st_count || !ws_count ||
        !vmin || !vmax || n < 1 || cols < 1 || n % cols || nlabels < 0) {
        set_error("band tables: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t m = nlabels + 1;
    DevBuf<uint32_t> tmin, tmax;
    DevBuf<unsigned long long> tcnt, kmin, kmax;
    DevBuf<int> scratch, err;
    MS_TRY(tmin.alloc((size_t)m, s));
    MS_TRY(tmax.alloc((size_t)m, s));
    MS_TRY(tcnt.alloc((size_t)m, s));
    MS_TRY(kmin.alloc((size_t)m, s));
    MS_TRY(kmax.alloc((size_t)m, s));
    MS_TRY(scratch.alloc((size_t)m, s));
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    unsigned gm = cdiv(m, 256);
    MS_LAUNCH(k_stats_init<uint32_t>, gm, 256, 0, s, tmin.p, tmax.p, st_sum, tcnt.p, m, 0xffffffffu);
    MS_LAUNCH(k_fill_u64, gm, 256, 0, s, kmin.p, ~0ull, scratch.p, INT32_MAX, m);
    MS_LAUNCH(k_fill_u64, gm, 256, 0, s, kmax.p, 0ull, scratch.p, INT32_MAX, m);
    MS_CUDA(cudaMemsetAsync(ws_count, 0, (size_t)m * sizeof(int64_t), s));
    prof_units(n);
    const int64_t rows = n / cols;
    const int tiles_x = (int)cdiv(cols, 64), ntiles = tiles_x * (int)cdiv(rows, 64);
    MS_LAUNCH(k_tables_a2<true>, ntiles, 256, 0, s, depths, labels, fnf, accum, wsheds, (int)rows, (int)cols, tiles_x, nlabels,
              tmin.p, tmax.p, st_sum, tcnt.p, kmin.p, kmax.p, (unsigned long long *)ws_count, err.p);
    MS_LAUNCH(k_stats_finish<float>, gm, 256, 0, s, tmin.p, tmax.p, tcnt.p, st_min, st_max, st_count, m);
    MS_LAUNCH(k_key_to_val, gm, 256, 0, s, kmin.p, vmin, m, 0);
    MS_LAUNCH(k_key_to_val, gm, 256, 0, s, kmax.p, vmax, m, 1);
    return MS_OK;
}

int ms_band_tables_b_dev(const int32_t *labels, const double *fnf, const double *accum, int64_t n, int64_t nlabels,
                         const double *vmin, const double *vmax, int64_t cell_offset, int64_t *idx_min,
                         int64_t *idx_max, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!labels || !fnf || !accum || !vmin || !vmax || !idx_min || !idx_max || n < 1 || nlabels < 0) {
        set_error("band tables: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t m = nlabels + 1;
    DevBuf<unsigned long long> kmin, kmax;
    DevBuf<int> imin, imax;
    MS_TRY(kmin.alloc((size_t)m, s));
    MS_TRY(kmax.alloc((size_t)m, s));
    MS_TRY(imin.alloc((size_t)m, s));
    MS_TRY(imax.alloc((size_t)m, s));
    unsigned gm = cdiv(m, 256);
    MS_LAUNCH(k_val_to_key, gm, 256, 0, s, vmin, kmin.p, imin.p, m);
    MS_LAUNCH(k_val_to_key, gm, 256, 0, s, vmax, kmax.p, imax.p, m);
    int64_t want = (n + 255) / 256;
    int blocks = (int)(want > 148 * 16 ? 148 * 16 : want);
    prof_units(n);
    MS_LAUNCH(k_tables_b<true>, blocks, 256, 0, s, labels, fnf, accum, n, nlabels, kmin.p, kmax.p, imin.p, imax.p);
    MS_LAUNCH(k_idx_global, gm, 256, 0, s, imin.p, cell_offset, idx_min, m);
    MS_LAUNCH(k_idx_global, gm, 256, 0, s, imax.p, cell_offset, idx_max, m);
    return MS_OK;
}

}  // extern "C"

namespace ms {

// ------------------------------------------------------------------------------------------------
// K10.  label.label_count (label.py:169-180, np.bincount) and K9 label.keep_labels (label.py:78-98)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_label_count(const int32_t *__restrict__ lab, int64_t n, int64_t nbins,
                                                     unsigned long long *cnt, int *err) {
    unsigned long long bg = 0;
    int64_t span = (int64_t)gridDim.x * blockDim.x;
    int64_t nround = (n + span - 1) / span;
    for (int64_t it = 0; it < nround; it++) {
        int64_t i = it * span + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        int lbl = -1;
        if (i < n) {
            lbl = lab[i];
            if (lbl < 0 || lbl >= nbins) { *err = 1; lbl = -1; }
        }
        if (lbl == 0) bg++;
        unsigned act = __ballot_sync(0xffffffffu, lbl > 0);
        if (lbl > 0) {
            unsigned g = __match_any_sync(act, lbl);
            if ((int)(__ffs(g) - 1) == (int)(threadIdx.x & 31)) atomicAdd(cnt + lbl, (unsigned long long)__popc(g));
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) bg += __shfl_xor_sync(0xffffffffu, bg, o);
    __shared__ unsigned long long sb[8];
    if ((threadIdx.x & 31) == 0) sb[threadIdx.x >> 5] = bg;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; k++) bg += sb[k];
        if (bg) atomicAdd(cnt, bg);
    }
}

int label_count_dev_impl(const int32_t *lab, int64_t n, int64_t nbins, int64_t *cnt, int *err_dev, cudaStream_t s) {
    if (!lab || !cnt || n < 1 || nbins < 1) { set_error("label_count: bad argument"); return MS_ERR_ARG; }
    MS_CUDA(cudaMemsetAsync(cnt, 0, (size_t)nbins * sizeof(int64_t), s));
    int64_t want = (n + 255) / 256;
    int blocks = (int)(want > 148 * 16 ? 148 * 16 : want);
    MS_LAUNCH(k_label_count, blocks, 256, 0, s, lab, n, nbins, (unsigned long long *)cnt, err_dev);
    return MS_OK;
}

__global__ void __launch_bounds__(256) k_keep_labels(const int32_t *__restrict__ lab, int64_t n,
                                                     const uint8_t *__restrict__ keep, int64_t nkeep,
                                                     uint8_t *__restrict__ out, int *err) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int l = lab[i];
    if (l < 0 || l >= nkeep) { *err = 1; out[i] = 0; return; }
    out[i] = __ldg(keep + l) ? 1 : 0;
}

int keep_labels_dev_impl(const int32_t *lab, int64_t n, const uint8_t *keep, int64_t nkeep, uint8_t *out,
                         int *err_dev, cudaStream_t s) {
    if (!lab || !keep || !out || n < 1 || nkeep < 1) { set_error("keep_labels: bad argument"); return MS_ERR_ARG; }
    MS_LAUNCH(k_keep_labels, cdiv(n, 256), 256, 0, s, lab, n, keep, nkeep, out, err_dev);
    return MS_OK;
}

}  // namespace ms

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
namespace {

struct ErrFlag {
    ms::DevBuf<int> d;
    cudaStream_t s;
    int init(cudaStream_t stream) {
        s = stream;
        MS_TRY(d.alloc(1, s));
        MS_CUDA(cudaMemsetAsync(d.p, 0, sizeof(int), s));
        return MS_OK;
    }
    // synchronises the stream
    int check(const char *what) {
        int64_t *h = ms::host_flags().h;
        MS_TRY(ms::readback(h + 16, d.p, sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        if (*(int *)(h + 16)) {
            ms::set_error("%s: a label lies outside the table", what);
            return MS_ERR_LABEL;
        }
        return MS_OK;
    }
};

size_t dtype_size(int dtype) {
    switch (dtype) {
        case MS_F32: case MS_I32: return 4;
        case MS_F64: case MS_I64: return 8;
        case MS_U8: return 1;
    }
    return 0;
}

}  // namespace

extern "C" {

int ms_connected_components_dev(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols,
                                int64_t *nlabels, void *stream) {
    MS_TRY(ms::ensure_init());
    cudaStream_t s = (cudaStream_t)stream;
    ms::DevBuf<int64_t> tot;
    MS_TRY(tot.alloc(1, s));
    MS_TRY(ms::cc_dev_impl(data, dtype, labels, rows, cols, tot.p, s));
    int64_t *h = ms::host_flags().h;
    MS_TRY(ms::readback(h, tot.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    if (nlabels) *nlabels = h[0];
    return MS_OK;
}

int ms_connected_components(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols,
                            int64_t *nlabels) {
    MS_TRY(ms::ensure_init());
    size_t es = dtype_size(dtype);
    if (!data || !labels || !es || rows < 1 || cols < 1) { ms::set_error("connected_components: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    uint8_t *d = nullptr;
    int32_t *l = nullptr;
    MS_TRY(hc.in((const uint8_t *)data, n * es, s, &d));
    MS_TRY(hc.out(n, &l));
    MS_TRY(ms_connected_components_dev(d, dtype, l, rows, cols, nlabels, s));
    MS_CUDA(cudaMemcpyAsync(labels, l, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(l, labels, n * sizeof(int32_t));
    return MS_OK;
}

int ms_label_range_dev(const int32_t *labels, int64_t n, int32_t *out_minmax_dev2, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!labels || !out_minmax_dev2 || n < 1) { ms::set_error("label_range: bad argument"); return MS_ERR_ARG; }
    return ms::label_range_dev_impl(labels, n, out_minmax_dev2, (cudaStream_t)stream);
}

int ms_label_range(const int32_t *labels, int64_t n, int32_t *out_min, int32_t *out_max) {
    MS_TRY(ms::ensure_init());
    if (!labels || n < 1) { ms::set_error("label_range: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    ms::HostCall hc;
    int32_t *l = nullptr;
    ms::DevBuf<int32_t> o;
    MS_TRY(hc.in(labels, (size_t)n, s, &l));
    MS_TRY(o.alloc(2, s));
    MS_TRY(ms::label_range_dev_impl(l, n, o.p, s));
    int32_t r[2];
    MS_CUDA(cudaMemcpyAsync(r, o.p, sizeof(r), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    if (out_min) *out_min = r[0];
    if (out_max) *out_max = r[1];
    return MS_OK;
}

int ms_label_stats_dev(const void *data, int dtype, const int32_t *labels, int64_t n, int64_t nlabels,
                       double *out_min, double *out_max, double *out_sum, int64_t *out_count, void *stream) {
    MS_TRY(ms::ensure_init());
    ErrFlag ef;
    MS_TRY(ef.init((cudaStream_t)stream));
    return ms::label_stats_dev_impl(data, dtype, labels, n, nlabels, out_min, out_max, out_sum, out_count, ef.d.p,
                                    (cudaStream_t)stream);
}

int ms_label_stats(const void *data, int dtype, const int32_t *labels, int64_t n, int64_t nlabels, double *out_min,
                   double *out_max, double *out_sum, int64_t *out_count) {
    MS_TRY(ms::ensure_init());
    size_t es = dtype_size(dtype);
    if (!data || !labels || (dtype != MS_F32 && dtype != MS_F64) || n < 1 || nlabels < 0) {
        ms::set_error("label_stats: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = nullptr;
    size_t m = (size_t)nlabels + 1;
    ms::HostCall hc;
    uint8_t *d = nullptr;
    int32_t *l = nullptr;
    ms::DevBuf<double> a, b, c;
    ms::DevBuf<int64_t> k;
    MS_TRY(hc.in((const uint8_t *)data, (size_t)n * es, s, &d));
    MS_TRY(hc.in(labels, (size_t)n, s, &l));
    MS_TRY(a.alloc(m, s)); MS_TRY(b.alloc(m, s)); MS_TRY(c.alloc(m, s)); MS_TRY(k.alloc(m, s));
    ErrFlag ef;
    MS_TRY(ef.init(s));
    MS_TRY(ms::label_stats_dev_impl(d, dtype, l, n, nlabels, a.p, b.p, c.p, k.p, ef.d.p, s));
    MS_TRY(ef.check("label_stats"));
    MS_CUDA(cudaMemcpyAsync(out_min, a.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_max, b.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_sum, c.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_count, k.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

int ms_label_extreme_index_dev(const double *data, const int32_t *labels, int64_t rows, int64_t cols,
                               int64_t nlabels, int want_max, double *out_value, int64_t *out_row, int64_t *out_col,
                               void *stream) {
    MS_TRY(ms::ensure_init());
    ErrFlag ef;
    MS_TRY(ef.init((cudaStream_t)stream));
    return ms::label_extreme_dev_impl(data, labels, rows, cols, nlabels, want_max, out_value, out_row, out_col,
                                      ef.d.p, (cudaStream_t)stream);
}

int ms_label_extreme_index(const double *data, const int32_t *labels, int64_t rows, int64_t cols, int64_t nlabels,
                           int want_max, double *out_value, int64_t *out_row, int64_t *out_col) {
    MS_TRY(ms::ensure_init());
    if (!data || !labels || rows < 1 || cols < 1 || nlabels < 0) { ms::set_error("label_min/max_index: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols), m = (size_t)nlabels + 1;
    ms::HostCall hc;
    double *d = nullptr;
    int32_t *l = nullptr;
    ms::DevBuf<double> v;
    ms::DevBuf<int64_t> r, c;
    MS_TRY(hc.in(data, n, s, &d));
    MS_TRY(hc.in(labels, n, s, &l));
    MS_TRY(v.alloc(m, s)); MS_TRY(r.alloc(m, s)); MS_TRY(c.alloc(m, s));
    ErrFlag ef;
    MS_TRY(ef.init(s));
    MS_TRY(ms::label_extreme_dev_impl(d, l, rows, cols, nlabels, want_max, v.p, r.p, c.p, ef.d.p, s));
    MS_TRY(ef.check("label_min/max_index"));
    MS_CUDA(cudaMemcpyAsync(out_value, v.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_row, r.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_col, c.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

int ms_label_count_dev(const int32_t *labels, int64_t n, int64_t nbins, int64_t *out_count, void *stream) {
    MS_TRY(ms::ensure_init());
    ErrFlag ef;
    MS_TRY(ef.init((cudaStream_t)stream));
    return ms::label_count_dev_impl(labels, n, nbins, out_count, ef.d.p, (cudaStream_t)stream);
}

int ms_label_count(const int32_t *labels, int64_t n, int64_t nbins, int64_t *out_count) {
    MS_TRY(ms::ensure_init());
    if (!labels || !out_count || n < 1 || nbins < 1) { ms::set_error("label_count: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    ms::HostCall hc;
    int32_t *l = nullptr;
    ms::DevBuf<int64_t> c;
    MS_TRY(hc.in(labels, (size_t)n, s, &l));
    MS_TRY(c.alloc((size_t)nbins, s));
    ErrFlag ef;
    MS_TRY(ef.init(s));
    MS_TRY(ms::label_count_dev_impl(l, n, nbins, c.p, ef.d.p, s));
    MS_TRY(ef.check("label_count"));
    MS_CUDA(cudaMemcpyAsync(out_count, c.p, (size_t)nbins * 8, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

int ms_keep_labels_dev(const int32_t *labels, int64_t n, const uint8_t *keep, int64_t nkeep, uint8_t *out,
                       void *stream) {
    MS_TRY(ms::ensure_init());
    ErrFlag ef;
    MS_TRY(ef.init((cudaStream_t)stream));
    return ms::keep_labels_dev_impl(labels, n, keep, nkeep, out, ef.d.p, (cudaStream_t)stream);
}

int ms_keep_labels(const int32_t *labels, int64_t n, const uint8_t *keep, int64_t nkeep, uint8_t *out) {
    MS_TRY(ms::ensure_init());
    if (!labels || !keep || !out || n < 1 || nkeep < 1) { ms::set_error("keep_labels: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    ms::HostCall hc;
    int32_t *l = nullptr;
    uint8_t *o = nullptr;
    ms::DevBuf<uint8_t> k;
    MS_TRY(hc.in(labels, (size_t)n, s, &l));
    MS_TRY(hc.out((size_t)n, &o));
    MS_TRY(k.alloc((size_t)nkeep, s));
    MS_CUDA(cudaMemcpyAsync(k.p, keep, (size_t)nkeep, cudaMemcpyHostToDevice, s));
    ErrFlag ef;
    MS_TRY(ef.init(s));
    MS_TRY(ms::keep_labels_dev_impl(l, n, k.p, nkeep, o, ef.d.p, s));
    MS_TRY(ef.check("keep_labels"));
    MS_CUDA(cudaMemcpyAsync(out, o, (size_t)n, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(o, out, (size_t)n);
    return MS_OK;
}

}  // extern "C"
