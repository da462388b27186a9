// flow.cu — K3 D8 flow direction, K4 flow accumulation, K7 local watersheds.
#include <math.h>

#include "common.cuh"

namespace ms {

// ------------------------------------------------------------------------------------------------
// K3.  flow.terrain_flowdirection (flow.py:142-167): interior stencil speedups/_flow.pyx:98-176 —
// dz = z - nbr (edge) or (z - nbr) * INV_SQRT2 (diagonal), float64, strict `>` against a running maximum
// that starts at 0, neighbours visited Up, UpRight, Right, DownRight, Down, DownLeft, Left, UpLeft, so
// the first maximum wins; 8 when no neighbour is lower.  Border rule flow.py:118-139 applied in the
// reference's assignment order (rows, then columns, then corners).
// ------------------------------------------------------------------------------------------------
// `open` (row bands): bit 0 / 1 = the first / last row is not the raster border (a halo row lies beyond it).
__global__ void __launch_bounds__(256) k_flowdir(const double *__restrict__ t, uint8_t *__restrict__ out, int rows,
                                                 int cols, int edges, double inv_sqrt2, int open) {
    int c = blockIdx.x * 64 + (threadIdx.x & 63);
    int r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= rows || c >= cols) return;
    size_t i = (size_t)r * cols + c;
    int code = 8;
    const bool top_border = (r == 0) && !(open & 1), bot_border = (r == rows - 1) && !(open & 2);
    if (!top_border && !bot_border && c >= 1 && c <= cols - 2) {
        const double *p = t + i;
        code = d8_code(*p, __ldg(p - cols), __ldg(p - cols + 1), __ldg(p + 1), __ldg(p + cols + 1), __ldg(p + cols),
                       __ldg(p + cols - 1), __ldg(p - 1), __ldg(p - cols - 1), inv_sqrt2);
    }
    if (edges) code = d8_border(code, top_border, bot_border, c, cols);
    out[i] = (uint8_t)code;
}

int flowdir_dev_impl(const double *t, uint8_t *out, int64_t rows, int64_t cols, int edges, cudaStream_t s,
                     int open) {
    if (!t || !out) { set_error("terrain_flowdirection: null pointer"); return MS_ERR_ARG; }
    if (rows < 1 || cols < 1 || rows * cols > (1ll << 30)) {
        set_error("terrain_flowdirection: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    const double inv_sqrt2 = 1.0 / pow(2.0, 0.5);     // _flow.pyx:93-94: SQRT2 = 2**0.5; INV_SQRT2 = 1 / SQRT2
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    MS_LAUNCH(k_flowdir, g2, 256, 0, s, t, out, (int)rows, (int)cols, edges, inv_sqrt2, open);
    return MS_OK;
}

// ------------------------------------------------------------------------------------------------
// K4 (flow.accumulated_flow) lives in accum.cu; d8_next below is shared with K7.
// ------------------------------------------------------------------------------------------------
__device__ inline bool d8_next(int r, int c, int d, int rows, int cols, int *nr, int *nc) {
    if (d > 7) return false;
    *nr = r + kDR[d];
    *nc = c + kDC[d];
    return *nr >= 0 && *nr < rows && *nc >= 0 && *nc < cols;
}

int accum_dev_impl(const uint8_t *fd, double *acc, int64_t rows, int64_t cols, cudaStream_t s);   // accum.cu

// ------------------------------------------------------------------------------------------------
// K7.  flow.watersheds_from_labels (flow.py:398-412; speedups/_flow.pyx:276-403).  The reference walks
// upstream from every border cell handing down the label of the last labelled cell.  Net effect: an
// `unassigned` cell takes the label of the first labelled cell on its downstream path, provided the
// path ends on the raster border (cells whose path dies at an interior no-direction cell are never
// visited and stay untouched).  Here: ptr = self for labelled / terminal cells, else the downstream
// cell; pointer jumping; gather.  The "path ends on the border" test needs a second forest (pointers
// that do not stop at labels) and is only run when an interior cell with code > 7 exists.
// ------------------------------------------------------------------------------------------------
template <typename L>
__global__ void __launch_bounds__(256) k_ws_ptr(const uint8_t *__restrict__ fd, const L *__restrict__ lab, int *ptr,
                                                int *ptr_full, int *interior_nodir, L unassigned, int rows,
                                                int cols) {
    int c = blockIdx.x * 64 + (threadIdx.x & 63);
    int r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= rows || c >= cols) return;
    int i = r * cols + c;
    int d = fd[i], nr, nc;
    bool moves = d8_next(r, c, d, rows, cols, &nr, &nc);
    int nxt = moves ? nr * cols + nc : i;
    if (ptr) ptr[i] = (lab[i] != unassigned) ? i : nxt;
    if (ptr_full) ptr_full[i] = nxt;
    if (interior_nodir && d > 7 && r > 0 && c > 0 && r < rows - 1 && c < cols - 1) *interior_nodir = 1;
}

// Tile form of k_ws_ptr + most of the pointer jumping (see k_descent_tile): in-tile paths are compressed in shared
// memory; a cell whose path leaves its tile goes on `list` for the global jumps.
// LABELS = false: out = ptr, the first labelled / terminal cell on the path; a listed cell holds the cell it enters
// next.  LABELS = true (labels >= 0, unassigned 0): out = the watershed raster itself - the in-tile root's label, or,
// for a listed cell, -(1 + the cell it enters next), the link encoding of forest_resolve_ids.
template <typename L, bool LABELS>
__global__ void __launch_bounds__(256) k_ws_tile(const uint8_t *__restrict__ fd, const L *__restrict__ lab, int *out,
                                                 int *interior_nodir, L unassigned, int rows, int cols, int tiles_x,
                                                 int *list, int *n_list) {
    __shared__ unsigned short sp[FT * FT];
    __shared__ int tgt[FT * FT];          // per tile-local root: >= 0 final (cell index or label), < 0: -(1 + cell in another tile)
    int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    int r0 = ty * FT, c0 = tx * FT, tid = threadIdx.x;
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        unsigned short p = (unsigned short)k;
        int t = 0;
        if (r < rows && c < cols) {
            int i = r * cols + c;
            const L v = lab[i];
            t = LABELS ? (int)v : i;
            int d = fd[i], nr, nc;
            if (interior_nodir && d > 7 && r > 0 && c > 0 && r < rows - 1 && c < cols - 1) *interior_nodir = 1;
            if (v == unassigned && d8_next(r, c, d, rows, cols, &nr, &nc)) {
                int tr = nr - r0, tc = nc - c0;
                if (tr >= 0 && tr < FT && tc >= 0 && tc < FT) p = (unsigned short)(tr * FT + tc);
                else t = -(1 + nr * cols + nc);
            }
        }
        sp[k] = p;
        tgt[k] = t;
    }
    __syncthreads();
    tile_pointer_double(sp);
    int mine[16], cnt = 0;
#pragma unroll 4
    for (int u = 0; u < 16; u++) {
        int k = tid + 256 * u;
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        mine[u] = -1;
        if (r < rows && c < cols) {
            int t = tgt[sp[k]];
            int i = r * cols + c;
            if (t < 0) {
                mine[u] = i;
                cnt++;
                if (!LABELS) t = -(t + 1);
            }
            out[i] = t;
        }
    }
    int pos = block_append_pos(cnt, n_list);
#pragma unroll 4
    for (int u = 0; u < 16; u++)
        if (mine[u] >= 0) list[pos++] = mine[u];
}

// LABELS = false: ptr[i] = the first labelled / terminal cell on i's path.  LABELS = true: out = the watershed labels
// (see k_ws_tile).  `nodir_flag` (optional) comes back in host_flags().h[8].
template <typename L, bool LABELS>
static int ws_resolve(const uint8_t *fd, const L *lab, int *out, int *nodir_flag, L unassigned, int64_t rows,
                      int64_t cols, int64_t *rounds_out, cudaStream_t s) {
    int64_t n = rows * cols;
    DevBuf<int> list, cnt;
    MS_TRY(list.alloc((size_t)n, s));
    MS_TRY(cnt.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(int), s));
    int tiles_x = (int)cdiv(cols, FT), tiles_y = (int)cdiv(rows, FT);
    prof_units(n);
    MS_LAUNCH((k_ws_tile<L, LABELS>), tiles_x * tiles_y, 256, 0, s, fd, lab, out, nodir_flag, unassigned, (int)rows,
              (int)cols, tiles_x, list.p, cnt.p);
    int64_t *h = host_flags().h;
    MS_TRY(ms::readback(h, cnt.p, sizeof(int), s));
    if (nodir_flag) MS_TRY(ms::readback(h + 8, nodir_flag, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    if (LABELS) return forest_resolve_ids(out, list.p, *(int *)h, rounds_out, s);
    return forest_resolve_list(out, list.p, *(int *)h, rounds_out, s);
}

template <typename L>
__global__ void __launch_bounds__(256) k_ws_assign(L *lab, const int *__restrict__ ptr,
                                                   const int *__restrict__ ptr_full, int64_t n, int rows, int cols) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int root = ptr[i];
    if (root == (int)i) return;
    if (ptr_full) {
        int t = ptr_full[i];
        int tr = t / cols, tc = t - tr * cols;
        if (!(tr == 0 || tc == 0 || tr == rows - 1 || tc == cols - 1)) return;
    }
    lab[i] = lab[root];     // roots never change, non-roots are never read: in place is safe
}

template <typename L>
int watersheds_dev_t(const uint8_t *fd, L *lab, int64_t rows, int64_t cols, L unassigned, int64_t *stats,
                     cudaStream_t s) {
    int64_t n = rows * cols;
    DevBuf<int> ptr, ptr_full, flag;
    MS_TRY(ptr.alloc((size_t)n, s));
    MS_TRY(flag.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    int64_t *h = host_flags().h;
    int64_t rounds = 0;
    MS_TRY((ws_resolve<L, false>(fd, lab, ptr.p, flag.p, unassigned, rows, cols, &rounds, s)));     // synchronises: h[8] is valid
    bool general = *(int *)(h + 8) != 0;
    if (general) {
        MS_TRY(ptr_full.alloc((size_t)n, s));
        MS_LAUNCH(k_ws_ptr<L>, g2, 256, 0, s, fd, lab, (int *)nullptr, ptr_full.p, (int *)nullptr, unassigned,
                  (int)rows, (int)cols);
        MS_TRY(forest_resolve(ptr_full.p, n, nullptr, s));
    }
    MS_LAUNCH(k_ws_assign<L>, cdiv(n, 256), 256, 0, s, lab, ptr.p, general ? ptr_full.p : (int *)nullptr, n,
              (int)rows, (int)cols);
    if (stats) stats[6] = rounds;
    return MS_OK;
}

int watersheds_dev_impl(const uint8_t *fd, void *lab, int label_bytes, int64_t rows, int64_t cols,
                        int64_t unassigned, int64_t *stats, cudaStream_t s) {
    if (!fd || !lab) { set_error("watersheds_from_labels: null pointer"); return MS_ERR_ARG; }
    if (rows < 1 || cols < 1 || rows * cols > (1ll << 30)) {
        set_error("watersheds_from_labels: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    if (label_bytes == 4) return watersheds_dev_t<int32_t>(fd, (int32_t *)lab, rows, cols, (int32_t)unassigned, stats, s);
    if (label_bytes == 8) return watersheds_dev_t<int64_t>(fd, (int64_t *)lab, rows, cols, unassigned, stats, s);
    set_error("watersheds_from_labels: label_bytes must be 4 or 8");
    return MS_ERR_ARG;
}

// The pipeline's K7 (labels int32 >= 0, unassigned 0): the tile pass reads `lab` and writes the watershed raster `ws`
// directly, and only the cells whose path leaves their tile are resolved afterwards - no copy of the labels, no ptr
// raster and no pass over every cell to gather lab[root].  A path can only end at an interior cell without a flow
// direction on a DEM with NaNs (the fallback D8); then the general form runs again from the untouched labels.
int watersheds_labels_dev_impl(const uint8_t *fd, const int32_t *lab, int32_t *ws, int64_t rows, int64_t cols,
                               int64_t *stats, cudaStream_t s) {
    if (!fd || !lab || !ws) { set_error("watersheds: null pointer"); return MS_ERR_ARG; }
    if (rows < 1 || cols < 1 || rows * cols > (1ll << 30)) {
        set_error("watersheds: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    DevBuf<int> flag;
    MS_TRY(flag.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
    int64_t rounds = 0;
    MS_TRY((ws_resolve<int32_t, true>(fd, lab, ws, flag.p, 0, rows, cols, &rounds, s)));     // h[8] is valid
    if (*(int *)(host_flags().h + 8)) {
        MS_CUDA(cudaMemcpyAsync(ws, lab, (size_t)(rows * cols) * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        return watersheds_dev_t<int32_t>(fd, ws, rows, cols, 0, stats, s);
    }
    if (stats) stats[6] = rounds;
    return MS_OK;
}


// ------------------------------------------------------------------------------------------------
// Row-band watersheds (SURVEY.md §8(e), K7).  Inside the band a path that leaves through an open band edge ends at
// a "band exit" root.  Phase 1 reports, for every cell of the first / last own row, what its path resolves to: a
// label, nothing (0), or "whatever band exit (side, col) resolves to"; and where each exit enters the neighbour.
// The host side chains these across bands (chain_resolve).  Phase 2 writes the labels, taking exit_label[] for
// cells whose root is an unlabelled band exit.  Only the int32, unassigned-label form with every path ending on
// the raster border is supported in band mode (the D8 surface of the no-flats fill has no interior sinks).
// ------------------------------------------------------------------------------------------------
__device__ inline bool band_exit_side(const uint8_t *fd, int i, int rows, int cols, int open, int *side, int *to) {
    int r = i / cols, c = i - r * cols;
    int d = fd[i];
    if (d > 7) return false;
    int nr = r + kDR[d], nc = c + kDC[d];
    if (nc < 0 || nc >= cols) return false;
    if (nr < 0 && (open & 1)) { *side = 0; *to = nc; return true; }
    if (nr >= rows && (open & 2)) { *side = 1; *to = nc; return true; }
    return false;
}

__global__ void __launch_bounds__(256) k_ws_band_out(const uint8_t *__restrict__ fd, const int32_t *__restrict__ lab,
                                                     const int *__restrict__ ptr, int32_t unassigned, int rows,
                                                     int cols, int open, int32_t *edge_res, int32_t *exit_to) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= 2 * cols) return;
    int side = k / cols, c = k - side * cols;
    int res = 0, to = -1;
    if (open & (1 << side)) {
        int i = (side ? rows - 1 : 0) * cols + c;
        int s2, t2;
        if (band_exit_side(fd, i, rows, cols, open, &s2, &t2) && s2 == side) to = t2;
        int root = ptr[i];
        int32_t v = lab[root];
        if (v != unassigned) res = v;
        else if (band_exit_side(fd, root, rows, cols, open, &s2, &t2)) res = -(1 + s2 * cols + (root % cols));
        else res = 0;
    }
    edge_res[k] = res;
    exit_to[k] = to;
}

__global__ void __launch_bounds__(256) k_chain_resolve(const int32_t *__restrict__ arr, int32_t *out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t v = arr[i];
    for (int guard = 0; v < 0 && guard < n; guard++) v = arr[-(v + 1)];
    out[i] = v < 0 ? 0 : v;
}

__global__ void __launch_bounds__(256) k_ws_assign_band(const uint8_t *__restrict__ fd, int32_t *lab,
                                                        const int *__restrict__ ptr, int32_t unassigned, int64_t n,
                                                        int rows, int cols, int open,
                                                        const int32_t *__restrict__ exit_label) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (lab[i] != unassigned && ptr[i] == (int)i) return;      // labelled cells are their own roots
    int root = ptr[i];
    int32_t v = lab[root];
    if (v == unassigned) {
        int s2, t2;
        if (band_exit_side(fd, root, rows, cols, open, &s2, &t2)) v = exit_label[s2 * cols + (root % cols)];
        else if (root == (int)i) return;                        // unlabelled terminal: stays as it is
    }
    if (root != (int)i || v != unassigned) lab[i] = v;
}

}  // namespace ms

extern "C" {

int ms_band_ws_local_dev(ms_band *B, const uint8_t *fd, const int32_t *labelled, int32_t unassigned, int32_t *edge_res,
                         int32_t *exit_to, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !fd || !labelled || !edge_res || !exit_to) { set_error("band watersheds: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t rows = B->rows, cols = B->cols, n = rows * cols;
    int *ptr = (int *)band_buf(B, BB_WS_PTR, (size_t)n * sizeof(int));
    if (!ptr) return MS_ERR_CUDA;
    DevBuf<int> flag;
    MS_TRY(flag.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
    int64_t *h = host_flags().h;
    MS_TRY((ws_resolve<int32_t, false>(fd, labelled, ptr, flag.p, unassigned, rows, cols, nullptr, s)));
    if (*(int *)(h + 8)) {
        set_error("band watersheds: an interior cell without flow direction (band mode needs every path to end on "
                  "the raster border)");
        return MS_ERR_ARG;
    }
    MS_LAUNCH(k_ws_band_out, cdiv(2 * cols, 256), 256, 0, s, fd, labelled, (const int *)ptr, unassigned, (int)rows,
              (int)cols, B->open, edge_res, exit_to);
    return MS_OK;
}

/* arr[i] >= 0: final value; arr[i] < 0: same as entry -(arr[i] + 1).  out[i] = the final value the chain ends at */
int ms_chain_resolve_dev(int64_t n, const int32_t *arr, int32_t *out, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (n < 0 || (n && (!arr || !out))) { set_error("chain_resolve: bad argument"); return MS_ERR_ARG; }
    if (n) MS_LAUNCH(k_chain_resolve, cdiv(n, 256), 256, 0, (cudaStream_t)stream, arr, out, (int)n);
    return MS_OK;
}

int ms_band_ws_finish_dev(ms_band *B, const uint8_t *fd, int32_t *labelled, int32_t unassigned,
                          const int32_t *exit_label, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !fd || !labelled || !B->buf[BB_WS_PTR] || (B->open && !exit_label)) { set_error("band watersheds: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t n = B->rows * B->cols;
    MS_LAUNCH(k_ws_assign_band, cdiv(n, 256), 256, 0, s, fd, labelled, (const int *)B->buf[BB_WS_PTR], unassigned, n,
              (int)B->rows, (int)B->cols, B->open, exit_label);
    return MS_OK;
}

int ms_flowdir_dev(const double *terrain, uint8_t *flowdir, int64_t rows, int64_t cols, int edges_flow_outward,
                   void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::flowdir_dev_impl(terrain, flowdir, rows, cols, edges_flow_outward, (cudaStream_t)stream, 0);
}

int ms_band_flowdir_dev(ms_band *B, const double *terrain, uint8_t *flowdir, int edges_flow_outward, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!B) { ms::set_error("band flowdir: null context"); return MS_ERR_ARG; }
    return ms::flowdir_dev_impl(terrain, flowdir, B->rows, B->cols, edges_flow_outward, (cudaStream_t)stream, B->open);
}

int ms_flowdir(const double *terrain, uint8_t *flowdir, int64_t rows, int64_t cols, int edges_flow_outward) {
    MS_TRY(ms::ensure_init());
    if (!terrain || !flowdir || rows < 1 || cols < 1) { ms::set_error("terrain_flowdirection: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    double *t = nullptr;
    uint8_t *o = nullptr;
    MS_TRY(hc.in(terrain, n, s, &t));
    MS_TRY(hc.out(n, &o));
    MS_TRY(ms::flowdir_dev_impl(t, o, rows, cols, edges_flow_outward, s, 0));
    MS_CUDA(cudaMemcpyAsync(flowdir, o, n, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(o, flowdir, n);
    return MS_OK;
}

int ms_accumulated_flow_dev(const uint8_t *flowdir, double *accum, int64_t rows, int64_t cols, void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::accum_dev_impl(flowdir, accum, rows, cols, (cudaStream_t)stream);
}

int ms_accumulated_flow(const uint8_t *flowdir, double *accum, int64_t rows, int64_t cols) {
    MS_TRY(ms::ensure_init());
    if (!flowdir || !accum || rows < 1 || cols < 1) { ms::set_error("accumulated_flow: bad argument"); return MS_ERR_ARG; }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    uint8_t *f = nullptr;
    double *a = nullptr;
    MS_TRY(hc.in(flowdir, n, s, &f));
    MS_TRY(hc.out(n, &a));
    MS_TRY(ms::accum_dev_impl(f, a, rows, cols, s));
    MS_CUDA(cudaMemcpyAsync(accum, a, n * sizeof(double), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(a, accum, n * sizeof(double));
    return MS_OK;
}

int ms_watersheds_from_labels_dev(const uint8_t *flowdir, void *labelled, int label_bytes, int64_t rows,
                                  int64_t cols, int64_t unassigned, void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::watersheds_dev_impl(flowdir, labelled, label_bytes, rows, cols, unassigned, nullptr,
                                   (cudaStream_t)stream);
}

int ms_watersheds_from_labels(const uint8_t *flowdir, void *labelled, int label_bytes, int64_t rows, int64_t cols,
                              int64_t unassigned) {
    MS_TRY(ms::ensure_init());
    if (!flowdir || !labelled || rows < 1 || cols < 1 || (label_bytes != 4 && label_bytes != 8)) {
        ms::set_error("watersheds_from_labels: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    uint8_t *f = nullptr, *l = nullptr;
    MS_TRY(hc.in(flowdir, n, s, &f));
    MS_TRY(hc.in((const uint8_t *)labelled, n * label_bytes, s, &l));
    // in place, on the device twin as on the host array (flow.py:398-412 mutates `labelled`)
    MS_TRY(ms::watersheds_dev_impl(f, l, label_bytes, rows, cols, unassigned, nullptr, s));
    MS_CUDA(cudaMemcpyAsync(labelled, l, n * label_bytes, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(l, labelled, n * label_bytes);
    return MS_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// SURVEY.md §8(f1).  net.pourpoint_network / net.next_downstream_label (net.py:142-192): from each pour point walk
// downstream (flow.trace_downstream, flow.py:279-301) to the first cell whose label is neither the start cell's nor
// the background.  That is K7 evaluated at the pour points: with a background label the walk uses K7's compressed
// forest (ptr = first non-background or terminal cell at or below a cell), so a step through any stretch of
// background costs one load; only stretches inside the pour point's own bluespot are walked cell by cell.
// Geometry wanted: the plain walk, once to count the cells and once to write them.
// ------------------------------------------------------------------------------------------------
namespace ms {

template <typename L, bool USE_PTR>
__global__ void __launch_bounds__(128) k_pp_downstream(const uint8_t *__restrict__ fd, const L *__restrict__ lab,
                                                       const int *__restrict__ ptr, int rows, int cols, int64_t np,
                                                       const int64_t *__restrict__ pp_row,
                                                       const int64_t *__restrict__ pp_col, L bg, int has_bg,
                                                       int64_t *down, uint8_t *found, int64_t *path_len,
                                                       const int64_t *__restrict__ path_off, int64_t *path_cells,
                                                       int *err) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= np) return;
    int r = (int)pp_row[k], c = (int)pp_col[k];
    int64_t steps = 0, limit = (int64_t)rows * cols;
    int64_t out = 0;
    uint8_t ok = 0;
    if (r >= 0 && r < rows && c >= 0 && c < cols) {
        int i = r * cols + c;
        const L src = lab[i];
        int64_t *pc = path_cells ? path_cells + path_off[k] : nullptr;
        if (pc) pc[0] = i;
        steps = 1;
        for (;;) {
            int nr, nc;
            if (!d8_next(r, c, fd[i], rows, cols, &nr, &nc)) break;
            i = nr * cols + nc;
            if (USE_PTR) {
                i = ptr[i];                     // skips background cells; identity for labelled / terminal cells
                nr = i / cols;
                nc = i - nr * cols;
            }
            r = nr;
            c = nc;
            if (pc) pc[steps] = i;
            steps++;
            L l = lab[i];
            if (l != src && !(has_bg && l == bg)) { out = (int64_t)l; ok = 1; break; }
            if (steps > limit) { *err = 1; break; }
        }
    }
    if (down) { down[k] = out; found[k] = ok; }
    if (path_len) path_len[k] = steps;
}

template <typename L>
static int pp_network_t(const uint8_t *fd, const L *lab, int64_t rows, int64_t cols, int64_t np, const int64_t *pp_row,
                        const int64_t *pp_col, int64_t bg, int has_bg, int64_t *down, uint8_t *found,
                        int64_t *path_len, cudaStream_t s) {
    int64_t n = rows * cols;
    DevBuf<int> err, ptr;
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    unsigned grid = cdiv(np, 128);
    if (np > 0) {
        // the forest pays off when there are many pour points; a handful (or a wanted geometry) walk cell by cell
        bool forest = has_bg && !path_len && np >= 64;
        if (forest) {
            MS_TRY(ptr.alloc((size_t)n, s));
            MS_TRY((ws_resolve<L, false>(fd, lab, ptr.p, nullptr, (L)bg, rows, cols, nullptr, s)));
            prof_units(np);
            MS_LAUNCH((k_pp_downstream<L, true>), grid, 128, 0, s, fd, lab, ptr.p, (int)rows, (int)cols, np, pp_row,
                      pp_col, (L)bg, has_bg, down, found, path_len, (const int64_t *)nullptr, (int64_t *)nullptr,
                      err.p);
        } else {
            prof_units(np);
            MS_LAUNCH((k_pp_downstream<L, false>), grid, 128, 0, s, fd, lab, (const int *)nullptr, (int)rows,
                      (int)cols, np, pp_row, pp_col, (L)bg, has_bg, down, found, path_len, (const int64_t *)nullptr,
                      (int64_t *)nullptr, err.p);
        }
    }
    int64_t *h = host_flags().h;
    MS_TRY(ms::readback(h, err.p, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    if (*(int *)h) { set_error("pourpoint_network: cyclic flow directions"); return MS_ERR_NOCONV; }
    return MS_OK;
}

int pp_network_dev_impl(const uint8_t *fd, const void *lab, int label_bytes, int64_t rows, int64_t cols, int64_t np,
                        const int64_t *pp_row, const int64_t *pp_col, int64_t bg, int has_bg, int64_t *down,
                        uint8_t *found, int64_t *path_len, cudaStream_t s) {
    if (!fd || !lab || (np > 0 && (!pp_row || !pp_col || !down || !found))) {
        set_error("pourpoint_network: null pointer");
        return MS_ERR_ARG;
    }
    if (rows < 1 || cols < 1 || rows * cols > (1ll << 30) || np < 0) {
        set_error("pourpoint_network: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    if (label_bytes == 4)
        return pp_network_t<int32_t>(fd, (const int32_t *)lab, rows, cols, np, pp_row, pp_col, bg, has_bg, down, found,
                                     path_len, s);
    if (label_bytes == 8)
        return pp_network_t<int64_t>(fd, (const int64_t *)lab, rows, cols, np, pp_row, pp_col, bg, has_bg, down, found,
                                     path_len, s);
    set_error("pourpoint_network: label_bytes must be 4 or 8");
    return MS_ERR_ARG;
}

template <typename L>
static int pp_paths_t(const uint8_t *fd, const L *lab, int64_t rows, int64_t cols, int64_t np, const int64_t *pp_row,
                      const int64_t *pp_col, int64_t bg, int has_bg, const int64_t *off, int64_t *cells,
                      cudaStream_t s) {
    DevBuf<int> err;
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    MS_LAUNCH((k_pp_downstream<L, false>), cdiv(np, 128), 128, 0, s, fd, lab, (const int *)nullptr, (int)rows,
              (int)cols, np, pp_row, pp_col, (L)bg, has_bg, (int64_t *)nullptr, (uint8_t *)nullptr,
              (int64_t *)nullptr, off, cells, err.p);
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_pourpoint_network_dev(const uint8_t *flowdir, const void *labelled, int label_bytes, int64_t rows,
                             int64_t cols, int64_t n_pp, const int64_t *pp_row, const int64_t *pp_col,
                             int64_t background, int has_background, int64_t *out_down, uint8_t *out_found,
                             void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::pp_network_dev_impl(flowdir, labelled, label_bytes, rows, cols, n_pp, pp_row, pp_col, background,
                                   has_background, out_down, out_found, nullptr, (cudaStream_t)stream);
}

int ms_pourpoint_network(const uint8_t *flowdir, const void *labelled, int label_bytes, int64_t rows, int64_t cols,
                         int64_t n_pp, const int64_t *pp_row, const int64_t *pp_col, int64_t background,
                         int has_background, int64_t *out_down, uint8_t *out_found, int64_t *out_path_offsets,
                         int64_t *out_path_cells, int64_t path_capacity) {
    MS_TRY(ms::ensure_init());
    if (!flowdir || !labelled || rows < 1 || cols < 1 || n_pp < 0 || (label_bytes != 4 && label_bytes != 8) ||
        (n_pp > 0 && (!pp_row || !pp_col || !out_down || !out_found))) {
        ms::set_error("pourpoint_network: bad argument");
        return MS_ERR_ARG;
    }
    if (rows * cols > (1ll << 30)) { ms::set_error("pourpoint_network: raster too large"); return MS_ERR_SHAPE; }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols), np = (size_t)n_pp;
    ms::DevBuf<uint8_t> f, l, fnd;
    ms::DevBuf<int64_t> pr, pc, dn, plen;
    MS_TRY(f.alloc(n, s));
    MS_TRY(l.alloc(n * label_bytes, s));
    MS_TRY(pr.alloc(np, s));
    MS_TRY(pc.alloc(np, s));
    MS_TRY(dn.alloc(np, s));
    MS_TRY(fnd.alloc(np, s));
    MS_CUDA(cudaMemcpyAsync(f.p, flowdir, n, cudaMemcpyHostToDevice, s));
    MS_CUDA(cudaMemcpyAsync(l.p, labelled, n * label_bytes, cudaMemcpyHostToDevice, s));
    if (np) {
        MS_CUDA(cudaMemcpyAsync(pr.p, pp_row, np * 8, cudaMemcpyHostToDevice, s));
        MS_CUDA(cudaMemcpyAsync(pc.p, pp_col, np * 8, cudaMemcpyHostToDevice, s));
    }
    if (out_path_offsets) MS_TRY(plen.alloc(np, s));
    MS_TRY(ms::pp_network_dev_impl(f.p, l.p, label_bytes, rows, cols, n_pp, pr.p, pc.p, background, has_background,
                                   dn.p, fnd.p, out_path_offsets ? plen.p : nullptr, s));
    if (np) {
        MS_CUDA(cudaMemcpyAsync(out_down, dn.p, np * 8, cudaMemcpyDeviceToHost, s));
        MS_CUDA(cudaMemcpyAsync(out_found, fnd.p, np, cudaMemcpyDeviceToHost, s));
    }
    if (out_path_offsets) {
        // lengths -> offsets on the host (n_pp is the number of bluespots, not of cells)
        if (np) MS_CUDA(cudaMemcpyAsync(out_path_offsets + 1, plen.p, np * 8, cudaMemcpyDeviceToHost, s));
        MS_TRY(ms::stream_sync(s));
        out_path_offsets[0] = 0;
        for (size_t k = 0; k < np; k++) out_path_offsets[k + 1] += out_path_offsets[k];
        int64_t total = out_path_offsets[np];
        if (np && total > 0 && total <= path_capacity && out_path_cells) {
            ms::DevBuf<int64_t> off, cells;
            MS_TRY(off.alloc(np + 1, s));
            MS_TRY(cells.alloc((size_t)total, s));
            MS_CUDA(cudaMemcpyAsync(off.p, out_path_offsets, (np + 1) * 8, cudaMemcpyHostToDevice, s));
            if (label_bytes == 4)
                MS_TRY(ms::pp_paths_t<int32_t>(f.p, (const int32_t *)l.p, rows, cols, n_pp, pr.p, pc.p, background,
                                               has_background, off.p, cells.p, s));
            else
                MS_TRY(ms::pp_paths_t<int64_t>(f.p, (const int64_t *)l.p, rows, cols, n_pp, pr.p, pc.p, background,
                                               has_background, off.p, cells.p, s));
            MS_CUDA(cudaMemcpyAsync(out_path_cells, cells.p, (size_t)total * 8, cudaMemcpyDeviceToHost, s));
        }
    }
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

}  // extern "C"
