// network.cu — SURVEY.md §8(f2): Network.rain_event (malstroem/network.py:75-129) on device, every rain event in
// one pass, and the StreamTool + RainTool chain on a finished ms_rasters (streams.py:66-100, rain.py:60-79).
//
// The bluespot network is a forest (node -> downstream node).  The reference walks each root's tree and evaluates
// the nodes leaves first; a node's inflow is Python's sum() over the spill of its upstream nodes in the order they
// were added.  Here:
//   1. upstream lists in insertion order: a stable sort of the node indices by parent (binary split radix sort on
//      the shared exclusive scan, one bit per pass) gives a CSR whose segments are ordered by node index;
//   2. evaluation leaves -> roots without levels: every leaf starts a walker; a node is evaluated by the walker
//      that delivers its last missing upstream value (one atomic countdown per node), which then carries on
//      downstream — the scheme of the flow-accumulation tracer (accum.cu), with the float sums taken in CSR order
//      so the result does not depend on which walker arrives last;
//   3. which nodes the reference reaches at all (those whose downstream chain ends at a root): pointer jumping.
// All arithmetic is float64 in the reference's order (-fmad=false), so results are bit-identical to the reference
// run under the same sum() flavour (sum_mode).
#include <math.h>

#include "common.cuh"

namespace ms {

constexpr int MAX_EVENTS = 16;
struct RainEvents {
    int ne;
    double mm[MAX_EVENTS];
};

__global__ void __launch_bounds__(256) k_net_count(const int32_t *__restrict__ parent, int n, int *cnt, int *bad) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = parent[i];
    if (p >= n || p < -2 || p == i) { *bad = 1; return; }
    if (p >= 0) atomicAdd(&cnt[p], 1);
}

__global__ void __launch_bounds__(256) k_net_keys(const int32_t *__restrict__ parent, int n, int *key, int *val) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = parent[i];
    key[i] = p >= 0 ? p : n;        // nodes without a downstream node sort behind every upstream list
    val[i] = i;
}

__global__ void __launch_bounds__(256) k_net_bitflag(const int *__restrict__ key, int n, int bit, int *flag) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = ((key[i] >> bit) & 1) ^ 1;
}

// stable split: zeros keep their order in front, ones keep theirs behind
__global__ void __launch_bounds__(256) k_net_split(const int *__restrict__ key, const int *__restrict__ val,
                                                   const int *__restrict__ pos0, const int64_t *__restrict__ total0,
                                                   int n, int bit, int *key_out, int *val_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int k = key[i];
    int z = pos0[i];
    int dst = ((k >> bit) & 1) ? (int)*total0 + (i - z) : z;
    key_out[dst] = k;
    val_out[dst] = val[i];
}

int radix_sort_split(int **key, int **val, int **key_alt, int **val_alt, int *flag, int64_t *total, int n, int bits,
                     cudaStream_t s) {
    unsigned g = cdiv(n, 256);
    for (int b = 0; b < bits; b++) {
        MS_LAUNCH(k_net_bitflag, g, 256, 0, s, *key, n, b, flag);
        MS_TRY(exclusive_scan_i32(flag, flag, n, total, s));
        MS_LAUNCH(k_net_split, g, 256, 0, s, *key, *val, flag, total, n, b, *key_alt, *val_alt);
        int *t = *key; *key = *key_alt; *key_alt = t;
        t = *val; *val = *val_alt; *val_alt = t;
    }
    return MS_OK;
}

__global__ void __launch_bounds__(256) k_net_present_ptr(const int32_t *__restrict__ parent, int n, int *ptr) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ptr[i] = parent[i] >= 0 ? parent[i] : i;
}

__global__ void __launch_bounds__(256) k_net_present(const int32_t *__restrict__ parent, const int *__restrict__ ptr,
                                                     int n, uint8_t *present) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) present[i] = parent[ptr[i]] == -1;
}

__global__ void __launch_bounds__(256) k_net_fill_nan(double *a, double *b, double *c, double *d, int64_t m) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double q = __longlong_as_double(0x7ff8000000000000ll);
    a[i] = q; b[i] = q; c[i] = q; d[i] = q;
}

// network.py:75-98 for one node and one event; child spills are final (their walkers fenced before the countdown)
__device__ inline void rain_node(int x, double mm, const double *__restrict__ area, const double *__restrict__ cap,
                                 const int *__restrict__ off, const int *__restrict__ child, int sum_mode,
                                 double *R, double *S, double *V, double *P) {
    double rv = __dmul_rn(__dmul_rn(area[x], mm), 0.001);
    double up = 0.0, comp = 0.0;
    int b = off[x], e = off[x + 1];
    for (int j = b; j < e; j++) {
        double y = __ldcg(&S[child[j]]);
        if (sum_mode == 0) { up = __dadd_rn(up, y); continue; }
        double t = __dadd_rn(up, y);            // Neumaier step, CPython >= 3.12 builtin sum()
        if (fabs(up) >= fabs(y)) comp = __dadd_rn(comp, __dadd_rn(__dsub_rn(up, t), y));
        else comp = __dadd_rn(comp, __dadd_rn(__dsub_rn(y, t), up));
        up = t;
    }
    if (sum_mode == 1 && comp != 0.0 && isfinite(comp)) up = __dadd_rn(up, comp);
    double total = __dadd_rn(rv, up);
    double c = cap[x];
    double filled = c < total ? c : total;                  // min(total, cap)
    double d = __dsub_rn(total, c);
    R[x] = rv;
    S[x] = d > 0.0 ? d : 0.0;                               // max(0, total - cap)
    V[x] = filled;
    P[x] = c != 0.0 ? __ddiv_rn(__dmul_rn(100.0, filled), c) : __longlong_as_double(0x7ff8000000000000ll);
}

__global__ void __launch_bounds__(128) k_net_rain(const int32_t *__restrict__ parent, const double *__restrict__ area,
                                                  const double *__restrict__ cap, const int *__restrict__ off,
                                                  const int *__restrict__ child, int *pending, int n, RainEvents ev,
                                                  int sum_mode, double *rainv, double *spillv, double *v,
                                                  double *pctv) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n || off[x + 1] != off[x]) return;             // walkers start at the leaves
    for (;;) {
        for (int e = 0; e < ev.ne; e++) {
            size_t o = (size_t)e * n;
            rain_node(x, ev.mm[e], area, cap, off, child, sum_mode, rainv + o, spillv + o, v + o, pctv + o);
        }
        int p = parent[x];
        if (p < 0) return;
        __threadfence();
        if (atomicSub(&pending[p], 1) != 1) return;         // someone else still owes p a value
        __threadfence();
        x = p;
    }
}

int rain_events_dev_impl(int64_t n64, const int32_t *parent, const double *area, const double *cap, int64_t ne,
                         const double *mm, int sum_mode, double *rainv, double *spillv, double *v, double *pctv,
                         uint8_t *present, cudaStream_t s) {
    if (n64 < 0 || n64 >= (1ll << 30) || ne < 0 || ne > MAX_EVENTS || (sum_mode != 0 && sum_mode != 1)) {
        set_error("rain_events: unsupported size (n = %lld, events = %lld) or sum_mode", (long long)n64, (long long)ne);
        return MS_ERR_ARG;
    }
    if (n64 == 0 || ne == 0) return MS_OK;
    if (!parent || !area || !cap || !mm || !rainv || !spillv || !v || !pctv) {
        set_error("rain_events: null pointer");
        return MS_ERR_ARG;
    }
    int n = (int)n64;
    unsigned g = cdiv(n, 256);
    DevBuf<int> cnt, off, key, val, key2, val2, flag, bad, ptr;
    DevBuf<int64_t> total;
    MS_TRY(cnt.alloc((size_t)n + 1, s));
    MS_TRY(off.alloc((size_t)n + 1, s));
    MS_TRY(key.alloc((size_t)n, s));
    MS_TRY(val.alloc((size_t)n, s));
    MS_TRY(key2.alloc((size_t)n, s));
    MS_TRY(val2.alloc((size_t)n, s));
    MS_TRY(flag.alloc((size_t)n, s));
    MS_TRY(bad.alloc(1, s));
    MS_TRY(total.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(cnt.p, 0, ((size_t)n + 1) * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
    MS_LAUNCH(k_net_count, g, 256, 0, s, parent, n, cnt.p, bad.p);
    MS_TRY(exclusive_scan_i32(cnt.p, off.p, (int64_t)n + 1, total.p, s));
    // upstream lists in insertion order: stable sort of node indices by parent, one bit per pass
    MS_LAUNCH(k_net_keys, g, 256, 0, s, parent, n, key.p, val.p);
    int bits = 1;
    while ((1ll << bits) <= n) bits++;                      // keys are 0..n
    int *ka = key.p, *va = val.p, *kb = key2.p, *vb = val2.p;
    MS_TRY(radix_sort_split(&ka, &va, &kb, &vb, flag.p, total.p, n, bits, s));
    MS_LAUNCH(k_net_fill_nan, cdiv((int64_t)n * ne, 256), 256, 0, s, rainv, spillv, v, pctv, (int64_t)n * ne);
    int64_t *h = host_flags().h;
    MS_TRY(ms::readback(h, bad.p, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    if (*(int *)h) { set_error("rain_events: parent index outside [-2, n) or a node that is its own parent"); return MS_ERR_ARG; }
    RainEvents ev;
    ev.ne = (int)ne;
    for (int e = 0; e < ev.ne; e++) ev.mm[e] = mm[e];
    prof_units(n);
    MS_LAUNCH(k_net_rain, cdiv(n, 128), 128, 0, s, parent, area, cap, off.p, va, cnt.p, n, ev, sum_mode, rainv, spillv,
              v, pctv);
    if (present) {
        MS_TRY(ptr.alloc((size_t)n, s));
        MS_LAUNCH(k_net_present_ptr, g, 256, 0, s, parent, n, ptr.p);
        int rc = forest_resolve(ptr.p, n, nullptr, s);
        if (rc != MS_OK && rc != MS_ERR_NOCONV) return rc;  // cycles: those nodes never reach a root -> not present
        MS_LAUNCH(k_net_present, g, 256, 0, s, parent, ptr.p, n, present);
    }
    return MS_OK;
}

// ---- StreamTool + RainTool on the pipeline's tables --------------------------------------------------------------
__global__ void __launch_bounds__(256) k_net_tables(const int64_t *__restrict__ down, const uint8_t *__restrict__ found,
                                                    const int64_t *__restrict__ ws_count,
                                                    const double *__restrict__ st_sum, double cell_area, int n,
                                                    int32_t *parent, double *area, double *cap) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    parent[i] = found[i] ? (int32_t)down[i] : -1;
    area[i] = __dmul_rn((double)ws_count[i], cell_area);    // bluespots.py:78  stats[2] * cell_area
    cap[i] = __dmul_rn(st_sum[i], cell_area);               // bluespots.py:77  stats[1]['sum'] * cell_area
}

// ---- row bands (SURVEY.md §8(e) for the §8(f) rows) -----------------------------------------------------------------
// On the D8 surface of the no-flats fill a bluespot's pour point (min of the surface, or max of the accumulated flow,
// over the bluespot) flows out of its bluespot with its first step and never comes back: the surface only falls and
// the accumulation only grows along a path.  So "the first label downstream that is neither mine nor background" is
// the watershed label (K7, already resolved across bands) of the cell the pour point flows into — one lookup, with
// the neighbours' edge rows of the watershed raster as halo.  Each band answers for the pour points it owns
// (everything else INT32_MIN, so a max all-reduce combines the bands); *err is raised if a lookup returns the pour
// point's own label, i.e. the raster is not such a surface (use the single-GPU walker then).
__global__ void __launch_bounds__(256) k_band_pp_parent(const uint8_t *__restrict__ fd, const int32_t *__restrict__ ws,
                                                        const int32_t *__restrict__ ws_above,
                                                        const int32_t *__restrict__ ws_below, int rows, int cols,
                                                        int64_t r0, int64_t R, int64_t n,
                                                        const int64_t *__restrict__ pp_row,
                                                        const int64_t *__restrict__ pp_col, int32_t *parent, int *err) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t r = pp_row[i], c = pp_col[i];
    if (r < r0 || r >= r0 + rows || c < 0 || c >= cols) { parent[i] = INT32_MIN; return; }
    int d = fd[(r - r0) * cols + c];
    int32_t out = -1;
    if (d <= 7) {
        int64_t nr = r + kDR[d], nc = c + kDC[d];
        if (nr >= 0 && nr < R && nc >= 0 && nc < cols) {
            int32_t v;
            if (nr < r0) v = ws_above ? ws_above[nc] : 0;
            else if (nr >= r0 + rows) v = ws_below ? ws_below[nc] : 0;
            else v = ws[(nr - r0) * cols + nc];
            if (v == (int32_t)i && i != 0) *err = 1;
            if (v != 0 && v != (int32_t)i) out = v;
        }
    }
    parent[i] = out;
}

int pp_network_dev_impl(const uint8_t *fd, const void *lab, int label_bytes, int64_t rows, int64_t cols, int64_t np,
                        const int64_t *pp_row, const int64_t *pp_col, int64_t bg, int has_bg, int64_t *down,
                        uint8_t *found, int64_t *path_len, cudaStream_t s);      // flow.cu

}  // namespace ms

extern "C" {

int ms_rain_events_dev(int64_t n, const int32_t *parent, const double *wshed_area, const double *bspot_vol,
                       int64_t n_events, const double *mm, int sum_mode, double *out_rainv, double *out_spillv,
                       double *out_v, double *out_pctv, uint8_t *out_present, void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::rain_events_dev_impl(n, parent, wshed_area, bspot_vol, n_events, mm, sum_mode, out_rainv, out_spillv,
                                    out_v, out_pctv, out_present, (cudaStream_t)stream);
}

int ms_rain_events(int64_t n, const int32_t *parent, const double *wshed_area, const double *bspot_vol,
                   int64_t n_events, const double *mm, int sum_mode, double *out_rainv, double *out_spillv,
                   double *out_v, double *out_pctv, uint8_t *out_present) {
    MS_TRY(ms::ensure_init());
    if (n < 0 || n_events < 0 || n_events > ms::MAX_EVENTS) { ms::set_error("rain_events: bad size"); return MS_ERR_ARG; }
    if (n == 0 || n_events == 0) return MS_OK;
    if (!parent || !wshed_area || !bspot_vol || !mm || !out_rainv || !out_spillv || !out_v || !out_pctv) {
        ms::set_error("rain_events: null pointer");
        return MS_ERR_ARG;
    }
    cudaStream_t s = nullptr;
    size_t m = (size_t)n * (size_t)n_events;
    ms::DevBuf<int32_t> p;
    ms::DevBuf<double> a, c, r, sp, v, pc;
    ms::DevBuf<uint8_t> pr;
    MS_TRY(p.alloc((size_t)n, s));
    MS_TRY(a.alloc((size_t)n, s));
    MS_TRY(c.alloc((size_t)n, s));
    MS_TRY(r.alloc(m, s));
    MS_TRY(sp.alloc(m, s));
    MS_TRY(v.alloc(m, s));
    MS_TRY(pc.alloc(m, s));
    MS_TRY(pr.alloc((size_t)n, s));
    MS_CUDA(cudaMemcpyAsync(p.p, parent, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    MS_CUDA(cudaMemcpyAsync(a.p, wshed_area, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    MS_CUDA(cudaMemcpyAsync(c.p, bspot_vol, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    MS_TRY(ms::rain_events_dev_impl(n, p.p, a.p, c.p, n_events, mm, sum_mode, r.p, sp.p, v.p, pc.p,
                                    out_present ? pr.p : nullptr, s));
    MS_CUDA(cudaMemcpyAsync(out_rainv, r.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_spillv, sp.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_v, v.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_pctv, pc.p, m * 8, cudaMemcpyDeviceToHost, s));
    if (out_present) MS_CUDA(cudaMemcpyAsync(out_present, pr.p, (size_t)n, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

int ms_bluespot_network_dev(const ms_rasters *io, double cell_area, int use_accum_pourpoints, int64_t n_events,
                            const double *mm, int sum_mode, int32_t *out_parent, double *out_rainv,
                            double *out_spillv, double *out_v, double *out_pctv, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!io || !out_parent || !io->flowdir || !io->labels || !io->ws_count || !io->st_sum) {
        ms::set_error("bluespot_network: null pointer");
        return MS_ERR_ARG;
    }
    const int64_t *pr = use_accum_pourpoints ? io->ppmax_row : io->ppmin_row;
    const int64_t *pc = use_accum_pourpoints ? io->ppmax_col : io->ppmin_col;
    if (!pr || !pc) { ms::set_error("bluespot_network: the pour-point table asked for is not part of the run"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    int64_t n = io->nlabels + 1;
    ms::DevBuf<int64_t> down;
    ms::DevBuf<uint8_t> found;
    ms::DevBuf<double> area, cap;
    MS_TRY(down.alloc((size_t)n, s));
    MS_TRY(found.alloc((size_t)n, s));
    MS_TRY(area.alloc((size_t)n, s));
    MS_TRY(cap.alloc((size_t)n, s));
    // streams.py:74: pourpoint_network(flowdir, labeled_bluespots, pourpoints_pix, 0)
    MS_TRY(ms::pp_network_dev_impl(io->flowdir, io->labels, 4, io->rows, io->cols, n, pr, pc, 0, 1, down.p, found.p,
                                   nullptr, s));
    MS_LAUNCH(ms::k_net_tables, ms::cdiv(n, 256), 256, 0, s, down.p, found.p, io->ws_count, io->st_sum, cell_area,
              (int)n, out_parent, area.p, cap.p);
    if (n_events > 0)
        MS_TRY(ms::rain_events_dev_impl(n, out_parent, area.p, cap.p, n_events, mm, sum_mode, out_rainv, out_spillv,
                                        out_v, out_pctv, nullptr, s));
    return MS_OK;
}

int ms_band_pp_parent_dev(const uint8_t *flowdir, const int32_t *wsheds, const int32_t *ws_above, const int32_t *ws_below,
                          int64_t band_rows, int64_t cols, int64_t first_row, int64_t total_rows, int64_t n,
                          const int64_t *pp_row, const int64_t *pp_col, int32_t *out_parent, void *stream) {
    MS_TRY(ms::ensure_init());
    if (!flowdir || !wsheds || !pp_row || !pp_col || !out_parent || band_rows < 1 || cols < 1 || n < 0) {
        ms::set_error("band pour-point network: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    ms::DevBuf<int> err;
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    if (n > 0)
        MS_LAUNCH(ms::k_band_pp_parent, ms::cdiv(n, 256), 256, 0, s, flowdir, wsheds, ws_above, ws_below, (int)band_rows,
                  (int)cols, first_row, total_rows, n, pp_row, pp_col, out_parent, err.p);
    int64_t *h = ms::host_flags().h;
    MS_TRY(ms::readback(h, err.p, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    if (*(int *)h) {
        ms::set_error("band pour-point network: a pour point flows back into its own bluespot (not a no-flats D8 surface)");
        return MS_ERR_ARG;
    }
    return MS_OK;
}

}  // extern "C"
