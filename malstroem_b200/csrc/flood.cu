// flood.cu — bluespot water levels after rain events and the water-depth raster of one event (DESIGN.md §4, "water levels").
//
// Level-pool approximation: the water a bluespot stores is one flat surface at level h with volume
// ca * sum_c max(0, h - z_c); that ignores that separate sub-pits of one bluespot may fill one after another.
// With the bluespot's values sorted, z_(1) <= ... <= z_(n), and S_j their prefix sums, the volume at h = z_(j) is
// ca * (j z_(j) - S_j), so the level of a volume v < cap is h = (T + S_k) / k, T = v / ca, k the last breakpoint
// at or below T.  The work is a segmented sort + scan over the wet cells:
//   1. group: cells per label (one atomic per run of one label), an exclusive scan to segment offsets, and a scatter
//      of every bluespot cell's order-preserving z key into its label's segment (one position reservation per run);
//      the same two passes check that the plain fill F is uniform over each label and record it (L_l);
//   2. labels whose every event is full, NaN or empty are answered from the counts (no sort);
//   3. the others are sorted and scanned by segment size: up to SEG_WARP cells one warp, up to SEG_CTA cells one CTA,
//      both in shared memory; larger segments ("lakes") go through the split radix sort of network.cu keyed on
//      (segment, z), then scanned in global memory by one CTA per 4096-cell chunk of a segment, the chunk sums of a
//      segment added in chunk order into per-chunk carries;
//   4. per event a binary search for k, and one for the wet count #{z < h}.
// Each segment's sorted values are identical bits whatever order the scatter's atomics took, and every float64 sum
// is taken in an order fixed by the segment's size, so levels and rasters are bitwise reproducible.
#include <math.h>

#include "common.cuh"

namespace ms {

constexpr int FL_CELLS = 16;      // consecutive cells per thread in the grouping passes
constexpr int SEG_WARP = 512;     // segments up to this size: one warp each
constexpr int SEG_CTA = 8192;     // up to this size: one CTA each; larger: global sort
constexpr int WARPS_A = 4;        // warps per CTA of the one-warp-per-segment kernel
constexpr int T_B = 256;          // threads of the one-CTA-per-segment kernels
constexpr int CHUNK_C = T_B * 16; // cells per scan chunk of a large segment
enum { FE_LABEL = MS_FLOOD_LABEL, FE_UNIFORM = MS_FLOOD_UNIFORM, FE_VOLUME = MS_FLOOD_VOLUME };
enum { CTL_ERR, CTL_NA, CTL_NB, CTL_NC, CTL_CELLS_C, CTL_N };

__device__ inline double zval(uint32_t k) { return (double)okey32_inv(k); }
__device__ inline double qnan() { return __longlong_as_double(0x7ff8000000000000ll); }

// Pass 1 (SCATTER = false): cnt[l] += cells of l (one atomic per run of one label among a thread's 16 cells), lkey[l]
// = okey32(F) of the label (a plain store: all writers of a uniform label store the same bits).  Pass 2 (SCATTER =
// true, cnt zeroed again): every cell of l > 0 writes okey32(z) into segment l, and is checked against lkey[l].
// Labels above `nlabels` are errors.  On a band, labels l <= lo belong to a lower band: pass 2 writes their cells to
// `send` at off[l] instead (the whole raster: lo = 0).
template <bool SCATTER>
__global__ void __launch_bounds__(256) k_flood_group(const int32_t *__restrict__ lab, const float *__restrict__ fil,
                                                     const float *__restrict__ dem, int64_t n, int64_t nlabels,
                                                     int *cnt, uint32_t *lkey, const int *__restrict__ off,
                                                     uint32_t *seg, int64_t lo, uint32_t *send, int *ctl) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * FL_CELLS;
    if (i0 >= n) return;
    const int m = n - i0 < FL_CELLS ? (int)(n - i0) : FL_CELLS;
    int err = 0;
    int a = __ldg(lab + i0);
    for (int j = 0; j < m;) {
        int e = j + 1, b = a;
        while (e < m && (b = __ldg(lab + i0 + e)) == a) e++;
        if (a < 0 || a > nlabels) {
            err |= FE_LABEL;
        } else if (a > 0) {
            if (!SCATTER) {
                const uint32_t k0 = okey32(__ldg(fil + i0 + j));
                for (int q = j + 1; q < e; q++)
                    if (okey32(__ldg(fil + i0 + q)) != k0) err |= FE_UNIFORM;
                atomicAdd(cnt + a, e - j);
                lkey[a] = k0;
            } else {
                const uint32_t L = lkey[a];
                uint32_t *dst = (a > lo ? seg : send) + off[a] + atomicAdd(cnt + a, e - j) - j;
                for (int q = j; q < e; q++) {
                    if (okey32(__ldg(fil + i0 + q)) != L) err |= FE_UNIFORM;
                    dst[q] = okey32(__ldg(dem + i0 + q));
                }
            }
        }
        a = b;
        j = e;
    }
    if (err) atomicOr(ctl + CTL_ERR, err);
}

// Labels l0 <= l < l1 every event of which is answered without the values (v NaN, full, or no cells; label 0) get
// their levels here; the rest go to the list of their size class.
__global__ void __launch_bounds__(256) k_flood_classify(const int *__restrict__ off, const uint32_t *__restrict__ lkey,
                                                        const double *__restrict__ st_sum, double ca,
                                                        const double *__restrict__ v, int nl1, int ne, int l0, int l1,
                                                        double *level, int64_t *wet, int *list_a, int *list_b,
                                                        int *list_c, int *size_c, int *ctl) {
    const int l = l0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= l1) return;
    const int cnt = off[l + 1] - off[l];
    const double L = cnt ? zval(lkey[l]) : qnan();
    const double cap = __dmul_rn(st_sum[l], ca);
    bool need = false;
    for (int e = 0; e < ne; e++) {
        const size_t o = (size_t)e * nl1 + l;
        const double x = v[o];
        if (l == 0 || cnt == 0 || isnan(x)) { level[o] = qnan(); wet[o] = 0; }
        else if (x < 0.0) atomicOr(ctl + CTL_ERR, FE_VOLUME);
        else if (x >= cap) { level[o] = L; wet[o] = cnt; }
        else need = true;
    }
    if (!need) return;
    if (cnt <= SEG_WARP) list_a[atomicAdd(ctl + CTL_NA, 1)] = l;
    else if (cnt <= SEG_CTA) list_b[atomicAdd(ctl + CTL_NB, 1)] = l;
    else {
        const int r = atomicAdd(ctl + CTL_NC, 1);
        list_c[r] = l;
        size_c[r] = cnt;
        atomicAdd(ctl + CTL_CELLS_C, cnt);
    }
}

template <int G>
__device__ inline void gsync() {
    if (G == 32) __syncwarp();
    else __syncthreads();
}

// Exclusive scan of one double per thread over a group of G threads (one warp, or the whole CTA): a shuffle scan per
// warp, then the warp totals added in warp order.  *total: the group's sum.
template <int G>
__device__ inline double group_exclusive_scan(double x, double *wtot, double *total) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    double inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(full, inc, o);
        if (lane >= o) inc = __dadd_rn(inc, y);
    }
    double ex = __shfl_up_sync(full, inc, 1);
    if (lane == 0) ex = 0.0;
    if (G == 32) {
        *total = __shfl_sync(full, inc, 31);
        return ex;
    }
    const int w = threadIdx.x >> 5;
    if (lane == 31) wtot[w] = inc;
    __syncthreads();
    double base = 0.0, tot = 0.0;
    for (int k = 0; k < G / 32; k++) {
        if (k == w) base = tot;
        tot = __dadd_rn(tot, wtot[k]);
    }
    __syncthreads();
    *total = tot;
    return __dadd_rn(base, ex);
}

// Inclusive float64 prefix sums p[i] = carry + z[b] + ... + z[i] over i in [b, e) by a group of G threads: thread t
// adds its contiguous share in order, the shares are combined by the fixed scan above.  Returns carry + the chunk sum.
template <int G>
__device__ inline double group_prefix(const uint32_t *k, double *p, int b, int e, int t, double carry, double *wtot) {
    const int c = (e - b + G - 1) / G;
    const int b0 = min(e, b + t * c), b1 = min(e, b0 + c);
    double sum = 0.0;
    for (int i = b0; i < b1; i++) sum = __dadd_rn(sum, zval(k[i]));
    double tot;
    double run = __dadd_rn(carry, group_exclusive_scan<G>(sum, wtot, &tot));
    for (int i = b0; i < b1; i++) {
        run = __dadd_rn(run, zval(k[i]));
        p[i] = run;
    }
    return __dadd_rn(carry, tot);
}

// Bitonic sort of s[0, n) in shared memory by a group of G threads (padded to a power of two with keys above every
// float's key).
template <int G>
__device__ inline void group_sort(uint32_t *s, int n, int t) {
    int p2 = 1;
    while (p2 < n) p2 <<= 1;
    for (int i = n + t; i < p2; i += G) s[i] = 0xffffffffu;
    gsync<G>();
    for (int k = 2; k <= p2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = t; i < p2; i += G) {
                const int x = i ^ j;
                if (x > i) {
                    const uint32_t a = s[i], b = s[x];
                    if ((a > b) == ((i & k) == 0)) { s[i] = b; s[x] = a; }
                }
            }
            gsync<G>();
        }
}

// prefix sum S_(i+1) of a segment: stored whole (small segments), or as the chunk-local prefix plus the carry of the
// sums of the segment's earlier chunks (large segments)
struct PlainPrefix {
    const double *p;
    __device__ double operator()(int i) const { return p[i]; }
};
struct ChunkPrefix {
    const double *p, *carry;
    __device__ double operator()(int i) const { return __dadd_rn(carry[i / CHUNK_C], p[i]); }
};

// The levels and wet counts of label l for events t0, t0 + stride, ... from its sorted keys k and prefix sums P.
template <class Prefix>
__device__ inline void solve_events(const uint32_t *k, Prefix P, int n, int l, double L, double cap, double ca,
                                    const double *__restrict__ v, int nl1, int ne, int t0, int stride, double *level,
                                    int64_t *wet) {
    for (int e = t0; e < ne; e += stride) {
        const size_t o = (size_t)e * nl1 + l;
        const double x = v[o];
        double h;
        int64_t w;
        if (isnan(x)) { h = qnan(); w = 0; }
        else if (x >= cap) { h = L; w = n; }
        else {
            const double T = __ddiv_rn(x, ca);
            int lo = 1, hi = n;           // largest j in [1, n] with j z_(j) - S_j <= T (j = 1 gives 0 <= T)
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (__dsub_rn(__dmul_rn((double)mid, zval(k[mid - 1])), P(mid - 1)) <= T) lo = mid;
                else hi = mid - 1;
            }
            h = __ddiv_rn(__dadd_rn(T, P(lo - 1)), (double)lo);
            if (h > L) h = L;
            int a = 0, b = n;             // #{ z < h }
            while (a < b) {
                const int mid = (a + b) >> 1;
                if (zval(k[mid]) < h) a = mid + 1;
                else b = mid;
            }
            w = a;
        }
        level[o] = h;
        wet[o] = w;
    }
}

// segments of at most SEG_WARP cells: one warp each
__global__ void __launch_bounds__(WARPS_A * 32) k_flood_seg_warp(const uint32_t *__restrict__ seg,
                                                                 const int *__restrict__ off,
                                                                 const uint32_t *__restrict__ lkey,
                                                                 const int *__restrict__ list, int nlist,
                                                                 const double *__restrict__ st_sum, double ca,
                                                                 const double *__restrict__ v, int nl1, int ne,
                                                                 double *level, int64_t *wet) {
    __shared__ uint32_t s_k[WARPS_A][SEG_WARP];
    __shared__ double s_p[WARPS_A][SEG_WARP];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int q = blockIdx.x * WARPS_A + w; q < nlist; q += gridDim.x * WARPS_A) {
        const int l = list[q], b = off[l], n = off[l + 1] - b;
        for (int i = lane; i < n; i += 32) s_k[w][i] = seg[b + i];
        group_sort<32>(s_k[w], n, lane);
        group_prefix<32>(s_k[w], s_p[w], 0, n, lane, 0.0, nullptr);
        __syncwarp();
        solve_events(s_k[w], PlainPrefix{s_p[w]}, n, l, zval(lkey[l]), __dmul_rn(st_sum[l], ca), ca, v, nl1, ne, lane, 32, level,
                     wet);
        __syncwarp();
    }
}

// segments of SEG_WARP < n <= SEG_CTA cells: one CTA each (dynamic shared memory: SEG_CTA keys + SEG_CTA doubles)
__global__ void __launch_bounds__(T_B) k_flood_seg_cta(const uint32_t *__restrict__ seg, const int *__restrict__ off,
                                                       const uint32_t *__restrict__ lkey,
                                                       const int *__restrict__ list, int nlist,
                                                       const double *__restrict__ st_sum, double ca,
                                                       const double *__restrict__ v, int nl1, int ne, double *level,
                                                       int64_t *wet) {
    extern __shared__ double s_dyn[];
    __shared__ double s_w[T_B / 32];
    double *s_p = s_dyn;
    uint32_t *s_k = reinterpret_cast<uint32_t *>(s_dyn + SEG_CTA);
    const int t = threadIdx.x;
    for (int q = blockIdx.x; q < nlist; q += gridDim.x) {
        const int l = list[q], b = off[l], n = off[l + 1] - b;
        for (int i = t; i < n; i += T_B) s_k[i] = seg[b + i];
        group_sort<T_B>(s_k, n, t);
        group_prefix<T_B>(s_k, s_p, 0, n, t, 0.0, s_w);
        __syncthreads();
        solve_events(s_k, PlainPrefix{s_p}, n, l, zval(lkey[l]), __dmul_rn(st_sum[l], ca), ca, v, nl1, ne, t, T_B, level, wet);
        __syncthreads();
    }
}

// largest r in [0, n) with a[r] <= x (a ascending, a[0] <= x)
__device__ inline int rank_of(const int *__restrict__ a, int n, int x) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (a[mid] <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// large segments: cell i of the sort input is cell i - coff[r] of segment r (label list_c[r]); value = r
__global__ void __launch_bounds__(256) k_flood_gather(const uint32_t *__restrict__ seg, const int *__restrict__ off,
                                                      const int *__restrict__ list_c, const int *__restrict__ coff,
                                                      int nc, int m, int *key, int *val) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int r = rank_of(coff, nc, i);
    key[i] = (int)seg[off[list_c[r]] + i - coff[r]];
    val[i] = r;
}

__global__ void __launch_bounds__(256) k_flood_nchunks(const int *__restrict__ size_c, int nc, int *nch) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nc) nch[r] = (size_c[r] + CHUNK_C - 1) / CHUNK_C;
}

// large segments, sorted by (segment, z): one CTA per CHUNK_C cells of a segment (chunks counted from the segment's
// start) writes the chunk-local inclusive prefix sums and the chunk's sum
__global__ void __launch_bounds__(T_B) k_flood_big_chunk(const uint32_t *__restrict__ sorted,
                                                         const int *__restrict__ size_c, const int *__restrict__ coff,
                                                         const int *__restrict__ choff, int nc,
                                                         const int64_t *__restrict__ nchunks, double *prefix,
                                                         double *ctot) {
    __shared__ double s_w[T_B / 32];
    const int q = blockIdx.x;
    if (q >= *nchunks) return;
    const int r = rank_of(choff, nc, q), b = (q - choff[r]) * CHUNK_C, n = size_c[r];
    const double t = group_prefix<T_B>(sorted + coff[r], prefix + coff[r], b, min(n, b + CHUNK_C), threadIdx.x, 0.0,
                                       s_w);
    if (threadIdx.x == 0) ctot[q] = t;
}

// carry of each chunk: the sum of the segment's earlier chunk sums, added in chunk order (one thread per segment)
__global__ void __launch_bounds__(128) k_flood_big_carry(const int *__restrict__ choff, const int *__restrict__ size_c,
                                                         int nc, const double *__restrict__ ctot, double *carry) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nc) return;
    const int c0 = choff[r], nch = (size_c[r] + CHUNK_C - 1) / CHUNK_C;
    double acc = 0.0;
    for (int c = 0; c < nch; c++) {
        carry[c0 + c] = acc;
        acc = __dadd_rn(acc, ctot[c0 + c]);
    }
}

// large segments: one thread per (segment, event)
__global__ void __launch_bounds__(128) k_flood_big_solve(const uint32_t *__restrict__ sorted,
                                                         const int *__restrict__ list_c, const int *__restrict__ size_c,
                                                         const int *__restrict__ coff, const int *__restrict__ choff,
                                                         int nc, const double *__restrict__ prefix,
                                                         const double *__restrict__ carry,
                                                         const uint32_t *__restrict__ lkey,
                                                         const double *__restrict__ st_sum, double ca,
                                                         const double *__restrict__ v, int nl1, int ne, double *level,
                                                         int64_t *wet) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (int64_t)nc * ne) return;
    const int r = (int)(q % nc), e = (int)(q / nc), l = list_c[r];
    solve_events(sorted + coff[r], ChunkPrefix{prefix + coff[r], carry + choff[r]}, size_c[r], l, zval(lkey[l]),
                 __dmul_rn(st_sum[l], ca), ca, v, nl1, ne, e, ne, level, wet);
}

__global__ void __launch_bounds__(256) k_water_depth(const float *__restrict__ dem, const float *__restrict__ fil,
                                                     const int32_t *__restrict__ lab, int64_t n, int64_t nlabels,
                                                     const double *__restrict__ level, float *out, int *ctl) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int l = lab[i];
    float d = 0.f;
    if (l < 0 || l > nlabels) {
        *ctl = FE_LABEL;
    } else if (l > 0) {
        const double h = __ldg(level + l);
        const float f = fil[i], z = dem[i];
        if (h == (double)f) d = __fsub_rn(f, z);                        // full: bitwise the fill's depths
        else if ((double)z < h) d = __double2float_rn(__dsub_rn(h, (double)z));
    }
    out[i] = d;
}

static int flood_check(const void *dem, const void *fil, const void *lab, int64_t rows, int64_t cols,
                       int64_t nlabels, const char *what) {
    if (!dem || !fil || !lab || rows < 1 || cols < 1 || rows * cols >= (1ll << 31) || nlabels < 0 ||
        nlabels >= (1ll << 31) - 2) {
        set_error("%s: null pointer or unsupported size (%lld x %lld, %lld labels)", what, (long long)rows,
                  (long long)cols, (long long)nlabels);
        return MS_ERR_ARG;
    }
    return MS_OK;
}

// Levels and wet counts of the labels l0 <= l < l1 from their segments: seg[off[l], off[l+1]) holds label l's z keys
// (any order), lkey[l] its fill key.  Labels outside the range are not touched.  ctl: CTL_N ints, counters zero,
// ctl[CTL_ERR] the grouping's flags.  *err: the flags after the classification (FE_VOLUME added); when they are not
// zero nothing else runs.
static int flood_solve(const int *off, const uint32_t *lkey, const uint32_t *seg, int l0, int l1,
                       const double *st_sum, double ca, const double *v, int nl1, int ne, double *level, int64_t *wet,
                       int *ctl, int *err, cudaStream_t s) {
    const int nr = l1 - l0;
    *err = 0;
    if (nr <= 0) return MS_OK;
    DevBuf<int> list_a, list_b, list_c, size_c;
    DevBuf<int64_t> total;
    MS_TRY(list_a.alloc((size_t)nr, s));
    MS_TRY(list_b.alloc((size_t)nr, s));
    MS_TRY(list_c.alloc((size_t)nr, s));
    MS_TRY(size_c.alloc((size_t)nr, s));
    MS_TRY(total.alloc(1, s));
    MS_LAUNCH(k_flood_classify, cdiv(nr, 256), 256, 0, s, off, lkey, st_sum, ca, v, nl1, ne, l0, l1, level, wet,
              list_a.p, list_b.p, list_c.p, size_c.p, ctl);
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, ctl, CTL_N * sizeof(int), s));
    MS_TRY(stream_sync(s));
    int c[CTL_N];
    for (int k = 0; k < CTL_N; k++) c[k] = ((int *)h)[k];
    *err = c[CTL_ERR];
    if (*err) return MS_OK;
    if (c[CTL_NA]) {
        prof_units(c[CTL_NA]);
        MS_LAUNCH(k_flood_seg_warp, cdiv(c[CTL_NA], WARPS_A), WARPS_A * 32, 0, s, seg, off, lkey, list_a.p,
                  c[CTL_NA], st_sum, ca, v, nl1, ne, level, wet);
    }
    if (c[CTL_NB]) {
        const size_t smem = (size_t)SEG_CTA * (sizeof(double) + sizeof(uint32_t));
        static bool attr = false;
        if (!attr) {
            MS_CUDA(cudaFuncSetAttribute(k_flood_seg_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr = true;
        }
        prof_units(c[CTL_NB]);
        MS_LAUNCH(k_flood_seg_cta, c[CTL_NB], T_B, smem, s, seg, off, lkey, list_b.p, c[CTL_NB], st_sum, ca, v,
                  nl1, ne, level, wet);
    }
    if (c[CTL_NC]) {
        const int nc = c[CTL_NC], m = c[CTL_CELLS_C];
        const int kmax = m / CHUNK_C + nc;              // chunks of all large segments, at most
        DevBuf<int> coff, choff, ka, va, kb, vb, flag;
        DevBuf<double> prefix, ctot, carry;
        DevBuf<int64_t> nchunks;
        MS_TRY(coff.alloc((size_t)nc, s));
        MS_TRY(choff.alloc((size_t)nc, s));
        MS_TRY(ka.alloc((size_t)m, s));
        MS_TRY(va.alloc((size_t)m, s));
        MS_TRY(kb.alloc((size_t)m, s));
        MS_TRY(vb.alloc((size_t)m, s));
        MS_TRY(flag.alloc((size_t)m, s));
        MS_TRY(prefix.alloc((size_t)m, s));
        MS_TRY(ctot.alloc((size_t)kmax, s));
        MS_TRY(carry.alloc((size_t)kmax, s));
        MS_TRY(nchunks.alloc(1, s));
        MS_TRY(exclusive_scan_i32(size_c.p, coff.p, nc, total.p, s));
        MS_LAUNCH(k_flood_nchunks, cdiv(nc, 256), 256, 0, s, size_c.p, nc, flag.p);
        MS_TRY(exclusive_scan_i32(flag.p, choff.p, nc, nchunks.p, s));
        prof_units(m);
        MS_LAUNCH(k_flood_gather, cdiv(m, 256), 256, 0, s, seg, off, list_c.p, coff.p, nc, m, ka.p, va.p);
        // LSD: stable by z key (32 bits), then stable by segment rank -> (segment, z) order
        int *k1 = ka.p, *v1 = va.p, *k2 = kb.p, *v2 = vb.p;
        MS_TRY(radix_sort_split(&k1, &v1, &k2, &v2, flag.p, total.p, m, 32, s));
        int rbits = 0;
        while ((1ll << rbits) < nc) rbits++;
        MS_TRY(radix_sort_split(&v1, &k1, &v2, &k2, flag.p, total.p, m, rbits, s));
        prof_units(m);
        MS_LAUNCH(k_flood_big_chunk, kmax, T_B, 0, s, (const uint32_t *)k1, size_c.p, coff.p, choff.p, nc, nchunks.p,
                  prefix.p, ctot.p);
        MS_LAUNCH(k_flood_big_carry, cdiv(nc, 128), 128, 0, s, choff.p, size_c.p, nc, ctot.p, carry.p);
        MS_LAUNCH(k_flood_big_solve, cdiv((int64_t)nc * ne, 128), 128, 0, s, (const uint32_t *)k1, list_c.p,
                  size_c.p, coff.p, choff.p, nc, prefix.p, carry.p, lkey, st_sum, ca, v, nl1, ne, level, wet);
    }
    return MS_OK;
}

static int flood_levels_impl(const float *dem, const float *fil, const int32_t *lab, int64_t rows, int64_t cols,
                             int64_t nlabels, const double *st_sum, double ca, int64_t ne64, const double *v,
                             double *level, int64_t *wet, cudaStream_t s) {
    const int64_t n = rows * cols;
    const int nl1 = (int)nlabels + 1, ne = (int)ne64;
    DevBuf<int> cnt, off, ctl;
    DevBuf<uint32_t> lkey, seg;
    DevBuf<int64_t> total;
    MS_TRY(cnt.alloc((size_t)nl1 + 1, s));
    MS_TRY(off.alloc((size_t)nl1 + 1, s));
    MS_TRY(lkey.alloc((size_t)nl1, s));
    MS_TRY(ctl.alloc(CTL_N, s));
    MS_TRY(total.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(cnt.p, 0, ((size_t)nl1 + 1) * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, CTL_N * sizeof(int), s));
    const unsigned g = cdiv(n, 256 * FL_CELLS);
    prof_units(n);
    MS_LAUNCH(k_flood_group<false>, g, 256, 0, s, lab, fil, dem, n, nlabels, cnt.p, lkey.p, off.p, seg.p, 0,
              nullptr, ctl.p);
    MS_TRY(exclusive_scan_i32(cnt.p, off.p, (int64_t)nl1 + 1, total.p, s));
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, total.p, sizeof(int64_t), s));
    MS_TRY(stream_sync(s));
    const int64_t ncells = h[0];
    MS_TRY(seg.alloc((size_t)ncells, s));
    MS_CUDA(cudaMemsetAsync(cnt.p, 0, ((size_t)nl1 + 1) * sizeof(int), s));
    prof_units(n);
    MS_LAUNCH(k_flood_group<true>, g, 256, 0, s, lab, fil, dem, n, nlabels, cnt.p, lkey.p, off.p, seg.p, 0, nullptr,
              ctl.p);
    int err = 0;
    MS_TRY(flood_solve(off.p, lkey.p, seg.p, 0, nl1, st_sum, ca, v, nl1, ne, level, wet, ctl.p, &err, s));
    if (err & FE_LABEL) { set_error("flood_levels: a label outside [0, %lld]", (long long)nlabels); return MS_ERR_LABEL; }
    if (err & FE_UNIFORM) {
        set_error("flood_levels: the fill is not uniform over a label (labels must be bluespots of this fill)");
        return MS_ERR_ARG;
    }
    if (err & FE_VOLUME) { set_error("flood_levels: a negative volume"); return MS_ERR_ARG; }
    return MS_OK;
}

// ---- the same on a band of a raster split by rows (BandPipeline.flood).  Band g owns the labels lo < l <= hi
// (the labels it numbered; their first cells lie in it); a label it sees at or below lo is owned by a lower band.  The
// owner of a label gathers every band's z keys of it into its own segment and solves it there with flood_solve, so the
// label's sorted keys, its count and with them the summation order are those of the whole-raster call.

// foreign labels: flag[l] = label l (1 <= l <= lo) has cells in this band
__global__ void __launch_bounds__(256) k_flood_foreign_flag(const int *__restrict__ cnt, int64_t lo, int *flag) {
    const int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l <= lo) flag[l] = l > 0 && cnt[l] > 0;
}

// the foreign list in label order: (label, count, fill key); res[0] = flags, res[2] = cells to send (off[lo + 1])
__global__ void __launch_bounds__(256) k_flood_foreign_list(const int *__restrict__ cnt,
                                                            const uint32_t *__restrict__ lkey,
                                                            const int *__restrict__ flag, const int *__restrict__ pos,
                                                            const int *__restrict__ off, int64_t lo, int32_t *list,
                                                            int64_t cap, int *ctl, int64_t *res) {
    const int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l <= lo && flag[l]) {
        const int64_t p = pos[l];
        if (p < cap) {
            list[3 * p] = (int32_t)l;
            list[3 * p + 1] = cnt[l];
            list[3 * p + 2] = (int32_t)lkey[l];
        } else {
            atomicOr(ctl + CTL_ERR, MS_FLOOD_CAPACITY);
        }
    }
    if (l == 0) res[2] = off[lo + 1];
}

// received runs: check the owner range and the fill key, reserve a place in the segment (after the owner's own
// cells: their count is in cnt[l] already).  res[0] = received cells, res[1] = the owner's own cells of its labels.
__global__ void __launch_bounds__(256) k_flood_recv(const int32_t *__restrict__ recv, int64_t nrecv, int64_t lo,
                                                    int64_t hi, int *cnt, const uint32_t *__restrict__ lkey,
                                                    const int *__restrict__ off, int *pos, int *ctl,
                                                    unsigned long long *res) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) res[1] = (unsigned long long)(off[hi + 1] - off[lo + 1]);
    if (i >= nrecv) return;
    const int64_t l = recv[3 * i];
    const int c = recv[3 * i + 1];
    if (l <= lo || l > hi || c <= 0) { atomicOr(ctl + CTL_ERR, FE_LABEL); return; }
    if ((uint32_t)recv[3 * i + 2] != lkey[l]) atomicOr(ctl + CTL_ERR, FE_UNIFORM);
    pos[i] = atomicAdd(cnt + l, c);
    atomicAdd(res, (unsigned long long)c);
}

// received keys: key j of run i goes to seg[off[l_i] + pos[i] + j]
__global__ void __launch_bounds__(256) k_flood_recv_copy(const int32_t *__restrict__ recv, int nrecv,
                                                         const int *__restrict__ roff, const int *__restrict__ pos,
                                                         const int *__restrict__ off,
                                                         const uint32_t *__restrict__ keys, int64_t nkeys,
                                                         uint32_t *seg) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nkeys) return;
    const int r = rank_of(roff, nrecv, (int)k);
    seg[off[recv[3 * r]] + pos[r] + (int)k - roff[r]] = keys[k];
}

__global__ void __launch_bounds__(256) k_flood_recv_counts(const int32_t *__restrict__ recv, int nrecv, int *c) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nrecv) c[i] = recv[3 * i + 1];
}

static int band_flood_count(const float *dem, const float *fil, const int32_t *lab, int64_t n, int64_t lo, int64_t hi,
                            int *cnt, uint32_t *lkey, int *off, int32_t *foreign, int64_t cap, int64_t *n_foreign,
                            int64_t *n_send, int *flags, cudaStream_t s) {
    DevBuf<int> ctl, flag, pos;
    DevBuf<int64_t> res;
    MS_TRY(ctl.alloc(CTL_N, s));
    MS_TRY(flag.alloc((size_t)lo + 1, s));
    MS_TRY(pos.alloc((size_t)lo + 1, s));
    MS_TRY(res.alloc(3, s));
    MS_CUDA(cudaMemsetAsync(cnt, 0, ((size_t)hi + 2) * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, CTL_N * sizeof(int), s));
    prof_units(n);
    MS_LAUNCH(k_flood_group<false>, cdiv(n, 256 * FL_CELLS), 256, 0, s, lab, fil, dem, n, hi, cnt, lkey, off,
              nullptr, 0, nullptr, ctl.p);
    // send offsets of the foreign labels (off[0 .. lo]), off[lo + 1] = their cells, off[hi + 1] - off[lo + 1] = the
    // cells of the band's own labels; no sum reaches 2^31 (a band holds at most 2^30 cells)
    MS_TRY(exclusive_scan_i32(cnt, off, hi + 2, res.p + 1, s));
    MS_LAUNCH(k_flood_foreign_flag, cdiv(lo + 1, 256), 256, 0, s, cnt, lo, flag.p);
    MS_TRY(exclusive_scan_i32(flag.p, pos.p, lo + 1, res.p + 1, s));
    MS_LAUNCH(k_flood_foreign_list, cdiv(lo + 1, 256), 256, 0, s, cnt, lkey, flag.p, pos.p, off, lo, foreign, cap,
              ctl.p, res.p);
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, res.p + 1, 2 * sizeof(int64_t), s));
    MS_TRY(readback(h + 2, ctl.p, sizeof(int), s));
    MS_TRY(stream_sync(s));
    *n_foreign = h[0] < cap ? h[0] : cap;
    *n_send = h[1];
    *flags = *(int *)(h + 2);
    return MS_OK;
}

static int band_flood_layout(int64_t lo, int64_t hi, int *cnt, const uint32_t *lkey, int *off, const int32_t *recv,
                             int64_t nrecv, int *recv_pos, int64_t *n_cells, int *flags, cudaStream_t s) {
    DevBuf<int> ctl;
    DevBuf<unsigned long long> res;
    DevBuf<int64_t> total;
    MS_TRY(ctl.alloc(CTL_N, s));
    MS_TRY(res.alloc(2, s));
    MS_TRY(total.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, CTL_N * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(res.p, 0, 2 * sizeof(unsigned long long), s));
    MS_LAUNCH(k_flood_recv, cdiv(nrecv > 0 ? nrecv : 1, 256), 256, 0, s, recv, nrecv, lo, hi, cnt, lkey, off,
              recv_pos, ctl.p, res.p);
    // segment offsets of the owned labels (off[lo + 1] = 0); wrong if the sum reaches 2^31, which is refused below.
    // The scan loads and stores 16-byte vectors, so it runs on copies that start on an allocation.
    const int64_t m = hi - lo + 1;
    DevBuf<int> a, b;
    MS_TRY(a.alloc((size_t)m, s));
    MS_TRY(b.alloc((size_t)m, s));
    MS_CUDA(cudaMemcpyAsync(a.p, cnt + lo + 1, (size_t)m * sizeof(int), cudaMemcpyDeviceToDevice, s));
    MS_TRY(exclusive_scan_i32(a.p, b.p, m, total.p, s));
    MS_CUDA(cudaMemcpyAsync(off + lo + 1, b.p, (size_t)m * sizeof(int), cudaMemcpyDeviceToDevice, s));
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, res.p, 2 * sizeof(int64_t), s));
    MS_TRY(readback(h + 2, ctl.p, sizeof(int), s));
    MS_TRY(stream_sync(s));
    *n_cells = h[0] + h[1];
    *flags = *(int *)(h + 2);
    if (*n_cells >= (1ll << 31)) {
        set_error("band_flood_layout: the labels of a band hold %lld cells with those of the other bands; at most "
                  "2^31 - 1 are supported", (long long)*n_cells);
        *flags |= MS_FLOOD_SIZE;
    }
    return MS_OK;
}

static int band_flood_scatter(const float *dem, const float *fil, const int32_t *lab, int64_t n, int64_t lo,
                              int64_t hi, int *cnt, const uint32_t *lkey, const int *off, uint32_t *seg,
                              uint32_t *send, int *flags, cudaStream_t s) {
    DevBuf<int> ctl;
    MS_TRY(ctl.alloc(CTL_N, s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, CTL_N * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(cnt, 0, ((size_t)hi + 2) * sizeof(int), s));
    prof_units(n);
    MS_LAUNCH(k_flood_group<true>, cdiv(n, 256 * FL_CELLS), 256, 0, s, lab, fil, dem, n, hi, cnt, (uint32_t *)lkey,
              off, seg, lo, send, ctl.p);
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, ctl.p, sizeof(int), s));
    MS_TRY(stream_sync(s));
    *flags = *(int *)h;
    return MS_OK;
}

static int band_flood_solve(int64_t nlabels, int64_t lo, int64_t hi, const int *off, const uint32_t *lkey,
                            uint32_t *seg, const int32_t *recv, int64_t nrecv, const int *recv_pos,
                            const uint32_t *recv_keys, int64_t n_recv_keys, const double *st_sum, double ca,
                            int64_t ne, const double *v, double *level, int64_t *wet, int *flags, cudaStream_t s) {
    if (nrecv > 0) {
        DevBuf<int> c, roff;
        DevBuf<int64_t> total;
        MS_TRY(c.alloc((size_t)nrecv, s));
        MS_TRY(roff.alloc((size_t)nrecv, s));
        MS_TRY(total.alloc(1, s));
        MS_LAUNCH(k_flood_recv_counts, cdiv(nrecv, 256), 256, 0, s, recv, (int)nrecv, c.p);
        MS_TRY(exclusive_scan_i32(c.p, roff.p, nrecv, total.p, s));
        int64_t *h = host_flags().h;
        MS_TRY(readback(h, total.p, sizeof(int64_t), s));
        MS_TRY(stream_sync(s));
        if (h[0] != n_recv_keys) {
            set_error("band_flood_solve: %lld received keys for runs of %lld cells", (long long)n_recv_keys,
                      (long long)h[0]);
            return MS_ERR_ARG;
        }
        prof_units(n_recv_keys);
        MS_LAUNCH(k_flood_recv_copy, cdiv(n_recv_keys, 256), 256, 0, s, recv, (int)nrecv, roff.p, recv_pos, off,
                  recv_keys, n_recv_keys, seg);
    }
    DevBuf<int> ctl;
    MS_TRY(ctl.alloc(CTL_N, s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, CTL_N * sizeof(int), s));
    return flood_solve(off, lkey, seg, (int)lo + 1, (int)hi + 1, st_sum, ca, v, (int)nlabels + 1, (int)ne, level, wet,
                       ctl.p, flags, s);
}

static int water_depth_impl(const float *dem, const float *fil, const int32_t *lab, int64_t rows, int64_t cols,
                            int64_t nlabels, const double *level, float *out, cudaStream_t s) {
    const int64_t n = rows * cols;
    DevBuf<int> ctl;
    MS_TRY(ctl.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(ctl.p, 0, sizeof(int), s));
    prof_units(n);
    MS_LAUNCH(k_water_depth, cdiv(n, 256), 256, 0, s, dem, fil, lab, n, nlabels, level, out, ctl.p);
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, ctl.p, sizeof(int), s));
    MS_TRY(stream_sync(s));
    if (*(int *)h) { set_error("water_depth: a label outside [0, %lld]", (long long)nlabels); return MS_ERR_LABEL; }
    return MS_OK;
}

}  // namespace ms

extern "C" {

static int flood_levels_args(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                             int64_t nlabels, const double *st_sum, double cell_area, int64_t n_events,
                             const double *v, const double *out_level, const int64_t *out_wet) {
    MS_TRY(ms::flood_check(dem, filled, labels, rows, cols, nlabels, "flood_levels"));
    if (!st_sum || !v || !out_level || !out_wet || n_events < 0 || n_events >= (1ll << 31) ||
        !(cell_area > 0.0) || !isfinite(cell_area)) {
        ms::set_error("flood_levels: null pointer, negative event count or cell_area not > 0 (%g)", cell_area);
        return MS_ERR_ARG;
    }
    return MS_OK;
}

int ms_flood_levels_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                        int64_t nlabels, const double *st_sum, double cell_area, int64_t n_events, const double *v,
                        double *out_level, int64_t *out_wet, void *stream) {
    MS_TRY(flood_levels_args(dem, filled, labels, rows, cols, nlabels, st_sum, cell_area, n_events, v, out_level,
                             out_wet));
    MS_TRY(ms::ensure_init());
    if (n_events == 0) return MS_OK;
    return ms::flood_levels_impl(dem, filled, labels, rows, cols, nlabels, st_sum, cell_area, n_events, v, out_level,
                                 out_wet, (cudaStream_t)stream);
}

int ms_flood_levels(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                    int64_t nlabels, const double *st_sum, double cell_area, int64_t n_events, const double *v,
                    double *out_level, int64_t *out_wet) {
    MS_TRY(flood_levels_args(dem, filled, labels, rows, cols, nlabels, st_sum, cell_area, n_events, v, out_level,
                             out_wet));
    MS_TRY(ms::ensure_init());
    if (n_events == 0) return MS_OK;
    cudaStream_t s = nullptr;
    const size_t n = (size_t)(rows * cols), nl1 = (size_t)nlabels + 1, m = nl1 * (size_t)n_events;
    ms::HostCall hc;
    float *d = nullptr, *f = nullptr;
    int32_t *l = nullptr;
    ms::DevBuf<double> ss, vv, lv;
    ms::DevBuf<int64_t> wt;
    MS_TRY(hc.in(dem, n, s, &d));
    MS_TRY(hc.in(filled, n, s, &f));
    MS_TRY(hc.in(labels, n, s, &l));
    MS_TRY(ss.alloc(nl1, s));
    MS_TRY(vv.alloc(m, s));
    MS_TRY(lv.alloc(m, s));
    MS_TRY(wt.alloc(m, s));
    MS_CUDA(cudaMemcpyAsync(ss.p, st_sum, nl1 * 8, cudaMemcpyHostToDevice, s));
    MS_CUDA(cudaMemcpyAsync(vv.p, v, m * 8, cudaMemcpyHostToDevice, s));
    MS_TRY(ms::flood_levels_impl(d, f, l, rows, cols, nlabels, ss.p, cell_area, n_events, vv.p, lv.p, wt.p, s));
    MS_CUDA(cudaMemcpyAsync(out_level, lv.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_CUDA(cudaMemcpyAsync(out_wet, wt.p, m * 8, cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

int ms_water_depth_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                       int64_t nlabels, const double *level, float *out_depth, void *stream) {
    MS_TRY(ms::flood_check(dem, filled, labels, rows, cols, nlabels, "water_depth"));
    if (!level || !out_depth) { ms::set_error("water_depth: null pointer"); return MS_ERR_ARG; }
    MS_TRY(ms::ensure_init());
    return ms::water_depth_impl(dem, filled, labels, rows, cols, nlabels, level, out_depth, (cudaStream_t)stream);
}

int ms_water_depth(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                   int64_t nlabels, const double *level, float *out_depth) {
    MS_TRY(ms::flood_check(dem, filled, labels, rows, cols, nlabels, "water_depth"));
    if (!level || !out_depth) { ms::set_error("water_depth: null pointer"); return MS_ERR_ARG; }
    MS_TRY(ms::ensure_init());
    cudaStream_t s = nullptr;
    const size_t n = (size_t)(rows * cols), nl1 = (size_t)nlabels + 1;
    ms::HostCall hc;
    float *d = nullptr, *f = nullptr;
    int32_t *l = nullptr;
    float *o = nullptr;
    ms::DevBuf<double> lv;
    MS_TRY(hc.in(dem, n, s, &d));
    MS_TRY(hc.in(filled, n, s, &f));
    MS_TRY(hc.in(labels, n, s, &l));
    MS_TRY(hc.out(n, &o));
    MS_TRY(lv.alloc(nl1, s));
    MS_CUDA(cudaMemcpyAsync(lv.p, level, nl1 * 8, cudaMemcpyHostToDevice, s));
    MS_TRY(ms::water_depth_impl(d, f, l, rows, cols, nlabels, lv.p, o, s));
    MS_CUDA(cudaMemcpyAsync(out_depth, o, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(o, out_depth, n * sizeof(float));
    return MS_OK;
}

static int band_flood_range(int64_t nlabels, int64_t lo, int64_t hi, const char *what) {
    if (nlabels < 0 || nlabels >= (1ll << 31) - 2 || lo < 0 || lo > hi || hi > nlabels) {
        ms::set_error("%s: the owned labels (%lld, %lld] are not a range of [1, %lld]", what, (long long)lo,
                      (long long)hi, (long long)nlabels);
        return MS_ERR_ARG;
    }
    return MS_OK;
}

int ms_band_flood_count_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                            int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, uint32_t *lkey, int32_t *off,
                            int32_t *foreign, int64_t capacity, int64_t *n_foreign, int64_t *n_send, int *flags,
                            void *stream) {
    MS_TRY(ms::flood_check(dem, filled, labels, rows, cols, nlabels, "band_flood_count"));
    MS_TRY(band_flood_range(nlabels, lo, hi, "band_flood_count"));
    if (!cnt || !lkey || !off || !foreign || capacity < 1 || !n_foreign || !n_send || !flags ||
        ((uintptr_t)cnt & 15) || ((uintptr_t)off & 15)) {
        ms::set_error("band_flood_count: null pointer, cnt / off not on a 16-byte boundary or capacity < 1");
        return MS_ERR_ARG;
    }
    MS_TRY(ms::ensure_init());
    return ms::band_flood_count(dem, filled, labels, rows * cols, lo, hi, cnt, lkey, off, foreign, capacity, n_foreign,
                                n_send, flags, (cudaStream_t)stream);
}

int ms_band_flood_layout_dev(int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, const uint32_t *lkey, int32_t *off,
                             const int32_t *recv, int64_t n_recv, int32_t *recv_pos, int64_t *n_cells, int *flags,
                             void *stream) {
    MS_TRY(band_flood_range(nlabels, lo, hi, "band_flood_layout"));
    if (!cnt || !lkey || !off || n_recv < 0 || n_recv >= (1ll << 31) || (n_recv && (!recv || !recv_pos)) ||
        !n_cells || !flags) {
        ms::set_error("band_flood_layout: null pointer or bad count of received runs (%lld)", (long long)n_recv);
        return MS_ERR_ARG;
    }
    MS_TRY(ms::ensure_init());
    return ms::band_flood_layout(lo, hi, cnt, lkey, off, recv, n_recv, recv_pos, n_cells, flags, (cudaStream_t)stream);
}

int ms_band_flood_scatter_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                              int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, const uint32_t *lkey,
                              const int32_t *off, uint32_t *seg, uint32_t *send, int *flags, void *stream) {
    MS_TRY(ms::flood_check(dem, filled, labels, rows, cols, nlabels, "band_flood_scatter"));
    MS_TRY(band_flood_range(nlabels, lo, hi, "band_flood_scatter"));
    if (!cnt || !lkey || !off || !flags) { ms::set_error("band_flood_scatter: null pointer"); return MS_ERR_ARG; }
    MS_TRY(ms::ensure_init());
    return ms::band_flood_scatter(dem, filled, labels, rows * cols, lo, hi, cnt, lkey, off, seg, send, flags,
                                  (cudaStream_t)stream);
}

int ms_band_flood_solve_dev(int64_t nlabels, int64_t lo, int64_t hi, const int32_t *off, const uint32_t *lkey,
                            uint32_t *seg, const int32_t *recv, int64_t n_recv, const int32_t *recv_pos,
                            const uint32_t *recv_keys, int64_t n_recv_keys, const double *st_sum, double cell_area,
                            int64_t n_events, const double *v, double *out_level, int64_t *out_wet, int *flags,
                            void *stream) {
    MS_TRY(band_flood_range(nlabels, lo, hi, "band_flood_solve"));
    if (!off || !lkey || !st_sum || !v || !out_level || !out_wet || !flags || n_recv < 0 || n_recv >= (1ll << 31) ||
        n_recv_keys < 0 || n_recv_keys >= (1ll << 31) || (n_recv && (!recv || !recv_pos)) ||
        (n_recv_keys && (!recv_keys || !seg)) || (!n_recv && n_recv_keys) || n_events < 0 ||
        n_events >= (1ll << 31) || !(cell_area > 0.0) || !isfinite(cell_area)) {
        ms::set_error("band_flood_solve: null pointer, bad count or cell_area not > 0 (%g)", cell_area);
        return MS_ERR_ARG;
    }
    MS_TRY(ms::ensure_init());
    *flags = 0;
    if (n_events == 0) return MS_OK;
    return ms::band_flood_solve(nlabels, lo, hi, off, lkey, seg, recv, n_recv, recv_pos, recv_keys, n_recv_keys, st_sum,
                                cell_area, n_events, v, out_level, out_wet, flags, (cudaStream_t)stream);
}

}  // extern "C"
