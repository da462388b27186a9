// primitives.cu — device-wide exclusive scan and forest pointer jumping, shared by the fill (catchment ids),
// connected components (scipy numbering) and watershed stages.
#include "common.cuh"

namespace ms {

// ------------------------------------------------------------------------------------------------
// exclusive scan of int32 values: reduce per 4096-element chunk, scan the chunk sums in one CTA,
// then rescan each chunk with its offset.  16 contiguous items per thread, 128-bit loads/stores.
// ------------------------------------------------------------------------------------------------
constexpr int SCAN_T = 256;
constexpr int SCAN_I = 16;
constexpr int SCAN_CH = SCAN_T * SCAN_I;

__device__ inline void load16(const int *p, int64_t base, int64_t n, int v[SCAN_I]) {
    if (base + SCAN_I <= n) {
        const int4 *q = reinterpret_cast<const int4 *>(p + base);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int4 t = q[k];
            v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < SCAN_I; k++) v[k] = (base + k < n) ? p[base + k] : -1;
    }
    if (base + SCAN_I > n) {
#pragma unroll
        for (int k = 0; k < SCAN_I; k++) if (base + k >= n) v[k] = 0;
    }
}

__device__ inline int block_exclusive_scan(int x, int *total) {
    __shared__ int wsum[SCAN_T / 32];
    __shared__ int tot;
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
        int s = lane < SCAN_T / 32 ? wsum[lane] : 0;
        int si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= o) si += y;
        }
        if (lane < SCAN_T / 32) wsum[lane] = si - s;
        if (lane == SCAN_T / 32 - 1) tot = si;
    }
    __syncthreads();
    int r = inc - x + wsum[w];
    if (total) *total = tot;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_T) k_scan_reduce(const int *in, int64_t n, int *bsum) {
    int64_t base = (int64_t)blockIdx.x * SCAN_CH + (int64_t)threadIdx.x * SCAN_I;
    int v[SCAN_I];
    load16(in, base, n, v);
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_I; k++) s += v[k];
    int tot;
    block_exclusive_scan(s, &tot);
    if (threadIdx.x == 0) bsum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) k_scan_bsums(int *bsum, int nb, int64_t *total) {
    __shared__ int wsum[32];
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int base = 0; base < nb; base += 1024) {
        int i = base + threadIdx.x;
        int x = i < nb ? bsum[i] : 0;
        int inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) wsum[w] = inc;
        __syncthreads();
        if (w == 0) {
            int s = wsum[lane], si = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, si, o);
                if (lane >= o) si += y;
            }
            wsum[lane] = si - s;
        }
        __syncthreads();
        int carry = carry_s;
        int ex = inc - x + wsum[w] + carry;
        if (i < nb) bsum[i] = ex;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = ex + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = (int64_t)carry_s;
}

__global__ void __launch_bounds__(SCAN_T) k_scan_final(const int *in, int *out, int64_t n, const int *bsum) {
    int64_t base = (int64_t)blockIdx.x * SCAN_CH + (int64_t)threadIdx.x * SCAN_I;
    int v[SCAN_I];
    load16(in, base, n, v);
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_I; k++) s += v[k];
    int ex = block_exclusive_scan(s, nullptr) + bsum[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_I; k++) {
        int t = v[k];
        v[k] = ex;
        ex += t;
    }
    if (base + SCAN_I <= n) {
        int4 *q = reinterpret_cast<int4 *>(out + base);
#pragma unroll
        for (int k = 0; k < 4; k++) q[k] = make_int4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    } else {
#pragma unroll
        for (int k = 0; k < SCAN_I; k++)
            if (base + k < n) out[base + k] = v[k];
    }
}

int exclusive_scan_i32(const int *flags, int *out, int64_t n, int64_t *total_dev, cudaStream_t s) {
    int nb = (int)cdiv(n, SCAN_CH);
    DevBuf<int> bsum;
    MS_TRY(bsum.alloc((size_t)nb, s));
    MS_LAUNCH(k_scan_reduce, nb, SCAN_T, 0, s, flags, n, bsum.p);
    MS_LAUNCH(k_scan_bsums, 1, 1024, 0, s, bsum.p, nb, total_dev);
    MS_LAUNCH(k_scan_final, nb, SCAN_T, 0, s, flags, out, n, bsum.p);
    return MS_OK;
}

// ------------------------------------------------------------------------------------------------
// forest pointer jumping.  ptr[i] is the parent cell (roots: ptr[i] == i).  Each round every cell hops
// up to JUMP_HOPS ancestors and writes the furthest one back (asynchronous, in place: a concurrent
// reader sees either the old or the new parent, both are ancestors).  Rounds repeat until no cell is
// more than one hop from its root.
// ------------------------------------------------------------------------------------------------
constexpr int JUMP_HOPS = 6;

__global__ void __launch_bounds__(256) k_forest_jump(int *ptr, int64_t n, int *changed) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = ptr[i];
    if (p == (int)i) return;
    int q = ptr[p];
    if (q == p) return;
    bool more = true;
#pragma unroll 1
    for (int h = 0; h < JUMP_HOPS; h++) {
        p = q;
        q = ptr[p];
        if (q == p) { more = false; break; }
    }
    ptr[i] = q;
    if (more) *changed = 1;
}

__global__ void __launch_bounds__(256) k_forest_jump_list(int *ptr, const int *__restrict__ list, int n, int *changed) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int i = list[k];
    int p = ptr[i];
    if (p == i) return;
    int q = ptr[p];
    if (q == p) return;
    bool more = true;
#pragma unroll 1
    for (int h = 0; h < JUMP_HOPS; h++) {
        p = q;
        q = ptr[p];
        if (q == p) { more = false; break; }
    }
    ptr[i] = q;
    if (more) *changed = 1;
}

int forest_resolve_list(int *ptr, const int *list, int n_list, int64_t *rounds_out, cudaStream_t s) {
    int rounds = 0;
    if (n_list > 0) {
        DevBuf<int> flag;
        MS_TRY(flag.alloc(1, s));
        int64_t *h = host_flags().h;
        for (;;) {
            MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
            prof_units(n_list);
            MS_LAUNCH(k_forest_jump_list, cdiv(n_list, 256), 256, 0, s, ptr, list, n_list, flag.p);
            MS_TRY(ms::readback(h, flag.p, sizeof(int), s));
            MS_TRY(ms::stream_sync(s));
            rounds++;
            if (*(int *)h == 0) break;
            if (rounds >= 64) {
                set_error("forest_resolve: no convergence after %d rounds (cyclic pointers)", rounds);
                return MS_ERR_NOCONV;
            }
        }
    }
    if (rounds_out) *rounds_out = rounds;
    return MS_OK;
}

// The same jumping on catchment ids (the fill): lab[i] >= 0 is final, lab[i] < 0 links cell i to cell -(1 + lab[i])
// further down its path.  Only the cells in `list` hold links; each round they hop up to JUMP_HOPS links and write the
// last value back (a concurrent reader sees the old or the new value, both lie on the cell's path).
__global__ void __launch_bounds__(256) k_forest_jump_ids(int *lab, const int *__restrict__ list, int n, int *changed) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int i = list[k];
    int v = lab[i];
    if (v >= 0) return;
#pragma unroll 1
    for (int h = 0; h < JUMP_HOPS && v < 0; h++) v = lab[-(v + 1)];
    lab[i] = v;
    if (v < 0) *changed = 1;
}

int forest_resolve_ids(int *lab, const int *list, int n_list, int64_t *rounds_out, cudaStream_t s) {
    int rounds = 0;
    if (n_list > 0) {
        DevBuf<int> flag;
        MS_TRY(flag.alloc(1, s));
        int64_t *h = host_flags().h;
        for (;;) {
            MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
            prof_units(n_list);
            MS_LAUNCH(k_forest_jump_ids, cdiv(n_list, 256), 256, 0, s, lab, list, n_list, flag.p);
            MS_TRY(ms::readback(h, flag.p, sizeof(int), s));
            MS_TRY(ms::stream_sync(s));
            rounds++;
            if (*(int *)h == 0) break;
            if (rounds >= 64) {
                set_error("forest_resolve_ids: no convergence after %d rounds (cyclic links)", rounds);
                return MS_ERR_NOCONV;
            }
        }
    }
    if (rounds_out) *rounds_out = rounds;
    return MS_OK;
}

int forest_resolve(int *ptr, int64_t n, int64_t *rounds_out, cudaStream_t s) {
    DevBuf<int> flag;
    MS_TRY(flag.alloc(1, s));
    int64_t *h = host_flags().h;
    int rounds = 0;
    for (;;) {
        MS_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
        MS_LAUNCH(k_forest_jump, cdiv(n, 256), 256, 0, s, ptr, n, flag.p);
        MS_TRY(ms::readback(h, flag.p, sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        rounds++;
        if (*(int *)h == 0) break;
        if (rounds >= 64) {
            set_error("forest_resolve: no convergence after %d rounds (cyclic pointers)", rounds);
            return MS_ERR_NOCONV;
        }
    }
    if (rounds_out) *rounds_out = rounds;
    return MS_OK;
}

}  // namespace ms
