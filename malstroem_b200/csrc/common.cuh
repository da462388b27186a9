// common.cuh — shared helpers of the sm_100a raster kernels (error handling, stream-ordered scratch
// memory, order-preserving float keys, D8 neighbour tables).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/malstroem_b200.h"

namespace ms {

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const char *fmt, ...);
extern int64_t g_launches;

#define MS_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            ms::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return MS_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

#define MS_TRY(call)                \
    do {                            \
        int r__ = (call);           \
        if (r__ != MS_OK) return r__; \
    } while (0)

// optional per-kernel CUDA-event timing (ms_profile): one event pair per launch on the launching stream
extern int g_prof;
extern int64_t g_prof_units;      // "units" (cells) the next launch processes; consumed by prof_begin
void prof_begin(const char *name, cudaStream_t s);
void prof_end(cudaStream_t s);
static inline void prof_units(int64_t u) { g_prof_units = u; }

// kernel launch + error check + launch counter
#define MS_LAUNCH(kernel, grid, block, smem, stream, ...)                                    \
    do {                                                                                     \
        if (ms::g_prof) ms::prof_begin(#kernel, (stream));                                   \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                          \
        if (ms::g_prof) ms::prof_end((stream));                                              \
        ms::g_launches++;                                                                    \
        cudaError_t e__ = cudaGetLastError();                                                \
        if (e__ != cudaSuccess) {                                                            \
            ms::set_error("%s:%d: launch %s -> %s", __FILE__, __LINE__, #kernel,             \
                          cudaGetErrorString(e__));                                          \
            return MS_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)

int ensure_init();

// host-side accounting (ms_host_counters): wall time spent waiting in stream syncs and in pool allocations
extern double g_host_t[4];      // [0] sync seconds, [1] sync count, [2] alloc seconds, [3] alloc count
int stream_sync(cudaStream_t s);
double now_s();

// ---- scratch memory: one device arena, stack discipline ------------------------------------------
// All scratch of a call is carved from one cudaMalloc'ed arena with bump allocation (frees pop the top; an
// out-of-order free is deferred until the blocks above it are gone).  Work of one call is ordered on one
// stream, so a block can be handed out again without waiting.  The arena grows (when empty) to the high-water
// mark of the previous call; a request that does not fit meanwhile is served by cudaMallocAsync.  This
// replaced per-buffer cudaMallocAsync, whose pool re-mapped physical memory for the changing 256 MB-class
// requests and cost 7-46 ms per step at 8192^2 (profiles/r01_host_overhead.txt).
void *arena_alloc(size_t bytes, cudaStream_t s);
void arena_free(void *p, cudaStream_t s);
// bytes the arena can still hand out without a cudaMallocAsync (0 before a call has sized it)
size_t arena_room();

template <typename T>
struct DevBuf {
    T *p = nullptr;
    cudaStream_t s = nullptr;
    DevBuf() {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    int alloc(size_t n, cudaStream_t stream) {
        release();
        s = stream;
        if (n == 0) n = 1;
        double t0 = now_s();
        p = (T *)arena_alloc(n * sizeof(T), stream);
        g_host_t[2] += now_s() - t0;
        g_host_t[3] += 1;
        if (!p) {
            set_error("device scratch allocation of %zu bytes failed", n * sizeof(T));
            return MS_ERR_CUDA;
        }
        return MS_OK;
    }
    void release() {
        if (p) arena_free(p, s);
        p = nullptr;
    }
    ~DevBuf() { release(); }
    operator T *() const { return p; }
};

// pinned host scalar(s) for flags / counters that come back every round
struct HostFlags {
    int64_t *h = nullptr;
    int init();
};
HostFlags &host_flags();
// A few counters from the device into host_flags() memory WITHOUT the copy engine: a one-warp kernel stores them into
// the (mapped) pinned buffer.  A cudaMemcpyAsync read-back queues behind whatever device-to-host copy is running - with
// the rasters of a host-buffer run leaving over the copy stream, every per-round read-back of the later stages stood
// behind gigabytes (32768^2: K2 + K3 done after 220 ms instead of 57).  bytes: a multiple of 4, at most 4096.
int readback(void *host_pinned, const void *dev, size_t bytes, cudaStream_t s);

static inline unsigned int cdiv(int64_t a, int64_t b) { return (unsigned int)((a + b - 1) / b); }

// ---- order-preserving keys ----------------------------------------------------------------------
// okey(a) < okey(b)  <=>  a < b  for non-NaN floats, with -0.0 canonicalised to +0.0
__host__ __device__ inline uint32_t okey32(float f) {
    f = f + 0.0f;
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    union { float f; uint32_t u; } v; v.f = f; uint32_t b = v.u;
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ inline float okey32_inv(uint32_t k) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    union { float f; uint32_t u; } v; v.u = b; return v.f;
#endif
}
__device__ inline unsigned long long okey64(double d) {
    d = d + 0.0;
    unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ inline double okey64_inv(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// ---- D8 neighbour order of the reference (flow.py:30-38, _flow.pyx:36-46):
//      0 Up, 1 UpRight, 2 Right, 3 DownRight, 4 Down, 5 DownLeft, 6 Left, 7 UpLeft, 8 none
__device__ __constant__ const int kDR[8] = {-1, -1, 0, 1, 1, 1, 0, -1};
__device__ __constant__ const int kDC[8] = {0, 1, 1, 1, 0, -1, -1, -1};

// K3's per-cell rule (speedups/_flow.pyx:98-176): dz = z - nbr (edge) or (z - nbr) * INV_SQRT2 (diagonal), float64,
// strict `>` against a running maximum that starts at 0, neighbours in the order above; 8 when none is lower.
#ifdef __CUDACC__
__device__ inline int d8_code(double z, double up, double ur, double rt, double dr, double dn, double dl, double lf,
                              double ul, double inv_sqrt2) {
    int code = 8;
    double dzmax = 0.0, dz;
    dz = __dsub_rn(z, up);                        if (dz > dzmax) { dzmax = dz; code = 0; }
    dz = __dmul_rn(__dsub_rn(z, ur), inv_sqrt2);  if (dz > dzmax) { dzmax = dz; code = 1; }
    dz = __dsub_rn(z, rt);                        if (dz > dzmax) { dzmax = dz; code = 2; }
    dz = __dmul_rn(__dsub_rn(z, dr), inv_sqrt2);  if (dz > dzmax) { dzmax = dz; code = 3; }
    dz = __dsub_rn(z, dn);                        if (dz > dzmax) { dzmax = dz; code = 4; }
    dz = __dmul_rn(__dsub_rn(z, dl), inv_sqrt2);  if (dz > dzmax) { dzmax = dz; code = 5; }
    dz = __dsub_rn(z, lf);                        if (dz > dzmax) { dzmax = dz; code = 6; }
    dz = __dmul_rn(__dsub_rn(z, ul), inv_sqrt2);  if (dz > dzmax) { dzmax = dz; code = 7; }
    return code;
}
// the border rule of flow.py:118-139 in the reference's assignment order (rows, then columns, then corners)
__device__ inline int d8_border(int code, bool top, bool bot, int c, int cols) {
    const int mc = cols - 1;
    if (top) code = 0;
    if (bot) code = 4;
    if (c == 0) code = 6;
    if (c == mc) code = 2;
    if (top && c == 0) code = 7;
    if (top && c == mc) code = 1;
    if (bot && c == 0) code = 5;
    if (bot && c == mc) code = 3;
    return code;
}
#endif

// ---- shared device primitives (scan.cu, forest.cu) ----------------------------------------------
// exclusive scan of int32 flags; out may alias flags; *total_dev receives the sum (int64 on device)
int exclusive_scan_i32(const int *flags, int *out, int64_t n, int64_t *total_dev, cudaStream_t s);
// stable LSD sort of int (key, val) pairs on key bits [0, bits), one binary split per bit (network.cu: the network's
// upstream lists, flood.cu's large segments).  The passes ping-pong between the buffers; on return *key / *val point
// at the sorted pairs and *key_alt / *val_alt at the other pair of buffers.  flag: n ints of scratch.
int radix_sort_split(int **key, int **val, int **key_alt, int **val_alt, int *flag, int64_t *total, int n, int bits,
                     cudaStream_t s);
// pointer jumping on a forest given as parent indices (roots point to themselves); in place.
// rounds_out (host, optional) receives the number of rounds.  MS_ERR_NOCONV after 64 rounds (cycles).
int forest_resolve(int *ptr, int64_t n, int64_t *rounds_out, cudaStream_t s);

// ---- row-band context (SURVEY.md §8(e)) ------------------------------------------------------------
// One band of a raster split by rows across GPUs.  Raster pointers handed to the band entry points point at the
// band's first own row; when `open & MS_OPEN_TOP` the row before it in memory is a halo row (the last row of the
// band above), when `open & MS_OPEN_BOTTOM` a halo row follows the last own row.  The context keeps the device
// state that has to survive between the phases of a stage (the exchanges happen on the host side in between).
enum BandBuf {
    BB_LAB, BB_COMP, BB_E, BB_FROZEN, BB_FRANK, BB_HASHK, BB_HASHV,
    BB_ACC_X, BB_ACC_X0, BB_ACC_ENTRY_NEXT, BB_ACC_NEXT, BB_ACC_INDEG, BB_ACC_INDEG0, BB_ACC_ISEXIT, BB_ACC_LOC16,
    BB_CC_PARENT, BB_CC_RANK, BB_WS_PTR, BB_NF_FLAG, BB_NF_SIDES, BB_NF_RING, BB_NF_CTL, BB_MISC, BB_NF_DG, BB_NF_TMETA,
    BB_NF_IRBAD, BB_NF_BANNED, BB_BLIST, BB_COUNT
};
}  // namespace ms
struct ms_band {
    int64_t rows, cols;
    int open;
    void *buf[ms::BB_COUNT];
    size_t cap[ms::BB_COUNT];
    int nC;            // catchments of the band (fill)
    int nF;            // frozen components (fill)
    int gid_base;      // global id of the band's first frozen component
    // no-flats solver fused over NVLink peer memory (noflats.cu): this band's shared block, the other ranks' blocks
    // as mapped here, and the device copy of the kernel's peer table
    void *nf_shared;
    void *nf_peer[16];
    int nf_peer_ipc[16];   // 1: mapped with cudaIpcOpenMemHandle (must be closed)
    int nf_rank, nf_world;
    void *nf_pp_dev;
    int n_blist;       // BB_BLIST: cells that still had a neighbour in another component when the local fill ended
    int nf_ban;        // BB_NF_BANNED holds seeds the verification stencil rejected (ms_band_nf_ban_dev)
};
namespace ms {
void *band_buf(ms_band *b, int slot, size_t bytes);      // grow-only cudaMalloc'ed buffer of the context

// pointer jumping restricted to the cells in `list` (device, n_list entries): every other cell already points at its
// root or at a listed cell.  Used after a tile-local compression (k_descent_tile, k_ws_tile).
int forest_resolve_list(int *ptr, const int *list, int n_list, int64_t *rounds_out, cudaStream_t s);
// the same for the fill's catchment ids (k_descent_tile): lab[i] >= 0 is an id, lab[i] < 0 a link to cell -(1 + lab[i]);
// only the cells in `list` hold links.  Afterwards every listed cell holds an id.
int forest_resolve_ids(int *lab, const int *list, int n_list, int64_t *rounds_out, cudaStream_t s);

#ifdef __CUDACC__
// ---- tile-local pointer compression (64x64 tiles, 256 threads, 16 cells per thread) -----------------------------
// sp[k] = tile-local parent of cell k (roots point at themselves).  Asynchronous pointer doubling in shared memory:
// a reader sees the old or the new parent, both are ancestors.
constexpr int FT = 64;
__device__ inline void tile_pointer_double(unsigned short *sp) {
    for (;;) {
        int changed = 0;
#pragma unroll 4
        for (int u = 0; u < 16; u++) {
            int k = threadIdx.x + 256 * u;
            unsigned short p = sp[k], pp = sp[p];
            if (pp != p) { sp[k] = pp; changed = 1; }
        }
        if (!__syncthreads_or(changed)) break;
    }
}

// block-aggregated append: `cnt` entries of this thread (in order) go to list_out at the returned position
__device__ inline int block_append_pos(int cnt, int *n_out) {
    __shared__ int wsum_[8];
    __shared__ int base_;
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) wsum_[w] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int k = 0; k < 8; k++) { int t = wsum_[k]; wsum_[k] = tot; tot += t; }
        base_ = tot ? atomicAdd(n_out, tot) : 0;
    }
    __syncthreads();
    return base_ + wsum_[w] + inc - cnt;
}
#endif

// ---- device twins of host rasters (cache.cu): used by the host-pointer entry points -----------------------------
void cache_begin_call();
void cache_end_call();
int cache_input(const void *host, size_t bytes, cudaStream_t s, void **dev_out);
int cache_output(size_t bytes, void **dev_out);
void cache_bind_host(void *dev, const void *host, size_t bytes);
void cache_bind_derived(void *dev, const void *src, int kind, double a, double b);
void *cache_find_derived(const void *src, int kind, double a, double b);
void cache_clear_all();
enum { CK_FILLED = 1, CK_DEPTHS = 2, CK_NOFLATS = 3 };
// one host-pointer call: inputs come from the cache (or are uploaded into it), results live in it afterwards
struct HostCall {
    HostCall() { cache_begin_call(); }
    ~HostCall() { cache_end_call(); }
    template <class T> int in(const T *host, size_t count, cudaStream_t s, T **dev) {
        void *p = nullptr;
        int rc = cache_input(host, count * sizeof(T), s, &p);
        *dev = (T *)p;
        return rc;
    }
    template <class T> int out(size_t count, T **dev) {
        void *p = nullptr;
        int rc = cache_output(count * sizeof(T), &p);
        *dev = (T *)p;
        return rc;
    }
};

// polygon.cu: frees the rings held for ms_polygonize_fetch
void poly_release();

// internal device-pointer stage entry points used by the pipeline (pipeline.cu)
// minmax_out (optional, 2 floats on the device): min / max of dtm, as minmax_dev computes them
int fill_terrain_dev_impl(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols,
                          int64_t *stats, cudaStream_t s, float *minmax_out = nullptr);

}  // namespace ms
