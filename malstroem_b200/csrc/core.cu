// core.cu — library state: device selection, stream-ordered memory pool, error string, pinned flags.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "tma.cuh"

namespace ms {

static thread_local char g_err[1024] = "";
int64_t g_launches = 0;
static int g_device = -1;
static HostFlags g_flags;

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

double g_host_t[4] = {0, 0, 0, 0};
double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
int stream_sync(cudaStream_t s) {
    double t0 = now_s();
    cudaError_t e = cudaStreamSynchronize(s);
    g_host_t[0] += now_s() - t0;
    g_host_t[1] += 1;
    if (e != cudaSuccess) {
        set_error("cudaStreamSynchronize -> %s", cudaGetErrorString(e));
        return MS_ERR_CUDA;
    }
    return MS_OK;
}

// ---- scratch arena ---------------------------------------------------------------------------------
struct ArenaBlock { size_t off, size; bool live; };
static char *g_arena = nullptr;
static size_t g_arena_cap = 0, g_arena_top = 0, g_arena_need = 0, g_overflow_live = 0;
static std::vector<ArenaBlock> g_blocks;
static cudaStream_t g_arena_stream = nullptr;
static std::map<void *, size_t> g_overflow;

void *arena_alloc(size_t bytes, cudaStream_t s) {
    bytes = (bytes + 511) & ~(size_t)511;
    if (s != g_arena_stream) {
        // blocks are recycled in stream order: switching streams must wait for the previous one
        if (g_arena) cudaStreamSynchronize(g_arena_stream);
        g_arena_stream = s;
    }
    if (g_blocks.empty() && g_overflow.empty() && g_arena_need > g_arena_cap) {
        if (g_arena) cudaFree(g_arena);
        g_arena = nullptr;
        size_t want = g_arena_need + (g_arena_need >> 3);
        if (cudaMalloc((void **)&g_arena, want) == cudaSuccess) g_arena_cap = want;
        else { g_arena_cap = 0; cudaGetLastError(); }
        g_arena_top = 0;
    }
    size_t virt = g_arena_top + g_overflow_live + bytes;
    if (virt > g_arena_need) g_arena_need = virt;
    if (g_arena && g_arena_top + bytes <= g_arena_cap) {
        g_blocks.push_back({g_arena_top, bytes, true});
        void *p = g_arena + g_arena_top;
        g_arena_top += bytes;
        return p;
    }
    void *p = nullptr;
    if (cudaMallocAsync(&p, bytes, s) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    g_overflow[p] = bytes;
    g_overflow_live += bytes;
    return p;
}

void arena_free(void *p, cudaStream_t s) {
    auto it = g_overflow.find(p);
    if (it != g_overflow.end()) {
        g_overflow_live -= it->second;
        g_overflow.erase(it);
        cudaFreeAsync(p, s);
        return;
    }
    size_t off = (size_t)((char *)p - g_arena);
    for (size_t k = g_blocks.size(); k-- > 0;)
        if (g_blocks[k].off == off) { g_blocks[k].live = false; break; }
    while (!g_blocks.empty() && !g_blocks.back().live) {
        g_arena_top = g_blocks.back().off;
        g_blocks.pop_back();
    }
}

size_t arena_room() { return g_arena ? g_arena_cap - g_arena_top : 0; }

// ---- per-kernel event timing -------------------------------------------------------------------
int g_prof = 0;
int64_t g_prof_units = 0;
struct ProfRec { const char *name; cudaEvent_t a, b; int64_t units; };
static std::vector<ProfRec> g_recs;
static std::vector<cudaEvent_t> g_evpool;

static cudaEvent_t ev_get() {
    if (!g_evpool.empty()) { cudaEvent_t e = g_evpool.back(); g_evpool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void prof_begin(const char *name, cudaStream_t s) {
    ProfRec r;
    r.name = name; r.a = ev_get(); r.b = ev_get(); r.units = g_prof_units;
    g_prof_units = 0;
    cudaEventRecord(r.a, s);
    g_recs.push_back(r);
}

void prof_end(cudaStream_t s) { cudaEventRecord(g_recs.back().b, s); }

int HostFlags::init() {
    if (h) return MS_OK;
    MS_CUDA(cudaHostAlloc((void **)&h, 64 * sizeof(int64_t), cudaHostAllocMapped | cudaHostAllocPortable));
    memset(h, 0, 64 * sizeof(int64_t));
    return MS_OK;
}
HostFlags &host_flags() { return g_flags; }

__global__ void k_readback(const uint32_t *__restrict__ src, uint32_t *dst_host, int words) {
    for (int k = threadIdx.x; k < words; k += blockDim.x) dst_host[k] = src[k];
    __threadfence_system();
}

int readback(void *host_pinned, const void *dev, size_t bytes, cudaStream_t s) {
    if ((bytes & 3) || bytes > 4096 || ((uintptr_t)dev & 3) || ((uintptr_t)host_pinned & 3)) {
        MS_CUDA(cudaMemcpyAsync(host_pinned, dev, bytes, cudaMemcpyDeviceToHost, s));
        return MS_OK;
    }
    MS_LAUNCH(k_readback, 1, 32, 0, s, (const uint32_t *)dev, (uint32_t *)host_pinned, (int)(bytes >> 2));
    return MS_OK;
}

static int init_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("no CUDA device available (%s): malstroem_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return MS_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        set_error("device %d out of range (have %d)", device, n);
        return MS_ERR_ARG;
    }
    MS_CUDA(cudaSetDevice(device));
    // keep freed scratch memory in the pool instead of returning it to the driver after every call
    cudaMemPool_t pool;
    MS_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thresh = UINT64_MAX;
    MS_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
    MS_TRY(g_flags.init());
    g_device = device;
    return MS_OK;
}

void *band_buf(ms_band *b, int slot, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b->cap[slot] >= bytes) return b->buf[slot];
    if (b->buf[slot]) {
        cudaDeviceSynchronize();
        cudaFree(b->buf[slot]);
        b->buf[slot] = nullptr;
        b->cap[slot] = 0;
    }
    size_t want = bytes + (bytes >> 3);
    void *p = nullptr;
    if (cudaMalloc(&p, want) != cudaSuccess) {
        cudaGetLastError();
        set_error("band context: cudaMalloc(%zu) failed", want);
        return nullptr;
    }
    b->buf[slot] = p;
    b->cap[slot] = want;
    return p;
}

// ---- TMA tensor maps (tma.cuh) ---------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int g_encode_tried = 0;

bool tma_map_2d(CUtensorMap *out, const void *base, int64_t rows, int64_t cols, int box_rows, int box_cols, bool is_float,
                bool nan_fill) {
    if (!g_encode_tried) {
        g_encode_tried = 1;
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            g_encode = (EncodeTiledFn)fn;
        else
            cudaGetLastError();
    }
    if (getenv("MS_TMA_DEBUG") && !g_encode) fprintf(stderr, "tma_map_2d: no cuTensorMapEncodeTiled entry point\n");
    if (!g_encode || ((uintptr_t)base & 15) || (cols & 3) || ((box_cols * 4) & 15) || box_rows > 256 || box_cols > 256 ||
        rows < 1 || cols < 1)
        return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(out, is_float ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_INT32, 2, (void *)base,
                          dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          nan_fill ? CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA : CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (getenv("MS_TMA_DEBUG"))
        fprintf(stderr, "tma_map_2d(base %p, %lld x %lld, box %d x %d) -> CUresult %d\n", base, (long long)rows,
                (long long)cols, box_rows, box_cols, (int)r);
    return r == CUDA_SUCCESS;
}

int ensure_init() {
    if (g_device >= 0) {
        // another library (torch) may have switched the current device of this thread
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && cur != g_device) MS_CUDA(cudaSetDevice(g_device));
        return MS_OK;
    }
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    return init_device(cur);
}

}  // namespace ms

extern "C" {

/* Host side of the row-band connected components (SURVEY.md §8(e), K5/K6): components that touch across a band edge
 * are merged; a merged component keeps its smallest root (global cell index).  root_top / root_bot hold, for each
 * of the G bands, the root of every cell of the band's first / last row (-1 = background), G * cols entries each.
 * Output: every distinct root seen on an interior band edge, ascending, with the root of its merged component.
 * Pure CPU code (a few thousand cells): runs identically on every rank. */
static int cc_boundary_merge(int nbands, int64_t cols, const int64_t *root_top, const int64_t *root_bot,
                             const int32_t *val_top, const int32_t *val_bot, int connect8, int64_t *out_root,
                             int64_t *out_global, int64_t capacity, int64_t *n_out) {
    if (nbands < 1 || cols < 1 || !root_top || !root_bot || !n_out || (!val_top != !val_bot)) { ms::set_error("cc_boundary_merge: bad argument"); return MS_ERR_ARG; }
    // distinct roots: cells of one component are consecutive along a row, so only the first cell of each run is kept
    // before sorting (a few thousand ids instead of 2 * cols per band edge)
    std::vector<int64_t> ids;
    for (int g = 0; g + 1 < nbands; g++) {
        const int64_t *rows2[2] = {root_bot + (int64_t)g * cols, root_top + (int64_t)(g + 1) * cols};
        for (int k = 0; k < 2; k++) {
            int64_t prev = -1;
            for (int64_t c = 0; c < cols; c++) {
                int64_t v = rows2[k][c];
                if (v >= 0 && v != prev) ids.push_back(v);
                prev = v;
            }
        }
    }
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    std::vector<int> parent(ids.size());
    for (size_t k = 0; k < ids.size(); k++) parent[k] = (int)k;
    auto find = [&](int x) {
        while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
        return x;
    };
    auto index_of = [&](int64_t v) { return (int)(std::lower_bound(ids.begin(), ids.end(), v) - ids.begin()); };
    for (int g = 0; g + 1 < nbands; g++) {
        const int64_t *bot = root_bot + (int64_t)g * cols, *top = root_top + (int64_t)(g + 1) * cols;
        const int32_t *vb = val_bot ? val_bot + (int64_t)g * cols : nullptr, *vt = val_top ? val_top + (int64_t)(g + 1) * cols : nullptr;
        int64_t last_a = -1, last_b = -1;
        for (int64_t c = 0; c < cols; c++) {
            int64_t a = bot[c];
            if (a < 0) continue;
            for (int64_t d = -1; d <= 1; d++) {
                if (c + d < 0 || c + d >= cols || (d != 0 && !connect8) || (vb && vb[c] != vt[c + d])) continue;
                int64_t b = top[c + d];
                if (b < 0 || (a == last_a && b == last_b)) continue;      // the same pair again along a run
                last_a = a;
                last_b = b;
                int x = find(index_of(a)), y = find(index_of(b));
                if (x == y) continue;
                if (x < y) parent[y] = x; else parent[x] = y;      // ids ascend with the cell index: smaller index wins
            }
        }
    }
    *n_out = (int64_t)ids.size();
    if ((int64_t)ids.size() > capacity) { ms::set_error("cc_boundary_merge: %zu roots do not fit capacity %lld", ids.size(), (long long)capacity); return MS_ERR_ARG; }
    for (size_t k = 0; k < ids.size(); k++) {
        if (out_root) out_root[k] = ids[k];
        if (out_global) out_global[k] = ids[find((int)k)];
    }
    return MS_OK;
}

int ms_cc_boundary_merge(int nbands, int64_t cols, const int64_t *root_top, const int64_t *root_bot,
                         int64_t *out_root, int64_t *out_global, int64_t capacity, int64_t *n_out) {
    return cc_boundary_merge(nbands, cols, root_top, root_bot, nullptr, nullptr, 1, out_root, out_global, capacity, n_out);
}

int ms_cc_boundary_merge_values(int nbands, int64_t cols, const int64_t *root_top, const int64_t *root_bot,
                                const int32_t *val_top, const int32_t *val_bot, int connect8, int64_t *out_root,
                                int64_t *out_global, int64_t capacity, int64_t *n_out) {
    if (!val_top || !val_bot) { ms::set_error("cc_boundary_merge_values: null value rows"); return MS_ERR_ARG; }
    return cc_boundary_merge(nbands, cols, root_top, root_bot, val_top, val_bot, connect8, out_root, out_global,
                             capacity, n_out);
}

int ms_version(void) { return 110; }

int ms_band_create(int64_t rows, int64_t cols, int open, ms_band **out) {
    MS_TRY(ms::ensure_init());
    if (!out || rows < 2 || cols < 3 || rows * cols > (1ll << 29) || (open & ~3) || ((open & 2) && (rows % 64))) {
        ms::set_error("ms_band_create: unsupported band %lld x %lld (open %d)", (long long)rows, (long long)cols, open);
        return MS_ERR_SHAPE;
    }
    ms_band *b = new ms_band();
    memset(b, 0, sizeof(*b));
    b->rows = rows;
    b->cols = cols;
    b->open = open;
    *out = b;
    return MS_OK;
}

int ms_band_destroy(ms_band *b) {
    if (!b) return MS_OK;
    cudaDeviceSynchronize();
    for (int k = 0; k < 16; k++)
        if (b->nf_peer[k] && b->nf_peer_ipc[k]) cudaIpcCloseMemHandle(b->nf_peer[k]);
    for (int k = 0; k < ms::BB_COUNT; k++)
        if (b->buf[k] && b->cap[k] != SIZE_MAX) cudaFree(b->buf[k]);      // SIZE_MAX: a view into nf_shared
    if (b->nf_shared) cudaFree(b->nf_shared);
    if (b->nf_pp_dev) cudaFree(b->nf_pp_dev);
    delete b;
    return MS_OK;
}

int ms_init(int device) {
    if (ms::g_device == device) return MS_OK;
    if (ms::g_device >= 0) {
        // the scratch arena, the pinned flags, the copy stream and the raster cache belong to the first device: a
        // second device in the same process would run on the first one's memory.  Multi-GPU = one process per GPU.
        ms::set_error("ms_init(%d): the library of this process is bound to device %d (one process per GPU; "
                      "ms_shutdown() first to rebind)", device, ms::g_device);
        return MS_ERR_ARG;
    }
    return ms::init_device(device);
}

int ms_shutdown(void) {
    if (ms::g_device < 0) return MS_OK;
    cudaDeviceSynchronize();
    ms::cache_clear_all();
    ms::poly_release();
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, ms::g_device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    if (ms::g_blocks.empty() && ms::g_arena) {
        cudaFree(ms::g_arena);
        ms::g_arena = nullptr;
        ms::g_arena_cap = ms::g_arena_top = 0;
        ms::g_device = -1;          // nothing of the old device is left: ms_init may bind another one
    }
    return MS_OK;
}

const char *ms_last_error(void) { return ms::g_err; }

int ms_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int64_t ms_kernel_launches(int reset) {
    int64_t v = ms::g_launches;
    if (reset) ms::g_launches = 0;
    return v;
}

int ms_host_counters(double *out4, int reset) {
    for (int k = 0; k < 4; k++) {
        if (out4) out4[k] = ms::g_host_t[k];
        if (reset) ms::g_host_t[k] = 0;
    }
    return MS_OK;
}

int ms_profile(int enable) {
    // enable > 1: also pre-create that many event pairs now, so that no cudaEventCreate falls inside a timed region
    for (int64_t k = (int64_t)ms::g_evpool.size(); k < 2ll * enable && enable > 1; k++) {
        cudaEvent_t e;
        MS_CUDA(cudaEventCreate(&e));
        ms::g_evpool.push_back(e);
    }
    ms::g_prof = enable ? 1 : 0;
    return MS_OK;
}

// one line per kernel: "<name> <launches> <total ms> <total units>"; clears the records
int ms_profile_report(char *buf, int64_t cap) {
    if (!buf || cap < 1) return MS_ERR_ARG;
    MS_CUDA(cudaDeviceSynchronize());
    struct Agg { int64_t n = 0; double ms = 0; int64_t units = 0; };
    std::map<std::string, Agg> agg;
    for (auto &r : ms::g_recs) {
        float t = 0;
        cudaEventElapsedTime(&t, r.a, r.b);
        Agg &a = agg[r.name];
        a.n++; a.ms += t; a.units += r.units;
        ms::g_evpool.push_back(r.a);
        ms::g_evpool.push_back(r.b);
    }
    ms::g_recs.clear();
    std::string out;
    char line[256];
    for (auto &kv : agg) {
        snprintf(line, sizeof(line), "%s %lld %.6f %lld\n", kv.first.c_str(), (long long)kv.second.n, kv.second.ms,
                 (long long)kv.second.units);
        out += line;
    }
    if ((int64_t)out.size() + 1 > cap) return MS_ERR_ARG;
    memcpy(buf, out.c_str(), out.size() + 1);
    return MS_OK;
}

void *ms_host_alloc(int64_t bytes) {
    void *p = nullptr;
    if (ms::ensure_init() != MS_OK) return nullptr;
    if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) {
        ms::set_error("cudaHostAlloc(%lld) failed", (long long)bytes);
        return nullptr;
    }
    return p;
}

int ms_host_free(void *p) {
    if (p) MS_CUDA(cudaFreeHost(p));
    return MS_OK;
}

}  // extern "C"
