// noflats.cu — K2: the epsilon-sloped ("no flats") depression fill in float64.
//
// Replaces fill.fill_terrain_no_flats (malstroem/algorithms/fill.py:174-232; sweep
// speedups/_fill.pyx:72-124): the fixed point of
//      W(c) = max( z(c), min( min4diag W + diag, min4edge W + short ) ),   W = z on the raster border,
// reached by the reference from W = +inf with raster-wide Gauss-Seidel sweeps.  For short, diag > 0 the
// fixed point is unique (SURVEY.md A.2), so any schedule that ends in a state where the equation holds
// at every interior cell has the reference's bits.
//
// Schedule used here ("seed, relax from above with a persistent tile solver, certify"):
//   k_nf_init    a dry cell (plain fill F == z) that has a strictly lower filled neighbour is seeded with
//                W = z; every other interior cell starts at +inf (these are the lake / flat cells, 20-35 %
//                of a fractal DEM).  Tiles holding a non-seed cell become active.
//   k_nf_solve   ONE cooperative launch, CTAs resident on every SM, fed by a device-side FIFO of active 64x64
//                tiles (ticket ring buffer; a counter of queued + running tiles ends the kernel).  A tile +
//                1-cell apron is held in shared memory and relaxed block-wise: the tile is 8x8 blocks of 8x8
//                cells, a 64-bit mask says which blocks may still change, a warp takes a dirty block (2 cells
//                per lane), iterates it until it is quiet and marks the neighbouring blocks whose edge it
//                changed.  Work therefore follows the wave fronts instead of sweeping 4096 cells per pass.  A
//                tile whose outer ring changed queues its neighbours (per-tile flag word = which of its sides
//                must be looked at).  No rounds, no host round trips: a wave moves on as soon as the tile it
//                leaves has been written back.
//   k_nf_verify  one stencil pass checks the equation everywhere.  Relaxed cells satisfy it by
//                construction; a seed can only fail by being too LOW (its lower neighbour is closer than
//                the accumulated epsilons).  Failing seeds are banned and the solve restarts — the result
//                that passes is certified by uniqueness.
//
// CAP (fast path, certified by the same verification): in the solver `sz` holds the plain fill F instead of z
// and candidates above F + capB are ignored.  Every candidate is an upper bound of the solution, the solution
// is >= F >= z so max(., z) never binds on a non-seed cell, and the solution lies within (#non-seed cells) *
// diag of F; a higher candidate (typically from a shore cell millimetres above a lake) can only be provisional
// garbage that the wave from the lake's outlet would overwrite.  Ignoring it is safe for a from-above
// relaxation (the cell just stays at +inf longer) and keeps the work proportional to the lake area.  If the
// verification fails, the solve is repeated without the cap.
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "common.cuh"
#include "tma.cuh"

namespace cg = cooperative_groups;

namespace ms {

constexpr int NF_T = 64;             // tile edge
constexpr int NF_LD = NF_T + 3;      // shared row stride in doubles (odd: spreads the rows of a block over banks)
constexpr int NF_SMEM = (NF_T + 2) * NF_LD * 8 + NF_T * NF_T * 4;
constexpr int NF_BLOCK_ITERS = 64;   // in-block iteration guard (a block that hits it stays dirty)

#ifdef NF_STATS
__device__ unsigned long long g_nf_dbg[16];
__device__ unsigned long long g_nf_log[4 * 262144];     // per visit: t_pop, t_loaded, t_end, tile | iters << 32
__device__ unsigned long long g_nf_hist[1024];          // per 65.5 us of the solve: visits started, ns spent in them
__device__ unsigned long long g_nf_t0;                  // earliest visit start seen (reset to ~0)
__device__ unsigned int g_nf_nlog;   // [0] tile iterations [1] block visits [2] block iterations [3] -, then per round (n, ns)
__device__ inline unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#endif

struct NfCtl {
    unsigned head, tail;   // FIFO tickets: next entry to take / next entry to fill
    int pending;           // tiles queued or being processed
    int done;              // 1: no work left; 2: a consumer gave up waiting (watchdog)
    int nonseed;           // cells k_nf_init left at +inf
    int nviol;             // cells failing k_nf_verify
    int visits;
    int reserved;
};

// wall-clock watchdog of the persistent solvers (ADVICE r1: a spin count trips under a profiler, compute-sanitizer or a
// time-sliced GPU): a consumer that has waited this long for work gives up and stops every CTA
constexpr unsigned long long NF_WATCHDOG_NS = 20ull * 1000ull * 1000ull * 1000ull;
__device__ inline unsigned long long nf_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ inline double dmin2(double a, double b) { return a <= b ? a : b; }
__device__ inline double dmin4(double a, double b, double c, double d) { return dmin2(dmin2(a, b), dmin2(c, d)); }

__global__ void __launch_bounds__(256) k_nf_init(const float *__restrict__ z, const float *__restrict__ F,
                                                 double *__restrict__ W, const uint8_t *__restrict__ banned,
                                                 int *tileflag, int *tilesides, NfCtl *ctl, int rows, int cols,
                                                 int tiles_x, int open) {
    int c = blockIdx.x * 64 + (threadIdx.x & 63);
    int r = blockIdx.y * 4 + (threadIdx.x >> 6);
    bool nonseed = false;
    if (r < rows && c < cols) {
        int i = r * cols + c;
        float zc = z[i];
        if ((r == 0 && !(open & 1)) || c == 0 || (r == rows - 1 && !(open & 2)) || c == cols - 1) {
            W[i] = (double)zc;
        } else {
            float f = F[i];
            float m = INFINITY;
#pragma unroll
            for (int dr = -1; dr <= 1; dr++)
#pragma unroll
                for (int dc = -1; dc <= 1; dc++) {
                    if (dr == 0 && dc == 0) continue;
                    m = fminf(m, __ldg(F + i + dr * cols + dc));
                }
            bool seed = (f == zc) && (m < f) && !(banned && banned[i]);
            W[i] = seed ? (double)zc : (double)INFINITY;
            nonseed = !seed;
        }
    }
    // the 4 rows x 64 columns of this CTA lie in one tile
    int cnt = __syncthreads_count(nonseed);
    int tile = ((blockIdx.y * 4) / NF_T) * tiles_x + blockIdx.x;
    if (threadIdx.x == 0 && cnt) {
        atomicAdd(&ctl->nonseed, cnt);
        tileflag[tile] = 16;
    }
    // sides of the tile along which a lake / flat cell lies (only those can be affected from outside)
    if (nonseed) {
        int lr = r & (NF_T - 1), lc = c & (NF_T - 1);
        int sides = (lr == 0 ? 1 : 0) | (lr == NF_T - 1 || r == rows - 2 ? 2 : 0) | (lc == 0 ? 4 : 0) |
                    (lc == NF_T - 1 || c == cols - 2 ? 8 : 0);
        if (sides) atomicOr(tilesides + tile, sides);
    }
}

// flagged tiles -> the FIFO (flags stay set: the solver clears a tile's flag word when it takes the tile)
__global__ void __launch_bounds__(256) k_nf_compact(const int *tileflag, int *ring, NfCtl *ctl, int ntiles) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntiles) return;
    if (tileflag[t]) {
        ring[atomicAdd(&ctl->tail, 1u)] = t;
        atomicAdd(&ctl->pending, 1);
    }
}

// ---- in-tile relaxation -------------------------------------------------------------------------------
// A warp relaxes one 8x8 block until it is quiet.  Lane l owns cells (row l/4, columns 2*(l%4), +1).  block()
// returns whether anything changed; `sides` bit 0/1/2/3 = the block's top / bottom / left / right edge changed,
// bit 4 = the iteration guard was hit (block must stay dirty).
__device__ inline unsigned nf_sides(unsigned bal) {
    unsigned sd = 0;
    if (bal & 0x0000000fu) sd |= 1u;
    if (bal & 0xf0000000u) sd |= 2u;
    if (bal & 0x11111111u) sd |= 4u;
    if (bal & 0x88888888u) sd |= 8u;
    return sd;
}

template <bool CAP>
struct RelaxF64 {
    double *sw;
    const float *sz;
    double sh, dg, capB;
    __device__ inline bool block(int b, unsigned *sides) const {
        const unsigned full = 0xffffffffu;
        int lane = threadIdx.x & 31;
        int lr = (b >> 3) * 8 + (lane >> 2), lc = (b & 7) * 8 + (lane & 3) * 2;
        double *p = sw + (lr + 1) * NF_LD + (lc + 1);
        float2 zz = *reinterpret_cast<const float2 *>(sz + lr * NF_T + lc);
        double z0 = (double)zz.x, z1 = (double)zz.y;
        double w0 = p[0], w1 = p[1];
        bool live = (w0 > z0) || (w1 > z1);
        *sides = 0;
        if (!__any_sync(full, live)) return false;
        unsigned sd = 0;
        bool any = false;
        for (int it = 0;; it++) {
            bool ch = false;
            if (live) {
                double a0 = p[-NF_LD - 1], a1 = p[-NF_LD], a2 = p[-NF_LD + 1], a3 = p[-NF_LD + 2];
                double l = p[-1], r = p[2];
                double c0 = p[NF_LD - 1], c1 = p[NF_LD], c2 = p[NF_LD + 1], c3 = p[NF_LD + 2];
                if (w0 > z0) {
                    double m = dmin2(__dadd_rn(dmin4(a0, a2, c0, c2), dg), __dadd_rn(dmin4(a1, l, w1, c1), sh));
                    if (!CAP) m = m >= z0 ? m : z0;
                    if (m < w0 && (!CAP || m <= z0 + capB)) { w0 = m; p[0] = m; ch = true; }
                }
                if (w1 > z1) {
                    double m = dmin2(__dadd_rn(dmin4(a1, a3, c1, c3), dg), __dadd_rn(dmin4(a2, w0, r, c2), sh));
                    if (!CAP) m = m >= z1 ? m : z1;
                    if (m < w1 && (!CAP || m <= z1 + capB)) { w1 = m; p[1] = m; ch = true; }
                }
            }
            __syncwarp();
            unsigned bal = __ballot_sync(full, ch);
            if (!bal) break;
            any = true;
            sd |= nf_sides(bal);
            if (it == NF_BLOCK_ITERS - 1) { sd |= 16u; break; }
        }
        *sides = sd;
        return any;
    }
};

// Integer form of the same relaxation for a tile whose lake / flat cells all lie in one float64 binade (the
// common case): there W = F + D * ulp with an integer D, `x (+) short` adds exactly sq ulps and `x (+) diag` rounds
// to exactly dq ulps more (SURVEY.md F4), so the relaxation is an integer chamfer distance transform.  Cells that
// cannot change (seeds, the raster border, cells outside the raster) are walls; they were taken into account as
// sources once, by k_nf_seedcand.
constexpr int NF_ILD = NF_T + 8;          // shared row stride in ints: even (64-bit pair loads), 8 banks per row
constexpr int D_INF = 0x3fffffff;         // lake cell not reached yet
constexpr int D_WALL = 0x40000000;        // not updatable, not a source
constexpr int D_LIMIT = 0x20000000;       // a tile whose distances get this large is left to the float64 form

__device__ inline int imin4(int a, int b, int c, int d) { return min(min(a, b), min(c, d)); }

constexpr int NF_NBIN = 8;               // binades a tile may span in the integer form

struct RelaxI32 {
    int *sd;
    const unsigned char *se;   // per interior cell: low byte of the binade exponent of its F
    const int2 *wtab;          // (short, diag) in ulps for binade elo + k
    int elo8;                  // low byte of the tile's lowest binade exponent
    int *overflow;             // set when a distance leaves the range the integer form is trusted for
    __device__ inline int2 weights(int lr, int lc) const {
        return wtab[(se[lr * NF_T + lc] - elo8) & (NF_NBIN - 1)];
    }
    __device__ inline bool block(int b, unsigned *sides) const {
        const unsigned full = 0xffffffffu;
        int lane = threadIdx.x & 31;
        int lr = (b >> 3) * 8 + (lane >> 2), lc = (b & 7) * 8 + (lane & 3) * 2;
        int *p = sd + (lr + 1) * NF_ILD + (lc + 1);
        int w0 = p[0], w1 = p[1];
        bool live = (w0 <= D_INF) || (w1 <= D_INF);
        *sides = 0;
        if (!__any_sync(full, live)) return false;
        // neighbouring lake cells share their F, hence their binade: a cell's own weights apply to all its inputs
        int sq = 0, dq = 0, sq1 = 0, dq1 = 0;
        if (live) {
            int2 wa = weights(lr, lc), wb = weights(lr, lc + 1);
            sq = wa.x; dq = wa.y; sq1 = wb.x; dq1 = wb.y;
        }
        unsigned sds = 0;
        bool any = false;
        for (int it = 0;; it++) {
            bool ch = false;
            if (live) {
                // the 3 x 4 window as six aligned pairs (the own cells are re-read with their neighbours)
                const int2 ua = *reinterpret_cast<const int2 *>(p - NF_ILD - 1), ub = *reinterpret_cast<const int2 *>(p - NF_ILD + 1);
                const int2 ma = *reinterpret_cast<const int2 *>(p - 1), mb = *reinterpret_cast<const int2 *>(p + 1);
                const int2 da = *reinterpret_cast<const int2 *>(p + NF_ILD - 1), db = *reinterpret_cast<const int2 *>(p + NF_ILD + 1);
                const int a0 = ua.x, a1 = ua.y, a2 = ub.x, a3 = ub.y, l = ma.x, r = mb.y;
                const int c0 = da.x, c1 = da.y, c2 = db.x, c3 = db.y;
                if (w0 <= D_INF) {
                    int m = min(imin4(a0, a2, c0, c2) + dq, imin4(a1, l, w1, c1) + sq);
                    if (m < w0) { w0 = m; p[0] = m; ch = true; if (m >= D_LIMIT) *overflow = 1; }
                }
                if (w1 <= D_INF) {
                    int m = min(imin4(a1, a3, c1, c3) + dq1, imin4(a2, w0, r, c2) + sq1);
                    if (m < w1) { w1 = m; p[1] = m; ch = true; if (m >= D_LIMIT) *overflow = 1; }
                }
            }
            __syncwarp();
            unsigned bal = __ballot_sync(full, ch);
            if (!bal) break;
            any = true;
            sds |= nf_sides(bal);
            if (it == NF_BLOCK_ITERS - 1) { sds |= 16u; break; }
        }
        *sides = sds;
        return any;
    }
};

struct NfTileShared {
    unsigned long long dirty[3];
    unsigned long long chgmask;
    int ring;          // bit 0/1/2/3: the tile's top / bottom / left / right ring changed
    int nb;            // neighbour tiles to queue: bit (dy+1)*3 + (dx+1)
    int grab[3];       // next dirty block to hand out (per iteration, rotating like `dirty`)
    unsigned char blist[64];   // the dirty blocks of the current iteration
    int2 wtab[NF_NBIN];
    int k;             // ticket
    int flags;         // side bits this tile was queued with
    int e, elo;        // largest / smallest binade exponent of the tile's lake cells (integer form needs e == elo)
    int bad;           // tile does not qualify for the integer form
    int dmax;          // largest finite distance loaded
    int any;           // sweeps: some warp changed a cell in the current round
};

// blocks of the tile that can be affected by what the tile was queued for (bit 4: everything)
__device__ inline unsigned long long nf_region(int flags) {
    if (flags & 16) return ~0ull;
    unsigned long long m = 0;
    if (flags & 1) m |= 0xffull;
    if (flags & 2) m |= 0xffull << 56;
    if (flags & 4) m |= 0x0101010101010101ull;
    if (flags & 8) m |= 0x8080808080808080ull;
    return m;
}

// Runs the dirty-block iteration of one tile to quiescence.  On entry S.dirty[0] holds the initial mask,
// S.dirty[1] = S.dirty[2] = S.chgmask = 0, S.ring = 0, all visible (a __syncthreads() has passed).
// `flush()` (called by all threads right after a __syncthreads) writes the blocks in S.chgmask back, queues the
// neighbours that can gain from the changed ring, and clears S.chgmask / S.ring.  It is called once, when the tile
// has settled.  Forwarding the ring before that (after iterations 1, 2, 4, ... or after every iteration) was
// measured at 8192^2: the kernel is throughput-bound for two thirds of its run (every CTA slot busy,
// profiles/r01_nf_timeline.txt), so the extra visits cost more than the shorter chains save (11.1 ms -> 12.9 /
// 13.8 ms).
template <class R, class F>
__device__ inline int nf_tile_iterate(const R &rx, NfTileShared &S, F &flush) {
    const int tid = threadIdx.x, lane = tid & 31;
    int it = 0;
    for (;; it++) {
        const unsigned long long m = S.dirty[it % 3];
        if (m == 0) break;
        if (tid == 0) { S.dirty[(it + 2) % 3] = 0; S.grab[(it + 2) % 3] = 0; }
        unsigned long long mark = 0, mine = 0;
        int rings = 0;
        // the warps take the dirty blocks off a counter: blocks differ a lot in how long they take to settle
        const int cnt = __popcll(m);
        if (tid < 64 && (m >> tid) & 1ull) S.blist[__popcll(m & ((1ull << tid) - 1ull))] = (unsigned char)tid;
        __syncthreads();
        for (;;) {
            int j = 0;
            if (lane == 0) j = atomicAdd(&S.grab[it % 3], 1);
            j = __shfl_sync(0xffffffffu, j, 0);
            if (j >= cnt) break;
            int b = S.blist[j];
            unsigned sd;
            if (!rx.block(b, &sd)) continue;
            int by = b >> 3, bx = b & 7;
            mine |= 1ull << b;
            if (sd & 16u) mark |= 1ull << b;
            // neighbouring blocks that read a changed edge (a corner cell belongs to both of its edges)
            unsigned long long row3 = ((0x7ull << bx) >> 1) & 0xffull;
            int ylo = by > 0 ? by - 1 : 0, yhi = by < 7 ? by + 1 : 7;
            if (sd & 1u) { if (by > 0) mark |= row3 << ((by - 1) * 8); else rings |= 1; }
            if (sd & 2u) { if (by < 7) mark |= row3 << ((by + 1) * 8); else rings |= 2; }
            if (sd & 4u) {
                if (bx > 0) { for (int y = ylo; y <= yhi; y++) mark |= 1ull << (y * 8 + bx - 1); }
                else rings |= 4;
            }
            if (sd & 8u) {
                if (bx < 7) { for (int y = ylo; y <= yhi; y++) mark |= 1ull << (y * 8 + bx + 1); }
                else rings |= 8;
            }
        }
        if (lane == 0) {
            if (mark) atomicOr(&S.dirty[(it + 1) % 3], mark);
            if (mine) atomicOr(&S.chgmask, mine);
            if (rings) atomicOr(&S.ring, rings);
        }
        __syncthreads();
    }
    if (S.chgmask) flush();
    return it;
}


// lake cell (w > f) -> integer distance; anything else -> wall.  Tracks the range of binades seen (elo..ehi).
__device__ inline int nf_binade(double fd) {
    int hi = __double2hiint(fd);
    int e = ((hi >> 20) & 0x7ff) - 1023;
    // values just above a negative power of two have the smaller magnitude: they live one binade lower
    if (fd < 0 && (hi & 0xfffff) == 0 && __double2loint(fd) == 0) e -= 1;
    return e;
}

__device__ inline int nf_to_int(double w, float f, int &bad, int &elo, int &ehi, int &dmax, unsigned char *e8) {
    double fd = (double)f;
    *e8 = 0;
    if (!(w > fd)) return D_WALL;
    int e = nf_binade(fd);
    if (fd == 0.0 || e < -900) { bad |= 1; return D_WALL; }
    *e8 = (unsigned char)(e & 0xff);
    elo = min(elo, e);
    ehi = max(ehi, e);
    if (w == INFINITY) return D_INF;
    int ew = ((__double2hiint(w) >> 20) & 0x7ff) - 1023;
    if (ew != e) { bad |= 2; return D_WALL; }
    double inv_ulp = __hiloint2double((1023 - (e - 52)) << 20, 0);
    double d = (w - fd) * inv_ulp;              // exact: same binade, both multiples of its ulp
    if (!(d < (double)D_LIMIT)) {
#ifdef NF_STATS
        if (atomicAdd(&g_nf_dbg[12], 1ull) == 1000ull) {
            g_nf_dbg[13] = (unsigned long long)__double_as_longlong(w);
            g_nf_dbg[14] = (unsigned long long)__double_as_longlong(fd);
        }
#endif
        bad |= 4;
        return D_WALL;
    }
    int di = (int)d;
    dmax = max(dmax, di);
    return di;
}

// tile flag word: bits 0-3 = sides of the tile whose apron changed, bit 4 = look at everything; NF_RUNNING while
// a CTA holds the tile.  "Side bits set and not running" means the tile is in the FIFO (exactly once).
constexpr int NF_SIDES = 31;
constexpr int NF_RUNNING = 256;
// FIFO capacity = tiles + this: a tile is queued at most once, and every CTA of the grid may hold a ticket for an
// entry that is not filled yet — two tickets must never share a slot (the grid is at most 148 SMs x 8 CTAs)
constexpr int NF_RING_SLACK = 2048;

// ---- row bands fused over NVLink peer memory (P2P) ---------------------------------------------------------
// Every band's solver (k_nf_solve_ir, below) runs at the same time, one cooperative launch per GPU.  A band's FIFO,
// tile flags and two "mailbox" rows (the neighbours' edge rows, i.e. this band's halo rows of the integer raster)
// live in one block that the neighbouring ranks map through CUDA IPC.  A tile on a band edge whose ring changed
// stores its edge row into the neighbour's mailbox and queues the neighbour's tile with system-scope atomics — the
// wave of a lake that spans bands runs on without a host round trip.  Termination: each band counts its queued +
// running tiles; the number of bands with a non-zero count lives on rank 0; whoever brings that to zero raises
// `done` on every rank.
constexpr int NF_MAXRANKS = 16;
struct NfPeer {
    int *tileflag;     // the neighbour band's tile flag words
    int *ring;         // ... its FIFO
    NfCtl *ctl;
    void *mail;        // ... its mailbox row facing this band (padded int32 distance row)
    int tiles_y, cap;
};
struct NfP2P {
    NfPeer up, down;                // null pointers where the band is not open
    void *mail_top, *mail_bot;      // this band's own halo rows of the integer raster (written by the neighbours)
    int *gactive;                   // rank 0: bands with queued or running tiles
    int *done_all[NF_MAXRANKS];     // every rank's ctl->done
    int world;
};

// queue `tile` on the FIFO (ring, ctl); with `sys` the FIFO may be another GPU's (or be fed by another GPU)
// (`remote`: the FIFO lives on another GPU - the entry is pushed out with a system-scope fence; a FIFO of this GPU that
// other GPUs also feed only needs the system-scope atomics)
__device__ inline void nf_push(int *ring, int cap, NfCtl *ctl, int tile, bool sys = false, int *gactive = nullptr,
                               bool remote = true) {
    if (sys) {
        if (atomicAdd_system(&ctl->pending, 1) == 0) atomicAdd_system(gactive, 1);      // the band wakes up
        unsigned idx = atomicAdd_system(&ctl->tail, 1u);
        volatile int *slot = ring + (idx % (unsigned)cap);
        for (unsigned spins = 0; *slot != -1 && spins < (1u << 23); spins++) __nanosleep(100);
        // never overwrite a slot that is still taken (a queued tile would be lost silently): stop the solve instead,
        // the host sees done == 2 and falls back
        if (*slot != -1) { atomicExch_system(&ctl->done, 2); return; }
        *slot = tile;
        if (remote) __threadfence_system();
        return;
    }
    atomicAdd(&ctl->pending, 1);
    unsigned idx = atomicAdd(&ctl->tail, 1u);
    volatile int *slot = ring + (idx % (unsigned)cap);
    // the ring holds every tile at most once, so the slot is free; wait if it is not (yet)
    for (unsigned spins = 0; *slot != -1 && spins < (1u << 23); spins++) __nanosleep(100);
    if (*slot != -1) { atomicExch(&ctl->done, 2); return; }
    *slot = tile;
}

// take the next FIFO entry (one thread of a solver CTA): wait for it to be filled unless all work is done, and free
// the slot.  Returns the tile, or -1 when the solve has ended.
__device__ __forceinline__ int nf_take(int *ring, int cap, NfCtl *ctl, bool p2p, const NfP2P *pp) {
    unsigned my = atomicAdd(&ctl->head, 1u);
    volatile int *slot = ring + (my % (unsigned)cap);
    int t = -1;
    const unsigned long long t_start = nf_globaltimer();
    for (unsigned spins = 0;; spins++) {
        t = *slot;
        if (t >= 0) break;
        if (*(volatile int *)&ctl->done) break;
        __nanosleep(100);
        // watchdog on the wall clock (never hang the GPU): generous, so that a profiler or a time-sliced GPU
        // does not trip it
        if ((spins & 1023u) == 1023u && nf_globaltimer() - t_start > NF_WATCHDOG_NS) {
            if (p2p) for (int k = 0; k < pp->world; k++) *(volatile int *)pp->done_all[k] = 2;      // every rank stops
            atomicExch(&ctl->done, 2);
            break;
        }
    }
    if (t >= 0) {
        *slot = -1;
        __threadfence();
    }
    return t;
}

// converts one loaded row pair of the integer form (cells 2*lane, 2*lane+1 and, for lanes 0/1, an apron column)
struct NfRowRegs {
    double w0, w1, wa;
    float f0, f1, fa;
};

template <bool CAP>
__global__ void __launch_bounds__(256, 4) k_nf_solve(const float *__restrict__ zsrc, double *W, int *ring, int cap,
                                                  int *tileflag, const int *__restrict__ tilesides, NfCtl *ctl, int rows, int cols, int tiles_x,
                                                  int tiles_y, double sh, double dg, int use_int, double capB,
                                                  int open) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sw = reinterpret_cast<double *>(smem_raw);
    float *sz = reinterpret_cast<float *>(smem_raw + (NF_T + 2) * NF_LD * 8);
    int *sdi = reinterpret_cast<int *>(smem_raw);
    unsigned char *se = smem_raw + (NF_T + 2) * NF_ILD * 4;          // integer form: binade byte per interior cell
    float *sfi = reinterpret_cast<float *>(se + NF_T * NF_T);        // integer form: F per interior cell (write-back)
    __shared__ NfTileShared S;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // rows the aprons may read: a band that continues above / below has a halo row there
    const int rlo = (open & 1) ? -1 : 0, rhi = rows + ((open & 2) ? 1 : 0);
    // halo rows of the surface: the ext rows of W
    const double *halo_top = W - (long long)cols;
    const double *halo_bot = W + (long long)rows * cols;
    if (*(volatile unsigned *)&ctl->tail == 0) return;      // nothing was queued (tail only grows)

    for (;;) {
        // The next tile is taken by thread 32 while thread 0 is still signing off the previous one (below): both are
        // chains of global atomics, and nobody touches S between the barrier that ends a visit and this point.
        if (tid == 32) {
            const int t = nf_take(ring, cap, ctl, false, nullptr);
            if (t >= 0) {
                // taken: while the tile runs, neighbours only leave their side bits; they are looked at when it ends
                S.flags = atomicExch(tileflag + t, NF_RUNNING) & NF_SIDES;
                S.dirty[1] = 0;
                S.dirty[2] = 0;
                S.chgmask = 0;
                S.ring = 0;
                S.nb = 0;
                S.grab[0] = S.grab[1] = S.grab[2] = 0;
                S.e = INT_MIN;
                S.elo = INT_MAX;
                S.bad = 0;
                S.dmax = 0;
                S.any = 0;
                atomicAdd(&ctl->visits, 1);
            }
            S.k = t;
        }
        __syncthreads();
        const int t = S.k;
        if (t < 0) break;
#ifdef NF_STATS
        long long tc0 = clock64(), tc1 = 0, tc2 = 0; int nit = 0;
        unsigned long long tg0 = gtimer(), tg1 = 0;
#endif
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        const int r0 = ty * NF_T, c0 = tx * NF_T;
        // queue the neighbour tiles named by S.nb: threads 0..8 take one neighbour each (after the tile's writes were
        // fenced), so the global atomics of all neighbours are in flight together instead of one thread's chain
        auto push_neighbours = [&]() {
            int nbm = S.nb;
                {
                    const int dy = tid / 3 - 1, dx = tid % 3 - 1;
                    if (tid >= 9 || (!dy && !dx)) return;
                    if (!(nbm & (1 << ((dy + 1) * 3 + (dx + 1))))) return;
                    int y = ty + dy, x = tx + dx;
                    // a tile of the neighbouring band: the host exchanges the halo rows and queues it there
                    if (x < 0 || x >= tiles_x || y < 0 || y >= tiles_y) return;
                    // which side of the neighbour looks at us
                    int bits = (dy < 0 ? 2 : 0) | (dy > 0 ? 1 : 0) | (dx < 0 ? 8 : 0) | (dx > 0 ? 4 : 0);
                    if (dy && dx) bits = dy < 0 ? 2 : 1;      // a corner: one block of that side is enough
                    int nb = y * tiles_x + x;
                    if (!(__ldg(tilesides + nb) & bits)) return;      // nothing there that could change
                    // an idle tile (no side bits yet, not running) is queued by whoever sets its first side bit
                    if (atomicOr(tileflag + nb, bits) == 0) nf_push(ring, cap, ctl, nb);
                }
        };
        bool solved = false;
        if (CAP && use_int) {
            // ---- integer form: load tile + apron (all loads of a batch in flight together), convert on the fly
            int bad = 0, elo = INT_MAX, ehi = INT_MIN, dmax = 0;
            const bool vec = ((cols & 1) == 0) && (c0 + NF_T <= cols);
#pragma unroll
            for (int half = 0; half < 2; half++) {
                NfRowRegs rg[5];
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    int lr = warp + 8 * (half * 5 + j);
                    int r = r0 + lr - 1;
                    rg[j].w0 = rg[j].w1 = rg[j].wa = 0.0;
                    rg[j].f0 = rg[j].f1 = rg[j].fa = 0.f;          // w == f: a wall
                    if (lr < NF_T + 2 && r >= rlo && r < rhi) {
                        const double *wr = r < 0 ? halo_top : (r >= rows ? halo_bot : W + (long long)r * cols);
                        const float *fr = zsrc + (long long)r * cols;
                        int c = c0 + 2 * lane;
                        if (vec) {
                            double2 wv = __ldcg(reinterpret_cast<const double2 *>(wr + c));
                            float2 fv = __ldg(reinterpret_cast<const float2 *>(fr + c));
                            rg[j].w0 = wv.x; rg[j].w1 = wv.y; rg[j].f0 = fv.x; rg[j].f1 = fv.y;
                        } else {
                            if (c < cols) { rg[j].w0 = __ldcg(wr + c); rg[j].f0 = __ldg(fr + c); }
                            if (c + 1 < cols) { rg[j].w1 = __ldcg(wr + c + 1); rg[j].f1 = __ldg(fr + c + 1); }
                        }
                        if (lane < 2) {
                            int ca = lane ? c0 + NF_T : c0 - 1;
                            if (ca >= 0 && ca < cols) { rg[j].wa = __ldcg(wr + ca); rg[j].fa = __ldg(fr + ca); }
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    int lr = warp + 8 * (half * 5 + j);
                    if (lr < NF_T + 2) {
                        int *row = sdi + lr * NF_ILD;
                        unsigned char e0, e1, ea;
                        row[1 + 2 * lane] = nf_to_int(rg[j].w0, rg[j].f0, bad, elo, ehi, dmax, &e0);
                        row[2 + 2 * lane] = nf_to_int(rg[j].w1, rg[j].f1, bad, elo, ehi, dmax, &e1);
                        if (lane < 2) row[lane ? NF_T + 1 : 0] = nf_to_int(rg[j].wa, rg[j].fa, bad, elo, ehi, dmax, &ea);
                        if (lr >= 1 && lr <= NF_T) {
                            se[(lr - 1) * NF_T + 2 * lane] = e0;
                            se[(lr - 1) * NF_T + 2 * lane + 1] = e1;
                            *reinterpret_cast<float2 *>(sfi + (lr - 1) * NF_T + 2 * lane) = make_float2(rg[j].f0, rg[j].f1);
                        }
                    }
                }
            }
#ifdef NF_STATS
            long long tl1 = clock64();
#endif
            dmax = __reduce_max_sync(0xffffffffu, dmax);
            elo = __reduce_min_sync(0xffffffffu, elo);
            ehi = __reduce_max_sync(0xffffffffu, ehi);
            bad = __reduce_or_sync(0xffffffffu, bad);
#ifdef NF_STATS
            if (lane == 0 && bad) { if (bad & 1) atomicAdd(&g_nf_dbg[6], 1ull); if (bad & 2) atomicAdd(&g_nf_dbg[7], 1ull); if (bad & 4) atomicAdd(&g_nf_dbg[8], 1ull); }
#endif
            if (lane == 0) {
                if (dmax) atomicMax(&S.dmax, dmax);
                if (ehi != INT_MIN) { atomicMin(&S.elo, elo); atomicMax(&S.e, ehi); }
                if (bad) S.bad = 1;
            }
            __syncthreads();
#ifdef NF_STATS
            if (tid == 0) { atomicAdd(&g_nf_dbg[13], (unsigned long long)(tl1 - tc0)); atomicAdd(&g_nf_dbg[14], (unsigned long long)(clock64() - tl1)); }
#endif
            bool ok = !S.bad && (S.e == INT_MIN || S.e - S.elo < NF_NBIN) && S.dmax < D_LIMIT;
#ifdef NF_STATS
            if (tid == 0 && !S.bad && !ok) atomicAdd(&g_nf_dbg[9], 1ull);
#endif
            if (ok && S.e != INT_MIN) {
                // weights per binade of the tile: short must be a whole number of ulps, diag must not sit on a
                // rounding tie, and both must leave room in the integer range
                if (tid < NF_NBIN) {
                    int e = S.elo + tid;
                    int2 wt = make_int2(0, 0);
                    if (e <= S.e) {
                        double inv_ulp = __longlong_as_double((long long)(1023 - (e - 52)) << 52);
                        double sqd = sh * inv_ulp, dqx = dg * inv_ulp, dqd = rint(dqx);
                        double fr2 = fabs(dqx - floor(dqx) - 0.5);
                        bool good = sqd >= 1.0 && sqd == rint(sqd) && dqd >= 1.0 && fr2 > 1e-9 &&
                                    dqd < (double)(1 << 27) && sqd < (double)(1 << 27);
                        if (good) wt = make_int2((int)sqd, (int)dqd);
                        else S.bad = 1;
                    }
                    S.wtab[tid] = wt;
                }
                __syncthreads();
                ok = !S.bad;
#ifdef NF_STATS
                if (tid == 0 && !ok) atomicAdd(&g_nf_dbg[10], 1ull);
#endif
            }
            if (ok && S.e == INT_MIN) {
                solved = true;                      // no lake cell in the tile or its apron: nothing to do
            } else if (ok) {
                if (tid == 0) S.dirty[0] = nf_region(S.flags);
                __syncthreads();
                RelaxI32 rx{sdi, se, S.wtab, S.elo & 0xff, &S.bad};
                auto flush = [&]() {
                    if (S.bad) return;              // the tile will be redone in float64: write nothing
                    // the blocks that changed: W = F + D * ulp (exact)
                    unsigned long long mm = S.chgmask;
                    for (int idx = 0; mm; idx++) {
                        int b = __ffsll((long long)mm) - 1;
                        mm &= mm - 1;
                        if ((idx & 7) != warp) continue;
                        int lr = (b >> 3) * 8 + (lane >> 2), lc = (b & 7) * 8 + (lane & 3) * 2;
                        int r = r0 + lr, c = c0 + lc;
                        const int *p = sdi + (lr + 1) * NF_ILD + (lc + 1);
                        if (r < rows) {
#pragma unroll
                            for (int q = 0; q < 2; q++) {
                                int d = p[q];
                                if (c + q < cols && d < D_INF) {
                                    size_t i = (size_t)r * cols + c + q;
                                    double fd = (double)sfi[lr * NF_T + lc + q];
                                    double ulp = __longlong_as_double((long long)(nf_binade(fd) - 52 + 1023) << 52);
                                    W[i] = __dadd_rn(fd, __dmul_rn((double)d, ulp));
                                }
                            }
                        }
                    }
                    // Which neighbours can actually gain from the new ring?  A ring cell with distance d improves an
                    // adjacent lake cell of the neighbour (held in the apron, possibly stale = too high, which only
                    // errs towards queueing) iff d + weight is below it.  Waves mostly run one way, so this drops
                    // the visit that would only bounce back to the tile the wave came from.
                    int side = tid >> 6, k = tid & 63;          // 0 top, 1 bottom, 2 left, 3 right
                    if (S.ring & (1 << side)) {
                        int lr = side == 0 ? 0 : (side == 1 ? NF_T - 1 : k);
                        int lc = side == 2 ? 0 : (side == 3 ? NF_T - 1 : k);
                        int d = sdi[(lr + 1) * NF_ILD + (lc + 1)];
                        int nbm = 0;
                        int2 wt = rx.weights(lr, lc);
                        if (d < D_INF) {
#pragma unroll
                            for (int o = -1; o <= 1; o++) {
                                // apron cell across this side, offset o along it
                                int ar = side == 0 ? -1 : (side == 1 ? NF_T : lr + o);
                                int ac = side == 2 ? -1 : (side == 3 ? NF_T : lc + o);
                                int da = sdi[(ar + 1) * NF_ILD + (ac + 1)];
                                int w = (o == 0) ? wt.x : wt.y;
                                if (da <= D_INF && d + w < da) {
                                    int dy = ar < 0 ? -1 : (ar >= NF_T ? 1 : 0), dx = ac < 0 ? -1 : (ac >= NF_T ? 1 : 0);
                                    nbm |= 1 << ((dy + 1) * 3 + (dx + 1));
                                }
                            }
                        }
                        nbm = __reduce_or_sync(0xffffffffu, nbm);
                        if (lane == 0 && nbm) atomicOr(&S.nb, nbm);
                    }
                    __threadfence();
                    __syncthreads();
                    push_neighbours();
                    __syncthreads();
                    if (tid == 0) {
                        S.nb = 0;
                        S.ring = 0;
                        S.chgmask = 0;
                    }
                    __syncthreads();
                };
#ifdef NF_STATS
                tc1 = clock64(); tg1 = gtimer();
#endif
                int its = nf_tile_iterate(rx, S, flush);
#ifdef NF_STATS
                nit = its;
#endif
                (void)its;
                solved = !S.bad;                    // a distance left the trusted range: redo the tile in float64
#ifdef NF_STATS
                if (tid == 0 && !solved) atomicAdd(&g_nf_dbg[11], 1ull);
#endif
            }
            if (!solved) __syncthreads();          // everybody is done with the integer tile before it is overwritten
        }
        if (!solved) {
            // ---- float64 form
#ifdef NF_STATS
            if (tid == 0) atomicAdd(&g_nf_dbg[5], 1ull);
#endif
            if (tid == 0) {
                S.dirty[0] = nf_region(S.flags);
                S.dirty[1] = 0;
                S.dirty[2] = 0;
                S.grab[0] = S.grab[1] = S.grab[2] = 0;
                S.chgmask = 0;
                S.ring = 0;
                S.nb = 0;
            }
            for (int q = tid; q < (NF_T + 2) * (NF_T + 2); q += 256) {
                int lr = q / (NF_T + 2), lc = q - lr * (NF_T + 2);
                int r = r0 + lr - 1, c = c0 + lc - 1;
                double v = INFINITY;
                if (r >= rlo && r < rhi && c >= 0 && c < cols)
                    v = __ldcg((r < 0 ? halo_top : (r >= rows ? halo_bot : W + (long long)r * cols)) + c);
                sw[lr * NF_LD + lc] = v;
            }
            for (int q = tid; q < NF_T * NF_T; q += 256) {
                int lr = q >> 6, lc = q & 63;
                int r = r0 + lr, c = c0 + lc;
                sz[q] = (r < rows && c < cols) ? __ldg(zsrc + (size_t)r * cols + c) : INFINITY;
            }
            __syncthreads();
#ifdef NF_STATS
            tc1 = clock64();
#endif
            RelaxF64<CAP> rx{sw, sz, sh, dg, capB};
            auto flush = [&]() {
                // the blocks that changed: a warp writes 8 rows of 8 doubles (lane: row l/4, 2 columns)
                unsigned long long mm = S.chgmask;
                for (int idx = 0; mm; idx++) {
                    int b = __ffsll((long long)mm) - 1;
                    mm &= mm - 1;
                    if ((idx & 7) != warp) continue;
                    int lr = (b >> 3) * 8 + (lane >> 2), lc = (b & 7) * 8 + (lane & 3) * 2;
                    int r = r0 + lr, c = c0 + lc;
                    const double *p = sw + (lr + 1) * NF_LD + (lc + 1);
                    if (r < rows) {
                        if (c < cols) W[(size_t)r * cols + c] = p[0];
                        if (c + 1 < cols) W[(size_t)r * cols + c + 1] = p[1];
                    }
                }
                __threadfence();
                __syncthreads();
                if (tid == 0) {
                    // every neighbour that sees a changed side (a diagonal one sees the corner cell, which belongs
                    // to both adjoining sides)
                    int rg = S.ring, nbm = 0;
                    for (int dy = -1; dy <= 1; dy++)
                        for (int dx = -1; dx <= 1; dx++) {
                            if (!dy && !dx) continue;
                            bool hit = (dy < 0 && (rg & 1)) || (dy > 0 && (rg & 2)) || (dx < 0 && (rg & 4)) ||
                                       (dx > 0 && (rg & 8));
                            if (hit) nbm |= 1 << ((dy + 1) * 3 + (dx + 1));
                        }
                    S.nb = nbm;
                }
                __syncthreads();
                push_neighbours();
                __syncthreads();
                if (tid == 0) {
                    S.nb = 0;
                    S.ring = 0;
                    S.chgmask = 0;
                }
                __syncthreads();
            };
            int its = nf_tile_iterate(rx, S, flush);
#ifdef NF_STATS
            nit = its;
#endif
            (void)its;
        }
#ifdef NF_STATS
        tc2 = clock64();
        if (tid == 0) {
            atomicAdd(&g_nf_dbg[1], (unsigned long long)(tc1 ? tc1 - tc0 : 0));
            atomicAdd(&g_nf_dbg[2], (unsigned long long)(tc1 ? tc2 - tc1 : 0));
            atomicAdd(&g_nf_dbg[3], (unsigned long long)nit);
            atomicMax(&g_nf_dbg[4], (unsigned long long)(tc1 ? tc2 - tc1 : 0));
            unsigned k = atomicAdd(&g_nf_nlog, 1u);
            if (k < 262144u) {
                g_nf_log[4 * k] = tg0; g_nf_log[4 * k + 1] = tg1; g_nf_log[4 * k + 2] = gtimer();
                g_nf_log[4 * k + 3] = (unsigned long long)t | ((unsigned long long)nit << 32);
            }
        }
#endif
        __syncthreads();
        if (tid == 0) {
            // this tile: side bits that arrived while it ran mean it has to run again
            if (atomicAnd(tileflag + t, ~NF_RUNNING) & NF_SIDES) nf_push(ring, cap, ctl, t);
            __threadfence();
            if (atomicSub(&ctl->pending, 1) == 1) atomicExch(&ctl->done, 1);
        }
    }
}

// k_nf_init + k_nf_seedcand in one pass (single-GPU capped path): a CTA holds z and F of a 64x64 tile with a 2-cell
// apron, works out which cells of the tile and of its 1-cell ring are seeds, and writes W for the tile: z on the
// raster border and for seeds; for a lake / flat cell the best candidate its fixed neighbours (seeds, border cells:
// W = z there) offer, unless that lies above F + capB, else +inf.  (Row bands keep the two-kernel form: the seed
// test of a halo-row cell would need a second halo row.)
constexpr int NI_A = NF_T + 4;          // tile + 2-cell apron

// With Dg != nullptr (the integer-raster solve, below) the kernel also writes the tile of the padded int32 raster
// Dg — lake / flat cell: its distance above F in ulps (D_INF: not reached yet), anything else: D_WALL — and
// tmeta[tile] = the binade range of the lake cells of the tile and its apron; *irbad is raised when a cell or tile
// does not qualify for the integer form.
// TMA = true (single GPU, raster describable by a tensor map): z and F of the tile + 2-cell apron arrive as two
// 68 x 72 boxes (cp.async.bulk.tensor.2d from column c0 - 4, see tma.cuh; NaN outside the raster - fminf ignores it
// like the +inf of the LDG -> STS form, and no cell outside the raster is ever read as a source).
constexpr int NI_LD_TMA = NF_T + 8;
template <bool TMA>
__global__ void __launch_bounds__(256) k_nf_init_tile(const float *__restrict__ z, const float *__restrict__ F,
                                                      double *__restrict__ W, int *tileflag, int *tilesides, NfCtl *ctl,
                                                      int rows, int cols, int tiles_x, double sh, double dg, double capB,
                                                      int *__restrict__ Dg, int P, int *tmeta, int *irbad, int open,
                                                      const uint8_t *__restrict__ fix_top,
                                                      const uint8_t *__restrict__ fix_bot,
                                                      const __grid_constant__ CUtensorMap zmap,
                                                      const __grid_constant__ CUtensorMap fmap) {
    constexpr int LDZ = TMA ? NI_LD_TMA : NI_A;       // shared row stride of z / F
    constexpr int XO = TMA ? 2 : 0;                   // shared column of raster column c0 - 2
    // Row band (open != 0): z and F have a halo row above / below the band where it is open; whether a cell of a
    // halo row is fixed would need a second halo row, so the neighbour says (fix_top / fix_bot, k_band_edgefix).
    const int rlo = (open & 1) ? -1 : 0, rhi = rows + ((open & 2) ? 1 : 0);
    __shared__ __align__(128) float sz[NI_A * LDZ], sf[NI_A * LDZ];
    __shared__ uint64_t bar;
    __shared__ unsigned char fixedc[(NF_T + 2) * (NF_T + 2)];      // 1: W = z there for good (seed or raster border)
    __shared__ int s_sides, s_elo, s_ehi, s_bad;
    int tile = blockIdx.x;
    int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    int r0 = ty * NF_T, c0 = tx * NF_T, tid = threadIdx.x;
    if (tid == 0) { s_sides = 0; s_elo = INT_MAX; s_ehi = INT_MIN; s_bad = 0; }
    if (TMA) {
        if (tid == 0) mbar_init(&bar, 1);
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&bar, (unsigned)(2 * sizeof(sz)));
            tma_load_2d(sz, &zmap, &bar, c0 - 4, r0 - 2);
            tma_load_2d(sf, &fmap, &bar, c0 - 4, r0 - 2);
        }
        mbar_wait(&bar, 0);
    } else {
        for (int k = tid; k < NI_A * NI_A; k += 256) {
            int lr = k / NI_A, lc = k - lr * NI_A;
            int r = r0 + lr - 2, c = c0 + lc - 2;
            bool in = r >= rlo && r < rhi && c >= 0 && c < cols;
            sz[k] = in ? z[(long long)r * cols + c] : INFINITY;
            sf[k] = in ? F[(long long)r * cols + c] : INFINITY;
        }
        __syncthreads();
    }
    for (int k = tid; k < (NF_T + 2) * (NF_T + 2); k += 256) {
        int lr = k / (NF_T + 2), lc = k - lr * (NF_T + 2);          // ring coordinates: cell (r0 + lr - 1, c0 + lc - 1)
        int r = r0 + lr - 1, c = c0 + lc - 1;
        unsigned char fx = 0;
        if (r >= rlo && r < rhi && c >= 0 && c < cols) {
            if (r < 0) fx = fix_top[c];
            else if (r >= rows) fx = fix_bot[c];
            else if ((r == 0 && !(open & 1)) || c == 0 || (r == rows - 1 && !(open & 2)) || c == cols - 1) fx = 1;
            else {
                const float *pf = sf + (lr + 1) * LDZ + (lc + 1) + XO;
                float f = *pf;
                float m = fminf(fminf(fminf(pf[-LDZ - 1], pf[-LDZ]), fminf(pf[-LDZ + 1], pf[-1])),
                                fminf(fminf(pf[1], pf[LDZ - 1]), fminf(pf[LDZ], pf[LDZ + 1])));
                fx = (f == sz[(lr + 1) * LDZ + (lc + 1) + XO]) && (m < f);
            }
        }
        fixedc[k] = fx;
        if (Dg && !fx && r >= rlo && r < rhi && c >= 0 && c < cols) {
            // a lake cell of the tile or its apron: its binade counts for the tile's weight table
            float f = sf[(lr + 1) * LDZ + (lc + 1) + XO];
            if (f == 0.f) atomicOr(&s_bad, 1);
            else {
                int e = nf_binade((double)f);
                if (e < -900) atomicOr(&s_bad, 1);
                // nearly every lake cell of a tile lies in the same binade: look before reducing (a third of the
                // tile's cells otherwise queue on these two words)
                if (e < *(volatile int *)&s_elo) atomicMin(&s_elo, e);
                if (e > *(volatile int *)&s_ehi) atomicMax(&s_ehi, e);
            }
        }
    }
    __syncthreads();
    int nonseed = 0, sides = 0;
    for (int k = tid; k < NF_T * NF_T; k += 256) {
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        if (r >= rows || c >= cols) {
            if (Dg) Dg[(size_t)(r + 1) * P + (c + 4)] = D_WALL;      // the padded raster covers whole tiles
            continue;
        }
        const unsigned char *fx = fixedc + (lr + 1) * (NF_T + 2) + (lc + 1);
        const float *pz = sz + (lr + 2) * LDZ + (lc + 2) + XO;
        double w;
        if (*fx) {
            w = (double)*pz;
        } else {
            double best = INFINITY;
#pragma unroll
            for (int dr = -1; dr <= 1; dr++)
#pragma unroll
                for (int dc = -1; dc <= 1; dc++) {
                    if (dr == 0 && dc == 0) continue;
                    if (!fx[dr * (NF_T + 2) + dc]) continue;
                    double cand = __dadd_rn((double)pz[dr * LDZ + dc], (dr != 0 && dc != 0) ? dg : sh);
                    best = dmin2(best, cand);
                }
            w = (best <= (double)sf[(lr + 2) * LDZ + (lc + 2) + XO] + capB) ? best : (double)INFINITY;
            nonseed++;
            sides |= (lr == 0 ? 1 : 0) | (lr == NF_T - 1 || r == rows - 2 ? 2 : 0) | (lc == 0 ? 4 : 0) |
                     (lc == NF_T - 1 || c == cols - 2 ? 8 : 0);
        }
        if (!Dg) W[(size_t)r * cols + c] = w;      // the integer-raster solve writes W once, at the end (k_nf_finish_ir)
        if (Dg) {
            int bad = 0, elo = 0, ehi = 0, dmax = 0;
            unsigned char e8;
            Dg[(size_t)(r + 1) * P + (c + 4)] = nf_to_int(w, sf[(lr + 2) * LDZ + (lc + 2) + XO], bad, elo, ehi, dmax, &e8);
            if (bad) atomicOr(&s_bad, 1);
        }
    }
    if (sides) atomicOr(&s_sides, sides);
    int cnt = __syncthreads_count(nonseed > 0);
    nonseed = 0;
    (void)nonseed;
    if (tid == 0 && cnt) {
        tileflag[tile] = 16;
        tilesides[tile] = s_sides;
    }
    if (Dg && tid == 0) {
        int span = s_ehi >= s_elo ? s_ehi - s_elo : 0;
        if (s_bad || span >= NF_NBIN) *irbad = 1;
        // [15:0] lowest binade exponent (signed), [19:16] span, bit 20: the tile or its apron holds a lake cell
        tmeta[tile] = s_ehi >= s_elo ? ((s_elo & 0xffff) | (span << 16) | (1 << 20)) : 0;
    }
}

// CAP only: the one time seeds (and the raster border) act as sources.  A lake / flat cell (still +inf) takes the
// best candidate its fixed neighbours offer, unless that lies above F + capB.  A neighbour is fixed iff W == F
// there (seed: W = z = F; border: W = z = F); lake cells hold +inf or, once written by this kernel, a value > F.
__global__ void __launch_bounds__(256) k_nf_seedcand(const float *__restrict__ F, double *W, const NfCtl *ctl,
                                                     int rows, int cols, double sh, double dg, double capB_in,
                                                     int open) {
    int c = blockIdx.x * 64 + (threadIdx.x & 63);
    int r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= rows || c < 1 || c >= cols - 1) return;
    if ((r == 0 && !(open & 1)) || (r == rows - 1 && !(open & 2))) return;
    size_t i = (size_t)r * cols + c;
    if (__ldcg(W + i) != INFINITY) return;
    const double capB = capB_in >= 0 ? capB_in : ((double)ctl->nonseed + 16.0) * dg * 1.001;
    double best = INFINITY;
#pragma unroll
    for (int dr = -1; dr <= 1; dr++)
#pragma unroll
        for (int dc = -1; dc <= 1; dc++) {
            if (dr == 0 && dc == 0) continue;
            size_t j = i + (long long)dr * cols + dc;
            double wn = __ldcg(W + j);
            if (wn != (double)__ldg(F + j)) continue;
            double cand = __dadd_rn(wn, (dr != 0 && dc != 0) ? dg : sh);
            best = dmin2(best, cand);
        }
    if (best <= (double)F[i] + capB) W[i] = best;
}

__global__ void __launch_bounds__(256) k_nf_verify(const float *__restrict__ z, const double *__restrict__ W,
                                                   uint8_t *banned, NfCtl *ctl, int rows, int cols, double sh,
                                                   double dg, int open) {
    int c = blockIdx.x * 64 + (threadIdx.x & 63);
    int r = blockIdx.y * 4 + (threadIdx.x >> 6);
    int bad = 0;
    if (r < rows && (r > 0 || (open & 1)) && c > 0 && (r < rows - 1 || (open & 2)) && c < cols - 1) {
        size_t i = (size_t)r * cols + c;
        const double *p = W + i;
        double d = dmin2(p[-cols - 1], dmin2(p[-cols + 1], dmin2(p[cols - 1], p[cols + 1])));
        double e = dmin2(p[-cols], dmin2(p[-1], dmin2(p[1], p[cols])));
        double m = dmin2(__dadd_rn(d, dg), __dadd_rn(e, sh));
        double zc = (double)z[i];
        double g = m >= zc ? m : zc;
        if (g != *p) {
            bad = 1;
            if (banned) banned[i] = 1;
        }
    }
    int cnt = __syncthreads_count(bad);
    if (threadIdx.x == 0 && cnt) atomicAdd(&ctl->nviol, cnt);
}


// =====================================================================================================
// Integer-raster solve (single GPU, capped fast path).  ncu on the W-based solver above showed where a tile visit
// goes: 40 % of all instructions convert the float64 tile + apron to the integer form and back, on every visit
// (profiles/r01c_nf_*).  Here the integer form is the state: k_nf_init_tile writes a padded int32 raster Dg
// (pitch P = 64 * tiles_x + 8, one wall row above and below, 4 wall columns left, >= 4 right, so every tile + apron
// is an in-bounds, 16-byte aligned 66 x 72 block), a visit copies that block to shared memory with cp.async (no
// registers, no conversion, one DRAM round trip), relaxes it, and stores the changed 8x8 blocks back as integers.
// W = F + D * ulp(F) is written once at the end, and verified in the same pass (k_nf_finish_ir).  The FIFO / flag protocol is the one of
// k_nf_solve.  Anything that does not fit the integer form (k_nf_init_tile's *irbad, a distance beyond D_LIMIT,
// weights that are not whole ulps) raises *irbad and the caller falls back to the W-based solver.
// =====================================================================================================
// In-tile relaxation of the integer-raster solver: LINE SWEEPS.  The four warps of a CTA are the four sweep
// directions of a chamfer distance transform (top->bottom, bottom->top, left->right, right->left); a sweep walks the
// 64 lines of the tile in its direction and relaxes every cell of a line from the three cells of the previous line
// that touch it (straight: + short, the two diagonals: + diag).  The previous line stays in registers (a lane owns
// cells k = lane and lane + 32 of every line, neighbours come by shuffle), the line's current values are loaded one
// step ahead, so the dependent chain of a step is shuffle -> add -> min -> compare (~45 cycles), and a wave crosses the
// tile in one sweep (~1.5 us) where the dirty-block iteration of round 1 took ~15 us (8 warps, two barriers and a
// 64-block work list per iteration: profiles/r01c_nf_solve_ir_raw.txt, 65 % of the warp samples at a barrier).
// The shared row stride is ODD (67 words): a row and a column of the tile are both 64 consecutive banks modulo 32, so
// all four directions read and write without bank conflicts through plain 4-byte accesses.  Rounds: a direction runs again when ANOTHER direction changed a cell in
// the previous round; the tile is settled when a round changes nothing.  A tile queued for a changed apron side starts
// with the one direction that reads that side.
constexpr int IR_LD = NF_T + 3;                 // 67: odd
constexpr int IR_SMEM = (NF_T + 2) * IR_LD * 4 + NF_T * NF_T;
constexpr int IR_NT = 128;
constexpr int IR_CTAS = 6;
// tail mode (edges forwarded after the first round) below grid >> IR_TAIL_SHIFT queued or running tiles
// (measured: shift 0 / 1 / 2 / 3 -> 3.15 / 3.21 / 3.42 / 3.47 ms at 8192^2, 38.8 / 38.8 / 38.6 / 38.8 ms at 32768^2; on two
// bands of 4096 / 16384 rows shift 0 gives 6.6 / 29.5 ms against 7.0 / 29.0: it helps where the tail dominates and costs
// where the bulk does)
constexpr int IR_TAIL_SHIFT = 2;

// the wall frame of the padded raster: row 0, the rows below the tiles, and 4 columns either side of every tile row
// (k_nf_init_tile writes everything inside, including the cells of edge tiles that lie beyond the raster)
__global__ void __launch_bounds__(256) k_ir_frame(int *Dg, int P, int inner_rows) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * (int64_t)P) {
        int64_t row = i < P ? 0 : inner_rows + 1;
        Dg[row * P + (i < P ? i : i - P)] = D_WALL;
        return;
    }
    i -= 2 * (int64_t)P;
    if (i >= 8 * (int64_t)inner_rows) return;
    int64_t row = 1 + i / 8;
    int k = (int)(i & 7);
    Dg[row * P + (k < 4 ? k : P - 8 + k)] = D_WALL;
}

struct IrShared {
    int k;             // tile taken off the FIFO (-1: none)
    int flags;         // side bits the tile was queued with
    int e, elo;        // largest / smallest binade exponent of the tile's lake cells
    int has;           // the tile or its apron holds a lake cell
    int bad;           // does not fit the integer form
    int chgdir[3];     // directions that changed a cell, per round (rotating)
    unsigned long long crow[3], ccol[3];   // rows / columns of the tile in which a cell changed, per round (rotating)
    unsigned long long rows, cols;         // ... during the whole visit (write-back, edges for the neighbours)
    int ring;          // bit 0/1/2/3: the tile's top / bottom / left / right edge changed
    int nb;            // neighbour tiles to queue: bit (dy+1)*3 + (dx+1)
    int mid;           // tail of the solve: forward the edges after the first round already
    int2 wtab[NF_NBIN];
};

// One sweep of the tile in direction `dir` (0 top->bottom, 1 bottom->top, 2 left->right, 3 right->left) by one warp.
// Cell (line, k) of the sweep sits at sd[org + line * SL + k * SK]; lines and k run -1..64 (apron included).
// `start`: first position (in sweep order: position p is line p of a forward sweep, line 63 - p of a backward one) to
// relax; `lastext`: from this position on the sweep stops at the first line it does not change (everything that
// could disturb the lines beyond lies behind it).
template <bool UNI, int dir>
__device__ __forceinline__ void ir_sweep(int *sd, const unsigned char *se, IrShared &S, const int lane, const int rnd,
                                         const int start, const int lastext) {
    const unsigned full = 0xffffffffu;
    constexpr bool rowsweep = dir < 2;
    constexpr int SL = rowsweep ? IR_LD : 1, SK = rowsweep ? 1 : IR_LD;
    constexpr int EL = rowsweep ? NF_T : 1, EK = rowsweep ? 1 : NF_T;      // the same walk over the binade bytes
    constexpr int step = (dir & 1) ? -1 : 1;
    const int first = (dir & 1) ? NF_T - 1 - start : start;                // line of position `start`
    const int org = IR_LD + 1;
    int *pa = sd + org + lane * SK + first * SL, *pb = pa + 32 * SK;       // the line being relaxed
    const int *pp = sd + org + (lane == 0 ? -1 : NF_T) * SK + first * SL;
    const unsigned char *ea = se + lane * EK + first * EL, *eb = ea + 32 * EK;
    const int elo8 = S.elo & 0xff;
    int2 wA = S.wtab[0], wB = wA;
    int pA = pa[-step * SL], pB = pb[-step * SL], pP = pp[-step * SL];
    int cA = pa[0], cB = pb[0], cP = pp[0];
    if (!UNI) {
        wA = S.wtab[(ea[0] - elo8) & (NF_NBIN - 1)];
        wB = S.wtab[(eb[0] - elo8) & (NF_NBIN - 1)];
    }
    // change bookkeeping without branches: one bit per step shifted into `hist` (the step at position start + j ends up
    // at bit n - 1 - j after n steps), per-lane "my cell A / B changed at some step" flags
    unsigned long long hist = 0;
    int everA = 0, everB = 0;
    const int srcl = (lane + 31) & 31, srcr = (lane + 1) & 31;
    const bool l0 = lane == 0, l31 = lane == 31;
    int p = start;
#pragma unroll 2
    for (; p < NF_T; p++) {
        // the next line's current values: independent of this step's result, in flight while it is computed
        const int nA = pa[step * SL], nB = pb[step * SL], nP = pp[step * SL];
        int2 nwA = wA, nwB = wB;
        if (!UNI) {
            const int o = p + 1 < NF_T ? step * EL : 0;
            nwA = S.wtab[(ea[o] - elo8) & (NF_NBIN - 1)];
            nwB = S.wtab[(eb[o] - elo8) & (NF_NBIN - 1)];
        }
        // a wall never moves: its candidate is pushed out of range (off the dependent chain: cA / cB were loaded a step ago)
        const int wallA = cA > D_INF ? 0x7fffffff : 0, wallB = cB > D_INF ? 0x7fffffff : 0;
        // neighbours of cell k on the previous line: k - 1 and k + 1 (cells 31 | 32 wrap between the two halves)
        const int X = l0 ? pB : pA, Y = l31 ? pA : pB;
        int lA = __shfl_sync(full, pA, srcl);
        const int rA = __shfl_sync(full, X, srcr);
        const int lB = __shfl_sync(full, Y, srcl);
        int rB = __shfl_sync(full, pB, srcr);
        lA = l0 ? pP : lA;
        rB = l31 ? pP : rB;
        const int candA = min(pA + wA.x, min(lA, rA) + wA.y) | wallA;
        const int candB = min(pB + wB.x, min(lB, rB) + wB.y) | wallB;
        const bool chA = candA < cA, chB = candB < cB;
        // the four warps work on the same tile at once: improvements go in as shared-memory min reductions (no result),
        // so a cell never rises and a value read one step early only costs another round.  Issued unconditionally (a
        // lane without an improvement reduces with INT_MAX): ptxas wraps a conditional ATOMS into a divergent branch
        // region, which costs more than the reduction (measured at 8192^2 / 32768^2: 4.03 / 41.5 ms against 4.46 / 43.8;
        // plain predicated stores with the sweeps restarted on the first changed line: 4.07 / 42.0 and more rounds)
        // (tried and dropped: skipping the two reductions on lines no lane improves - a vote and a uniform branch per
        // step - and plain stores when only one direction sweeps: 3.37 -> 4.00 ms at 8192^2, 38.6 -> 45.1 ms at 32768^2;
        // the branch costs the step more scheduling freedom than the reductions cost LSU time)
        atomicMin(pa, chA ? candA : 0x7fffffff);
        atomicMin(pb, chB ? candB : 0x7fffffff);
        hist = (hist << 1) | (unsigned long long)(chA | chB);
        everA |= chA;
        everB |= chB;
        pA = chA ? candA : cA;
        pB = chB ? candB : cB;
        pP = cP;
        cA = nA; cB = nB; cP = nP;
        wA = nwA; wB = nwB;
        pa += step * SL; pb += step * SL; pp += step * SL;
        if (!UNI) { ea += step * EL; eb += step * EL; }
        if (p >= lastext && !__any_sync(full, chA | chB)) { p++; break; }
    }
    const int n = p - start;                       // steps done
    // lines that changed (any lane), as a mask over line numbers
    unsigned hlo = __reduce_or_sync(full, (unsigned)hist), hhi = __reduce_or_sync(full, (unsigned)(hist >> 32));
    unsigned long long lines = ((unsigned long long)hhi << 32) | hlo;
    if (n > 0 && lines) {
        lines = __brevll(lines) >> (64 - n);       // bit j = step j, i.e. position start + j
        lines <<= start;                           // bit = position
        if (dir & 1) lines = __brevll(lines);      // position p is line 63 - p
    }
    const unsigned balA = __ballot_sync(full, everA), balB = __ballot_sync(full, everB);      // cells k = lane / lane + 32
    if (lane == 0 && lines) {
        const unsigned long long cells = ((unsigned long long)balB << 32) | balA;
        const unsigned long long r = rowsweep ? lines : cells, c = rowsweep ? cells : lines;
        atomicOr(&S.crow[rnd % 3], r);
        atomicOr(&S.ccol[rnd % 3], c);
        atomicOr(&S.chgdir[rnd % 3], 1 << dir);
    }
}

template <bool P2P>
__global__ void __launch_bounds__(IR_NT, IR_CTAS) k_nf_solve_ir(const float *__restrict__ F, int *Dg, int P, int *ring, int cap,
                                                        int *tileflag, const int *__restrict__ tilesides,
                                                        const int *__restrict__ tmeta, NfCtl *ctl, int *irbad, int rows,
                                                        int cols, int tiles_x, int tiles_y, double sh, double dg,
                                                        const NfP2P *pp) {
    // pp != nullptr: one band of a raster split across GPUs, every band's kernel running at the same time (see "row
    // bands fused over NVLink peer memory" above).  The rows above / below the band are mailbox rows (padded like a row
    // of Dg) the neighbours store their edge rows into; an edge tile whose edge row changed stores it into the
    // neighbour's mailbox and queues the neighbour's tiles with system-scope atomics.
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int *sd = reinterpret_cast<int *>(smem_raw);
    unsigned char *se = smem_raw + (NF_T + 2) * IR_LD * 4;
    __shared__ IrShared S;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr bool p2p = P2P;       // compiled twice: the single-GPU form carries none of the peer code
    if (!p2p && (*(volatile unsigned *)&ctl->tail == 0 || *(volatile int *)irbad)) return;      // nothing queued / not for this form
    const int *mail_top = p2p ? (const int *)pp->mail_top : nullptr, *mail_bot = p2p ? (const int *)pp->mail_bot : nullptr;
    const bool open_top = p2p && pp->up.tileflag, open_bot = p2p && pp->down.tileflag;

    for (;;) {
        // thread 32 takes the next tile while thread 0 still signs off the previous one
        if (tid == 32) {
            const int t = nf_take(ring, cap, ctl, p2p, pp);
            if (t >= 0) {
                S.flags = (p2p ? atomicExch_system(tileflag + t, NF_RUNNING) : atomicExch(tileflag + t, NF_RUNNING)) & NF_SIDES;
                S.ring = 0;
                S.nb = 0;
                S.bad = 0;
                S.rows = S.cols = 0;
                S.chgdir[0] = S.chgdir[1] = S.chgdir[2] = 0;
                S.crow[0] = S.crow[1] = S.crow[2] = 0;
                S.ccol[0] = S.ccol[1] = S.ccol[2] = 0;
                int meta = __ldg(tmeta + t);
                S.elo = (int)(short)(meta & 0xffff);
                S.e = S.elo + ((meta >> 16) & 15);
                S.has = (meta >> 20) & 1;
                S.mid = *(volatile int *)&ctl->pending < (int)(gridDim.x >> IR_TAIL_SHIFT);
                atomicAdd(&ctl->visits, 1);
            }
            S.k = t;
        }
        __syncthreads();
        const int t = S.k;
        if (t < 0) break;
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        const int r0 = ty * NF_T, c0 = tx * NF_T;
#ifdef NF_STATS
        unsigned long long tg0 = gtimer(), tg1 = tg0, tg2 = tg0; int nrounds = 0;
#endif
        if (S.has) {
            // ---- tile + apron: 66 rows x 18 chunks of 16 bytes (columns c0 - 4 .. c0 + 67 of the padded raster, L2 only:
            // other SMs write these lines), the 66 x 66 cells of interest stored at the odd stride
            const int *src0 = Dg + (size_t)r0 * P + c0;        // row r0 - 1, column c0 - 4 of the padded raster
            constexpr int NCH = (NF_T + 2) * 18;
            int fin = 0;       // a finite distance somewhere in the block: without one nothing can move
#pragma unroll 1
            for (int q0 = tid; q0 < NCH; q0 += IR_NT * 5) {
                int4 v[5];
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    int q = q0 + j * IR_NT;
                    if (q < NCH) {
                        int lr = q / 18, ch = q - lr * 18;
                        const int *src = src0 + (size_t)lr * P + ch * 4;
                        // the row above the first / below the last tile row of an open band: the neighbour's edge row
                        if (lr == 0 && ty == 0 && open_top) src = mail_top + c0 + ch * 4;
                        if (lr == NF_T + 1 && ty == tiles_y - 1 && open_bot) src = mail_bot + c0 + ch * 4;
                        v[j] = __ldcg(reinterpret_cast<const int4 *>(src));
                    }
                }
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    int q = q0 + j * IR_NT;
                    if (q < NCH) {
                        int lr = q / 18, ch = q - lr * 18;
                        int *dst = sd + lr * IR_LD + ch * 4 - 3;      // column c0 - 4 + 4 ch + m -> k + 1 = 4 ch + m - 3
                        if (ch == 0) { dst[3] = v[j].w; fin |= v[j].w < D_INF; }                       // k = -1
                        else if (ch == 17) { dst[0] = v[j].x; fin |= v[j].x < D_INF; }                 // k = 64 (the rest lies beyond the apron)
                        else {
                            dst[0] = v[j].x; dst[1] = v[j].y; dst[2] = v[j].z; dst[3] = v[j].w;
                            fin |= min(min(v[j].x, v[j].y), min(v[j].z, v[j].w)) < D_INF;
                        }
                    }
                }
            }
            const bool uni = S.e == S.elo;
            if (!uni) {
                // several binades in the tile: the per-cell binade byte comes from F
                for (int q = tid; q < NF_T * NF_T; q += IR_NT) {
                    int r = r0 + (q >> 6), c = c0 + (q & 63);
                    se[q] = (r < rows && c < cols) ? (unsigned char)(nf_binade((double)__ldg(F + (size_t)r * cols + c)) & 0xff) : 0;
                }
            }
            // weights per binade: short must be a whole number of ulps, diag must not sit on a rounding tie
            if (tid < NF_NBIN) {
                int e = S.elo + tid;
                int2 wt = make_int2(0, 0);
                if (e <= S.e) {
                    double inv_ulp = __longlong_as_double((long long)(1023 - (e - 52)) << 52);
                    double sqd = sh * inv_ulp, dqx = dg * inv_ulp, dqd = rint(dqx);
                    double fr2 = fabs(dqx - floor(dqx) - 0.5);
                    bool good = sqd >= 1.0 && sqd == rint(sqd) && dqd >= 1.0 && fr2 > 1e-9 &&
                                dqd < (double)(1 << 27) && sqd < (double)(1 << 27);
                    if (good) wt = make_int2((int)sqd, (int)dqd);
                    else S.bad = 1;
                }
                S.wtab[tid] = wt;
            }
            fin = __syncthreads_or(fin);
#ifdef NF_STATS
            tg1 = tg2 = gtimer();
#endif
            // Write-back + neighbour activation: the rows that changed since the last flush go back to the raster, the
            // neighbours that can gain from the changed edges are queued.  Called by all threads, at the end of the visit
            // and - while the solve is in its tail (few tiles queued or running: the time is a chain of visits along
            // the biggest lakes) - once after the first round, which carries the wave across the tile: the next tile of
            // the chain starts while this one is still checking itself.
            auto flush = [&]() {
            // ---- the rows that changed go back (two coalesced 128-byte stores per row)
            unsigned long long mm = S.rows;
            const int ringbits = ((mm & 1ull) ? 1 : 0) | ((mm >> 63) ? 2 : 0) | ((S.cols & 1ull) ? 4 : 0) | ((S.cols >> 63) ? 8 : 0);
            for (int idx = 0; mm; idx++) {
                int lr = __ffsll((long long)mm) - 1;
                mm &= mm - 1;
                if ((idx & (IR_NT / 32 - 1)) != warp) continue;
                const int *srow = sd + (lr + 1) * IR_LD + 1;
                int *drow = Dg + (size_t)(r0 + lr + 1) * P + (c0 + 4);
                const int va = srow[lane], vb = srow[lane + 32];
                __stcg(drow + lane, va);
                __stcg(drow + lane + 32, vb);
                // a distance beyond what the integer form is trusted for: the float64 form takes over
                if ((va >= D_LIMIT && va < D_INF) || (vb >= D_LIMIT && vb < D_INF)) S.bad = 1;
                // an edge row of the band also goes into the neighbour's mailbox (peer memory over NVLink)
                if (p2p) {
                    int *peer = nullptr;
                    if (lr == 0 && ty == 0 && open_top) peer = (int *)pp->up.mail;
                    if (lr == NF_T - 1 && ty == tiles_y - 1 && open_bot) peer = (int *)pp->down.mail;
                    if (peer) { peer[c0 + 4 + lane] = va; peer[c0 + 4 + lane + 32] = vb; }
                }
            }
            // (Reading the apron lines again before this decision - the neighbours may have lowered their cells since
            // the visit loaded them - was measured: 14 % / 7 % fewer visits at 8192^2 / 32768^2 (30 % of all visits
            // change nothing), but the same kernel time, 3.44 / 38.4 ms, and the same 30.0 ms on two bands: the visits
            // it saves are the cheap ones, and every flush pays one more trip to L2.  Dropped.)
            // ---- neighbours that can gain from the new edge cells: a lake cell of their side of the apron that
            // lies above (edge cell + weight)
            const bool uni2 = uni;
            for (int sidx = tid; sidx < 4 * NF_T; sidx += IR_NT) {
                const int side = sidx >> 6, k = sidx & 63;      // 0 top, 1 bottom, 2 left, 3 right (warp-uniform)
                int nbm = 0;
                if (ringbits & (1 << side)) {
                    int lr = side == 0 ? 0 : (side == 1 ? NF_T - 1 : k);
                    int lc = side == 2 ? 0 : (side == 3 ? NF_T - 1 : k);
                    int d = sd[(lr + 1) * IR_LD + (lc + 1)];
                    if (d < D_INF) {
#pragma unroll
                        for (int o = -1; o <= 1; o++) {
                            int ar = side == 0 ? -1 : (side == 1 ? NF_T : lr + o);
                            int ac = side == 2 ? -1 : (side == 3 ? NF_T : lc + o);
                            int da = sd[(ar + 1) * IR_LD + (ac + 1)];
                            if (da <= D_INF) {
                                // the weight is the TARGET cell's (adjacent lake cells share their binade)
                                int2 wt = uni2 ? S.wtab[0] : S.wtab[(se[lr * NF_T + lc] - (S.elo & 0xff)) & (NF_NBIN - 1)];
                                int w = (o == 0) ? wt.x : wt.y;
                                if (d + w < da) {
                                    int dy = ar < 0 ? -1 : (ar >= NF_T ? 1 : 0), dx = ac < 0 ? -1 : (ac >= NF_T ? 1 : 0);
                                    nbm |= 1 << ((dy + 1) * 3 + (dx + 1));
                                }
                            }
                        }
                    }
                }
                nbm = __reduce_or_sync(0xffffffffu, nbm);
                if (lane == 0 && nbm) atomicOr(&S.nb, nbm);
            }
            // order the tile's stores before the flags / FIFO entries that announce them.  Only a tile on an open
            // band edge has stored into (or will queue a tile of) another GPU: everything else stays on this GPU,
            // where the device-scope fence is enough (a system-scope fence per visit cost 3x in the banded solve)
            const bool peer_touch = p2p && ((ty == 0 && open_top) || (ty == tiles_y - 1 && open_bot));
            if (peer_touch) __threadfence_system(); else __threadfence();
            __syncthreads();
            if (tid < 9 && tid != 4) {
                const int dy = tid / 3 - 1, dx = tid % 3 - 1;
                const int y = ty + dy, x = tx + dx;
                if ((S.nb & (1 << tid)) && x >= 0 && x < tiles_x) {
                    int bits = (dy < 0 ? 2 : 0) | (dy > 0 ? 1 : 0) | (dx < 0 ? 8 : 0) | (dx > 0 ? 4 : 0);
                    if (dy && dx) bits = dy < 0 ? 2 : 1;      // a corner: the row sweep from that side reads it
                    if (y >= 0 && y < tiles_y) {
                        int nb = y * tiles_x + x;
                        if (__ldg(tilesides + nb) & bits) {
                            if (p2p) { if (atomicOr_system(tileflag + nb, bits) == 0) nf_push(ring, cap, ctl, nb, true, pp->gactive, false); }
                            else if (atomicOr(tileflag + nb, bits) == 0) nf_push(ring, cap, ctl, nb);
                        }
                    } else if (p2p) {
                        // the tile lies in the neighbouring band: its flag word and FIFO are on another GPU
                        const NfPeer &q = y < 0 ? pp->up : pp->down;
                        if (q.tileflag) {
#ifdef NF_STATS
                            unsigned long long tq0 = gtimer();
#endif
                            int nbq = (y < 0 ? q.tiles_y - 1 : 0) * tiles_x + x;
                            if (atomicOr_system(q.tileflag + nbq, bits) == 0) nf_push(q.ring, q.cap, q.ctl, nbq, true, pp->gactive);
#ifdef NF_STATS
                            atomicAdd(&g_nf_dbg[0], 1ull);
                            atomicAdd(&g_nf_dbg[1], gtimer() - tq0);
#endif
                        }
                    }
                }
            }
                __syncthreads();
                if (tid == 0) { S.rows = 0; S.cols = 0; S.nb = 0; }
                __syncthreads();
            };
            if (!S.bad && fin) {
                // round 0: everything (first visit), or the one direction that reads the apron side that changed
                int dirs = (S.flags & 16) ? 15 : (S.flags & 15);
                bool whole = (S.flags & 16) != 0;
                unsigned long long mrow = 0, mcol = 0;       // rows / columns changed in the previous round
                for (int rnd = 0;; rnd++) {
                    if (tid == 0) { S.chgdir[(rnd + 1) % 3] = 0; S.crow[(rnd + 1) % 3] = 0; S.ccol[(rnd + 1) % 3] = 0; }
                    if ((dirs >> warp) & 1) {
                        // positions (sweep order) this direction has to look at: the line after the first changed one ...
                        int start = 0, lastext = rnd == 0 && whole ? NF_T : 0;
                        if (rnd > 0) {
                            unsigned long long m = warp < 2 ? mrow : mcol;
                            if (warp & 1) m = __brevll(m);
                            start = __ffsll((long long)m);               // first changed position + 1 (m != 0 here)
                            lastext = 64 - __clzll((long long)m);        // ... up to the one after the last changed one
                        }
                        if (start < NF_T) {
                            if (uni) {
                                if (warp == 0) ir_sweep<true, 0>(sd, se, S, lane, rnd, start, lastext);
                                else if (warp == 1) ir_sweep<true, 1>(sd, se, S, lane, rnd, start, lastext);
                                else if (warp == 2) ir_sweep<true, 2>(sd, se, S, lane, rnd, start, lastext);
                                else ir_sweep<true, 3>(sd, se, S, lane, rnd, start, lastext);
                            } else {
                                if (warp == 0) ir_sweep<false, 0>(sd, se, S, lane, rnd, start, lastext);
                                else if (warp == 1) ir_sweep<false, 1>(sd, se, S, lane, rnd, start, lastext);
                                else if (warp == 2) ir_sweep<false, 2>(sd, se, S, lane, rnd, start, lastext);
                                else ir_sweep<false, 3>(sd, se, S, lane, rnd, start, lastext);
                            }
                        }
                    }
                    __syncthreads();
                    const int cd = S.chgdir[rnd % 3];
                    mrow = S.crow[rnd % 3];
                    mcol = S.ccol[rnd % 3];
                    if (tid == 0) { S.rows |= mrow; S.cols |= mcol; }
                    if (cd == 0 || S.bad) {
                        if (tid == 0) atomicAdd(&ctl->reserved, rnd + 1);
#ifdef NF_STATS
                        nrounds = rnd + 1; tg2 = gtimer();
#endif
                        break;
                    }
                    dirs = (cd & (cd - 1)) ? 15 : (15 & ~cd);
                    if (rnd == 0 && S.mid) {
                        __syncthreads();           // S.rows / S.cols of round 0 are in place
                        if (S.rows) flush();
                    }
                }
                __syncthreads();
            }
            if (!S.bad && S.rows) flush();
            __syncthreads();
            if (S.bad && tid == 0) atomicExch(irbad, 1);
        }
#ifdef NF_STATS
        if (tid == 0) {                 // activity over time, all visits
            atomicMin(&g_nf_t0, tg0);
            long long rel = (long long)(tg0 - *(volatile unsigned long long *)&g_nf_t0);
            unsigned b = rel < 0 ? 0u : (unsigned)(rel >> 16);
            if (b > 511u) b = 511u;
            atomicAdd(&g_nf_hist[2 * b], 1ull);
            atomicAdd(&g_nf_hist[2 * b + 1], gtimer() - tg0);
        }
#ifdef NF_STATS_TAIL
        if (tid == 0 && S.mid) {        // only the visits of the tail (a raster with more visits than log entries)
#else
        if (tid == 0) {
#endif
            unsigned k = atomicAdd(&g_nf_nlog, 1u);
            if (k < 262144u) {
                unsigned long long rel = tg2 - tg1; if (rel > 0xffffffull) rel = 0xffffffull;
                g_nf_log[4 * k] = tg0; g_nf_log[4 * k + 1] = tg1; g_nf_log[4 * k + 2] = gtimer();
                g_nf_log[4 * k + 3] = (unsigned long long)(unsigned)t | ((unsigned long long)(nrounds & 0xff) << 32) | (rel << 40);
            }
        }
#endif
        __syncthreads();
        if (tid == 0) {
            // side bits that arrived while the tile ran mean it has to run again
            if (p2p) {
                if (atomicAnd_system(tileflag + t, ~NF_RUNNING) & NF_SIDES) nf_push(ring, cap, ctl, t, true, pp->gactive, false);
                // the band runs dry: one band less is active; the last one ends every rank's kernel (system-scope fence:
                // this is the point at which another GPU may conclude that everything this band wrote is in place)
                __threadfence();
                if (atomicSub_system(&ctl->pending, 1) == 1) {
                    __threadfence_system();
                    if (atomicSub_system(pp->gactive, 1) == 1)
                        for (int k = 0; k < pp->world; k++) *(volatile int *)pp->done_all[k] = 1;
                }
            } else {
                if (atomicAnd(tileflag + t, ~NF_RUNNING) & NF_SIDES) nf_push(ring, cap, ctl, t);
                __threadfence();
                if (atomicSub(&ctl->pending, 1) == 1) atomicExch(&ctl->done, 1);
            }
        }
    }
}

// Row band: the fixed flags (seed or raster border: W = z for good) of the band's first and last own row, for the
// neighbours' k_nf_init_tile.  blockIdx.y = 0: first row -> ftop, 1: last row -> fbot.
__global__ void __launch_bounds__(256) k_band_edgefix(const float *__restrict__ z, const float *__restrict__ F,
                                                      uint8_t *ftop, uint8_t *fbot, int rows, int cols, int open) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    int r = blockIdx.y ? rows - 1 : 0;
    long long i = (long long)r * cols + c;
    unsigned char fx;
    if ((r == 0 && !(open & 1)) || c == 0 || (r == rows - 1 && !(open & 2)) || c == cols - 1) fx = 1;
    else {
        float f = F[i], m = INFINITY;
#pragma unroll
        for (int dr = -1; dr <= 1; dr++)
#pragma unroll
            for (int dc = -1; dc <= 1; dc++) {
                if (dr == 0 && dc == 0) continue;
                m = fminf(m, __ldg(F + i + (long long)dr * cols + dc));
            }
        fx = (f == z[i]) && (m < f);
    }
    (blockIdx.y ? fbot : ftop)[c] = fx;
}

// Row band: the band's first / last own row of the integer raster (whole padded rows) -> the neighbours' mailboxes
__global__ void __launch_bounds__(256) k_band_ir_publish(const int *__restrict__ Dg, int P, int rows, const NfP2P *pp) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P) return;
    int *peer = blockIdx.y ? (int *)pp->down.mail : (int *)pp->up.mail;
    if (!peer) return;
    peer[k] = Dg[(size_t)(blockIdx.y ? rows : 1) * P + k];
}

// End of the integer-raster solve: W is written once, and verified on the way.  A CTA rebuilds the float64 surface
// of a 64x64 tile + apron in shared memory — lake / flat cell: W = F + D * ulp(F) (exact: one binade, D * ulp is a
// multiple of ulp below 2^29 ulps; +inf if the solve never reached the cell), anything else: W = z — stores the
// tile and checks W == max(z, min(min4diag W + diag, min4edge W + short)) at every interior cell (SURVEY.md A.2:
// passing it certifies the surface, however it was computed).  Violations are counted in ctl->nviol.  With the tile and
// its apron in shared memory the D8 flow direction of every cell of the tile (K3, flow.py:142-167, edges flowing
// outward) is one more stencil over the same data: written to `flowdir` when the caller wants it (the pipeline), which
// saves K3's own pass over the float64 surface.  It is only valid if the verification passes.
__global__ void __launch_bounds__(256) k_nf_finish_ir(const float *__restrict__ z, const float *__restrict__ F,
                                                      const int *__restrict__ Dg, int P, double *__restrict__ W,
                                                      NfCtl *ctl, int rows, int cols, int tiles_x, double sh, double dg,
                                                      uint8_t *__restrict__ flowdir, double inv_sqrt2, int open,
                                                      const int *__restrict__ mail_top, const int *__restrict__ mail_bot) {
    // Row band (open != 0): the rows above / below the band are the neighbours' edge rows - z and F from the halo rows
    // of the band's rasters, the distances from the mailbox rows the neighbours wrote (padded like a row of Dg).
    const int rlo = (open & 1) ? -1 : 0, rhi = rows + ((open & 2) ? 1 : 0);
    constexpr int LD = NF_T + 2;
    __shared__ double sW[LD * LD];
    const int tile = blockIdx.x, tid = threadIdx.x;
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int r0 = ty * NF_T, c0 = tx * NF_T;
    // 66 x 66 cells, 18 per thread in three batches of six: the loads of a batch do not depend on each other's
    // values (z and F are read whether or not the cell turns out to be a lake cell), so they are all in flight together
#pragma unroll 1
    for (int batch = 0; batch < 3; batch++) {
        int dv[6];
        float zv[6], fv[6];
#pragma unroll
        for (int j = 0; j < 6; j++) {
            int k = tid + 256 * (batch * 6 + j);
            int lr = k / LD, lc = k - lr * LD;
            int r = r0 + lr - 1, c = c0 + lc - 1;
            dv[j] = D_WALL; zv[j] = INFINITY; fv[j] = 0.f;
            if (k < LD * LD && r >= rlo && r < rhi && c >= 0 && c < cols) {
                long long i = (long long)r * cols + c;
                dv[j] = r < 0 ? __ldg(mail_top + c + 4) : (r >= rows ? __ldg(mail_bot + c + 4) : __ldg(Dg + (size_t)(r + 1) * P + (c + 4)));
                zv[j] = __ldg(z + i);
                fv[j] = __ldg(F + i);
            }
        }
#pragma unroll
        for (int j = 0; j < 6; j++) {
            int k = tid + 256 * (batch * 6 + j);
            if (k >= LD * LD) continue;
            double w = (double)zv[j];                   // seeds, border cells; +inf outside the raster
            if (dv[j] == D_INF) w = INFINITY;           // a lake cell the solve never reached
            else if (dv[j] < D_INF) {
                double fd = (double)fv[j];
                double ulp = __longlong_as_double((long long)(nf_binade(fd) - 52 + 1023) << 52);
                w = __dadd_rn(fd, __dmul_rn((double)dv[j], ulp));
            }
            sW[k] = w;
        }
    }
    __syncthreads();
    int bad = 0;
    for (int k = tid; k < NF_T * NF_T; k += 256) {
        int lr = k >> 6, lc = k & 63;
        int r = r0 + lr, c = c0 + lc;
        if (r >= rows || c >= cols) continue;
        const double *p = sW + (lr + 1) * LD + (lc + 1);
        size_t i = (size_t)r * cols + c;
        double w = *p;
        W[i] = w;
        int code = 8;
        if ((r > 0 || (open & 1)) && c > 0 && (r < rows - 1 || (open & 2)) && c < cols - 1) {
            double d4 = dmin2(p[-LD - 1], dmin2(p[-LD + 1], dmin2(p[LD - 1], p[LD + 1])));
            double e4 = dmin2(p[-LD], dmin2(p[-1], dmin2(p[1], p[LD])));
            double m = dmin2(__dadd_rn(d4, dg), __dadd_rn(e4, sh));
            double zc = (double)__ldg(z + i);
            double g = m >= zc ? m : zc;
            if (g != w) bad = 1;
            if (flowdir) code = d8_code(w, p[-LD], p[-LD + 1], p[1], p[LD + 1], p[LD], p[LD - 1], p[-1], p[-LD - 1], inv_sqrt2);
        }
        if (flowdir) flowdir[i] = (uint8_t)d8_border(code, r == 0 && !(open & 1), r == rows - 1 && !(open & 2), c, cols);
    }
    int cnt = __syncthreads_count(bad);
    if (tid == 0 && cnt) atomicAdd(&ctl->nviol, cnt);
}

}  // namespace ms

/* The cap of the fast path: candidates more than this above the plain fill are ignored.  The solution exceeds the
 * plain fill by (geodesic steps to the lake's outlet) * diag at most; 4 * (rows + cols) steps covers every lake that
 * does not wind back and forth across the whole raster, and is far below the millimetre-scale gaps to shore cells
 * that the cap is there to keep out (a bound derived from the number of lake cells reaches a millimetre at 8192^2
 * and stops filtering).  A lake that needs more is caught by the verification and solved by the uncapped path. */
extern "C" double ms_nf_cap_bound(int64_t rows, int64_t cols, double diag_eps) {
    return 4.0 * (double)(rows + cols) * diag_eps;
}

namespace ms {

int g_nf_use_int = 1;      // MS_NF_INT=0 in the environment keeps every tile in the float64 form (debugging)

template <bool CAP>
static int nf_launch_solve(const float *zsrc, double *W, int *ring, int cap, int *tileflag, const int *tilesides,
                           NfCtl *ctl, int rows,
                           int cols, int tiles_x, int tiles_y, int ntiles, double sh, double dg, int use_int,
                           double capB, int open, int64_t units, cudaStream_t s) {
    static int grid_blocks = 0;
    if (!grid_blocks) {
        MS_CUDA(cudaFuncSetAttribute(k_nf_solve<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, NF_SMEM));
        int dev = 0, sms = 0, per_sm = 0;
        MS_CUDA(cudaGetDevice(&dev));
        MS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        MS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_nf_solve<CAP>, 256, NF_SMEM));
        if (per_sm < 1) { set_error("fill_terrain_no_flats: solver kernel does not fit on an SM"); return MS_ERR_CUDA; }
        grid_blocks = sms * per_sm;
    }
    void *args[] = {(void *)&zsrc, (void *)&W, (void *)&ring, (void *)&cap, (void *)&tileflag, (void *)&tilesides,
                    (void *)&ctl,
                    (void *)&rows, (void *)&cols, (void *)&tiles_x, (void *)&tiles_y, (void *)&sh, (void *)&dg,
                    (void *)&use_int, (void *)&capB, (void *)&open};
    // consumers wait on the FIFO, so every CTA must be resident: cooperative launch guarantees it (or fails)
    int g = grid_blocks < ntiles ? grid_blocks : ntiles;
    prof_units(units);
    if (g_prof) prof_begin(CAP ? "k_nf_solve<true>" : "k_nf_solve<false>", s);
    cudaError_t e = cudaLaunchCooperativeKernel((const void *)k_nf_solve<CAP>, dim3(g), dim3(256), args, NF_SMEM, s);
    if (g_prof) prof_end(s);
    g_launches++;
    if (e != cudaSuccess) {
        set_error("%s:%d: cooperative launch k_nf_solve -> %s", __FILE__, __LINE__, cudaGetErrorString(e));
        return MS_ERR_CUDA;
    }
    return MS_OK;
}

static int nf_launch_solve_ir(const float *F, int *Dg, int P, int *ring, int cap, int *tileflag, const int *tilesides,
                              const int *tmeta, NfCtl *ctl, int *irbad, int rows, int cols, int tiles_x, int tiles_y,
                              int ntiles, double sh, double dg, int64_t units, cudaStream_t s, const NfP2P *pp = nullptr) {
    static int grid_blocks_of[2] = {0, 0};
    const void *kern = pp ? (const void *)k_nf_solve_ir<true> : (const void *)k_nf_solve_ir<false>;
    int &grid_blocks = grid_blocks_of[pp ? 1 : 0];
    if (!grid_blocks) {
        MS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, IR_SMEM));
        int dev = 0, sms = 0, per_sm = 0;
        MS_CUDA(cudaGetDevice(&dev));
        MS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        MS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, IR_NT, IR_SMEM));
        if (per_sm < 1) { set_error("fill_terrain_no_flats: solver kernel does not fit on an SM"); return MS_ERR_CUDA; }
        grid_blocks = sms * per_sm;
    }
    void *args[] = {(void *)&F, (void *)&Dg, (void *)&P, (void *)&ring, (void *)&cap, (void *)&tileflag,
                    (void *)&tilesides, (void *)&tmeta, (void *)&ctl, (void *)&irbad, (void *)&rows, (void *)&cols,
                    (void *)&tiles_x, (void *)&tiles_y, (void *)&sh, (void *)&dg, (void *)&pp};
    int g = (grid_blocks < ntiles || pp) ? grid_blocks : ntiles;
    prof_units(units);
    if (g_prof) prof_begin("k_nf_solve_ir", s);
    cudaError_t e = cudaLaunchCooperativeKernel(kern, dim3(g), dim3(IR_NT), args, IR_SMEM, s);
    if (g_prof) prof_end(s);
    g_launches++;
    if (e != cudaSuccess) {
        set_error("%s:%d: cooperative launch k_nf_solve_ir -> %s", __FILE__, __LINE__, cudaGetErrorString(e));
        return MS_ERR_CUDA;
    }
    return MS_OK;
}

// flowdir_out (optional): the D8 flow directions of the result with edges flowing outward (K3); *flowdir_done says
// whether they were written (the integer-raster path does it in its finishing pass, the others do not).
int fill_no_flats_dev_impl(const float *dtm, const float *filled, double sh, double dg, double *out,
                           int64_t rows, int64_t cols, int64_t *stats, cudaStream_t s, uint8_t *flowdir_out,
                           int *flowdir_done) {
    if (flowdir_done) *flowdir_done = 0;
    if (!dtm || !out) { set_error("fill_terrain_no_flats: null pointer"); return MS_ERR_ARG; }
    if (rows < 3 || cols < 3 || rows * cols > (1ll << 30)) {
        set_error("fill_terrain_no_flats: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    if (!(sh >= 0) || !(dg >= 0)) { set_error("fill_terrain_no_flats: short/diag must be >= 0"); return MS_ERR_ARG; }
    int64_t n = rows * cols;
    DevBuf<float> ftmp;
    if (!filled) {
        MS_TRY(ftmp.alloc((size_t)n, s));
        MS_TRY(fill_terrain_dev_impl(dtm, ftmp.p, nullptr, rows, cols, nullptr, s));
        filled = ftmp.p;
    }
    static bool env_done = false;
    if (!env_done) {
        const char *e = getenv("MS_NF_INT");
        if (e && e[0] == '0') g_nf_use_int = 0;
        env_done = true;
    }
    int tiles_x = (int)cdiv(cols, NF_T), tiles_y = (int)cdiv(rows, NF_T);
    int ntiles = tiles_x * tiles_y;
    int cap_ring = ntiles + NF_RING_SLACK;          // a tile is in the FIFO at most once
    DevBuf<int> tileflag, tilesides, ring;
    DevBuf<uint8_t> banned;
    DevBuf<NfCtl> ctl;
    MS_TRY(tileflag.alloc((size_t)ntiles, s));
    MS_TRY(tilesides.alloc((size_t)ntiles, s));
    MS_TRY(ring.alloc((size_t)cap_ring, s));
    MS_TRY(ctl.alloc(1, s));
    bool cap = sh > 0 && dg > 0;      // capped fast path first; a verification failure falls back to the generic one
    const double cap_bound = ms_nf_cap_bound(rows, cols, dg);
    // integer-raster form of the capped solve: padded int32 raster (see k_nf_solve_ir)
    bool use_ir = cap && g_nf_use_int;
    const int P = tiles_x * NF_T + 8;
    const size_t dg_cells = (size_t)P * ((size_t)tiles_y * NF_T + 2);
    DevBuf<int> Dg, tmeta, irbad;
    if (use_ir) {
        MS_TRY(Dg.alloc(dg_cells, s));
        MS_TRY(tmeta.alloc((size_t)ntiles, s));
        MS_TRY(irbad.alloc(1, s));
    }
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    int64_t visits = 0, tries = 0, rounds = 0;
    for (;;) {
        tries++;
        MS_CUDA(cudaMemsetAsync(tileflag.p, 0, (size_t)ntiles * sizeof(int), s));
        MS_CUDA(cudaMemsetAsync(tilesides.p, 0, (size_t)ntiles * sizeof(int), s));
        MS_CUDA(cudaMemsetAsync(ring.p, 0xff, (size_t)cap_ring * sizeof(int), s));
        MS_CUDA(cudaMemsetAsync(ctl.p, 0, sizeof(NfCtl), s));
        const bool ir = cap && use_ir;
        if (ir) {
            const int inner_rows = tiles_y * NF_T;
            MS_LAUNCH(k_ir_frame, cdiv(2 * (int64_t)P + 8 * (int64_t)inner_rows, 256), 256, 0, s, Dg.p, P, inner_rows);
            MS_CUDA(cudaMemsetAsync(irbad.p, 0, sizeof(int), s));
        }
        if (cap) {
            CUtensorMap zmap, fmap;
            memset(&zmap, 0, sizeof(zmap));
            memset(&fmap, 0, sizeof(fmap));
            if (tma_map_2d(&zmap, dtm, rows, cols, NI_A, NI_LD_TMA, true, true) &&
                tma_map_2d(&fmap, filled, rows, cols, NI_A, NI_LD_TMA, true, true))
                MS_LAUNCH(k_nf_init_tile<true>, ntiles, 256, 0, s, dtm, filled, out, tileflag.p, tilesides.p, ctl.p, (int)rows,
                          (int)cols, tiles_x, sh, dg, cap_bound, ir ? Dg.p : (int *)nullptr, P, tmeta.p, irbad.p, 0,
                          (const uint8_t *)nullptr, (const uint8_t *)nullptr, zmap, fmap);
            else
                MS_LAUNCH(k_nf_init_tile<false>, ntiles, 256, 0, s, dtm, filled, out, tileflag.p, tilesides.p, ctl.p, (int)rows,
                          (int)cols, tiles_x, sh, dg, cap_bound, ir ? Dg.p : (int *)nullptr, P, tmeta.p, irbad.p, 0,
                          (const uint8_t *)nullptr, (const uint8_t *)nullptr, zmap, fmap);
        }
        else
            MS_LAUNCH(k_nf_init, g2, 256, 0, s, dtm, filled, out, banned.p, tileflag.p, tilesides.p, ctl.p, (int)rows,
                      (int)cols, tiles_x, 0);
        MS_LAUNCH(k_nf_compact, cdiv(ntiles, 256), 256, 0, s, tileflag.p, ring.p, ctl.p, ntiles);
        if (ir) {
            MS_TRY(nf_launch_solve_ir(filled, Dg.p, P, ring.p, cap_ring, tileflag.p, tilesides.p, tmeta.p, ctl.p, irbad.p,
                                      (int)rows, (int)cols, tiles_x, tiles_y, ntiles, sh, dg, n, s));
            prof_units(n);
            MS_LAUNCH(k_nf_finish_ir, ntiles, 256, 0, s, dtm, filled, Dg.p, P, out, ctl.p, (int)rows, (int)cols, tiles_x, sh,
                      dg, flowdir_out, 1.0 / pow(2.0, 0.5), 0, (const int *)nullptr, (const int *)nullptr);      // _flow.pyx:93-94: INV_SQRT2 = 1 / 2**0.5
        } else if (cap) {
            MS_TRY(nf_launch_solve<true>(filled, out, ring.p, cap_ring, tileflag.p, tilesides.p, ctl.p, (int)rows, (int)cols, tiles_x,
                                         tiles_y, ntiles, sh, dg, g_nf_use_int, cap_bound, 0, n, s));
        } else {
            MS_TRY(nf_launch_solve<false>(dtm, out, ring.p, cap_ring, tileflag.p, tilesides.p, ctl.p, (int)rows, (int)cols, tiles_x,
                                          tiles_y, ntiles, sh, dg, 0, 0.0, 0, n, s));
        }
        if (!ir) MS_LAUNCH(k_nf_verify, g2, 256, 0, s, dtm, out, banned.p, ctl.p, (int)rows, (int)cols, sh, dg, 0);
        MS_TRY(ms::readback(h, ctl.p, sizeof(NfCtl), s));
        int *h_irbad = (int *)(h + 1);
        *h_irbad = 0;
        if (ir) MS_TRY(ms::readback(h_irbad, irbad.p, sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        visits += h->visits;
        rounds += h->reserved;
        if (ir && *h_irbad) {       // something does not fit the integer form: the W-based solver takes over
            use_ir = false;
            continue;
        }
        if (h->done != 1 && h->tail != 0) {
            set_error("fill_terrain_no_flats: tile solver stopped early (done=%d, pending=%d)", h->done, h->pending);
            return MS_ERR_NOCONV;
        }
        if (h->nviol == 0) {
            if (ir && flowdir_out && flowdir_done) *flowdir_done = 1;
            break;
        }
        if (cap) {          // the heuristic cap (or a seed) was wrong somewhere: redo without it
            cap = false;
            continue;
        }
        if (!banned.p) {
            // first failure: allocate the ban map and mark the failing seeds
            MS_TRY(banned.alloc((size_t)n, s));
            MS_CUDA(cudaMemsetAsync(banned.p, 0, (size_t)n, s));
            MS_LAUNCH(k_nf_verify, g2, 256, 0, s, dtm, out, banned.p, ctl.p, (int)rows, (int)cols, sh, dg, 0);
        }
        if (tries > 1000) {
            set_error("fill_terrain_no_flats: seed verification did not settle");
            return MS_ERR_NOCONV;
        }
    }
    if (stats) { stats[0] = tries; stats[1] = visits; stats[2] = tries - 1; stats[3] = rounds; }
    return MS_OK;
}


// =====================================================================================================
// Row-band no-flats fill (SURVEY.md §8(e), K2).  The band solves its own rows with the halo rows as fixed data;
// the host side exchanges the first / last own row with the neighbours and calls the solver again on the tiles
// along a band edge whose halo changed, until no band changes any more; the verification stencil (with halos)
// certifies the result as in the single-GPU case.
// =====================================================================================================
__global__ void __launch_bounds__(256) k_nf_activate_edges(int *tileflag, const int *__restrict__ tilesides,
                                                           int tiles_x, int tiles_y, int which) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= tiles_x) return;
    if ((which & 1) && (tilesides[x] & 1)) atomicOr(tileflag + x, 1);
    int t = (tiles_y - 1) * tiles_x + x;
    if ((which & 2) && (tilesides[t] & 2)) atomicOr(tileflag + t, 2);
}

struct NfBandBufs {
    int *tileflag, *tilesides, *ring;
    NfCtl *ctl;
    int tiles_x, tiles_y, ntiles, cap_ring;
};

static int nf_band_bufs(ms_band *B, NfBandBufs *o) {
    o->tiles_x = (int)cdiv(B->cols, NF_T);
    o->tiles_y = (int)cdiv(B->rows, NF_T);
    o->ntiles = o->tiles_x * o->tiles_y;
    o->cap_ring = o->ntiles + NF_RING_SLACK;
    o->tileflag = (int *)band_buf(B, BB_NF_FLAG, (size_t)o->ntiles * sizeof(int));
    o->tilesides = (int *)band_buf(B, BB_NF_SIDES, (size_t)o->ntiles * sizeof(int));
    o->ring = (int *)band_buf(B, BB_NF_RING, (size_t)o->cap_ring * sizeof(int));
    o->ctl = (NfCtl *)band_buf(B, BB_NF_CTL, sizeof(NfCtl));
    if (!o->tileflag || !o->tilesides || !o->ring || !o->ctl) return MS_ERR_CUDA;
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_band_nf_init_dev(ms_band *B, const float *dem, const float *filled, double *fnf, int64_t *nonseed,
                        void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !filled || !fnf) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    MS_CUDA(cudaMemsetAsync(nb.tileflag, 0, (size_t)nb.ntiles * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.tilesides, 0, (size_t)nb.ntiles * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.ctl, 0, sizeof(NfCtl), s));
    dim3 g2(cdiv(B->cols, 64), cdiv(B->rows, 4));
    MS_LAUNCH(k_nf_init, g2, 256, 0, s, dem, filled, fnf, B->nf_ban ? (const uint8_t *)B->buf[BB_NF_BANNED] : (const uint8_t *)nullptr,
              nb.tileflag, nb.tilesides, nb.ctl, (int)B->rows, (int)B->cols, nb.tiles_x, B->open);
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::stream_sync(s));
    if (nonseed) *nonseed = h->nonseed;
    return MS_OK;
}

/* Seed repair in band mode (the single-GPU loop of fill_no_flats_dev_impl): a seed is a dry cell with a strictly lower
 * filled neighbour, taken as W = z; next to a lake whose surface has risen above it by the time the wave arrives that
 * is wrong, the stencil fails there, and the cell has to be relaxed like a lake cell.  reset != 0: forget the band's
 * ban map (start of a stage).  Otherwise: run the verification stencil (incl. halo rows) on fnf, mark every failing
 * cell in the ban map (kept across calls, so bans accumulate) and return the count; ms_band_nf_init_dev then treats
 * the marked cells as non-seeds. */
int ms_band_nf_ban_dev(ms_band *B, const float *dem, const double *fnf, double short_eps, double diag_eps, int reset,
                       int64_t *nviol, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    if (reset) { B->nf_ban = 0; return MS_OK; }
    if (!dem || !fnf || !nviol) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    const size_t n = (size_t)B->rows * (size_t)B->cols;
    uint8_t *banned = (uint8_t *)band_buf(B, BB_NF_BANNED, n);
    if (!banned) return MS_ERR_CUDA;
    if (!B->nf_ban) MS_CUDA(cudaMemsetAsync(banned, 0, n, s));
    B->nf_ban = 1;
    MS_CUDA(cudaMemsetAsync(nb.ctl, 0, sizeof(NfCtl), s));
    dim3 g2(cdiv(B->cols, 64), cdiv(B->rows, 4));
    MS_LAUNCH(k_nf_verify, g2, 256, 0, s, dem, fnf, banned, nb.ctl, (int)B->rows, (int)B->cols, short_eps, diag_eps, B->open);
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::stream_sync(s));
    *nviol = h->nviol;
    return MS_OK;
}

/* mode 0: first solve after ms_band_nf_init_dev (+ halo exchange of fnf); mode 1: solve again after the halo rows
 * named by `edges` (bit 0 top, bit 1 bottom) changed.  cap = 1: capped fast path (cap_bound = the bound on
 * solution - plain fill, the same on every band); cap = 0: generic float64 path.  *changed_edges: bit 0 / 1 = the
 * band's first / last own row may have changed (conservative: any tile of that row wrote something). */
int ms_band_nf_solve_dev(ms_band *B, const float *dem, const float *filled, double *fnf, double short_eps,
                         double diag_eps, double cap_bound, int cap, int mode, int edges, int64_t *tile_visits,
                         void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !filled || !fnf) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    int rows = (int)B->rows, cols = (int)B->cols;
    dim3 g2(cdiv(cols, 64), cdiv(rows, 4));
    MS_CUDA(cudaMemsetAsync(nb.ring, 0xff, (size_t)nb.cap_ring * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.ctl, 0, sizeof(NfCtl), s));
    if (mode == 0) {
        if (cap) MS_LAUNCH(k_nf_seedcand, g2, 256, 0, s, filled, fnf, nb.ctl, rows, cols, short_eps, diag_eps, cap_bound, B->open);
    } else {
        MS_LAUNCH(k_nf_activate_edges, cdiv(nb.tiles_x, 256), 256, 0, s, nb.tileflag, nb.tilesides, nb.tiles_x, nb.tiles_y, edges);
    }
    MS_LAUNCH(k_nf_compact, cdiv(nb.ntiles, 256), 256, 0, s, nb.tileflag, nb.ring, nb.ctl, nb.ntiles);
    if (cap)
        MS_TRY(nf_launch_solve<true>(filled, fnf, nb.ring, nb.cap_ring, nb.tileflag, nb.tilesides, nb.ctl, rows, cols,
                                     nb.tiles_x, nb.tiles_y, nb.ntiles, short_eps, diag_eps, g_nf_use_int, cap_bound,
                                     B->open, B->rows * B->cols, s));
    else
        MS_TRY(nf_launch_solve<false>(dem, fnf, nb.ring, nb.cap_ring, nb.tileflag, nb.tilesides, nb.ctl, rows, cols,
                                      nb.tiles_x, nb.tiles_y, nb.ntiles, short_eps, diag_eps, 0, 0.0, B->open,
                                      B->rows * B->cols, s));
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::stream_sync(s));
    if (h->done != 1 && h->tail != 0) {
        set_error("band no-flats: tile solver stopped early (done=%d, pending=%d)", h->done, h->pending);
        return MS_ERR_NOCONV;
    }
    if (tile_visits) *tile_visits = h->visits;
    return MS_OK;
}


// ---- P2P: shared block, peer mapping, solve -----------------------------------------------------------------
}  // extern "C"

namespace ms {
struct NfSharedLayout {
    size_t off_gactive, off_flag, off_sides, off_ring, off_mtop, off_mbot, total;
    int tiles_x, tiles_y, ntiles, cap;
};
static NfSharedLayout nf_layout(int64_t rows, int64_t cols) {
    NfSharedLayout L;
    L.tiles_x = (int)cdiv(cols, NF_T);
    L.tiles_y = (int)cdiv(rows, NF_T);
    L.ntiles = L.tiles_x * L.tiles_y;
    L.cap = L.ntiles + NF_RING_SLACK;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 255) & ~(size_t)255; return at; };
    take(sizeof(NfCtl));                       // the control block is at offset 0
    L.off_gactive = take(sizeof(int));
    L.off_flag = take((size_t)L.ntiles * sizeof(int));
    L.off_sides = take((size_t)L.ntiles * sizeof(int));
    L.off_ring = take((size_t)L.cap * sizeof(int));
    // a mailbox row holds the padded int32 row of the integer raster
    size_t mail = ((size_t)L.tiles_x * NF_T + 8) * sizeof(int);
    L.off_mtop = take(mail);
    L.off_mbot = take(mail);
    L.total = o;
    return L;
}

__global__ void k_nf_arm(NfCtl *ctl, int *gactive) {
    if (ctl->pending > 0) atomicAdd_system(gactive, 1);
}
}  // namespace ms

extern "C" {

/* info (80 bytes): CUDA IPC handle of the band's shared block, its address in this process, the process id */
int ms_band_nf_shared_create(ms_band *B, void *info80) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !info80) { set_error("band no-flats P2P: null pointer"); return MS_ERR_ARG; }
    if (!B->nf_shared) {
        NfSharedLayout L = nf_layout(B->rows, B->cols);
        void *p = nullptr;
        MS_CUDA(cudaMalloc(&p, L.total));
        MS_CUDA(cudaMemset(p, 0, L.total));
        B->nf_shared = p;
        // the solver state of this band lives in the block, where the neighbours can reach it
        int slots[4] = {BB_NF_CTL, BB_NF_FLAG, BB_NF_SIDES, BB_NF_RING};
        size_t offs[4] = {0, L.off_flag, L.off_sides, L.off_ring};
        for (int k = 0; k < 4; k++) {
            if (B->buf[slots[k]] && B->cap[slots[k]] != SIZE_MAX) cudaFree(B->buf[slots[k]]);
            B->buf[slots[k]] = (char *)p + offs[k];
            B->cap[slots[k]] = SIZE_MAX;
        }
    }
    unsigned char *out = (unsigned char *)info80;
    cudaIpcMemHandle_t h;
    MS_CUDA(cudaIpcGetMemHandle(&h, B->nf_shared));
    memcpy(out, &h, 64);
    unsigned long long addr = (unsigned long long)(uintptr_t)B->nf_shared, pid = (unsigned long long)getpid();
    memcpy(out + 64, &addr, 8);
    memcpy(out + 72, &pid, 8);
    return MS_OK;
}

/* infos: world x 80 bytes as written by ms_band_nf_shared_create on every rank; rows_all: own rows of every band */
int ms_band_nf_shared_open(ms_band *B, int rank, int world, const void *infos, const int64_t *rows_all) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->nf_shared || !infos || !rows_all || world < 1 || world > NF_MAXRANKS || rank < 0 || rank >= world) {
        set_error("band no-flats P2P: bad argument");
        return MS_ERR_ARG;
    }
    const unsigned char *in = (const unsigned char *)infos;
    unsigned long long mypid = (unsigned long long)getpid();
    for (int k = 0; k < world; k++) {
        if (B->nf_peer[k]) continue;
        if (k == rank) { B->nf_peer[k] = B->nf_shared; continue; }
        unsigned long long addr, pid;
        memcpy(&addr, in + 80 * k + 64, 8);
        memcpy(&pid, in + 80 * k + 72, 8);
        if (pid == mypid) {
            B->nf_peer[k] = (void *)(uintptr_t)addr;      // a band of the same process: same address space
        } else {
            cudaIpcMemHandle_t h;
            memcpy(&h, in + 80 * k, 64);
            void *p = nullptr;
            MS_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            B->nf_peer[k] = p;
            B->nf_peer_ipc[k] = 1;
        }
    }
    B->nf_rank = rank;
    B->nf_world = world;
    NfP2P pp;
    memset(&pp, 0, sizeof(pp));
    NfSharedLayout me = nf_layout(B->rows, B->cols);
    pp.mail_top = (void *)((char *)B->nf_shared + me.off_mtop);
    pp.mail_bot = (void *)((char *)B->nf_shared + me.off_mbot);
    pp.world = world;
    pp.gactive = (int *)((char *)B->nf_peer[0] + nf_layout(rows_all[0], B->cols).off_gactive);
    for (int k = 0; k < world; k++) pp.done_all[k] = &((NfCtl *)B->nf_peer[k])->done;
    for (int side = 0; side < 2; side++) {
        int k = side ? rank + 1 : rank - 1;
        if (k < 0 || k >= world || !(B->open & (side ? 2 : 1))) continue;
        NfSharedLayout L = nf_layout(rows_all[k], B->cols);
        char *base = (char *)B->nf_peer[k];
        NfPeer q;
        q.tileflag = (int *)(base + L.off_flag);
        q.ring = (int *)(base + L.off_ring);
        q.ctl = (NfCtl *)base;
        q.mail = (void *)(base + (side ? L.off_mtop : L.off_mbot));      // the row of theirs that faces this band
        q.tiles_y = L.tiles_y;
        q.cap = L.cap;
        if (side) pp.down = q; else pp.up = q;
    }
    if (!B->nf_pp_dev) MS_CUDA(cudaMalloc(&B->nf_pp_dev, sizeof(NfP2P)));
    MS_CUDA(cudaMemcpy(B->nf_pp_dev, &pp, sizeof(pp), cudaMemcpyHostToDevice));
    return MS_OK;
}

/* P2P step 2 (all ranks prepared): a band with queued tiles counts itself active.  The caller synchronises again. */
int ms_band_nf_p2p_arm_dev(ms_band *B, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->nf_pp_dev) { set_error("band no-flats P2P: not set up"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfP2P pp;
    MS_CUDA(cudaMemcpy(&pp, B->nf_pp_dev, sizeof(pp), cudaMemcpyDeviceToHost));
    MS_LAUNCH(k_nf_arm, 1, 1, 0, s, (NfCtl *)B->nf_shared, pp.gactive);
    MS_TRY(ms::stream_sync(s));
    return MS_OK;
}

/* ---- integer-raster form of the P2P solve (the single-GPU solver k_nf_solve_ir across bands) -------------------
 * 1. ms_band_nf_ir_edgefix_dev: fixed flags of the band's first / last own row; the caller hands them to the
 *    neighbours (they are the flags of the neighbours' halo rows).
 * 2. ms_band_nf_ir_prepare_dev: padded int32 raster of the band (k_nf_init_tile with the halo rows), the band's edge
 *    rows stored into the neighbours' mailboxes, FIFO := tiles with lake cells.  *queued = tiles queued, *irbad = the
 *    band does not fit the integer form.  The caller synchronises all ranks, then ms_band_nf_p2p_arm_dev, synchronises
 *    again, then
 * 3. ms_band_nf_ir_solve_launch_dev / _wait_dev: every band's k_nf_solve_ir at once; ends when no band has work left.
 * 4. ms_band_nf_ir_finish_dev: W = F + D ulp(F) written once, verified against the fixed-point equation with the
 *    halo rows (*nviol), D8 codes of the band's rows written on the way (K3 fused, edges of the RASTER flow outward). */
int ms_band_nf_ir_edgefix_dev(ms_band *B, const float *dem, const float *filled, uint8_t *fix_top, uint8_t *fix_bot,
                              void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !filled || !fix_top || !fix_bot) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    MS_LAUNCH(k_band_edgefix, dim3(cdiv(B->cols, 256), 2), 256, 0, s, dem, filled, fix_top, fix_bot, (int)B->rows,
              (int)B->cols, B->open);
    return MS_OK;
}

int ms_band_nf_ir_prepare_dev(ms_band *B, const float *dem, const float *filled, double short_eps, double diag_eps,
                              double cap_bound, const uint8_t *fix_top, const uint8_t *fix_bot, int64_t *queued,
                              int *irbad_out, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->nf_pp_dev || !dem || !filled || !queued || !irbad_out) {
        set_error("band no-flats P2P: not set up");
        return MS_ERR_ARG;
    }
    if (((B->open & 1) && !fix_top) || ((B->open & 2) && !fix_bot)) { set_error("band no-flats: halo flags missing"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    const int P = nb.tiles_x * NF_T + 8;
    const int inner_rows = nb.tiles_y * NF_T;
    int *Dg = (int *)band_buf(B, BB_NF_DG, (size_t)P * ((size_t)inner_rows + 2) * sizeof(int));
    int *tmeta = (int *)band_buf(B, BB_NF_TMETA, (size_t)nb.ntiles * sizeof(int));
    int *irbad = (int *)band_buf(B, BB_NF_IRBAD, sizeof(int));
    if (!Dg || !tmeta || !irbad) return MS_ERR_CUDA;
    NfSharedLayout L = nf_layout(B->rows, B->cols);
    char *base = (char *)B->nf_shared;
    MS_CUDA(cudaMemsetAsync(nb.tileflag, 0, (size_t)nb.ntiles * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.tilesides, 0, (size_t)nb.ntiles * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.ring, 0xff, (size_t)nb.cap_ring * sizeof(int), s));
    MS_CUDA(cudaMemsetAsync(nb.ctl, 0, sizeof(NfCtl), s));
    MS_CUDA(cudaMemsetAsync(irbad, 0, sizeof(int), s));
    if (B->nf_rank == 0) MS_CUDA(cudaMemsetAsync(base + L.off_gactive, 0, sizeof(int), s));
    MS_LAUNCH(k_ir_frame, cdiv(2 * (int64_t)P + 8 * (int64_t)inner_rows, 256), 256, 0, s, Dg, P, inner_rows);
    prof_units(B->rows * B->cols);
    CUtensorMap nomap;
    memset(&nomap, 0, sizeof(nomap));
    MS_LAUNCH(k_nf_init_tile<false>, nb.ntiles, 256, 0, s, dem, filled, (double *)nullptr, nb.tileflag, nb.tilesides, nb.ctl,
              (int)B->rows, (int)B->cols, nb.tiles_x, short_eps, diag_eps, cap_bound, Dg, P, tmeta, irbad, B->open, fix_top,
              fix_bot, nomap, nomap);
    MS_LAUNCH(k_band_ir_publish, dim3(cdiv(P, 256), 2), 256, 0, s, Dg, P, (int)B->rows, (const NfP2P *)B->nf_pp_dev);
    // (queueing the tile rows next to an open band edge first - so that what crosses the edge reaches the neighbour
    // early - was measured at N = 2: 30.4 vs 30.0 ms, no gain; both bands are saturated for 27 of the 30 ms)
    MS_LAUNCH(k_nf_compact, cdiv(nb.ntiles, 256), 256, 0, s, nb.tileflag, nb.ring, nb.ctl, nb.ntiles);
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    int *h_irbad = (int *)(h + 1);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::readback(h_irbad, irbad, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    *queued = h->pending;
    *irbad_out = *h_irbad;
    return MS_OK;
}

/* launch: returns as soon as the solver kernel and the read-back of its control block are queued (the host may do
 * CPU work meanwhile; no other library call on this band until wait); wait: the result. */
int ms_band_nf_ir_solve_launch_dev(ms_band *B, const float *filled, double short_eps, double diag_eps, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->nf_pp_dev || !filled) { set_error("band no-flats P2P: not set up"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    const int P = nb.tiles_x * NF_T + 8;
    int *Dg = (int *)B->buf[BB_NF_DG], *tmeta = (int *)B->buf[BB_NF_TMETA], *irbad = (int *)B->buf[BB_NF_IRBAD];
    if (!Dg || !tmeta || !irbad) { set_error("band no-flats P2P: ms_band_nf_ir_prepare_dev first"); return MS_ERR_ARG; }
    MS_TRY(nf_launch_solve_ir(filled, Dg, P, nb.ring, nb.cap_ring, nb.tileflag, nb.tilesides, tmeta, nb.ctl, irbad,
                              (int)B->rows, (int)B->cols, nb.tiles_x, nb.tiles_y, nb.ntiles, short_eps, diag_eps,
                              B->rows * B->cols, s, (const NfP2P *)B->nf_pp_dev));
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    int *h_irbad = (int *)(h + 1);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::readback(h_irbad, irbad, sizeof(int), s));
    return MS_OK;
}

int ms_band_nf_ir_solve_wait_dev(ms_band *B, int64_t *tile_visits, int *irbad_out, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !irbad_out) { set_error("band no-flats P2P: null pointer"); return MS_ERR_ARG; }
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    int *h_irbad = (int *)(h + 1);
    MS_TRY(ms::stream_sync((cudaStream_t)stream));
    if (tile_visits) *tile_visits = h->visits;
    *irbad_out = *h_irbad;
    if (h->done != 1) {
        set_error("band no-flats P2P: solver stopped early (done=%d, pending=%d)", h->done, h->pending);
        return MS_ERR_NOCONV;
    }
    return MS_OK;
}

int ms_band_nf_ir_finish_dev(ms_band *B, const float *dem, const float *filled, double *fnf, uint8_t *flowdir,
                             double short_eps, double diag_eps, int64_t *nviol, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !B->nf_pp_dev || !dem || !filled || !fnf || !nviol) { set_error("band no-flats P2P: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    const int P = nb.tiles_x * NF_T + 8;
    int *Dg = (int *)B->buf[BB_NF_DG];
    if (!Dg) { set_error("band no-flats P2P: ms_band_nf_ir_prepare_dev first"); return MS_ERR_ARG; }
    NfSharedLayout L = nf_layout(B->rows, B->cols);
    char *base = (char *)B->nf_shared;
    MS_CUDA(cudaMemsetAsync(&nb.ctl->nviol, 0, sizeof(int), s));
    prof_units(B->rows * B->cols);
    MS_LAUNCH(k_nf_finish_ir, nb.ntiles, 256, 0, s, dem, filled, Dg, P, fnf, nb.ctl, (int)B->rows, (int)B->cols, nb.tiles_x,
              short_eps, diag_eps, flowdir, 1.0 / pow(2.0, 0.5), B->open, (const int *)(base + L.off_mtop),
              (const int *)(base + L.off_mbot));
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::stream_sync(s));
    *nviol = h->nviol;
    return MS_OK;
}

int ms_band_nf_verify_dev(ms_band *B, const float *dem, const double *fnf, double short_eps, double diag_eps,
                          int64_t *nviol, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!B || !dem || !fnf || !nviol) { set_error("band no-flats: null pointer"); return MS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    NfBandBufs nb;
    MS_TRY(nf_band_bufs(B, &nb));
    MS_CUDA(cudaMemsetAsync(nb.ctl, 0, sizeof(NfCtl), s));
    dim3 g2(cdiv(B->cols, 64), cdiv(B->rows, 4));
    MS_LAUNCH(k_nf_verify, g2, 256, 0, s, dem, fnf, (uint8_t *)nullptr, nb.ctl, (int)B->rows, (int)B->cols, short_eps,
              diag_eps, B->open);
    NfCtl *h = (NfCtl *)(host_flags().h + 32);
    MS_TRY(ms::readback(h, nb.ctl, sizeof(NfCtl), s));
    MS_TRY(ms::stream_sync(s));
    *nviol = h->nviol;
    return MS_OK;
}

int ms_fill_terrain_no_flats_dev(const float *dtm, const float *filled, double short_eps, double diag_eps,
                                 double *out, int64_t rows, int64_t cols, int64_t *stats, void *stream) {
    MS_TRY(ms::ensure_init());
    int64_t st[4] = {0, 0, 0, 0};       // the internal form also counts sweep rounds; the ABI documents three entries
    int rc = ms::fill_no_flats_dev_impl(dtm, filled, short_eps, diag_eps, out, rows, cols, st, (cudaStream_t)stream,
                                        nullptr, nullptr);
    if (stats) { stats[0] = st[0]; stats[1] = st[1]; stats[2] = st[2]; }
    return rc;
}

int ms_fill_terrain_no_flats(const float *dtm, double short_eps, double diag_eps, double *out, int64_t rows,
                             int64_t cols) {
    MS_TRY(ms::ensure_init());
    if (!dtm || !out) { ms::set_error("fill_terrain_no_flats: null pointer"); return MS_ERR_ARG; }
    if (rows < 3 || cols < 3 || rows * cols > (1ll << 30)) {
        ms::set_error("fill_terrain_no_flats: unsupported shape %lld x %lld", (long long)rows, (long long)cols);
        return MS_ERR_SHAPE;
    }
    cudaStream_t s = nullptr;
    size_t n = (size_t)(rows * cols);
    ms::HostCall hc;
    float *d = nullptr;
    MS_TRY(hc.in(dtm, n, s, &d));
    // asked for twice by the tool layer (dem.py:80, bluespots.py:203-205): the second time it is still on the device
    double *o = (double *)ms::cache_find_derived(d, ms::CK_NOFLATS, short_eps, diag_eps);
    if (!o) {
        // the plain fill of this DEM, if fill_terrain has just computed it (dem.py:67)
        const float *f = (const float *)ms::cache_find_derived(d, ms::CK_FILLED, 0, 0);
        MS_TRY(hc.out(n, &o));
        MS_TRY(ms::fill_no_flats_dev_impl(d, f, short_eps, diag_eps, o, rows, cols, nullptr, s, nullptr, nullptr));
        ms::cache_bind_derived(o, d, ms::CK_NOFLATS, short_eps, diag_eps);
    }
    MS_CUDA(cudaMemcpyAsync(out, o, n * sizeof(double), cudaMemcpyDeviceToHost, s));
    MS_TRY(ms::stream_sync(s));
    ms::cache_bind_host(o, out, n * sizeof(double));
    return MS_OK;
}

#ifdef NF_STATS
int ms_nf_log(unsigned long long *out, unsigned *n, int reset) {
    if (n) cudaMemcpyFromSymbol(n, ms::g_nf_nlog, sizeof(unsigned));
    if (out) cudaMemcpyFromSymbol(out, ms::g_nf_log, sizeof(unsigned long long) * 4 * 262144);
    if (reset) { unsigned z = 0; cudaMemcpyToSymbol(ms::g_nf_nlog, &z, sizeof(z)); }
    return 0;
}

int ms_nf_hist(unsigned long long *out1024, int reset) {
    if (out1024) cudaMemcpyFromSymbol(out1024, ms::g_nf_hist, sizeof(unsigned long long) * 1024);
    if (reset) {
        static unsigned long long z[1024];
        cudaMemcpyToSymbol(ms::g_nf_hist, z, sizeof(z));
        unsigned long long big = ~0ull;
        cudaMemcpyToSymbol(ms::g_nf_t0, &big, sizeof(big));
    }
    return 0;
}

int ms_nf_debug(unsigned long long *out, int n, int reset) {
    if (out) cudaMemcpyFromSymbol(out, ms::g_nf_dbg, sizeof(unsigned long long) * n);
    if (reset) { static unsigned long long z[16]; cudaMemcpyToSymbol(ms::g_nf_dbg, z, sizeof(z)); }
    return 0;
}
#endif

}  // extern "C"
