/*
 * malstroem_b200.h — C ABI of the B200-native (sm_100a) raster hot path of SDFIdk/malstroem.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / numpy types.  Every entry point
 * replaces one function of the reference's `malstroem.algorithms` layer (the layer its own native
 * plugin, malstroem/algorithms/speedups/__init__.py:37-78, rebinds); the reference file:line each one
 * stands in for is cited beside it.  The Python mirror in malstroem_b200/algorithms/ binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - rasters are C-contiguous row-major, `rows x cols`, rows*cols < 2^30 per device
 *   - functions without a suffix take HOST pointers and do H2D / compute / D2H themselves (blocking);
 *     `_dev` functions take DEVICE pointers plus a cudaStream_t (passed as void*) and only enqueue work,
 *     except where a count has to come back to the host (documented per function)
 *   - return value: 0 = ok, negative = error (MS_ERR_*); ms_last_error() gives the message
 *   - there is no CPU fallback anywhere: without a CUDA device every call fails with MS_ERR_CUDA
 */
#ifndef MALSTROEM_B200_H
#define MALSTROEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MS_OK 0
#define MS_ERR_CUDA (-1)   /* CUDA runtime / driver error, or no device */
#define MS_ERR_ARG (-2)    /* bad argument (null pointer, unsupported dtype code) */
#define MS_ERR_SHAPE (-3)  /* rows/cols too small (< 3) or raster too large for 30-bit cell indices */
#define MS_ERR_LABEL (-4)  /* a label lies outside [0, nlabels] (reference: IndexError / undefined) */
#define MS_ERR_NOCONV (-5) /* an iteration hit its safety cap (cyclic flow directions) */

/* dtype codes for `const void *data` arguments */
#define MS_F32 0
#define MS_F64 1
#define MS_U8 2
#define MS_I32 3
#define MS_I64 4

/* ---- library ---------------------------------------------------------------------------------- */
int ms_version(void);
int ms_init(int device);                 /* select device, create the memory pool; idempotent */
int ms_shutdown(void);
/* Device twins of host rasters (csrc/cache.cu): the host-pointer entry points below keep the device buffer of every
 * raster they upload or return, keyed on (host address, size, sampled fingerprint of the host bytes), so that the
 * call sequence of DemTool.process / BluespotTool.process (dem.py:67-91, bluespots.py:158-206) uploads each array
 * once, fill_terrain_no_flats reuses fill_terrain's result, and its second call (bluespots.py:203-205) is a copy.
 * An array rewritten IN PLACE between two calls must be followed by ms_cache_clear() (the fingerprint samples ~2000
 * words); MS_CACHE=0 in the environment switches the cache off.  stats: out5 = inputs found on the device, inputs
 * uploaded, derived results reused, evictions, bytes held. */
int ms_cache_clear(void);
int ms_cache_forget(const void *host);      /* the host array at this address is gone: drop its twin */
int ms_cache_stats(int64_t *out5);
const char *ms_last_error(void);
int ms_device_count(void);
/* launches of this library's own kernels since the last reset (bench.py's `gpu_launches`) */
int64_t ms_kernel_launches(int reset);
/* per-kernel CUDA-event timing on the launching stream: ms_profile(n >= 1) starts recording one event pair per
 * launch (n > 1 pre-creates n pairs first), ms_profile(0) stops; ms_profile_report() synchronises the device and writes one line per kernel
 * ("<name> <launches> <total ms> <total units>") into buf, then clears the records */
int ms_profile(int enable);
/* host-side accounting since the last reset: out4 = {seconds waiting in stream syncs, number of syncs,
 * seconds inside pool allocations, number of allocations} */
int ms_host_counters(double *out4, int reset);
int ms_profile_report(char *buf, int64_t cap);
/* pinned host memory for the host-pointer entry points (optional; pageable memory also works) */
void *ms_host_alloc(int64_t bytes);
int ms_host_free(void *p);

/* ---- fill ------------------------------------------------------------------------------------- */
/* fill.fill_terrain(dtm) — malstroem/algorithms/fill.py:112-171 (sweeps: speedups/_fill.pyx:28-70).
 * `depths` (= filled - dtm, malstroem/dem.py:71) may be NULL. */
int ms_fill_terrain(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols);
int ms_fill_terrain_dev(const float *dtm, float *filled, float *depths, int64_t rows, int64_t cols,
                        void *stream);

/* the data pass of fill.minimum_safe_short_and_diag(dem) — fill.py:235-250: min and max of the raster
 * (short = 1024 ulp64(max|z|), diag = short * 2**0.5 are two scalar operations done by the caller) */
int ms_minmax_f32(const float *dem, int64_t n, float *out_min, float *out_max);
int ms_minmax_f32_dev(const float *dem, int64_t n, float *out_minmax_dev2, void *stream);

/* fill.fill_terrain_no_flats(dtm, short, diag) — fill.py:174-232 (speedups/_fill.pyx:72-124).
 * `filled` (the plain fill of the same dtm) may be NULL; then it is computed internally.
 * stats (may be NULL): [0] = relaxation rounds, [1] = tile visits, [2] = seed re-verification passes */
int ms_fill_terrain_no_flats(const float *dtm, double short_eps, double diag_eps, double *out,
                             int64_t rows, int64_t cols);
int ms_fill_terrain_no_flats_dev(const float *dtm, const float *filled, double short_eps, double diag_eps,
                                 double *out, int64_t rows, int64_t cols, int64_t *stats, void *stream);

/* ---- flow ------------------------------------------------------------------------------------- */
/* flow.terrain_flowdirection(terrain, edges_flow_outward) — flow.py:142-167; stencil
 * speedups/_flow.pyx:98-176; border rule flow.py:118-139 */
int ms_flowdir(const double *terrain, uint8_t *flowdir, int64_t rows, int64_t cols, int edges_flow_outward);
int ms_flowdir_dev(const double *terrain, uint8_t *flowdir, int64_t rows, int64_t cols,
                   int edges_flow_outward, void *stream);

/* flow.accumulated_flow(flowdir) — flow.py:344-364; speedups/_flow.pyx:225-273 */
int ms_accumulated_flow(const uint8_t *flowdir, double *accum, int64_t rows, int64_t cols);
int ms_accumulated_flow_dev(const uint8_t *flowdir, double *accum, int64_t rows, int64_t cols, void *stream);

/* flow.watersheds_from_labels(flowdir, labelled, unassigned) — flow.py:398-412;
 * speedups/_flow.pyx:276-403.  In place; label_bytes = 4 (int32) or 8 (int64). */
int ms_watersheds_from_labels(const uint8_t *flowdir, void *labelled, int label_bytes, int64_t rows,
                              int64_t cols, int64_t unassigned);
int ms_watersheds_from_labels_dev(const uint8_t *flowdir, void *labelled, int label_bytes, int64_t rows,
                                  int64_t cols, int64_t unassigned, void *stream);

/* ---- label ------------------------------------------------------------------------------------ */
/* label.connected_components(data) — label.py:19-40 (scipy.ndimage.label, 8-connectivity, components
 * numbered by first cell in row-major order).  Foreground = data != 0.  *nlabels comes back to the
 * host (the _dev form synchronises the stream for it). */
int ms_connected_components(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols,
                            int64_t *nlabels);
int ms_connected_components_dev(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols,
                                int64_t *nlabels, void *stream);

/* max (and min) label of an int32 raster: the `nlabels = np.max(labelled)` default of label.py:57,116,150 */
int ms_label_range(const int32_t *labels, int64_t n, int32_t *out_min, int32_t *out_max);
int ms_label_range_dev(const int32_t *labels, int64_t n, int32_t *out_minmax_dev2, void *stream);

/* label.label_stats(data, labelled, nlabels) — label.py:43-75; speedups/_label.pyx:31-97.
 * data dtype MS_F32 or MS_F64; tables have nlabels+1 entries. */
int ms_label_stats(const void *data, int dtype, const int32_t *labels, int64_t n, int64_t nlabels,
                   double *out_min, double *out_max, double *out_sum, int64_t *out_count);
int ms_label_stats_dev(const void *data, int dtype, const int32_t *labels, int64_t n, int64_t nlabels,
                       double *out_min, double *out_max, double *out_sum, int64_t *out_count, void *stream);

/* label.label_min_index / label_max_index(data, labelled, nlabels) — label.py:101-166;
 * speedups/_label.pyx:99-164.  data is float64; first cell in raster order wins ties; labels never
 * seen keep value = +inf / -inf and row = col = -1. */
int ms_label_extreme_index(const double *data, const int32_t *labels, int64_t rows, int64_t cols,
                           int64_t nlabels, int want_max, double *out_value, int64_t *out_row,
                           int64_t *out_col);
int ms_label_extreme_index_dev(const double *data, const int32_t *labels, int64_t rows, int64_t cols,
                               int64_t nlabels, int want_max, double *out_value, int64_t *out_row,
                               int64_t *out_col, void *stream);

/* label.label_count(labelled) — label.py:169-180 (np.bincount); nbins = max label + 1 */
int ms_label_count(const int32_t *labels, int64_t n, int64_t nbins, int64_t *out_count);
int ms_label_count_dev(const int32_t *labels, int64_t n, int64_t nbins, int64_t *out_count, void *stream);

/* label.keep_labels(labelled, keep_label, background) — label.py:78-98: out[i] = keep[labels[i]] */
int ms_keep_labels(const int32_t *labels, int64_t n, const uint8_t *keep, int64_t nkeep, uint8_t *out);
int ms_keep_labels_dev(const int32_t *labels, int64_t n, const uint8_t *keep, int64_t nkeep, uint8_t *out,
                       void *stream);


/* ---- row bands: one raster split by rows across GPUs (SURVEY.md §8(e)) --------------------------------
 * The reference has no distributed path (SURVEY.md F8); these entry points are the per-band halves of the stage
 * functions above, with the exchange steps left to the caller (malstroem_b200/bands.py drives them over
 * torch.distributed / NCCL).  Conventions: every raster pointer points at the band's FIRST OWN row; if the band is
 * open at the top (MS_OPEN_TOP: another band continues above) the row before it in memory is a halo row holding the
 * neighbour's last own row, likewise MS_OPEN_BOTTOM and the row after the last own row.  A band that is open at
 * the bottom must have a multiple of 64 rows.  rows * cols <= 2^29 per band.  All pointers are device pointers
 * unless stated; functions returning a count synchronise the stream. */
#define MS_OPEN_TOP 1
#define MS_OPEN_BOTTOM 2
typedef struct ms_band ms_band;
int ms_band_create(int64_t rows, int64_t cols, int open, ms_band **out);
int ms_band_destroy(ms_band *band);

/* fill.fill_terrain (fill.py:112-171) on a band.  local: Boruvka contraction inside the band; components whose
 * lowest way out crosses a band edge stay "frozen" (*n_frozen of them).  edge_ids: global ids (gid_base + rank + 1;
 * 0 = outside) of the components of the first / last own row, to be exchanged as halo ids.  edges: the boundary
 * graph of this band (frozen components x their neighbours, lowest cell-pair edge each), at most `capacity`.
 * ms_graph_minimax_dev: minimax height to node 0 over the union of all bands' edges (every rank solves the same
 * small graph).  finish: filled (and depths = filled - dem, may be NULL) for the band. */
int ms_band_fill_local_dev(ms_band *band, const float *dem, int64_t *n_frozen, void *stream);
int ms_band_fill_edge_ids_dev(ms_band *band, int64_t gid_base, int32_t *gid_top, int32_t *gid_bot, void *stream);
int ms_band_fill_edges_dev(ms_band *band, const float *dem, const int32_t *halo_gid_top, const int32_t *halo_gid_bot,
                           int32_t *edge_a, int32_t *edge_b, float *edge_w, int64_t capacity, int64_t *n_edges,
                           void *stream);
int ms_graph_minimax_dev(int64_t n_nodes, const int32_t *edge_a, const int32_t *edge_b, const float *edge_w,
                         int64_t n_edges, float *out_x, void *stream);
int ms_band_fill_finish_dev(ms_band *band, const float *dem, const float *graph_x, float *filled, float *depths,
                            void *stream);

/* fill.fill_terrain_no_flats (fill.py:174-232) on a band: init (needs the halo rows of `filled`; returns the
 * band's count of lake / flat cells), solve (mode 0: first solve, after the halo rows of fnf were exchanged; mode 1:
 * again after the halo rows named by `edges` changed), verify (the fixed-point stencil incl. halo rows). */
double ms_nf_cap_bound(int64_t rows, int64_t cols, double diag_eps);   /* rows = of the WHOLE raster */
int ms_band_nf_init_dev(ms_band *band, const float *dem, const float *filled, double *fnf, int64_t *nonseed,
                        void *stream);
int ms_band_nf_solve_dev(ms_band *band, const float *dem, const float *filled, double *fnf, double short_eps,
                         double diag_eps, double cap_bound, int cap, int mode, int edges, int64_t *tile_visits,
                         void *stream);
int ms_band_nf_verify_dev(ms_band *band, const float *dem, const double *fnf, double short_eps, double diag_eps,
                          int64_t *nviol, void *stream);
/* seed repair (the retry loop of fill.fill_terrain_no_flats' device form, here per band): reset != 0 forgets the
 * band's ban map; otherwise the stencil runs on fnf, every failing cell is added to the ban map (ms_band_nf_init_dev
 * then treats it as a lake cell, not as a seed) and their count is returned. */
int ms_band_nf_ban_dev(ms_band *band, const float *dem, const double *fnf, double short_eps, double diag_eps, int reset,
                       int64_t *nviol, void *stream);
/* The same solve fused over NVLink peer memory, on the INTEGER RASTER of the single-GPU path (fill.py:174-232 /
 * _fill.pyx:72-124 as above): every band's solver kernel runs at the same time and the bands feed each other's tile
 * queues and halo rows directly (system-scope atomics and stores into blocks mapped through CUDA IPC), instead of one
 * host-driven halo exchange per crossing of a band edge.  create: allocates the band's shared block, info80 (HOST,
 * 80 bytes) describes it; open: maps every rank's block (infos: world x 80 bytes gathered from all ranks, rows_all:
 * own rows of every band; HOST pointers).  Per solve: edgefix: fixed flags (seed or raster border) of the band's
 * first / last own row (cols bytes each) - the caller hands them to the neighbours, whose halo rows they describe.
 * prepare: the band's padded int32 distance raster, its edge rows stored into the neighbours' mailboxes (peer
 * memory), FIFO := tiles holding lake cells; *queued, *irbad (the band does not fit the integer form).  All ranks
 * synchronise, arm (a band with queued tiles counts itself active), synchronise, solve (all ranks at once; skipped
 * when no rank has queued tiles): solve_launch returns once the solver kernel is queued, and the host is free for
 * CPU work until solve_wait (no library call on this band in between).  finish: the float64 surface written once and
 * verified against the fixed-point equation with the halo rows (*nviol), the D8 codes of the band's rows
 * (flow.py:142-167, edges of the raster flowing outward) on the way.  When any rank reports irbad, a solver error or
 * a violation, the host-driven init / solve / verify calls above take over on every rank. */
int ms_band_nf_shared_create(ms_band *band, void *info80);
int ms_band_nf_shared_open(ms_band *band, int rank, int world, const void *infos, const int64_t *rows_all);
int ms_band_nf_ir_edgefix_dev(ms_band *band, const float *dem, const float *filled, uint8_t *fix_top, uint8_t *fix_bot,
                              void *stream);
int ms_band_nf_ir_prepare_dev(ms_band *band, const float *dem, const float *filled, double short_eps, double diag_eps,
                              double cap_bound, const uint8_t *fix_top, const uint8_t *fix_bot, int64_t *queued,
                              int *irbad, void *stream);
int ms_band_nf_p2p_arm_dev(ms_band *band, void *stream);
int ms_band_nf_ir_solve_launch_dev(ms_band *band, const float *filled, double short_eps, double diag_eps, void *stream);
int ms_band_nf_ir_solve_wait_dev(ms_band *band, int64_t *tile_visits, int *irbad, void *stream);
int ms_band_nf_ir_finish_dev(ms_band *band, const float *dem, const float *filled, double *fnf, uint8_t *flowdir,
                             double short_eps, double diag_eps, int64_t *nviol, void *stream);

/* flow.terrain_flowdirection (flow.py:142-167) on a band (needs the halo rows of the terrain) */
int ms_band_flowdir_dev(ms_band *band, const double *terrain, uint8_t *flowdir, int edges_flow_outward, void *stream);

/* flow.accumulated_flow (flow.py:344-364) on a band (needs the halo rows of flowdir).  local: arrays of 2 * cols
 * entries (first the top row's cells, then the bottom row's): exit_to = column at which the path leaving the band
 * at this cell enters the neighbour (-1: not an exit), exit_val = the count it carries from inside the band,
 * entry_root = side * cols + col of the band exit this cell's own path ends at (-1: it ends inside the band).
 * ms_forest_accumulate_dev: totals over the forest of all bands' exits.  finish: halo_total_top / _bot[c] = total
 * of the neighbour's edge-row cell in column c (used where that cell flows into this band). */
int ms_band_accum_local_dev(ms_band *band, const uint8_t *flowdir, int32_t *exit_to, double *exit_val,
                            int32_t *entry_root, void *stream);
int ms_forest_accumulate_dev(int64_t n, const int32_t *parent, double *totals, void *stream);
int ms_band_accum_finish_dev(ms_band *band, const uint8_t *flowdir, const double *halo_total_top,
                             const double *halo_total_bot, double *accum, void *stream);

/* label.connected_components (label.py:19-40) on a band.  local: roots (global cell index = cell_offset + local
 * index, -1 = background) of the first / last own row.  ms_cc_boundary_merge (HOST pointers, CPU): merges the
 * components that touch across band edges; out_root ascending, out_global = smallest root of the merged component.
 * count: `rerooted` = local indices of this band's roots that are not their component's smallest; returns how many
 * components the band numbers.  root_labels: final labels of roots this band owns.  finish: writes the labels. */
int ms_band_cc_local_dev(ms_band *band, const void *data, int dtype, int64_t cell_offset, int64_t *root_top,
                         int64_t *root_bot, void *stream);
int ms_cc_boundary_merge(int nbands, int64_t cols, const int64_t *root_top, const int64_t *root_bot,
                         int64_t *out_root, int64_t *out_global, int64_t capacity, int64_t *n_out);
/* The same merge for regions of equal value (label polygonisation on bands): val_top / val_bot hold the cells' values
 * (G * cols each, like the roots); two cells across a band edge join only if their values are equal, and diagonal
 * neighbours only if connect8 != 0.  ms_cc_boundary_merge is this merge with every non-negative root joining its three
 * neighbours. */
int ms_cc_boundary_merge_values(int nbands, int64_t cols, const int64_t *root_top, const int64_t *root_bot,
                                const int32_t *val_top, const int32_t *val_bot, int connect8, int64_t *out_root,
                                int64_t *out_global, int64_t capacity, int64_t *n_out);
int ms_band_cc_count_dev(ms_band *band, const int32_t *rerooted, int64_t n_rerooted, int64_t *count, void *stream);
int ms_band_cc_root_labels_dev(ms_band *band, const int32_t *roots, int64_t n_roots, int64_t label_offset,
                               int32_t *labels_out, void *stream);
int ms_band_cc_finish_dev(ms_band *band, const int32_t *rerooted, const int32_t *rerooted_label, int64_t n_rerooted,
                          int64_t label_offset, int32_t *labels, void *stream);

/* flow.watersheds_from_labels (flow.py:398-412) on a band, int32 labels.  local: edge_res[2 * cols] = what each cell
 * of the first / last own row resolves to: >= 0 a label (0: none), < 0: -(1 + side * cols + col) of the band exit it
 * waits for; exit_to as above.  ms_chain_resolve_dev follows such references to their final value.  finish:
 * exit_label[side * cols + col] = label for cells draining through that exit. */
int ms_band_ws_local_dev(ms_band *band, const uint8_t *flowdir, const int32_t *labelled, int32_t unassigned,
                         int32_t *edge_res, int32_t *exit_to, void *stream);
int ms_chain_resolve_dev(int64_t n, const int32_t *arr, int32_t *out, void *stream);
int ms_band_ws_finish_dev(ms_band *band, const uint8_t *flowdir, int32_t *labelled, int32_t unassigned,
                          const int32_t *exit_label, void *stream);

/* All per-label tables of a band in two fused passes over its rasters.  Phase A: partial label_stats(depths, labels),
 * label_count(wsheds) and the extreme values of fnf (min) / accum (max) per label, +-inf where the band does not see
 * a label: combine across bands with min / max / sum all-reduces.  Phase B: with the GLOBAL extremes, the smallest
 * global flat index holding each (INT64_MAX: not in this band): combine with a min all-reduce. */
int ms_band_tables_a_dev(const float *depths, const int32_t *labels, const double *fnf, const double *accum,
                         const int32_t *wsheds, int64_t n, int64_t cols, int64_t nlabels, double *st_min, double *st_max,
                         double *st_sum, int64_t *st_count, int64_t *ws_count, double *vmin, double *vmax,
                         void *stream);
int ms_band_tables_b_dev(const int32_t *labels, const double *fnf, const double *accum, int64_t n, int64_t nlabels,
                         const double *vmin, const double *vmax, int64_t cell_offset, int64_t *idx_min,
                         int64_t *idx_max, void *stream);

/* ---- the whole path, device resident (what bench.py times) -------------------------------------- */
typedef struct ms_rasters {
    int64_t rows, cols;
    const float *dem;   /* in  : float32 DEM                                   (dem.py:56)            */
    float *filled;      /* out : fill_terrain                                   (dem.py:67)            */
    float *depths;      /* out : filled - dem                                   (dem.py:71)            */
    double *fnf;        /* out : fill_terrain_no_flats                          (dem.py:80)            */
    uint8_t *flowdir;   /* out : terrain_flowdirection                          (dem.py:83)            */
    double *accum;      /* out : accumulated_flow                               (dem.py:89)  may be NULL */
    int32_t *labels;    /* out : connected_components(depths)                   (bluespots.py:159)     */
    int32_t *wsheds;    /* out : watersheds_from_labels                         (bluespots.py:183-185) */
    /* per-label tables, device memory with room for table_capacity entries (>= nlabels + 1) */
    int64_t table_capacity;
    double *st_min, *st_max, *st_sum; /* label_stats(depths, labels)            (bluespots.py:160)     */
    int64_t *st_count;
    int64_t *ws_count;                /* label_count(wsheds)                    (bluespots.py:186)     */
    double *ppmin_value;              /* label_min_index(fnf, labels)           (bluespots.py:205)     */
    int64_t *ppmin_row, *ppmin_col;
    double *ppmax_value;              /* label_max_index(accum, labels)         (bluespots.py:198)  may be NULL */
    int64_t *ppmax_row, *ppmax_col;
    /* results that come back to the host */
    int64_t nlabels;
    double short_eps, diag_eps;
    int64_t stats[8]; /* [0] Boruvka rounds, [1] catchments, [2] no-flats rounds, [3] tile visits,
                         [4] seed re-verifications, [5] pointer-jump rounds (fill), [6] (wsheds) */
} ms_rasters;

/* DEM in HBM -> every raster and table of the path in HBM.  Synchronises the stream a few times for
 * convergence flags and counts. */
int ms_pipeline_dev(ms_rasters *io, void *stream);

/* The same with the finished rasters shipped to (pinned) host buffers while the later stages run: every non-NULL
 * pointer of `host` receives its raster through a second stream as soon as the stage that produces it is done.
 * The copies are complete after ms_copies_wait().  (The host-buffer front end of malstroem_b200.pipeline uses this;
 * what the reference's tool layer writes to GeoTIFFs — dem.py:67-93, bluespots.py:159-216 — is exactly this set.) */
typedef struct ms_host_out {
    float *filled, *depths;
    double *fnf;
    uint8_t *flowdir;
    double *accum;
    int32_t *labels, *wsheds;
} ms_host_out;
int ms_pipeline_host_dev(ms_rasters *io, const ms_host_out *host, void *stream);
int ms_copies_wait(void);

/* ---- the bluespot filter of BluespotTool.process (bluespots.py:158-170: raw labels -> raw stats -> filterbluespots ->
 * keep_labels -> connected_components) ------------------------------------------------------------------------------
 * A filter is a postfix program over three per-label variables (malstroem_b200/bluespot_filter.py compiles the CLI's
 * `-filter` text into it): area = (double)count * cell_area, maxdepth = max, volume = sum * cell_area, from the raw
 * label_stats of the depths.  Every operation is one IEEE float64 operation (the library builds with -fmad=false), so
 * decisions are bitwise numpy's.  Comparisons push 1.0 / 0.0; truthiness is x != 0 (NaN is true, as in Python); the
 * program keeps a label when its result is true.  Label 0 is never kept.  At most MS_BF_MAX_OPS operations and a stack
 * of MS_BF_MAX_STACK values; a malformed program is MS_ERR_ARG before any device work. */
#define MS_BF_MAX_OPS 64
#define MS_BF_MAX_STACK 16
enum {
    MS_BF_AREA = 1, MS_BF_MAXDEPTH, MS_BF_VOLUME, MS_BF_CONST, /* push a variable, or imm[k]                 */
    MS_BF_NEG, MS_BF_NOT,                                       /* -x, (x == 0)                              */
    MS_BF_ADD, MS_BF_SUB, MS_BF_MUL, MS_BF_DIV,                 /* a op b (b on top of the stack)            */
    MS_BF_LT, MS_BF_LE, MS_BF_GT, MS_BF_GE, MS_BF_EQ, MS_BF_NE, /* a op b -> 1.0 / 0.0                       */
    MS_BF_AND, MS_BF_OR                                         /* (a != 0) op (b != 0) -> 1.0 / 0.0         */
};
typedef struct ms_bluespot_filter {
    int32_t n_ops;
    int32_t op[MS_BF_MAX_OPS];
    double imm[MS_BF_MAX_OPS]; /* the constant of an MS_BF_CONST at the same position */
    double cell_area;
} ms_bluespot_filter;

/* keep decisions of labels 1..nlabels from their raw stats (device tables of nlabels + 1 entries; only max, sum and
 * count are read) as a rank-compaction table: lut_out[l] = rank of l among the kept labels (1, 2, ...), 0 for a
 * dropped label and for label 0.  *nkept comes back to the host (synchronises the stream).  `filter` is a HOST
 * pointer. */
int ms_bluespot_filter_dev(const ms_bluespot_filter *filter, int64_t nlabels, const double *st_max,
                           const double *st_sum, const int64_t *st_count, int32_t *lut_out, int64_t *nkept,
                           void *stream);
/* labels[c] = lut[labels[c]] in place, lut with nlabels + 1 entries: the second connected_components of
 * bluespots.py:170, which only renumbers the kept components (SURVEY.md A.6).  MS_ERR_LABEL for a label outside
 * [0, nlabels] (synchronises the stream). */
int ms_relabel_dev(int32_t *labels, int64_t n, int64_t nlabels, const int32_t *lut, void *stream);
/* ms_pipeline_host_dev with the bluespot filter between the labels and the watersheds: raw labels, raw label_stats of
 * the depths, keep decisions, relabel; io->nlabels = the kept bluespots, every raster and table after the labels is
 * the filtered one (the labels are shipped after the relabel).  *nlabels_raw (may be NULL) = the raw bluespots.
 * filter == NULL is ms_pipeline_host_dev. */
int ms_pipeline_filtered_host_dev(ms_rasters *io, const ms_host_out *host, const ms_bluespot_filter *filter,
                                  int64_t *nlabels_raw, void *stream);

/* ---- SURVEY.md §8(f): the bluespot network on device ------------------------------------------------ */
/* net.pourpoint_network / net.next_downstream_label (malstroem/algorithms/net.py:142-192; the walk is
 * flow.trace_downstream, flow.py:279-301).  For each of the n_pp start cells (pp_row, pp_col): out_down = the first
 * label on the downstream path that differs from the start cell's label and, when has_background, from `background`;
 * out_found = 0 when the path ends first (Python None).  labelled: int32 (label_bytes 4) or int64 (8).
 * Geometry (net.py:166-167), host form only: when out_path_offsets != NULL it receives n_pp + 1 offsets into
 * out_path_cells (flat cell indices of the cells visited, start cell first, answering cell last); the cells are
 * written only if out_path_offsets[n_pp] <= path_capacity — otherwise call again with a larger buffer.
 * MS_ERR_NOCONV on cyclic flow directions (the reference would not return). */
int ms_pourpoint_network(const uint8_t *flowdir, const void *labelled, int label_bytes, int64_t rows, int64_t cols,
                         int64_t n_pp, const int64_t *pp_row, const int64_t *pp_col, int64_t background,
                         int has_background, int64_t *out_down, uint8_t *out_found, int64_t *out_path_offsets,
                         int64_t *out_path_cells, int64_t path_capacity);
int ms_pourpoint_network_dev(const uint8_t *flowdir, const void *labelled, int label_bytes, int64_t rows,
                             int64_t cols, int64_t n_pp, const int64_t *pp_row, const int64_t *pp_col,
                             int64_t background, int has_background, int64_t *out_down, uint8_t *out_found,
                             void *stream);

/* Network.rain_event (malstroem/network.py:75-129) for n_events rain depths at once.  Nodes in insertion order;
 * parent[i] = index of the downstream node, -1 = root (dstrnodeid None), -2 = an id that is not a node.  Outputs
 * are [n_events][n] row-major: rainv, spillv, v, pctv (NaN where the reference gives None: capacity 0);
 * out_present[i] = 0 for nodes the reference never reaches from a root (their values are unspecified).
 * Upstream spill is summed in insertion order of the upstream nodes, sum_mode 0 = plain float addition (sum()
 * before CPython 3.12), 1 = Neumaier compensated (sum() from CPython 3.12 on).  `mm` is a HOST array in both forms
 * (n_events <= 16). */
int ms_rain_events(int64_t n, const int32_t *parent, const double *wshed_area, const double *bspot_vol,
                   int64_t n_events, const double *mm, int sum_mode, double *out_rainv, double *out_spillv,
                   double *out_v, double *out_pctv, uint8_t *out_present);
int ms_rain_events_dev(int64_t n, const int32_t *parent, const double *wshed_area, const double *bspot_vol,
                       int64_t n_events, const double *mm, int sum_mode, double *out_rainv, double *out_spillv,
                       double *out_v, double *out_pctv, uint8_t *out_present, void *stream);

/* The chain StreamTool + RainTool run on BluespotTool's tables (streams.py:66-100, rain.py:60-79), device resident,
 * straight from a finished ms_rasters: node i = bluespot label i (label 0 included, as the reference does —
 * bluespots.py:74), pour point = ppmin (or ppmax when use_accum_pourpoints), wshed_area = ws_count * cell_area,
 * bspot_vol = st_sum * cell_area.  out_parent[nlabels + 1] = downstream label or -1; event tables as above,
 * [n_events][nlabels + 1].  All outputs are device memory. */
int ms_bluespot_network_dev(const ms_rasters *io, double cell_area, int use_accum_pourpoints, int64_t n_events,
                            const double *mm, int sum_mode, int32_t *out_parent, double *out_rainv,
                            double *out_spillv, double *out_v, double *out_pctv, void *stream);

/* The pour-point network for one band of a raster split by rows (one band per GPU): out_parent[i] = downstream
 * bluespot of label i (-1: none) for the pour points (GLOBAL row / column) inside rows [first_row, first_row +
 * band_rows), INT32_MIN for all others — combine the bands with a max all-reduce.  wsheds is the band's finished
 * watershed raster, ws_above / ws_below the neighbours' facing rows of theirs (NULL at the raster's edge).  Valid on
 * the D8 surface of the no-flats fill, where a pour point leaves its bluespot with its first step (MS_ERR_ARG
 * otherwise).  Synchronises the stream. */
int ms_band_pp_parent_dev(const uint8_t *flowdir, const int32_t *wsheds, const int32_t *ws_above, const int32_t *ws_below,
                          int64_t band_rows, int64_t cols, int64_t first_row, int64_t total_rows, int64_t n,
                          const int64_t *pp_row, const int64_t *pp_col, int32_t *out_parent, void *stream);

/* synthetic fractal DEM (malstroem_b200/synth.py, bit-identical), generated in place on the device */
int ms_synth_fractal_dev(float *dem, int64_t rows, int64_t cols, int64_t row0, int64_t col0, int seed,
                         void *stream);

/* ---- SURVEY.md 8(f3): the raster codec of malstroem/io.py (GeoTIFF: tiled, deflate, predictor 2) on the device.
 * The container (header, tag directory) is host-side bookkeeping (malstroem_b200/io.py); these touch every byte.
 * ms_tiff_encode_dev replaces the compression inside RasterWriter.write (io.py:112-139): the raster (device, row
 * major, sample_bytes 1 / 2 / 4 / 8) becomes one zlib stream (RFC 1950 / 1951, what TIFF compression 8 holds) per
 * 256 x 256 tile in row-major tile order, tile k at out + k * slot (slot >= ms_tiff_tile_slot(sample_bytes)),
 * sizes[k] bytes long; predictor 1 = none, 2 = horizontal differencing.  ms_tiff_pack_dev lines the streams up.
 * ms_tiff_decode_dev replaces RasterReader.read (io.py:52-72): nblocks zlib streams (tiles, or strips with
 * block_w = cols; any conforming deflate stream) are inflated into `scratch`, the predictor is undone, the blocks are
 * cropped into the rows x cols raster, and samples equal to the file's nodata value (subst_mode 1: np.isclose, 2:
 * np.isnan, 0: no substitution - io.py:69-71) become `subst`.  compressed = 0: `scratch` already holds the raw blocks. */
int64_t ms_tiff_tile_slot(int sample_bytes);
int ms_tiff_encode_dev(const void *raster, int sample_bytes, int64_t rows, int64_t cols, int predictor, void *out,
                       int64_t slot, uint32_t *sizes, void *stream);
int ms_tiff_pack_dev(const void *slots, int64_t slot, const uint32_t *sizes, const uint64_t *offs, int64_t ntiles,
                     void *packed, void *stream);
int ms_tiff_decode_dev(const void *in, const uint64_t *in_off, const uint32_t *in_len, int64_t nblocks, int block_w,
                       int block_h, int sample_bytes, int sample_format, int predictor, void *scratch, void *raster,
                       int64_t rows, int64_t cols, int subst_mode, double nodata, double subst, int compressed,
                       void *stream);
/* ms_tiff_decode_rows_dev: one window of file rows, for a row band (RasterReader.read_rows).  The nblocks streams are
 * the whole block rows from block row block_row0 on (k * blocks_x tiles, or k strips) and must cover file rows
 * [out_row0, out_row0 + out_rows); `raster` is out_rows x cols and receives them, file row r at raster row
 * r - out_row0; `rows` stays the file's row count.  The short last strip of a striped file is accepted only when the
 * window's block rows include the file's last one.  ms_tiff_decode_dev is the window (0, 0, rows). */
int ms_tiff_decode_rows_dev(const void *in, const uint64_t *in_off, const uint32_t *in_len, int64_t nblocks,
                            int block_w, int block_h, int sample_bytes, int sample_format, int predictor, void *scratch,
                            void *raster, int64_t rows, int64_t cols, int64_t block_row0, int64_t out_row0,
                            int64_t out_rows, int subst_mode, double nodata, double subst, int compressed, void *stream);

/* ---- SURVEY.md 8(f4): label polygonisation.  Replaces vector.py:42-87 (vectorize_labels_file), i.e.
 * gdal.Polygonize(band, band.GetMaskBand(), layer, 0, ['8CONNECTED=8']): one polygon per 8-connected (connect8 = 0:
 * 4-connected) region of equal cell value, cells equal to `nodata` (has_nodata != 0) in none.  The rings stay on the
 * device; counts3[0..2] = rings, vertices, boundary edges.  ms_polygonize_fetch copies them to caller-allocated host
 * arrays and releases them: ring k owns vertices [off[k], off[k+1]) (lattice corners: row 0..rows, col 0..cols; only
 * the corners of the outline, without a repeated closing vertex; the region lies on the right-hand side walking the
 * ring on the screen), ring_value = the cells' value, ring_cell = a cell of the ring's region touching it,
 * ring_region = the first cell of the region in raster order (the same for an exterior ring and its holes),
 * ring_hole = 1 for a hole.  Rings come ordered by their first boundary cell in raster order. */
int ms_polygonize_dev(const int32_t *labels, int64_t rows, int64_t cols, int connect8, int has_nodata, int32_t nodata,
                      int64_t *counts3, void *stream);
int ms_polygonize(const int32_t *labels, int64_t rows, int64_t cols, int connect8, int has_nodata, int32_t nodata,
                  int64_t *counts3);
int ms_polygonize_fetch(int64_t *ring_vertex_offset, int32_t *ring_value, int64_t *ring_cell, int64_t *ring_region,
                        uint8_t *ring_hole, int32_t *vertex_row, int32_t *vertex_col);

/* Label polygonisation on a row band (malstroem_b200/vector.py polygonize_band; DESIGN.md 8(f4)).  `lab` points at
 * the band's first row of `rows` x `cols` cells; halo bit 0 / 1: the row above (lab - cols) / below (lab + rows * cols)
 * holds the neighbouring band's edge row.  Every buffer is the caller's, on the device unless named host; edge numbers
 * are the band's own (0 .. n_edges - 1, in raster order: by cell, then top / right / bottom / left); the band's global
 * edge numbers start at the sum of the lower bands' n_edges.  At most 2^30 cells and 2^31 - 1024 edges per band.
 *  count: eoff[rows * cols] = first edge of every cell; *n_edges (host); row_eoff / row_mask [2 cols] = first edge and
 *    side mask (bit 0 top .. 3 left) of the first and the last row's cells, for the neighbours' halo.
 *  edges: halo_eoff (global) / halo_mask [2 cols] = the neighbours' row_eoff + their base / row_mask for the rows
 *    above and below (ignored where the halo bit is clear).  Writes ecell[n_edges] = (cell << 2) | side, succ = local
 *    successor (an exit, whose successor lies in another band: itself), lead = ring key << 32 (key: leader | 2^31 on a
 *    ring closed in the band, else the slot of the exit ending the edge's chain), rank = steps to the leader / exit
 *    << 32.  Exit slots [4 cols]: 2 c + {0, 1} for the top / left side of first-row cell c, 2 cols + 2 c + {0, 1} for
 *    the right / bottom side of last-row cell c: exit_edge (-1: none), exit_next = global successor, exit_corner = 1
 *    if that successor turns.
 *  place: units = closed rings (head: the leader) and segments (head: the entry), numbered in head order; ishead,
 *    uidx, ulen, ustart, placed, corner, vidx [n_edges] as for one GPU (corner at a segment's first edge: 0); per exit
 *    slot seg_entry, seg_min (smallest edge), seg_tmin (its position from the entry).  counts2 (host) = units,
 *    vertices.
 *  emit: vrow / vcol [nverts] (global lattice rows, row0 = the band's first row), the unit table [units]: u_head,
 *    u_len, u_vstart, u_vcount, u_value, u_root (global cell index of the region root within the band), u_slot (-1:
 *    a closed ring); root_rows [2 cols]: region roots of the first and last row (-1: nodata), for
 *    ms_cc_boundary_merge_values. */
int ms_band_poly_count_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                           int32_t nodata, int32_t *eoff, int64_t *n_edges, int32_t *row_eoff, uint8_t *row_mask,
                           void *stream);
int ms_band_poly_edges_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                           int32_t nodata, const int32_t *eoff, int64_t n_edges, const int64_t *halo_eoff,
                           const uint8_t *halo_mask, uint32_t *ecell, int32_t *succ, uint64_t *lead, uint64_t *rank,
                           int32_t *exit_edge, int64_t *exit_next, uint8_t *exit_corner, void *stream);
int ms_band_poly_place_dev(int64_t cols, int64_t n_edges, const uint32_t *ecell, const int32_t *succ,
                           const uint64_t *lead, const uint64_t *rank, int32_t *ishead, int32_t *uidx, int32_t *ulen,
                           int32_t *ustart, uint32_t *placed, int32_t *corner, int32_t *vidx, int32_t *seg_entry,
                           int32_t *seg_min, int32_t *seg_tmin, int64_t *counts2, void *stream);
int ms_band_poly_emit_dev(const int32_t *lab, int64_t rows, int64_t cols, int halo, int connect8, int has_nodata,
                          int32_t nodata, int64_t row0, int64_t n_edges, const uint32_t *ecell, const uint64_t *lead,
                          const int32_t *ishead, const int32_t *uidx, const int32_t *ulen, const int32_t *ustart,
                          const uint32_t *placed, const int32_t *corner, const int32_t *vidx, int64_t nverts,
                          int32_t *vrow, int32_t *vcol, int32_t *u_head, int32_t *u_len, int32_t *u_vstart,
                          int32_t *u_vcount, int32_t *u_value, int64_t *u_root, int32_t *u_slot, int64_t *root_rows,
                          void *stream);

/* ---- Bluespot water levels and water-depth rasters after rain events.
 * Bluespot l >= 1 is the set of cells with labels == l; z = dem widened to float64, F = the plain fill (uniform over
 * a bluespot: L_l), ca = cell_area > 0, cap_l = st_sum[l] * ca, v = the stored volume of a bluespot per event
 * (e.g. the `v` of ms_rain_events / ms_bluespot_network_dev), row-major [n_events][nlabels+1].
 * Level-pool approximation: a bluespot's water is one flat surface at level h holding ca * sum max(0, h - z_c); this
 * ignores that separate sub-pits of one bluespot may fill one after another.
 * ms_flood_levels: level[e][l] and wet[e][l] (cells with z < level), both [n_events][nlabels+1]:
 *   v NaN -> NaN, 0;  v >= cap_l -> L_l, #cells of l;  otherwise, with z_(1) <= ... <= z_(n) the bluespot's values,
 *   S_j = z_(1) + ... + z_(j), T = v / ca and k = max{ j : j * z_(j) - S_j <= T }: h = min(L_l, (T + S_k) / k),
 *   wet = #{ z_c < h };  label 0 -> NaN, 0.  Results are bitwise reproducible.  MS_ERR_ARG for bad sizes, null
 *   pointers or cell_area <= 0 (before any device work), for a label whose F is not uniform and for a negative v;
 *   MS_ERR_LABEL for a label outside [0, nlabels].
 * ms_water_depth: the depth raster of one event's levels (nlabels+1 entries): level_l == L_l -> F - z in float32
 *   (bitwise the `depths` raster of the fill); z < level_l -> (float)(level_l - z) from float64; 0 elsewhere and
 *   outside bluespots.  MS_ERR_LABEL for a label outside [0, nlabels]. */
int ms_flood_levels_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                        int64_t nlabels, const double *st_sum, double cell_area, int64_t n_events, const double *v,
                        double *out_level, int64_t *out_wet, void *stream);
int ms_flood_levels(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                    int64_t nlabels, const double *st_sum, double cell_area, int64_t n_events, const double *v,
                    double *out_level, int64_t *out_wet);
int ms_water_depth_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                       int64_t nlabels, const double *level, float *out_depth, void *stream);
int ms_water_depth(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                   int64_t nlabels, const double *level, float *out_depth);

/* The same levels on a raster split by rows (malstroem_b200/bands.py BandPipeline.flood), one band per call, all
 * pointers device memory, dem / filled / labels the band's own rows.  Band g owns the labels it numbered, lo < l <= hi
 * (lo = the sum of the earlier bands' counts); a label of the band at or below lo is "foreign": its owner is a lower
 * band.  Per-label arrays: cnt and off nlabels + 2 entries, lkey nlabels + 1, kept between the phases; cnt and off
 * must start on 16-byte boundaries (the scans load and store 16-byte vectors).
 *   count:   the band's cells per label, checks (labels in [0, hi], F uniform within the band), send offsets in off
 *            and the foreign list: (label, count, F key) int32 triples in label order, at most `capacity` (a foreign
 *            label touches the band's first or last row, so 2 * cols suffice); *n_send = cells of foreign labels.
 *   layout:  the owner's received triples (every sender's list part for the owner, any order): counts added, F keys
 *            checked against its own, segment offsets of its labels in off; recv_pos[i] = where run i starts in its
 *            label's segment.  *n_cells = cells of its segments (the seg buffer to allocate).
 *   scatter: z keys of the band's cells: owned labels' into seg, foreign labels' into send (n_send keys, label
 *            order, so the part for each owner is contiguous).
 *   solve:   the received key runs (concatenated in the order of the received triples, n_recv_keys = the sum of
 *            their counts, else MS_ERR_ARG) into their segments, then the
 *            levels and wet counts of the owned labels into out_level / out_wet [n_events][nlabels + 1] (other
 *            columns untouched), bitwise those of ms_flood_levels_dev on the whole raster with the same st_sum and v.
 * The return value reports bad arguments and CUDA errors only.  Errors of the data come back in *flags (combine them
 * across the bands, then stop): MS_FLOOD_LABEL a label outside [0, hi] or a triple outside the owner's range,
 * MS_FLOOD_UNIFORM F not uniform over a label (within the band or across bands), MS_FLOOD_VOLUME a negative v,
 * MS_FLOOD_SIZE an owner's segments reaching 2^31 cells, MS_FLOOD_CAPACITY more foreign labels than `capacity` (labels
 * that are not connected components).  Each phase synchronises the stream. */
#define MS_FLOOD_LABEL 1
#define MS_FLOOD_UNIFORM 2
#define MS_FLOOD_VOLUME 4
#define MS_FLOOD_SIZE 8
#define MS_FLOOD_CAPACITY 16
int ms_band_flood_count_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                            int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, uint32_t *lkey, int32_t *off,
                            int32_t *foreign, int64_t capacity, int64_t *n_foreign, int64_t *n_send, int *flags,
                            void *stream);
int ms_band_flood_layout_dev(int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, const uint32_t *lkey, int32_t *off,
                             const int32_t *recv, int64_t n_recv, int32_t *recv_pos, int64_t *n_cells, int *flags,
                             void *stream);
int ms_band_flood_scatter_dev(const float *dem, const float *filled, const int32_t *labels, int64_t rows, int64_t cols,
                              int64_t nlabels, int64_t lo, int64_t hi, int32_t *cnt, const uint32_t *lkey,
                              const int32_t *off, uint32_t *seg, uint32_t *send, int *flags, void *stream);
int ms_band_flood_solve_dev(int64_t nlabels, int64_t lo, int64_t hi, const int32_t *off, const uint32_t *lkey,
                            uint32_t *seg, const int32_t *recv, int64_t n_recv, const int32_t *recv_pos,
                            const uint32_t *recv_keys, int64_t n_recv_keys, const double *st_sum, double cell_area,
                            int64_t n_events, const double *v, double *out_level, int64_t *out_wet, int *flags,
                            void *stream);

#ifdef __cplusplus
}
#endif
#endif
