// pipeline.cu — the whole raster hot path on device-resident data (what bench.py times):
// DEM -> fill (+depths) -> short/diag -> no-flats fill -> D8 -> accumulation -> bluespot labels ->
// [bluespot filter] -> label stats -> watersheds (+counts) -> pour points.  Order and operands follow DemTool.process
// (malstroem/dem.py:53-93) and BluespotTool.process (malstroem/bluespots.py:138-216).  The bluespot filter
// (bluespots.py:160-170) runs when the caller gives one (ms_pipeline_filtered_host_dev): raw label stats, keep
// decisions and a relabel of the kept labels by rank (bfilter.cu); bench.py runs without a filter.
#include <math.h>

#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"

namespace ms {
int fill_no_flats_dev_impl(const float *dtm, const float *filled, double sh, double dg, double *out, int64_t rows,
                           int64_t cols, int64_t *stats, cudaStream_t s, uint8_t *flowdir_out, int *flowdir_done);
int flowdir_dev_impl(const double *t, uint8_t *out, int64_t rows, int64_t cols, int edges, cudaStream_t s, int open);
int accum_dev_impl(const uint8_t *fd, double *acc, int64_t rows, int64_t cols, cudaStream_t s);
int watersheds_labels_dev_impl(const uint8_t *fd, const int32_t *lab, int32_t *ws, int64_t rows, int64_t cols,
                               int64_t *stats, cudaStream_t s);
int cc_dev_impl(const void *data, int dtype, int32_t *labels, int64_t rows, int64_t cols, int64_t *nlabels_dev,
                cudaStream_t s);
int label_stats_dev_impl(const void *data, int dtype, const int32_t *lab, int64_t n, int64_t nlabels, double *omin,
                         double *omax, double *osum, int64_t *ocnt, int *err_dev, cudaStream_t s);
int label_extreme_dev_impl(const double *data, const int32_t *lab, int64_t rows, int64_t cols, int64_t nlabels,
                           int want_max, double *oval, int64_t *orow, int64_t *ocol, int *err_dev, cudaStream_t s);
int label_count_dev_impl(const int32_t *lab, int64_t n, int64_t nbins, int64_t *cnt, int *err_dev, cudaStream_t s);
int pipeline_tables_dev_impl(const float *depths, const int32_t *lab, const double *fnf, const double *accum,
                             const int32_t *ws, int64_t rows, int64_t cols, int64_t nlabels, double *st_min,
                             double *st_max, double *st_sum, int64_t *st_count, int64_t *ws_count, double *pmin_v,
                             int64_t *pmin_r, int64_t *pmin_c, double *pmax_v, int64_t *pmax_r, int64_t *pmax_c,
                             int *err_dev, cudaStream_t s);
int bluespot_filter_dev_impl(const ms_bluespot_filter *f, int64_t nlabels, const double *st_max, const double *st_sum,
                             const int64_t *st_count, int32_t *lut, int64_t *nkept, cudaStream_t s);
int relabel_dev_impl(int32_t *lab, int64_t n, int64_t nlabels, const int32_t *lut, int *err_dev, cudaStream_t s);
int check_bluespot_filter(const ms_bluespot_filter *f);
}  // namespace ms

namespace {
// device -> host copies of finished rasters on a second stream, so that they overlap the stages that follow
cudaStream_t g_copy_stream = nullptr;
cudaEvent_t g_copy_ev[8];
int g_copy_n = 0;

// MS_SHIP_TRACE=1: time every shipped raster on the copy stream (printed by ms_copies_wait) - where the PCIe time of
// the host-buffer path goes
struct ShipTrace { cudaEvent_t ready, t0, t1; size_t bytes; };
ShipTrace g_trace[16];
int g_trace_n = 0, g_trace_on = -1;
cudaEvent_t g_trace_origin = nullptr;

int ship(void *dst, const void *src, size_t bytes, cudaStream_t s) {
    if (!dst) return MS_OK;
    if (!g_copy_stream) {
        MS_CUDA(cudaStreamCreateWithFlags(&g_copy_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 8; k++) MS_CUDA(cudaEventCreateWithFlags(&g_copy_ev[k], cudaEventDisableTiming));
    }
    if (g_trace_on < 0) { const char *e = getenv("MS_SHIP_TRACE"); g_trace_on = e && e[0] == '1'; }
    cudaEvent_t ev = g_copy_ev[g_copy_n++ & 7];
    ShipTrace *t = nullptr;
    if (g_trace_on && g_trace_n < 16) {
        t = &g_trace[g_trace_n++];
        if (!t->ready) { cudaEventCreate(&t->ready); cudaEventCreate(&t->t0); cudaEventCreate(&t->t1); }
        t->bytes = bytes;
        ev = t->ready;
    }
    MS_CUDA(cudaEventRecord(ev, s));
    MS_CUDA(cudaStreamWaitEvent(g_copy_stream, ev, 0));
    if (t) MS_CUDA(cudaEventRecord(t->t0, g_copy_stream));
    // In pieces: the stages that follow read small counters back every round (Boruvka, pointer jumping, label
    // counts), and a device-to-host read-back queues behind whatever the copy engine is busy with - behind one
    // 8.6 GB copy the compute stream stood still for 170 ms (MS_SHIP_TRACE: 32768^2 host-buffer step 739 ms).
    // Between pieces of 32 MB (0.6 ms) the engine takes the read-back.
    const size_t piece = (size_t)32 << 20;
    for (size_t off = 0; off < bytes; off += piece) {
        const size_t nb = bytes - off < piece ? bytes - off : piece;
        MS_CUDA(cudaMemcpyAsync((char *)dst + off, (const char *)src + off, nb, cudaMemcpyDeviceToHost, g_copy_stream));
    }
    if (t) MS_CUDA(cudaEventRecord(t->t1, g_copy_stream));
    return MS_OK;
}
}  // namespace

extern "C" int ms_copies_wait(void) {
    if (g_copy_stream) MS_CUDA(cudaStreamSynchronize(g_copy_stream));
    if (g_trace_on > 0 && g_trace_n) {
        for (int k = 0; k < g_trace_n; k++) {
            float ready = 0, a = 0, b = 0;
            cudaEventElapsedTime(&ready, g_trace_origin ? g_trace_origin : g_trace[0].ready, g_trace[k].ready);
            cudaEventElapsedTime(&a, g_trace_origin ? g_trace_origin : g_trace[0].ready, g_trace[k].t0);
            cudaEventElapsedTime(&b, g_trace[k].t0, g_trace[k].t1);
            fprintf(stderr, "[ship] raster %d: ready at %.1f ms, copy starts at %.1f ms, %.2f GB in %.1f ms = %.1f GB/s\n", k,
                    ready, a, g_trace[k].bytes / 1e9, b, g_trace[k].bytes / 1e6 / b);
        }
        g_trace_n = 0;
    }
    return MS_OK;
}

namespace {
// bluespots.py:160-170: raw label_stats(depths, labels) -> filterbluespots -> keep_labels -> connected_components,
// the last two as one relabel by rank.  The raw stats go into the pipeline's own tables when it has all four (the
// table passes overwrite them with the filtered ones), into scratch otherwise.
int filter_labels(ms_rasters *io, const ms_bluespot_filter *filter, int *err_dev, cudaStream_t s) {
    using namespace ms;
    const int64_t n = io->rows * io->cols, m = io->nlabels + 1;
    DevBuf<double> smin, smax, ssum;
    DevBuf<int64_t> scnt;
    double *tmin = io->st_min, *tmax = io->st_max, *tsum = io->st_sum;
    int64_t *tcnt = io->st_count;
    if (!tmin || !tmax || !tsum || !tcnt) {
        MS_TRY(smin.alloc((size_t)m, s)); MS_TRY(smax.alloc((size_t)m, s));
        MS_TRY(ssum.alloc((size_t)m, s)); MS_TRY(scnt.alloc((size_t)m, s));
        tmin = smin.p; tmax = smax.p; tsum = ssum.p; tcnt = scnt.p;
    }
    MS_TRY(label_stats_dev_impl(io->depths, MS_F32, io->labels, n, io->nlabels, tmin, tmax, tsum, tcnt, err_dev, s));
    DevBuf<int32_t> lut;
    MS_TRY(lut.alloc((size_t)m, s));
    int64_t nkept = 0;
    MS_TRY(bluespot_filter_dev_impl(filter, io->nlabels, tmax, tsum, tcnt, lut.p, &nkept, s));
    MS_TRY(relabel_dev_impl(io->labels, n, io->nlabels, lut.p, err_dev, s));
    io->nlabels = nkept;
    return MS_OK;
}
}  // namespace

extern "C" int ms_pipeline_dev(ms_rasters *io, void *stream) { return ms_pipeline_host_dev(io, nullptr, stream); }

extern "C" int ms_pipeline_host_dev(ms_rasters *io, const ms_host_out *host, void *stream) {
    return ms_pipeline_filtered_host_dev(io, host, nullptr, nullptr, stream);
}

extern "C" int ms_pipeline_filtered_host_dev(ms_rasters *io, const ms_host_out *host, const ms_bluespot_filter *filter,
                                             int64_t *nlabels_raw, void *stream) {
    using namespace ms;
    if (host && g_trace_on > 0) {
        if (!g_trace_origin) cudaEventCreate(&g_trace_origin);
        cudaEventRecord(g_trace_origin, (cudaStream_t)stream);
    }
    MS_TRY(ensure_init());
    cudaStream_t s = (cudaStream_t)stream;
    static const ms_host_out no_host = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (!host) host = &no_host;
    if (!io || !io->dem || !io->filled || !io->depths || !io->fnf || !io->flowdir || !io->labels || !io->wsheds) {
        set_error("pipeline: null raster pointer");
        return MS_ERR_ARG;
    }
    if (filter) MS_TRY(check_bluespot_filter(filter));
    int64_t rows = io->rows, cols = io->cols, n = rows * cols;
    for (int k = 0; k < 8; k++) io->stats[k] = 0;
    int64_t *h = host_flags().h;

    // dem.py:67-72, and dem.py:79's min / max of the DEM (fill.py:235-250), which the fill's tile pass reduces
    DevBuf<float> mm;
    MS_TRY(mm.alloc(2, s));
    MS_TRY(fill_terrain_dev_impl(io->dem, io->filled, io->depths, rows, cols, io->stats, s, mm.p));
    MS_TRY(ship(host->filled, io->filled, (size_t)n * sizeof(float), s));
    MS_TRY(ship(host->depths, io->depths, (size_t)n * sizeof(float), s));
    MS_TRY(ms::readback(h + 24, mm.p, 2 * sizeof(float), s));
    MS_TRY(ms::stream_sync(s));
    float lo = ((float *)(h + 24))[0], hi = ((float *)(h + 24))[1];
    double maxval = (double)fmaxf(fabsf(hi), fabsf(lo));
    io->short_eps = (nextafter(maxval, (double)INFINITY) - maxval) * 1024.0;
    io->diag_eps = io->short_eps * pow(2.0, 0.5);
    // dem.py:80-83
    int64_t nfstats[4] = {0, 0, 0, 0};
    int flowdir_done = 0;      // the integer-raster no-flats solve writes the D8 codes in its finishing pass
    MS_TRY(fill_no_flats_dev_impl(io->dem, io->filled, io->short_eps, io->diag_eps, io->fnf, rows, cols, nfstats, s,
                                  io->flowdir, &flowdir_done));
    io->stats[2] = nfstats[0]; io->stats[3] = nfstats[1]; io->stats[4] = nfstats[2]; io->stats[7] = nfstats[3];
    MS_TRY(ship(host->fnf, io->fnf, (size_t)n * sizeof(double), s));
    if (!flowdir_done) MS_TRY(flowdir_dev_impl(io->fnf, io->flowdir, rows, cols, 1, s, 0));
    MS_TRY(ship(host->flowdir, io->flowdir, (size_t)n, s));
    // dem.py:87-91
    if (io->accum) {
        MS_TRY(accum_dev_impl(io->flowdir, io->accum, rows, cols, s));
        MS_TRY(ship(host->accum, io->accum, (size_t)n * sizeof(double), s));
    }
    // bluespots.py:158-160
    DevBuf<int64_t> tot;
    DevBuf<int> err;
    MS_TRY(tot.alloc(1, s));
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    MS_TRY(cc_dev_impl(io->depths, MS_F32, io->labels, rows, cols, tot.p, s));
    MS_TRY(ms::readback(h, tot.p, sizeof(int64_t), s));
    MS_TRY(ms::stream_sync(s));
    io->nlabels = h[0];
    if (nlabels_raw) *nlabels_raw = io->nlabels;
    if (io->nlabels + 1 > io->table_capacity) {
        set_error("pipeline: %lld labels do not fit table_capacity %lld", (long long)io->nlabels,
                  (long long)io->table_capacity);
        return MS_ERR_ARG;
    }
    if (filter) MS_TRY(filter_labels(io, filter, err.p, s));
    MS_TRY(ship(host->labels, io->labels, (size_t)n * sizeof(int32_t), s));
    // every table asked for (the usual case): two fused passes over the rasters (labels.cu: k_tables_a2 / k_tables_b)
    const bool fused = io->st_min && io->st_max && io->st_sum && io->st_count && io->ws_count && io->ppmin_value &&
                       io->ppmin_row && io->ppmin_col;
    if (io->st_min && !fused)
        MS_TRY(label_stats_dev_impl(io->depths, MS_F32, io->labels, n, io->nlabels, io->st_min, io->st_max, io->st_sum,
                                    io->st_count, err.p, s));
    // bluespots.py:183-186
    MS_TRY(watersheds_labels_dev_impl(io->flowdir, io->labels, io->wsheds, rows, cols, io->stats, s));
    MS_TRY(ship(host->wsheds, io->wsheds, (size_t)n * sizeof(int32_t), s));
    if (fused) {
        // bluespots.py:160, 186, 195-206 (both pour-point variants)
        MS_TRY(pipeline_tables_dev_impl(io->depths, io->labels, io->fnf, io->accum, io->wsheds, rows, cols, io->nlabels,
                                        io->st_min, io->st_max, io->st_sum, io->st_count, io->ws_count, io->ppmin_value,
                                        io->ppmin_row, io->ppmin_col, io->accum ? io->ppmax_value : nullptr, io->ppmax_row,
                                        io->ppmax_col, err.p, s));
        return MS_OK;
    }
    if (io->ws_count) MS_TRY(label_count_dev_impl(io->wsheds, n, io->nlabels + 1, io->ws_count, err.p, s));
    // bluespots.py:195-206 (both pour-point variants)
    if (io->ppmin_value)
        MS_TRY(label_extreme_dev_impl(io->fnf, io->labels, rows, cols, io->nlabels, 0, io->ppmin_value, io->ppmin_row,
                                      io->ppmin_col, err.p, s));
    if (io->ppmax_value && io->accum)
        MS_TRY(label_extreme_dev_impl(io->accum, io->labels, rows, cols, io->nlabels, 1, io->ppmax_value, io->ppmax_row,
                                      io->ppmax_col, err.p, s));
    return MS_OK;
}
