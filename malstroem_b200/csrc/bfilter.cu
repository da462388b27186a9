// bfilter.cu — the bluespot filter of BluespotTool.process (bluespots.py:158-170) on the device: keep decisions of
// the raw labels from their raw stats (a postfix program compiled from the CLI's -filter text by
// malstroem_b200/bluespot_filter.py), the rank-compaction table of the kept labels, and the relabel pass that stands in
// for the second connected_components (a filter drops whole components, so the kept ones keep their cell sets and
// the scipy numbering of them is their raw-label order: SURVEY.md A.6).
#include <math.h>

#include "common.cuh"

namespace ms {

constexpr int BF_T = 128;

// One thread per label l in [0, nlabels + 1]: keep[l] = the program's decision (label 0: never), keep[nlabels + 1] = 0
// (the terminator the scan turns into the kept total).  Every thread runs the same program, so the loop is uniform;
// the operand stack lives in shared memory, one column per thread.  Each operation is one IEEE float64 operation.
__global__ void __launch_bounds__(BF_T) k_bluespot_keep(const __grid_constant__ ms_bluespot_filter f, int64_t nlabels,
                                                        const double *__restrict__ st_max,
                                                        const double *__restrict__ st_sum,
                                                        const int64_t *__restrict__ st_count, int *__restrict__ keep) {
    __shared__ double stk[MS_BF_MAX_STACK][BF_T];
    const int t = threadIdx.x;
    const int64_t l = (int64_t)blockIdx.x * BF_T + t;
    if (l > nlabels + 1) return;
    if (l == 0 || l == nlabels + 1) { keep[l] = 0; return; }
    const double area = __dmul_rn((double)st_count[l], f.cell_area);
    const double maxdepth = st_max[l];
    const double volume = __dmul_rn(st_sum[l], f.cell_area);
    int sp = 0;
    for (int pc = 0; pc < f.n_ops; pc++) {
        const int op = f.op[pc];
        if (op <= MS_BF_CONST) {
            stk[sp++][t] = op == MS_BF_AREA ? area : op == MS_BF_MAXDEPTH ? maxdepth : op == MS_BF_VOLUME ? volume
                                                                                                      : f.imm[pc];
            continue;
        }
        const double b = stk[sp - 1][t];
        if (op == MS_BF_NEG) { stk[sp - 1][t] = -b; continue; }
        if (op == MS_BF_NOT) { stk[sp - 1][t] = b == 0.0 ? 1.0 : 0.0; continue; }
        const double a = stk[sp - 2][t];
        double r;
        switch (op) {
            case MS_BF_ADD: r = __dadd_rn(a, b); break;
            case MS_BF_SUB: r = __dsub_rn(a, b); break;
            case MS_BF_MUL: r = __dmul_rn(a, b); break;
            case MS_BF_DIV: r = __ddiv_rn(a, b); break;
            case MS_BF_LT: r = a < b ? 1.0 : 0.0; break;
            case MS_BF_LE: r = a <= b ? 1.0 : 0.0; break;
            case MS_BF_GT: r = a > b ? 1.0 : 0.0; break;
            case MS_BF_GE: r = a >= b ? 1.0 : 0.0; break;
            case MS_BF_EQ: r = a == b ? 1.0 : 0.0; break;
            case MS_BF_NE: r = a != b ? 1.0 : 0.0; break;
            case MS_BF_AND: r = (a != 0.0 && b != 0.0) ? 1.0 : 0.0; break;
            default: r = (a != 0.0 || b != 0.0) ? 1.0 : 0.0; break;      // MS_BF_OR (validated on the host)
        }
        stk[--sp - 1][t] = r;
    }
    keep[l] = stk[0][t] != 0.0 ? 1 : 0;
}

// ex = exclusive scan of keep over nlabels + 2 entries: lut[l] = rank of a kept l = ex[l + 1], 0 for a dropped one
__global__ void __launch_bounds__(256) k_keep_lut(const int *__restrict__ ex, int64_t nlabels, int32_t *__restrict__ lut) {
    int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l > nlabels) return;
    const int a = ex[l], b = ex[l + 1];
    lut[l] = b != a ? b : 0;
}

// labels[c] = lut[labels[c]], four cells per thread with 16-byte accesses from the first aligned cell `head` on; the
// thread of quad 0 also does the cells before it.
__device__ inline int32_t relabel_one(int32_t v, int64_t nlabels, const int32_t *__restrict__ lut, int *err) {
    if ((uint32_t)v > (uint64_t)nlabels) { *err = 1; return v; }
    return __ldg(lut + v);
}

__global__ void __launch_bounds__(256) k_relabel(int32_t *lab, int64_t n, int64_t head, int64_t nlabels,
                                                 const int32_t *__restrict__ lut, int *err) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i = head + 4 * q;
    if (q == 0)
        for (int64_t k = 0; k < head && k < n; k++) lab[k] = relabel_one(lab[k], nlabels, lut, err);
    if (i + 4 <= n) {
        int4 v = *reinterpret_cast<const int4 *>(lab + i);
        v.x = relabel_one(v.x, nlabels, lut, err);
        v.y = relabel_one(v.y, nlabels, lut, err);
        v.z = relabel_one(v.z, nlabels, lut, err);
        v.w = relabel_one(v.w, nlabels, lut, err);
        *reinterpret_cast<int4 *>(lab + i) = v;
    } else {
        for (int64_t k = i; k < n; k++) lab[k] = relabel_one(lab[k], nlabels, lut, err);
    }
}

int check_bluespot_filter(const ms_bluespot_filter *f) {
    if (!f) { set_error("bluespot filter: null program"); return MS_ERR_ARG; }
    if (f->n_ops < 1 || f->n_ops > MS_BF_MAX_OPS) {
        set_error("bluespot filter: %d operations (1 ... %d)", f->n_ops, MS_BF_MAX_OPS);
        return MS_ERR_ARG;
    }
    if (!(f->cell_area > 0.0) || !isfinite(f->cell_area)) {
        set_error("bluespot filter: cell_area must be finite and > 0 (%g)", f->cell_area);
        return MS_ERR_ARG;
    }
    int sp = 0;
    for (int k = 0; k < f->n_ops; k++) {
        const int op = f->op[k];
        if (op < MS_BF_AREA || op > MS_BF_OR) { set_error("bluespot filter: bad op code %d at %d", op, k); return MS_ERR_ARG; }
        const int pops = op <= MS_BF_CONST ? 0 : op <= MS_BF_NOT ? 1 : 2;
        if (sp < pops) { set_error("bluespot filter: stack underflow at operation %d", k); return MS_ERR_ARG; }
        sp += op <= MS_BF_CONST ? 1 : op <= MS_BF_NOT ? 0 : -1;
        if (sp > MS_BF_MAX_STACK) {
            set_error("bluespot filter: stack deeper than %d at operation %d", MS_BF_MAX_STACK, k);
            return MS_ERR_ARG;
        }
    }
    if (sp != 1) { set_error("bluespot filter: the program leaves %d values", sp); return MS_ERR_ARG; }
    return MS_OK;
}

// keep decisions + LUT; *nkept (host) comes back through the pinned flags (synchronises the stream)
int bluespot_filter_dev_impl(const ms_bluespot_filter *f, int64_t nlabels, const double *st_max, const double *st_sum,
                             const int64_t *st_count, int32_t *lut, int64_t *nkept, cudaStream_t s) {
    MS_TRY(check_bluespot_filter(f));
    if (nlabels < 0 || nlabels >= INT32_MAX - 2 || !st_max || !st_sum || !st_count || !lut) {
        set_error("bluespot filter: bad argument");
        return MS_ERR_ARG;
    }
    const int64_t m2 = nlabels + 2;
    DevBuf<int> keep;
    DevBuf<int64_t> tot;
    MS_TRY(keep.alloc((size_t)m2, s));
    MS_TRY(tot.alloc(1, s));
    prof_units(m2);
    MS_LAUNCH(k_bluespot_keep, cdiv(m2, BF_T), BF_T, 0, s, *f, nlabels, st_max, st_sum, st_count, keep.p);
    MS_TRY(exclusive_scan_i32(keep.p, keep.p, m2, tot.p, s));
    prof_units(nlabels + 1);
    MS_LAUNCH(k_keep_lut, cdiv(nlabels + 1, 256), 256, 0, s, keep.p, nlabels, lut);
    int64_t *h = host_flags().h;
    MS_TRY(readback(h, tot.p, sizeof(int64_t), s));
    MS_TRY(stream_sync(s));
    if (nkept) *nkept = h[0];
    return MS_OK;
}

int relabel_dev_impl(int32_t *lab, int64_t n, int64_t nlabels, const int32_t *lut, int *err_dev, cudaStream_t s) {
    if (!lab || !lut || n < 1 || nlabels < 0) { set_error("relabel: bad argument"); return MS_ERR_ARG; }
    const int64_t head = ((16 - ((uintptr_t)lab & 15)) & 15) / 4;
    const int64_t quads = n > head ? (n - head + 3) / 4 : 1;
    prof_units(n);
    MS_LAUNCH(k_relabel, cdiv(quads, 256), 256, 0, s, lab, n, head, nlabels, lut, err_dev);
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_bluespot_filter_dev(const ms_bluespot_filter *filter, int64_t nlabels, const double *st_max,
                           const double *st_sum, const int64_t *st_count, int32_t *lut_out, int64_t *nkept,
                           void *stream) {
    MS_TRY(ms::ensure_init());
    return ms::bluespot_filter_dev_impl(filter, nlabels, st_max, st_sum, st_count, lut_out, nkept,
                                        (cudaStream_t)stream);
}

int ms_relabel_dev(int32_t *labels, int64_t n, int64_t nlabels, const int32_t *lut, void *stream) {
    MS_TRY(ms::ensure_init());
    cudaStream_t s = (cudaStream_t)stream;
    ms::DevBuf<int> err;
    MS_TRY(err.alloc(1, s));
    MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
    MS_TRY(ms::relabel_dev_impl(labels, n, nlabels, lut, err.p, s));
    int64_t *h = ms::host_flags().h;
    MS_TRY(ms::readback(h + 16, err.p, sizeof(int), s));
    MS_TRY(ms::stream_sync(s));
    if (*(int *)(h + 16)) {
        ms::set_error("relabel: a label lies outside [0, %lld]", (long long)nlabels);
        return MS_ERR_LABEL;
    }
    return MS_OK;
}

}  // extern "C"
