// Checks of a solve's keywords, shared by libbsgp (bsgp_kernels.cu) and the test-only host emulation: plain C++, no CUDA
// call.  A batch either shares one bsgp_params or gives every image its own row (bsgp_solve_batch_rows); both go through
// check_batch_params, which also fixes the per-image stride of the trace outputs.
#pragma once
#include <stdio.h>
#include <string.h>

#include "../../include/bsgp.h"
#include "bsgp_smem.h"

namespace bsgp {

// One set of keywords and the inputs / outputs it needs.  `where` names the row in messages ("" for a shared set).
inline int check_params_row(const bsgp_params* q, const bsgp_inputs* in, const bsgp_outputs* out, const char* where, char* err,
                            size_t errlen) {
    const char* msg = nullptr;
    char mem[48];
    snprintf(mem, sizeof mem, "M and M_alpha must be in 1..%d", kMaxMem);
    if (q->divergence != BSGP_DIV_KL && q->divergence != BSGP_DIV_BETA) msg = "bad divergence";
    else if (q->init_recon < 0 || q->init_recon > 3) msg = "init_recon must be 0..3";
    else if (q->proj_type < 0 || q->proj_type > 1) msg = "proj_type must be 0 or 1";
    else if (q->stop_criterion < 0 || q->stop_criterion > 4) msg = "stop_criterion must be 0..4";
    else if (q->maxit < 1) msg = "MAXIT must be >= 1";
    else if (q->m < 1 || q->m > kMaxMem || q->m_alpha < 1 || q->m_alpha > kMaxMem) msg = mem;
    else if (q->has_flux && !in->flux) msg = "has_flux set but inputs.flux is NULL";
    else if (q->divergence == BSGP_DIV_BETA && !in->beta0) msg = "beta-divergence needs inputs.beta0";
    else if (q->init_recon == 1 && !in->x0) msg = "init_recon = 1 needs inputs.x0";
    else if (q->errflag && (!in->obj || !out->err)) msg = "errflag needs inputs.obj and outputs.err";
    if (!msg) return BSGP_OK;
    snprintf(err, errlen, "%s%s", where, msg);
    return BSGP_E_ARG;
}

// The fields that describe the operator and the plan rather than the solve: equal in every row of a batch.
inline bool same_operator(const bsgp_params* a, const bsgp_params* b) {
    return memcmp(a->region, b->region, sizeof a->region) == 0 && a->div_a == b->div_a && a->div_at == b->div_at &&
           a->adjoint_second_psf == b->adjoint_second_psf;
}

// The keywords of a batch: `prm` shared by all images (rows == NULL), or rows[0 .. batch-1], one per image.  On success
// *trace_stride is the per-image stride of discr, times, stop_value and trace_* (err: trace_stride + 1), the largest
// maxit + 1 of the batch.
inline int check_batch_params(const bsgp_params* prm, const bsgp_params* rows, int batch, const bsgp_inputs* in,
                              const bsgp_outputs* out, int* trace_stride, char* err, size_t errlen) {
    if (!rows) {
        const int rc = check_params_row(prm, in, out, "", err, errlen);
        if (rc) return rc;
        *trace_stride = prm->maxit + 1;
        return BSGP_OK;
    }
    int stride = 0;
    for (int i = 0; i < batch; ++i) {
        char where[48];
        snprintf(where, sizeof where, "row %d: ", i);
        const int rc = check_params_row(&rows[i], in, out, where, err, errlen);
        if (rc) return rc;
        if (!same_operator(&rows[i], &rows[0])) {
            snprintf(err, errlen, "row %d: region, div_a, div_at and adjoint_second_psf describe the operator and must equal row 0's", i);
            return BSGP_E_ARG;
        }
        if (rows[i].maxit + 1 > stride) stride = rows[i].maxit + 1;
    }
    *trace_stride = stride;
    return BSGP_OK;
}

// The observations of a batch (bsgp_inputs.source, host memory): without a map, image i is observation i; with one, every
// entry must name one of n_sources >= 1 observations, since the kernels index gn, bkg, x0, obj and the PSF spectra with it.
inline int check_sources(const bsgp_inputs* in, int batch, char* err, size_t errlen) {
    if (!in->source) return BSGP_OK;
    if (in->n_sources < 1) {
        snprintf(err, errlen, "n_sources must be >= 1 with a source map (got %d)", in->n_sources);
        return BSGP_E_ARG;
    }
    for (int i = 0; i < batch; ++i)
        if (in->source[i] < 0 || in->source[i] >= in->n_sources) {
            snprintf(err, errlen, "solve %d: source %d is outside 0..%d", i, in->source[i], in->n_sources - 1);
            return BSGP_E_ARG;
        }
    return BSGP_OK;
}

// The number of observations a batch reads: n_sources with a map, else one per image.
inline int observation_count(const bsgp_inputs* in, int batch) { return in->source ? in->n_sources : batch; }

// Iterate snapshots (bsgp_outputs.snap_x / snap_every / snap_count): an interval >= 0, and a destination when it is > 0.
inline int check_snapshots(const bsgp_outputs* out, char* err, size_t errlen) {
    if (out->snap_every < 0) {
        snprintf(err, errlen, "snap_every must be >= 0 (got %d)", out->snap_every);
        return BSGP_E_ARG;
    }
    if (out->snap_every > 0 && !out->snap_x) {
        snprintf(err, errlen, "snap_every = %d needs outputs.snap_x", out->snap_every);
        return BSGP_E_ARG;
    }
    return BSGP_OK;
}

// Snapshot slots per solve for a batch whose trace stride (check_batch_params) is the largest maxit + 1: the iterates
// after 0, k, 2k, ... <= maxit passes.
inline int snapshot_slots(int trace_stride, int snap_every) { return (trace_stride - 1) / snap_every + 1; }

// PSF spectra set on the plan: one for all, or one per observation.
inline int check_psf_count(int n_psf, const bsgp_inputs* in, int batch, char* err, size_t errlen) {
    if (n_psf == 1 || n_psf == observation_count(in, batch)) return BSGP_OK;
    if (in->source) snprintf(err, errlen, "bsgp_set_psf was called with %d PSFs; need 1 or n_sources (%d)", n_psf, in->n_sources);
    else snprintf(err, errlen, "bsgp_set_psf was called with %d PSFs; need 1 or batch (%d)", n_psf, batch);
    return BSGP_E_STATE;
}

}  // namespace bsgp
