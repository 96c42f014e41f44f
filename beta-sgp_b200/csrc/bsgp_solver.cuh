// One complete SGP / beta-SGP restoration of one image by one thread-block cluster.
//
// This is the body of the persistent solve kernel: every loop of the reference (outer iteration
// sgp.py:302-425 / 748-882, line search :328-349 / :776-800, projection root-find
// flux_conserve_proj.py:38-142) runs here with ordinary control flow.  All threads of all CTAs of
// the cluster execute the scalar controller (`solve_image`) redundantly on bit-identical
// all-reduced sums, so the control flow is uniform across the cluster and no scalar is ever
// broadcast or sent to the host.
//
// Structure.  The controller is inlined into the kernel; every pass over the pixels is a separate
// NON-inlined "phase" function (ph_*), so each pass gets its own register allocation (no spills
// from the controller's long-lived state) and the kernel stays small enough for the instruction
// cache.  Phases read the per-image constants (`ImgState`, one copy per CTA in shared memory), take
// the few changing scalars by value and return their partial sums by value; the controller does the
// cluster all-reduce.  Each phase starts with a block barrier because consecutive phases map
// pixels to threads differently.
//
// `Ctx` supplies: tid, nt, rank, G, sync(), cluster_sync(), allreduce_sum(double*, k),
// allreduce_min(double&), allreduce_max(double&), now().  DeviceCtx (bsgp_device.cuh) is the
// product; tests/host_emul provides a one-thread emulation of the same code.
//
// Numerics follow the reference's operand order with non-contracted arithmetic (bsgp_math.cuh);
// deliberate deviations, all at rounding level:
//   * the projection evaluates (c + lambda) * X instead of (c + lambda) / D with D = 1/X,
//   * den^beta = den^(beta-1) * den and den^(beta-2) = den^(beta-1) / den (one pow per pixel),
//   * reductions are tree sums in fp64 (numpy: pairwise / BLAS dot).
#pragma once
#include <type_traits>

#include "../../include/bsgp.h"
#include "bsgp_conv.cuh"
#include "bsgp_project.cuh"
#include "bsgp_smem.h"

#ifndef BSGP_U_TRIAL
#define BSGP_U_TRIAL 2
#endif
#ifndef BSGP_U_TP
#define BSGP_U_TP 4
#endif
#ifndef BSGP_U_PE
#define BSGP_U_PE 8
#endif

namespace bsgp {

enum Buf { B_GN = 0, B_BKG, B_X, B_G, B_XTF, B_D, B_DTF, B_T1, NBUF };

template <typename T> struct SolveArgs {
    bsgp_params p;
    ConvGeom g;
    int batch;
    // inputs
    const T* gn; const T* bkg; int bkg_is_image; const double* flux; const double* beta0; const T* x0; const T* obj; const int* order;
    // tables
    const cplx<T>* twx; const cplx<T>* twy; cplx<T>* tf; cplx<T>* tf_adj; int n_psf;
    // per-cluster global scratch
    T* work; size_t work_stride; cplx<T>* spec; size_t spec_stride;
    int resident_mask;              // bit b: Buf b lives in shared memory
    // outputs
    T* x_out; int* iters; int* status; double* discr; double* times; double* stop_value; double* err;
    double* beta_final; int* proj_evals; int* ls_trials; double* scalars;
    double* tr_alpha; double* tr_lambda; double* tr_beta; int* tr_trials; int* tr_evals;
    int* queue;
    const int* ready;               // [batch] or NULL: queue item i may start once ready[i] != 0 (pipelined upload, bsgp_solve_batch_pinned)
};

// A mixed batch (bsgp_solve_batch_rows): image i solves with its own keywords rows[i] (device, [batch]); the operator fields
// (region, divisors, adjoint kernel) still come from SolveArgs::p.  trace_stride: the per-image stride of discr / times /
// stop_value / trace_* (err: + 1), the largest maxit + 1 of the rows.  Only the ROWS kernels take it: a launch without rows
// runs kernels compiled exactly as before the feature existed.
// source: [batch] (device) or NULL: the observation each solve reads (bsgp_inputs.source).  A launch with a map always runs
// the ROWS kernels (the host expands shared keywords into equal rows), so the kernels without rows never see one.
// snap: [batch][n_snap][..] (device) or NULL: iterate snapshots (bsgp_outputs.snap_x), every snap_every-th pass; a slot
// holds the whole grid, or with snap_crop the valid window a.p.region (a wrapped plan: the caller's image shape).
// snap_count: [batch] or NULL.  Like a source map, snapshots always run the ROWS kernels.
struct RowArgs {
    const bsgp_params* rows; int trace_stride; const int* source;
    void* snap; int* snap_count; int snap_every, n_snap, snap_crop;
};
struct NoRow {};
// the observation solve `img` reads: gn, bkg, x0, obj and the PSF spectra are indexed by it
BSGP_DEV int source_of(int img) { return img; }
BSGP_DEV int source_of(int img, const RowArgs& ra) { return ra.source ? ra.source[img] : img; }
// the keywords the controller reads: the image's own copy of its row, or the batch's
BSGP_DEV const bsgp_params& image_params(const bsgp_params& own, const bsgp_params&) { return own; }
BSGP_DEV const bsgp_params& image_params(const NoRow&, const bsgp_params& shared) { return shared; }

// Per-image constants of one CTA (shared memory).  Pointers address this CTA's slab of each array.
template <typename T> struct ImgState {
    T* gn; T* bkg; T* x; T* g; T* xtf; T* d; T* dtf; T* t1;
    const T* gn_raw; const T* bkg_raw; const T* x0_raw; const T* truth; T* x_out;
    const cplx<T>* twx; const cplx<T>* twy; cplx<T>* spec; cplx<T>* tf; cplx<T>* tf_at;
    unsigned ws_off, ppx_off;        // FFT workspace and position table: byte offsets into dynamic shared memory
    unsigned twx_off, twy_off;       // twiddle tables in shared memory, or kNoSmem (then twx / twy are used)
    int tw_split;                    // the shared-memory tables are two-level (long transforms)
    ConvGeom geom;
    int nslab, bkg_img, init_recon, has_cap, pflag, want_err, stop2;
    int x_ones;                      // the projection's X is 1, not clip(x): initial projection, first iteration from x = 0
    int masked, reg[4];              // zero-padded operator: valid window [reg0, reg1) x [reg2, reg3) of the FFT grid
    T bkg_raw_s, scaling, bkg_s, null_fill, x_const, cap, xlo, xhi;
    T div_a, div_at;                 // output divisors of A / A^T (zero-padded operator; 1 otherwise)
};

struct R2 { double a, b; };
struct R3 { double a, b, c; };
struct R7 { double v[7]; };

enum { F_FIRST = 4 };

// divergence constants for the current beta (sgp.py:452-458)
template <typename T> struct DivK {
    int kind;            // 0 KL (sgp), 1 beta generic, 2 beta == 0, 3 beta == 1
    T b, bm1, k, k2, k3;
};
template <typename T> BSGP_DEV DivK<T> make_divk(int divergence, double beta) {
    DivK<T> d;
    d.b = (T)beta; d.bm1 = (T)(beta - 1.0); d.k = d.k2 = d.k3 = (T)0;
    if (divergence == BSGP_DIV_KL) { d.kind = 0; return d; }
    if (beta == 0.0) { d.kind = 2; return d; }
    if (beta == 1.0) { d.kind = 3; return d; }
    d.kind = 1;
    const double k = 1.0 / nmul(beta, beta - 1.0);
    d.k = (T)k; d.k2 = (T)nmul(k, beta - 1.0); d.k3 = (T)nmul(k, beta);
    return d;
}

// One pixel of the objective at den = x_tf_try + bkg.  Adds its terms to acc[0..3] and returns the
// quantity cached for the gradient: gn/den (KL) or den^(beta-1) (beta-divergence).
//   KL    : acc0 += gn*log(gn/den), acc1 += x_tf_try                               sgp.py:333-334
//   beta  : acc0 += k*gn^b (only if want_s1), acc1 += k(b-1)*den^b, acc2 += k*b*gn*den^(b-1)   sgp.py:457-458
//   b == 0: acc0 += gn/den, acc1 += log(gn/den)                                     sgp.py:453
//   b == 1: acc0 += gn*log(gn/den), acc1 += gn, acc2 += den                         sgp.py:455
// KIND is compile-time in the solver's phases: each phase exists once per divergence kind, so a solve only ever touches
// the code of its own kind - the phases that evaluate the objective are the largest functions of the kernel (an inlined
// pow() per pixel of every pair and row).  The data-only term of the generic beta-divergence, s1 = sum k*gn^beta, changes
// only when beta does: it has its own small pass (ph_s1) instead of a second pow() in every objective phase.
template <int KIND, bool CALL = false, typename T> BSGP_DEV T objective_pixel_k(const DivK<T>& dk, T gnv, T den, T xtf_try, KSum* acc) {
    if (KIND == 0) {
        const T ratio = ndiv(gnv, den);
        acc[0].add((double)nmul(gnv, mlog_sel<CALL>(ratio)));
        acc[1].add((double)xtf_try);
        return ratio;
    }
    if (KIND == 1) {
        const T p1 = mpow_sel<CALL>(den, dk.bm1);
        acc[1].add((double)nmul(dk.k2, nmul(p1, den)));
        acc[2].add((double)nmul(nmul(dk.k3, gnv), p1));
        return p1;
    }
    const T ratio = ndiv(gnv, den);
    if (KIND == 2) {
        acc[0].add((double)ratio);
        acc[1].add((double)mlog_sel<CALL>(ratio));
        return ndiv((T)1, den);
    }
    acc[0].add((double)nmul(gnv, mlog_sel<CALL>(ratio)));
    acc[1].add((double)gnv);
    acc[2].add((double)den);
    return (T)1;
}
template <typename T> BSGP_DEV T objective_pixel(const DivK<T>& dk, T gnv, T den, T xtf_try, bool want_s1, KSum* acc) {
    if (dk.kind == 0) return objective_pixel_k<0>(dk, gnv, den, xtf_try, acc);
    if (dk.kind == 1) {
        if (want_s1) acc[0].add((double)nmul(dk.k, mpow(gnv, dk.b)));
        return objective_pixel_k<1>(dk, gnv, den, xtf_try, acc);
    }
    if (dk.kind == 2) return objective_pixel_k<2>(dk, gnv, den, xtf_try, acc);
    return objective_pixel_k<3>(dk, gnv, den, xtf_try, acc);
}

// call phase FN<T, MK, KIND>(...) with the divergence kind as a compile-time constant
#define BSGP_DISPATCH_KIND(dk, FN, ...)                         \
    ((dk).kind == 0 ? FN<T, MK, 0>(__VA_ARGS__)                  \
     : (dk).kind == 1 ? FN<T, MK, 1>(__VA_ARGS__)                \
     : (dk).kind == 2 ? FN<T, MK, 2>(__VA_ARGS__)                \
                      : FN<T, MK, 3>(__VA_ARGS__))

template <typename T> BSGP_DEV double objective_value(const DivK<T>& dk, const double* acc, double s1, double flux, double npix) {
    if (dk.kind == 0) return (acc[0] + acc[1]) - flux;
    if (dk.kind == 1) return (s1 + acc[1]) - acc[2];
    if (dk.kind == 2) return (acc[0] - acc[1]) - npix;
    return (acc[0] - acc[1]) + acc[2];
}

// per-pixel d D_beta / d beta, sgp.py:495 (term order kept)
template <bool CALL = false, typename T> BSGP_DEV T dbeta_pixel(T x, T y, T b) {
    const T bm1 = b - (T)1;
    const T ypb1 = mpow_sel<CALL>(y, bm1), ypb = nmul(ypb1, y), xpb = mpow_sel<CALL>(x, b), ly = mlog_sel<CALL>(y), lx = mlog_sel<CALL>(x);
    const T bm1sq = nmul(bm1, bm1), bbm1 = nmul(b, bm1), bsq = nmul(b, b);
    T s = ndiv(nmul(nmul(-x, ypb1), ly), bm1);
    s = nadd(s, ndiv(nmul(x, ypb1), bm1sq));
    s = nadd(s, ndiv(nmul(xpb, lx), bbm1));
    s = nsub(s, ndiv(xpb, nmul(b, bm1sq)));
    s = nadd(s, ndiv(nmul(ypb, ly), b));
    s = nsub(s, ndiv(xpb, nmul(bsq, bm1)));
    s = nsub(s, ndiv(ypb, bsq));
    return s;
}

template <typename T> BSGP_DEV T clip_bounds(T v, T lo, T hi) {   // sgp.py:355-357
    if (v < lo) v = lo;
    if (v > hi) v = hi;
    return v;
}

// x(lambda) of the projection: min(cap, max(0, (c + lambda) * X))      flux_conserve_proj.py:22-24
template <typename T> BSGP_DEV T proj_point(T c, T X, T lam, bool has_cap, T cap) {
    T v = nmul(nadd(c, lam), X);
    v = (v <= (T)0) ? (T)0 : v;
    if (has_cap) v = (v >= cap) ? cap : v;
    return v;
}

// -------------------------------------------------------------------------------------------------
// Valid region.  With the zero-padded operator (the reference's astropy closure, sgp.py:121-161) the
// image occupies a centred window [r0, r1) x [c0, c1) of the power-of-two FFT grid the kernel works on;
// everything outside is padding: it holds zeros in every array, contributes to no sum, and operator
// outputs that land there are discarded.  With the circular operator the region is the whole grid and
// `on` is 0 (every test below folds to true).
// -------------------------------------------------------------------------------------------------
struct Region { int on, r0, r1, c0, c1, row_off, lg_nx, colmask; };
template <bool MK, typename T, class Ctx> BSGP_DEV Region region_of(const Ctx& ctx, const ImgState<T>* S) {
    Region R;
    R.on = MK;
    if (!MK) { R.r0 = R.r1 = R.c0 = R.c1 = R.row_off = R.lg_nx = R.colmask = 0; return R; } R.r0 = S->reg[0]; R.r1 = S->reg[1]; R.c0 = S->reg[2]; R.c1 = S->reg[3];
    R.row_off = ctx.rank * S->geom.rows_per_cta; R.lg_nx = S->geom.lg_nx; R.colmask = S->geom.nx - 1;
    return R;
}
template <bool MK> BSGP_DEV bool inside(const Region& R, int i) {
    if (!MK) return true;
    const int row = R.row_off + (i >> R.lg_nx), col = i & R.colmask;
    return row >= R.r0 && row < R.r1 && col >= R.c0 && col < R.c1;
}

// -------------------------------------------------------------------------------------------------
// setup phases (sgp.py:166-217, 248-257)
// -------------------------------------------------------------------------------------------------
// sum(gn), sum(gn - bkg), max(gn) over the raw slab
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R3 ph_stats(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    const T* gr = S->gn_raw; const T* br = S->bkg_raw; const bool bimg = S->bkg_img != 0; const T bs = S->bkg_raw_s;
    const Region R = region_of<MK>(ctx, S);
    double mx = -INFINITY, s0 = 0.0, s1 = 0.0;
    auto fetch = [&](int i) { In2<T> r; r.a = ld2(gr, i); r.b = bimg ? ld2(br, i) : mk2(bs, bs); return r; };
    auto one = [&](bool m, T v, T b) {
        if (!m) return;
        mx = ((double)v > mx) ? (double)v : mx;
        s0 += (double)v;
        s1 += (double)nsub(v, b);
    };
    auto body = [&](int i, const In2<T>& in) { one(inside<MK>(R, i), in.a.x, in.b.x); one(inside<MK>(R, i + 1), in.a.y, in.b.y); };
    pair_loop<4>(ctx, S->nslab, fetch, body);
    R3 r; r.a = s0; r.b = s1; r.c = mx;
    return r;
}

// gn = gn_raw / scaling; returns the smallest positive scaled value
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_scale_gn(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    const T* gr = S->gn_raw; T* gn = S->gn; const T scaling = S->scaling;
    const Region R = region_of<MK>(ctx, S);
    double vmin = INFINITY;
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(gr, i); return r; };
    auto body = [&](int i, const In1<T>& in) {
        const bool m0 = inside<MK>(R, i), m1 = inside<MK>(R, i + 1);
        const V2<T> v = mk2(m0 ? ndiv(in.a.x, scaling) : (T)0, m1 ? ndiv(in.a.y, scaling) : (T)0);
        st2(gn, i, v);
        if (m0 && v.x > (T)0 && (double)v.x < vmin) vmin = (double)v.x;
        if (m1 && v.y > (T)0 && (double)v.y < vmin) vmin = (double)v.y;
    };
    pair_loop<4>(ctx, S->nslab, fetch, body);
    return vmin;
}

// null-pixel fix, scaled background, start image; returns sum(gn - bkg)
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_init(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    T* gn = S->gn; T* bkgb = S->bkg; T* x = S->x; const T* br = S->bkg_raw; const T* x0 = S->x0_raw;
    const bool bimg = S->bkg_img != 0; const int init = S->init_recon;
    const T scaling = S->scaling, null_fill = S->null_fill, bkg_s = S->bkg_s, x_const = S->x_const;
    const Region R = region_of<MK>(ctx, S);
    double sum = 0.0;
    auto fetch = [&](int i) {
        In3<T> r; r.a = ld2(gn, i); r.b = bimg ? ld2(br, i) : mk2(bkg_s, bkg_s); r.c = (init == 1) ? ld2(x0, i) : mk2((T)0, (T)0);
        return r;
    };
    auto one = [&](bool m, T v0, T braw, T x0v, T& gfix, T& bk, T& xv) {
        if (!m) { gfix = (T)0; bk = (T)0; xv = (T)0; return; }
        gfix = (v0 <= (T)0) ? null_fill : v0;
        bk = bimg ? ndiv(braw, scaling) : bkg_s;
        sum += (double)nsub(gfix, bk);
        if (init == 0) xv = (T)0;
        else if (init == 1) xv = ndiv(x0v, scaling);
        else if (init == 2) xv = v0;                      // gn.copy() before the null-pixel fix (sgp.py:171)
        else xv = x_const;
    };
    auto body = [&](int i, const In3<T>& in) {
        V2<T> gf, bk, xv;
        one(inside<MK>(R, i), in.a.x, in.b.x, in.c.x, gf.x, bk.x, xv.x);
        one(inside<MK>(R, i + 1), in.a.y, in.b.y, in.c.y, gf.y, bk.y, xv.y);
        if (gf.x != in.a.x || gf.y != in.a.y) st2(gn, i, gf);
        if (bimg) st2(bkgb, i, bk);
        st2(x, i, xv);
    };
    pair_loop<4>(ctx, S->nslab, fetch, body);
    return sum;
}

// initial projection, step 1: pflag 0 -> x = max(x, 0); pflag 1 -> c = x (x_ones: X = 1)
template <typename T, class Ctx> BSGP_NOINLINE void ph_proj_init_load(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    T* x = S->x; T* cbuf = S->d; const bool pflag = S->pflag != 0;
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(x, i); return r; };
    auto body = [&](int i, const In1<T>& in) {
        if (pflag) st2(cbuf, i, in.a);
        else st2(x, i, mk2((in.a.x < (T)0) ? (T)0 : in.a.x, (in.a.y < (T)0) ? (T)0 : in.a.y));
    };
    pair_loop<4>(ctx, S->nslab, fetch, body);
}

// r(lambda) + b = sum_i x_i(lambda) over the slab; X = clip(x) is recomputed from x     flux_conserve_proj.py:22-25
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_proj_eval(Ctx ctx, const ImgState<T>* S, T lam) {
    ctx.sync();
    const T* cbuf = S->d; const T* x = S->x; const bool has_cap = S->has_cap != 0; const T cap = S->cap;
    const T xlo = S->xlo, xhi = S->xhi;
    const bool ones = S->x_ones != 0;
    const Region R = region_of<MK>(ctx, S);
    double s = 0.0;
    auto fetch = [&](int i) { In2<T> r; r.a = ld2(cbuf, i); r.b = ones ? mk2((T)0, (T)0) : ld2(x, i); return r; };
    auto X = [&](T xv) { return ones ? (T)1 : clip_bounds(xv, xlo, xhi); };
    auto body = [&](int i, const In2<T>& in) {
        if (inside<MK>(R, i)) s += (double)proj_point(in.a.x, X(in.b.x), lam, has_cap, cap);
        if (inside<MK>(R, i + 1)) s += (double)proj_point(in.a.y, X(in.b.y), lam, has_cap, cap);
    };
    pair_loop<BSGP_U_PE>(ctx, S->nslab, fetch, body);
    return s;
}

template <typename T, bool MK, class Ctx> BSGP_NOINLINE void ph_proj_init_store(Ctx ctx, const ImgState<T>* S, T lam) {
    ctx.sync();
    const T* cbuf = S->d; T* x = S->x; const bool has_cap = S->has_cap != 0; const T cap = S->cap;
    const Region R = region_of<MK>(ctx, S);
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(cbuf, i); return r; };
    auto body = [&](int i, const In1<T>& in) {
        st2(x, i, mk2(inside<MK>(R, i) ? proj_point(in.a.x, (T)1, lam, has_cap, cap) : (T)0,
                      inside<MK>(R, i + 1) ? proj_point(in.a.y, (T)1, lam, has_cap, cap) : (T)0));
    };
    pair_loop<4>(ctx, S->nslab, fetch, body);
}

// errflag, iteration 0: |x - obj|^2, |obj|^2                            sgp.py:240-244, 255-257
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R2 ph_err0(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    const T* truth = S->truth; const T* x = S->x; const T scaling = S->scaling;
    const Region R = region_of<MK>(ctx, S);
    double e0 = 0.0, e1 = 0.0;
    auto fetch = [&](int i) { In2<T> r; r.a = ld2(truth, i); r.b = ld2(x, i); return r; };
    auto one = [&](bool m, T tr, T xv) {
        if (!m) return;
        const T t = ndiv(tr, scaling);
        const T e = nsub(xv, t);
        e0 += (double)nmul(e, e);
        e1 += (double)nmul(t, t);
    };
    auto body = [&](int i, const In2<T>& in) { one(inside<MK>(R, i), in.a.x, in.b.x); one(inside<MK>(R, i + 1), in.a.y, in.b.y); };
    pair_loop<4>(ctx, S->nslab, fetch, body);
    R2 r; r.a = e0; r.b = e1;
    return r;
}

// -------------------------------------------------------------------------------------------------
// row passes of the PSF operator with the neighbouring elementwise work fused in.  `div` is the operator's
// output divisor: 1 for the circular operator, the kernel-weight constant of the zero-padded one.
// -------------------------------------------------------------------------------------------------
// producer: plain copy of x (which = 0) or gn (which = 1); both are zero in the padding
template <typename T, bool MK, class Ctx> BSGP_NOINLINE void ph_rf_copy(Ctx ctx, const ImgState<T>* S, int which) {
    ctx.sync();
    const T* src = which ? S->gn : S->x;
    auto pf = [&](int i) { In1<T> r; r.a = ld2(src, i); return r; };
    auto pe = [&](int, const In1<T>& in) -> V2<T> { return in.a; };
    conv_rows_forward<2, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, pf, pe);
}

// consumer of A(x): x_tf, objective terms, gradient cache                sgp.py:260-265 / 702-709
template <typename T, bool MK, int KIND, class Ctx> BSGP_NOINLINE R3 ph_ri_obj0_k(Ctx ctx, const ImgState<T>* S, DivK<T> dk) {
    const T* gn = S->gn; const T* bkgb = S->bkg; T* xtf = S->xtf; T* t1 = S->t1;
    const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s; const T div = S->div_a;
    const Region R = region_of<MK>(ctx, S);
    KSum acc[3];
    acc[0].clear(); acc[1].clear(); acc[2].clear();
    auto cf = [&](int i) { In2<T> r; r.a = ld2(gn, i); r.b = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); return r; };
    auto one = [&](bool m, T gnv, T bk, T v, T& xt, T& p) {
        if (!m) { xt = (T)0; p = (T)0; return; }
        xt = MK ? ndiv(v, div) : v;
        p = objective_pixel_k<KIND, Ctx::kSmall>(dk, gnv, nadd(xt, bk), xt, acc);
    };
    auto ca = [&](int i, const In2<T>& in, V2<T> v) {
        V2<T> xt, p;
        one(inside<MK>(R, i), in.a.x, in.b.x, v.x, xt.x, p.x);
        one(inside<MK>(R, i + 1), in.a.y, in.b.y, v.y, xt.y, p.y);
        st2(xtf, i, xt);
        st2(t1, i, p);
    };
    conv_rows_inverse<1, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, cf, ca);
    R3 r; r.a = acc[0].value(); r.b = acc[1].value(); r.c = acc[2].value();
    return r;
}

// producer of the gradient's A^T argument: gn/den (KL, cached) or gn*den^(beta-2) = gn*(den^(beta-1)/den).
// Unless F_FIRST, the accepted step is applied to x_tf on the way (x_tf += lam*d_tf, sgp.py:340).
template <typename T, bool MK, class Ctx> BSGP_NOINLINE void ph_rf_grad(Ctx ctx, const ImgState<T>* S, int kind, T lam, int flags) {
    ctx.sync();
    const T* gn = S->gn; const T* bkgb = S->bkg; T* xtf = S->xtf; const T* dtf = S->dtf; const T* t1 = S->t1;
    const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s; const bool first = (flags & F_FIRST) != 0;
    const Region R = region_of<MK>(ctx, S);
    auto pf = [&](int i) {
        In5<T> r; r.a = ld2(xtf, i); r.b = first ? mk2((T)0, (T)0) : ld2(dtf, i); r.c = ld2(t1, i);
        r.d = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); r.e = ld2(gn, i); return r;
    };
    auto pe = [&](int i, const In5<T>& in) -> V2<T> {
        V2<T> xt = in.a;
        if (!first) { xt = mk2(nadd(in.a.x, nmul(lam, in.b.x)), nadd(in.a.y, nmul(lam, in.b.y))); st2(xtf, i, xt); }
        if (kind == 0) return in.c;                        // the cache is zero in the padding
        return mk2(inside<MK>(R, i) ? nmul(in.e.x, ndiv(in.c.x, nadd(xt.x, in.d.x))) : (T)0,
                   inside<MK>(R, i + 1) ? nmul(in.e.y, ndiv(in.c.y, nadd(xt.y, in.d.y))) : (T)0);
    };
    conv_rows_forward<1, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, pf, pe);
}

// consumer: g = 1 - w (KL) or den^(beta-1) - w                            sgp.py:262 / 705
template <typename T, bool MK, class Ctx> BSGP_NOINLINE void ph_ri_grad0(Ctx ctx, const ImgState<T>* S, int kind) {
    const T* t1 = S->t1; T* gr = S->g; const T div = S->div_at;
    const Region R = region_of<MK>(ctx, S);
    auto cf = [&](int i) { In1<T> r; r.a = ld2(t1, i); return r; };
    auto one = [&](bool m, T p1, T w) -> T {
        if (!m) return (T)0;
        if (MK) w = ndiv(w, div);
        return (kind == 0) ? nsub((T)1, w) : nsub(p1, w);
    };
    auto ca = [&](int i, const In1<T>& in, V2<T> w) { st2(gr, i, mk2(one(inside<MK>(R, i), in.a.x, w.x), one(inside<MK>(R, i + 1), in.a.y, w.y))); };
    conv_rows_inverse<2, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, cf, ca);
}

// consumer: bounds of the scaling matrix from y = flux/(flux+bkg) * A^T(gn)     sgp.py:268-270 / 712-714
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R2 ph_ri_bounds(Ctx ctx, const ImgState<T>* S, double flux) {
    const T* bkgb = S->bkg; const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s; const T div = S->div_at;
    const Region R = region_of<MK>(ctx, S);
    double lo = INFINITY, hi = -INFINITY;
    auto cf = [&](int i) { In1<T> r; r.a = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); return r; };
    auto one = [&](bool m, T b, T w) {
        if (!m) return;
        if (MK) w = ndiv(w, div);
        const T ratio = (T)ndiv(flux, nadd(flux, (double)b));
        const double yv = (double)nmul(ratio, w);
        if (yv > 0.0 && yv < lo) lo = yv;
        if (yv > hi) hi = yv;
    };
    auto ca = [&](int i, const In1<T>& in, V2<T> w) { one(inside<MK>(R, i), in.a.x, w.x); one(inside<MK>(R, i + 1), in.a.y, w.y); };
    conv_rows_inverse<2, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, cf, ca);
    R2 r; r.a = lo; r.b = hi;
    return r;
}

// -------------------------------------------------------------------------------------------------
// iteration phases (sgp.py:302-425 / 748-882)
// -------------------------------------------------------------------------------------------------
// proj_type 1: X = clip(x), c = (x - alpha X g) / X                              sgp.py:311-316
// X is not stored: ph_proj_eval and ph_rf_dir recompute it from x.
// Also returns the slab sums of x(lambda) for lambda = 0, +1, -1: the root-find always starts with lambda = 0 and
// then tries +1 or -1 (flux_conserve_proj.py:7,22,33,58), so its first two evaluations need no pass of their own.
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R3 ph_trial_point(Ctx ctx, const ImgState<T>* S, T al) {
    ctx.sync();
    const T* x = S->x; const T* gr = S->g; T* cbuf = S->d;
    const T xlo = S->xlo, xhi = S->xhi, cap = S->cap;
    const bool has_cap = S->has_cap != 0, ones = S->x_ones != 0;
    const Region R = region_of<MK>(ctx, S);
    double s0 = 0.0, sp = 0.0, sm = 0.0;
    auto fetch = [&](int i) { In2<T> r; r.a = ld2(x, i); r.b = ld2(gr, i); return r; };
    auto one = [&](bool m, T xv, T gv) -> T {
        if (!m) return (T)0;
        const T X = ones ? (T)1 : clip_bounds(xv, xlo, xhi);
        const T y = nsub(xv, nmul(al, nmul(X, gv)));
        const T co = nmul(y, ndiv((T)1, X));
        s0 += (double)proj_point(co, X, (T)0, has_cap, cap);
        sp += (double)proj_point(co, X, (T)1, has_cap, cap);
        sm += (double)proj_point(co, X, (T)-1, has_cap, cap);
        return co;
    };
    auto body = [&](int i, const In2<T>& in) {
        st2(cbuf, i, mk2(one(inside<MK>(R, i), in.a.x, in.b.x), one(inside<MK>(R, i + 1), in.a.y, in.b.y)));
    };
    pair_loop<BSGP_U_TP>(ctx, S->nslab, fetch, body);
    R3 r; r.a = s0; r.b = sp; r.c = sm;
    return r;
}

// producer of A(d): d = y - x with y the projected trial point; returns the slab part of gd = d.g   sgp.py:311-321
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_rf_dir(Ctx ctx, const ImgState<T>* S, T al, T lam_proj) {
    ctx.sync();
    const T* x = S->x; const T* gr = S->g; T* dbuf = S->d;
    const T xlo = S->xlo, xhi = S->xhi, cap = S->cap;
    const bool has_cap = S->has_cap != 0, pflag = S->pflag != 0, ones = S->x_ones != 0;
    const Region R = region_of<MK>(ctx, S);
    double gd = 0.0;
    auto pf = [&](int i) { In3<T> r; r.a = ld2(x, i); r.b = ld2(gr, i); r.c = pflag ? ld2(dbuf, i) : mk2((T)0, (T)0); return r; };
    auto one = [&](bool m, T xv, T gv, T cv) -> T {
        if (!m) return (T)0;
        const T X = ones ? (T)1 : clip_bounds(xv, xlo, xhi);
        T y;
        if (pflag) {
            y = proj_point(cv, X, lam_proj, has_cap, cap);
        } else {
            y = nsub(xv, nmul(al, nmul(X, gv)));
            y = (y < (T)0) ? (T)0 : y;
        }
        const T d = nsub(y, xv);
        gd += (double)nmul(d, gv);
        return d;
    };
    auto pe = [&](int i, const In3<T>& in) -> V2<T> {
        const V2<T> d = mk2(one(inside<MK>(R, i), in.a.x, in.b.x, in.c.x), one(inside<MK>(R, i + 1), in.a.y, in.b.y, in.c.y));
        st2(dbuf, i, d);
        return d;
    };
    conv_rows_forward<1, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, pf, pe);
    return gd;
}

// consumer of A(d): d_tf, first line-search trial (lam = 1) fused            sgp.py:326-334
template <typename T, bool MK, int KIND, class Ctx> BSGP_NOINLINE R3 ph_ri_trial_k(Ctx ctx, const ImgState<T>* S, DivK<T> dk) {
    const T* gn = S->gn; const T* bkgb = S->bkg; const T* xtf = S->xtf; T* dtf = S->dtf; T* t1 = S->t1;
    const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s; const T div = S->div_a;
    const Region R = region_of<MK>(ctx, S);
    KSum acc[3];
    acc[0].clear(); acc[1].clear(); acc[2].clear();
    auto cf = [&](int i) { In3<T> r; r.a = ld2(xtf, i); r.b = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); r.c = ld2(gn, i); return r; };
    auto one = [&](bool m, T xtfv, T bk, T gnv, T v, T& dt, T& p) {
        if (!m) { dt = (T)0; p = (T)0; return; }
        dt = MK ? ndiv(v, div) : v;
        const T xt = nadd(xtfv, dt);                       // lam = 1
        p = objective_pixel_k<KIND, Ctx::kSmall>(dk, gnv, nadd(xt, bk), xt, acc);
    };
    auto ca = [&](int i, const In3<T>& in, V2<T> v) {
        V2<T> dt, p;
        one(inside<MK>(R, i), in.a.x, in.b.x, in.c.x, v.x, dt.x, p.x);
        one(inside<MK>(R, i + 1), in.a.y, in.b.y, in.c.y, v.y, dt.y, p.y);
        st2(dtf, i, dt);
        st2(t1, i, p);
    };
    conv_rows_inverse<1, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, cf, ca);
    R3 r; r.a = acc[0].value(); r.b = acc[1].value(); r.c = acc[2].value();
    return r;
}

// slab part of s1 = sum k * gn^beta, the data-only term of the generic beta-divergence       sgp.py:457
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_s1(Ctx ctx, const ImgState<T>* S, T k, T b) {
    ctx.sync();
    const T* gn = S->gn;
    const Region R = region_of<MK>(ctx, S);
    KSum acc;
    acc.clear();
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(gn, i); return r; };
    auto body = [&](int i, const In1<T>& in) {
        if (inside<MK>(R, i)) acc.add((double)nmul(k, mpow_sel<Ctx::kSmall>(in.a.x, b)));
        if (inside<MK>(R, i + 1)) acc.add((double)nmul(k, mpow_sel<Ctx::kSmall>(in.a.y, b)));
    };
    pair_loop<1>(ctx, S->nslab, fetch, body);
    return acc.value();
}

// slab part of sum dD_beta/dbeta at the rejected trial point               sgp.py:798-800
template <typename T, bool MK, class Ctx> BSGP_NOINLINE double ph_dbeta(Ctx ctx, const ImgState<T>* S, T lam, T b) {
    ctx.sync();
    const T* gn = S->gn; const T* bkgb = S->bkg; const T* xtf = S->xtf; const T* dtf = S->dtf;
    const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s;
    const Region R = region_of<MK>(ctx, S);
    double db = 0.0;
    auto fetch = [&](int i) {
        In4<T> r; r.a = ld2(xtf, i); r.b = ld2(dtf, i); r.c = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); r.d = ld2(gn, i); return r;
    };
    auto body = [&](int i, const In4<T>& in) {
        if (inside<MK>(R, i)) db += (double)dbeta_pixel<Ctx::kSmall>(in.d.x, nadd(nadd(in.a.x, nmul(lam, in.b.x)), in.c.x), b);
        if (inside<MK>(R, i + 1)) db += (double)dbeta_pixel<Ctx::kSmall>(in.d.y, nadd(nadd(in.a.y, nmul(lam, in.b.y)), in.c.y), b);
    };
    pair_loop<1>(ctx, S->nslab, fetch, body);
    return db;
}

// one more line-search trial: objective at x_tf + lam d_tf                  sgp.py:329-334
template <typename T, bool MK, int KIND, class Ctx> BSGP_NOINLINE R3 ph_trial_k(Ctx ctx, const ImgState<T>* S, T lam, DivK<T> dk) {
    ctx.sync();
    const T* gn = S->gn; const T* bkgb = S->bkg; const T* xtf = S->xtf; const T* dtf = S->dtf; T* t1 = S->t1;
    const bool bimg = S->bkg_img != 0; const T bkg_s = S->bkg_s;
    const Region R = region_of<MK>(ctx, S);
    KSum acc[3];
    acc[0].clear(); acc[1].clear(); acc[2].clear();
    auto fetch = [&](int i) {
        In4<T> r; r.a = ld2(xtf, i); r.b = ld2(dtf, i); r.c = bimg ? ld2(bkgb, i) : mk2(bkg_s, bkg_s); r.d = ld2(gn, i); return r;
    };
    auto one = [&](bool m, T xtfv, T dtfv, T bk, T gnv) -> T {
        if (!m) return (T)0;
        const T xt = nadd(xtfv, nmul(lam, dtfv));
        return objective_pixel_k<KIND, Ctx::kSmall>(dk, gnv, nadd(xt, bk), xt, acc);
    };
    auto body = [&](int i, const In4<T>& in) {
        V2<T> p;
        p.x = one(inside<MK>(R, i), in.a.x, in.b.x, in.c.x, in.d.x);
        p.y = one(inside<MK>(R, i + 1), in.a.y, in.b.y, in.c.y, in.d.y);
        st2(t1, i, p);
    };
    pair_loop<BSGP_U_TRIAL>(ctx, S->nslab, fetch, body);
    R3 r; r.a = acc[0].value(); r.b = acc[1].value(); r.c = acc[2].value();
    return r;
}

// Iterate snapshots (RowArgs::snap): the slot one phase stores x * scaling into, like ph_store_out.  crop: the slot holds
// the valid window [reg0, reg1) x [reg2, reg3) row by row (masked kernels only), else the whole grid.
template <typename T> struct SnapDst { T* dst; int crop; };
struct NoSnap {};
template <bool MK, typename T, class Ctx>
BSGP_DEV void snap_store2(const Ctx& ctx, const ImgState<T>* S, const Region& R, const SnapDst<T>& sn, int i, V2<T> v) {
    const T scaling = S->scaling;
    const V2<T> o = mk2(nmul(v.x, scaling), nmul(v.y, scaling));
    if constexpr (MK) {
        if (sn.crop) {
            const size_t w = (size_t)(R.c1 - R.c0);
            const int row = R.row_off + (i >> R.lg_nx), col = i & R.colmask;      // i is even: both pixels share the row
            if (inside<MK>(R, i)) sn.dst[(size_t)(row - R.r0) * w + (size_t)(col - R.c0)] = o.x;
            if (inside<MK>(R, i + 1)) sn.dst[(size_t)(row - R.r0) * w + (size_t)(col + 1 - R.c0)] = o.y;
            return;
        }
    }
    st2(sn.dst + (size_t)ctx.rank * S->nslab, i, o);
}
template <bool MK, typename T, class Ctx> BSGP_DEV void snap_store2(const Ctx&, const ImgState<T>*, const Region&, const NoSnap&, int, V2<T>) {}

// consumer of A^T(.): new gradient, y_k, Barzilai-Borwein sums, stop-rule / error sums   sgp.py:343-365, 394-402
// The next iterate x + lam*d goes into the d array (d is dead after this pass); the controller swaps the x and d
// pointers when the loop continues, so x keeps the previous iterate when it stops.  ph_ri_bb_snap (mixed-batch kernels,
// on the passes that take a snapshot) also stores that iterate into the snapshot slot `sn`.
template <typename T, bool MK, class Ctx, class Sn> BSGP_DEV R7 ri_bb_body(Ctx& ctx, const ImgState<T>* S, T lam, int kind, const Sn& sn) {
    const T* t1 = S->t1; T* gr = S->g; T* dbuf = S->d; const T* x = S->x; const T* truth = S->truth;
    const T xlo = S->xlo, xhi = S->xhi, scaling = S->scaling, div = S->div_at;
    const bool want_err = S->want_err != 0, stop2 = S->stop2 != 0;
    const Region R = region_of<MK>(ctx, S);
    double bb[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) bb[k] = 0.0;
    auto cf = [&](int i) {
        In5<T> r; r.a = ld2(t1, i); r.b = ld2(gr, i); r.c = ld2(dbuf, i); r.d = ld2(x, i);
        r.e = want_err ? ld2(truth, i) : mk2((T)0, (T)0); return r;
    };
    auto one = [&](bool m, T p1, T gold, T dv, T xv, T tr, T w, T& xo) -> T {
        if (!m) { xo = (T)0; return (T)0; }
        if (MK) w = ndiv(w, div);
        const T gnew = (kind == 0) ? nsub((T)1, w) : nsub(p1, w);
        const T yk = nsub(gnew, gold);
        const T sk = nmul(lam, dv);
        const T xn = nadd(xv, sk);                                // x + lam*d (:329,337)
        const T X = clip_bounds(xn, xlo, xhi);
        const T sk2 = nmul(sk, ndiv((T)1, X));
        const T yk2 = nmul(yk, X);
        bb[0] += (double)sk2 * (double)yk;
        bb[1] += (double)yk2 * (double)sk;
        bb[2] += (double)sk2 * (double)sk2;
        bb[3] += (double)yk2 * (double)yk2;
        if (stop2) { bb[4] += (double)sk * (double)sk; bb[5] += (double)xn * (double)xn; }
        if (want_err) { const T e = nsub(xn, ndiv(tr, scaling)); bb[6] += (double)nmul(e, e); }
        xo = xn;
        return gnew;
    };
    auto ca = [&](int i, const In5<T>& in, V2<T> w) {
        V2<T> gnew, xn;
        gnew.x = one(inside<MK>(R, i), in.a.x, in.b.x, in.c.x, in.d.x, in.e.x, w.x, xn.x);
        gnew.y = one(inside<MK>(R, i + 1), in.a.y, in.b.y, in.c.y, in.d.y, in.e.y, w.y, xn.y);
        st2(gr, i, gnew);
        st2(dbuf, i, xn);
        snap_store2<MK>(ctx, S, R, sn, i, xn);
    };
    conv_rows_inverse<1, MK>(ctx, S->geom, S->ws_off, S->twx, S->twx_off, S->tw_split, S->ppx_off, S->spec, cf, ca);
    R7 r;
#pragma unroll
    for (int k = 0; k < 7; ++k) r.v[k] = bb[k];
    return r;
}
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R7 ph_ri_bb(Ctx ctx, const ImgState<T>* S, T lam, int kind) {
    return ri_bb_body<T, MK>(ctx, S, lam, kind, NoSnap{});
}
template <typename T, bool MK, class Ctx> BSGP_NOINLINE R7 ph_ri_bb_snap(Ctx ctx, const ImgState<T>* S, T lam, int kind, SnapDst<T> sn) {
    return ri_bb_body<T, MK>(ctx, S, lam, kind, sn);
}

// snapshot slot 0: the start image after the initial projection (mixed-batch kernels only)
template <typename T, bool MK, class Ctx> BSGP_NOINLINE void ph_store_snap(Ctx ctx, const ImgState<T>* S, SnapDst<T> sn) {
    ctx.sync();
    const T* x = S->x;
    const Region R = region_of<MK>(ctx, S);
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(x, i); return r; };
    auto body = [&](int i, const In1<T>& in) { snap_store2<MK>(ctx, S, R, sn, i, in.a); };
    pair_loop<4>(ctx, S->nslab, fetch, body);
}

// where solve `img` keeps snapshot slot j (RowArgs::snap)
template <typename T> BSGP_DEV SnapDst<T> snap_slot(const SolveArgs<T>& a, const RowArgs& ra, int img, int j) {
    const int* r = a.p.region;
    const size_t per = ra.snap_crop ? (size_t)(r[1] - r[0]) * (size_t)(r[3] - r[2]) : (size_t)a.g.ny * a.g.nx;
    SnapDst<T> sn;
    sn.dst = (T*)ra.snap + ((size_t)img * ra.n_snap + (size_t)j) * per;
    sn.crop = ra.snap_crop;
    return sn;
}

// x_out = x * scaling                                                        sgp.py:428
template <typename T, class Ctx> BSGP_NOINLINE void ph_store_out(Ctx ctx, const ImgState<T>* S) {
    ctx.sync();
    const T* x = S->x; T* out = S->x_out; const T scaling = S->scaling;
    auto fetch = [&](int i) { In1<T> r; r.a = ld2(x, i); return r; };
    auto body = [&](int i, const In1<T>& in) { st2(out, i, mk2(nmul(in.a.x, scaling), nmul(in.a.y, scaling))); };
    pair_loop<4>(ctx, S->nslab, fetch, body);
}

// the two column passes between a producer and a consumer
template <typename T, bool MK, class Ctx> BSGP_DEV void conv_middle(Ctx& ctx, const ImgState<T>* S, cplx<T>* tf, int mode) {
    ctx.cluster_sync();
    conv_cols<MK>(ctx, &S->geom, S->ws_off, S->twy, S->twy_off, S->tw_split, S->spec, tf, mode);
    ctx.cluster_sync();
}

// -------------------------------------------------------------------------------------------------
// the controller
// -------------------------------------------------------------------------------------------------
// Controller scalars of one solve.  Every lane of every warp runs the scalar controller redundantly on bit-identical
// all-reduced sums (uniform control flow, nothing is broadcast), but its state does not live in registers: each WARP
// owns one copy of this block in shared memory (Ctx::ctl) and all of its lanes store the same values to it.  Nothing of
// the controller is therefore alive in registers across the calls of the non-inlined phases, reductions and root-find
// (round 1: ~100 live scalars, 260 M local-memory loads per launch that missed the carved-out L1), and those callees can
// be real functions instead of 40 inlined copies (the kernel's main body shrank from 18.5 k to a few thousand
// instructions).  A warp never reads another warp's copy, so no barrier orders the accesses; within a warp every lane
// reads back what it, or a lane in lock step with it, has just written.
template <typename T> struct CtlState {
    double flux, tol, discr_coeff, npix_d, truth_sq, t_start, sum_raw;
    double alpha, tau, lr, beta_p, s1, fv, x_low, x_upp, f_prev, lam, gd, f_ref;
    double pre[3];                                   // sums of x(lambda) at lambda = 0, +1, -1 delivered by ph_trial_point
    double alpha_hist[kMaxMem], f_hist[kMaxMem];     // Valpha / Fold (sgp.py:214-215)
    DivK<T> dk;
    T al, lam_proj;
    int status, total_evals, total_trials, iter, trials, evals;
    int have_pre, s1_valid, keep_going;
};

// all-reduce of K doubles as a real function (the execution context travels by value, its parity comes back)
template <int K> struct ArOut { double v[K]; int parity; };
template <int OP, int K, class Ctx> BSGP_NOINLINE ArOut<K> ar_call(Ctx ctx, ArOut<K> io) {
    ctx.allreduce(OP, io.v, K);
    io.parity = ctx.parity;
    return io;
}
// small-image kernels: every sum of two or more values goes through one eight-wide function (DeviceCtxSmall::allreduce_sum8)
template <class Ctx> BSGP_NOINLINE ArOut<8> ar_sum8_call(Ctx ctx, ArOut<8> io) {
    ctx.allreduce_sum8(io.v);
    io.parity = ctx.parity;
    return io;
}
template <int OP, int K, class Ctx> BSGP_DEV void allreduce_fn(Ctx& ctx, double* v) {
    if constexpr (Ctx::kSmall && OP == 0 && K > 1) {
        ArOut<8> io;
#pragma unroll
        for (int j = 0; j < 8; ++j) io.v[j] = j < K ? v[j] : 0.0;
        io.parity = 0;
        io = ar_sum8_call(ctx, io);
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = io.v[j];
        ctx.parity = io.parity;
    } else {
        ArOut<K> io;
#pragma unroll
        for (int j = 0; j < K; ++j) io.v[j] = v[j];
        io.parity = 0;
        io = ar_call<OP, K>(ctx, io);
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = io.v[j];
        ctx.parity = io.parity;
    }
}

// The projection root-find of one call (initial projection or one iteration), as a real function: the residual
// r(lambda) = sum_i x_i(lambda) - flux comes from the fused sums of ph_trial_point where it can, else from one pass.
struct RfOut { ProjResult pr; int parity; };
template <typename T, bool MK, class Ctx> BSGP_NOINLINE RfOut rootfind_call(Ctx ctx, const ImgState<T>* S, const CtlState<T>* W, int max_projs) {
    const double flux = W->flux;
    const bool have_pre = W->have_pre != 0;
    const double p0 = W->pre[0], p1 = W->pre[1], p2 = W->pre[2];
    auto proj_eval = [&](double lam) -> double {
        if (have_pre) {
            if (lam == 0.0) return p0 - flux;
            if (lam == 1.0) return p1 - flux;
            if (lam == -1.0) return p2 - flux;
        }
        double s = ph_proj_eval<T, MK>(ctx, S, (T)lam);
        allreduce_fn<0, 1>(ctx, &s);
        return s - flux;
    };
    RfOut out;
    out.pr = flux_rootfind(proj_eval, flux, max_projs);
    out.parity = ctx.parity;
    return out;
}

// Barzilai-Borwein steps and their alternation, learning-rate schedule, bookkeeping and stop rules of one iteration
// (sgp.py:366-425 / 818-882).  bb: the seven all-reduced sums of ph_ri_bb.  Returns the value compared with tol.
// ROWS only separates the instantiations of the kernels with and without rows (bsgp_solve_kernel.cuh, RowCtx)
template <typename T, bool ROWS = false> BSGP_NOINLINE double ctl_finish_iteration(const bsgp_params* Pp, CtlState<T>* W, R7 bbr) {
    const bsgp_params& P = *Pp;
    const double* bb = bbr.v;
    const int MA = P.m_alpha;
    const double alpha_prev = W->alpha;
    const double bk = bb[0], ck = bb[1];
    double a1, a2;
    if (bk <= 0.0) a1 = py_min(nmul(10.0, alpha_prev), P.alpha_max);
    else a1 = py_min(P.alpha_max, py_max(P.alpha_min, bb[2] / bk));
    if (ck <= 0.0) a2 = py_min(nmul(10.0, alpha_prev), P.alpha_max);
    else a2 = py_min(P.alpha_max, py_max(P.alpha_min, ck / bb[3]));
    W->alpha_hist[MA - 1] = a2;
    double amin = W->alpha_hist[0];
    for (int k = 1; k < MA; ++k) amin = py_min(amin, W->alpha_hist[k]);
    const int iter = W->iter;
    double tau = W->tau, alpha;
    if (iter <= 20) alpha = amin;
    else if (a2 / a1 < tau) { alpha = amin; tau = nmul(tau, 0.9); }
    else { alpha = a1; tau = nmul(tau, 1.1); }
    W->alpha = alpha; W->tau = tau;
    if (P.divergence == BSGP_DIV_BETA && P.schedule_lr) W->lr = nmul(P.lr, exp(nmul(-P.lr_exp_param, (double)iter)));   // :842-844, epoch == iter
    // ---- bookkeeping and stop rules (:390-425)
    const int it1 = iter + 1;
    W->iter = it1;
    const double fv = W->fv;
    double stop_val = 0.0;
    int keep_going = 1;
    if (P.stop_criterion == 2) {
        stop_val = bb[4] / bb[5];
        keep_going = stop_val > W->tol;
    } else if (P.stop_criterion == 3) {
        stop_val = (W->f_prev - fv) / fv;
        keep_going = (stop_val > W->tol) && (stop_val >= 0.0);
    } else if (P.stop_criterion == 4) {
        stop_val = nmul(W->discr_coeff, fv);
        keep_going = stop_val > W->tol;
    }
    if (it1 > P.maxit) keep_going = 0;
    W->keep_going = keep_going;
    return stop_val;
}

// x <- x + lam*d: ph_ri_bb has stored the new iterate in the d array, so the x and d arrays swap roles.  When the loop stops
// nothing is swapped and x still holds the previous iterate, which is what the reference returns (sgp.py:424-425).  Only
// thread 0 of each CTA writes S: every thread read it before the all-reduce that followed ph_ri_bb, and the next phase
// opens with a barrier.  A real function: a thread-index test in the controller's loop costs it registers across every
// phase call.
template <typename T, class Ctx> BSGP_NOINLINE void ctl_accept_step(Ctx ctx, ImgState<T>* S, int keep_going) {
    if (ctx.tid != 0) return;
    S->x_ones = 0;
    if (keep_going) { T* t = S->x; S->x = S->d; S->d = t; }
}

template <typename T, bool MK, bool ROWS = false, class Ctx>
BSGP_DEV void solve_image(Ctx& ctx, const SolveArgs<T>& a, ImgState<T>* S, T* const* buf, cplx<T>* tf, cplx<T>* tf_adj, int img,
                          const RowArgs& ra = RowArgs{}) {
    // A mixed batch: every thread keeps its own copy of the image's row, in local memory (its address reaches
    // ctl_finish_iteration), the way a launch without rows reads SolveArgs::p.  The operator fields are equal in every row
    // (bsgp_rows.h) and always come from a.p, where a wrapped plan sets them for its grid.
    typename std::conditional<ROWS, bsgp_params, NoRow>::type own;
    if constexpr (ROWS) {
        own = ra.rows[img];
        for (int k = 0; k < 4; ++k) own.region[k] = a.p.region[k];
        own.div_a = a.p.div_a; own.div_at = a.p.div_at; own.adjoint_second_psf = a.p.adjoint_second_psf;
    }
    const bsgp_params& P = image_params(own, a.p);
    CtlState<T>* W = ctx.template ctl<CtlState<T>>();
    constexpr bool masked = MK;                                          // zero-padded operator: the image is a window of the grid
    const bool leader = (ctx.rank == 0 && ctx.tid == 0);
    const bool pflag = P.proj_type == 1;
    const bool is_beta = P.divergence == BSGP_DIV_BETA;
    const bool want_err = P.errflag && a.obj != nullptr && a.err != nullptr;
    const size_t stride = ROWS ? (size_t)ra.trace_stride : (size_t)(P.maxit + 1);
    const size_t toff = (size_t)img * stride;

    ctx.sync();                      // the previous image's last phase may still be reading S
    {
        const int nslab = a.g.rows_per_cta * a.g.nx;
        const size_t npix = (size_t)a.g.ny * a.g.nx;
        // inputs at the offset of the observation the solve reads, the restored image at the solve's own
        int obs = img;
        if constexpr (ROWS) obs = source_of(img, ra);
        const size_t goff = (size_t)obs * npix + (size_t)ctx.rank * nslab;
        const size_t xoff = (size_t)img * npix + (size_t)ctx.rank * nslab;
        const bool bkg_img = a.bkg_is_image != 0;
        const T bkg_raw_s = bkg_img ? (T)0 : a.bkg[obs];
        if (ctx.tid == 0) {
            S->gn = buf[B_GN]; S->bkg = buf[B_BKG]; S->x = buf[B_X]; S->g = buf[B_G];
            S->xtf = buf[B_XTF]; S->d = buf[B_D]; S->dtf = buf[B_DTF]; S->t1 = buf[B_T1];
            S->gn_raw = a.gn + goff;
            S->bkg_raw = bkg_img ? a.bkg + goff : a.gn + goff;             // never dereferenced when !bkg_img
            S->x0_raw = (P.init_recon == 1) ? a.x0 + goff : a.gn + goff;
            S->truth = want_err ? a.obj + goff : a.gn + goff;
            S->x_out = a.x_out + xoff;
            S->tf = tf;
            // A^T: conj(TF) of the same PSF (sgp.py:110), or the spectrum of a second kernel, psf.conj().T (sgp.py:157)
            S->tf_at = P.adjoint_second_psf ? tf_adj : tf;
            S->nslab = nslab; S->bkg_img = bkg_img; S->init_recon = P.init_recon; S->has_cap = P.has_sat != 0;
            S->pflag = pflag; S->want_err = want_err; S->stop2 = (P.stop_criterion == 2);
            S->x_ones = 1;                                                  // the initial projection: c = x, X = 1
            S->bkg_raw_s = bkg_raw_s;
            S->masked = masked; S->reg[0] = P.region[0]; S->reg[1] = P.region[1]; S->reg[2] = P.region[2]; S->reg[3] = P.region[3];
            S->div_a = masked ? (T)P.div_a : (T)1; S->div_at = masked ? (T)P.div_at : (T)1;
        }
        W->npix_d = masked ? (double)(P.region[1] - P.region[0]) * (double)(P.region[3] - P.region[2]) : (double)npix;
        W->t_start = ctx.now();
    }
    const int mode_at = P.adjoint_second_psf ? CONV_TF : CONV_CTF;

    // ------------------------------------------------------------------ setup (sgp.py:166-217)
    {
        const R3 st = ph_stats<T, MK>(ctx, S);
        double v2[2] = {st.a, st.b};
        double mx = st.c;
        allreduce_fn<0, 2>(ctx, v2);
        allreduce_fn<2, 1>(ctx, &mx);
        const T scaling = P.scale_data ? (T)mx : (T)1;
        const T bkg_s = ndiv(S->bkg_raw_s, scaling);
        if (ctx.tid == 0) { S->scaling = scaling; S->bkg_s = bkg_s; }
        W->sum_raw = v2[0];
        W->flux = v2[1];                                                 // sum(gn - bkg) of the raw data, until ph_init refines it
    }
    {
        double vmin = ph_scale_gn<T, MK>(ctx, S);
        allreduce_fn<1, 1>(ctx, &vmin);
        const T eps = Eps<T>::v();
        const T scaling = S->scaling;
        const double flux_in = P.has_flux ? a.flux[img] : 0.0;
        if (ctx.tid == 0) {
            S->null_fill = nmul(nmul((T)vmin, eps), eps);
            S->x_const = ndiv(nmul((T)ndiv(P.has_flux ? flux_in : W->flux, W->npix_d), (T)1), scaling);
            S->cap = (P.has_sat != 0) ? nsub(ndiv((T)P.ccd_sat_level, scaling), eps) : (T)0;
            S->xlo = (T)0; S->xhi = (T)0;
        }
        double v1 = ph_init<T, MK>(ctx, S);
        allreduce_fn<0, 1>(ctx, &v1);
        W->flux = P.has_flux ? ndiv(flux_in, (double)scaling) : v1;

        double tol = 0.0;                                                   // sgp.py:185-190, 291-294
        if (P.stop_criterion == 2 || P.stop_criterion == 3) tol = P.tol_convergence;
        else if (P.stop_criterion == 4) tol = 1.0 + 1.0 / (W->sum_raw / W->npix_d);
        if (P.verbose && P.stop_criterion == 2) tol = nmul(tol, tol);
        W->tol = tol;
        W->discr_coeff = nmul(2.0 / W->npix_d, (double)scaling);
    }
    W->status = BSGP_ST_OK;
    W->total_evals = 0; W->total_trials = 0;
    W->have_pre = 0;
    if (pflag && !(W->flux > 0.0 && is_finite(W->flux))) W->status = BSGP_ST_BAD_FLUX;

    // ------------------------------------------------------------------ initial projection (:248-253)
    if (W->status == BSGP_ST_OK) {
        ph_proj_init_load<T>(ctx, S);
        if (pflag) {
            const RfOut rf = rootfind_call<T, MK>(ctx, S, W, P.max_projs);
            ctx.parity = rf.parity;
            const ProjResult pr = rf.pr;
            W->total_evals += pr.evals;
            if (pr.status != PROJ_OK) W->status = BSGP_ST_PROJ_NO_BRACKET;
            ph_proj_init_store<T, MK>(ctx, S, (T)pr.lambda);
        }
    }
    if constexpr (ROWS) {
        if (ra.snap) ph_store_snap<T, MK>(ctx, S, snap_slot(a, ra, img, 0));     // slot 0: what MAXIT = 1 returns
    }

    W->truth_sq = 1.0;
    if (want_err && W->status == BSGP_ST_OK) {                          // :240-244, 255-257
        const R2 e = ph_err0<T, MK>(ctx, S);
        double e2[2] = {e.a, e.b};
        allreduce_fn<0, 2>(ctx, e2);
        W->truth_sq = e2[1];
        if (leader) a.err[(size_t)img * (stride + 1)] = sqrt(e2[0] / e2[1]);
    }

    W->beta_p = is_beta ? a.beta0[img] : 1.0;
    W->dk = make_divk<T>(P.divergence, W->beta_p);
    W->s1 = 0.0;              // sum k*gn^beta for the current beta
    W->s1_valid = 0;
    auto refresh_s1 = [&]() {                                            // after beta changed (and once at the start)
        if (W->dk.kind == 1 && !W->s1_valid) {
            double s = ph_s1<T, MK>(ctx, S, W->dk.k, W->dk.b);
            allreduce_fn<0, 1>(ctx, &s);
            W->s1 = s; W->s1_valid = 1;
        }
    };
    W->fv = 0.0; W->x_low = 0.0; W->x_upp = 0.0;

    if (W->status == BSGP_ST_OK) {
        // ---------------------------------------------------------------- x_tf = A(x), objective (:260-265)
        ph_rf_copy<T, MK>(ctx, S, 0);
        conv_middle<T, MK>(ctx, S, S->tf, CONV_TF);
        double acc[3];
        {
            const R3 o = BSGP_DISPATCH_KIND(W->dk, ph_ri_obj0_k, ctx, S, W->dk);
            acc[0] = o.a; acc[1] = o.b; acc[2] = o.c;
        }
        allreduce_fn<0, 3>(ctx, acc);
        refresh_s1();
        W->fv = objective_value(W->dk, acc, W->s1, W->flux, W->npix_d);
        // ---------------------------------------------------------------- gradient
        ph_rf_grad<T, MK>(ctx, S, W->dk.kind, (T)0, F_FIRST);
        conv_middle<T, MK>(ctx, S, S->tf_at, mode_at);
        ph_ri_grad0<T, MK>(ctx, S, W->dk.kind);
        // ---------------------------------------------------------------- scaling-matrix bounds (:268-273)
        ph_rf_copy<T, MK>(ctx, S, 1);
        conv_middle<T, MK>(ctx, S, S->tf_at, mode_at);
        const R2 lh = ph_ri_bounds<T, MK>(ctx, S, W->flux);
        double lo = lh.a, hi = lh.b;
        allreduce_fn<1, 1>(ctx, &lo);
        allreduce_fn<2, 1>(ctx, &hi);
        if (!(lo < INFINITY)) W->status = BSGP_ST_EMPTY_BOUNDS;
        double x_low = lo, x_upp = hi;
        if (x_upp / x_low < 50.0) { x_low = x_low / 10.0; x_upp = x_upp * 10.0; }
        W->x_low = x_low; W->x_upp = x_upp;
        if (ctx.tid == 0) { S->xlo = (T)x_low; S->xhi = (T)x_upp; }
    }

    if (leader) {
        a.discr[toff] = nmul(W->discr_coeff, W->fv);
        a.times[toff] = 0.0;
        if (a.stop_value) a.stop_value[toff] = 0.0;
    }

    // ------------------------------------------------------------------ main loop (sgp.py:302-425)
    W->alpha = P.alpha; W->tau = P.tau; W->lr = P.lr;
    {
        const int M = P.m, MA = P.m_alpha;
        for (int k = 0; k < MA; ++k) W->alpha_hist[k] = P.alpha_max;
        for (int k = 0; k < M; ++k) W->f_hist[k] = -1e30;
    }
    if (ctx.tid == 0) S->x_ones = (P.init_recon == 0);                 // X = 1 in the first iteration from a zero start
    W->iter = 1;
    W->keep_going = (W->status == BSGP_ST_OK);

    while (W->keep_going) {
        // history shift (:306-308)
        {
            const int M = P.m, MA = P.m_alpha;
            for (int k = 0; k < MA - 1; ++k) W->alpha_hist[k] = W->alpha_hist[k + 1];
            for (int k = 0; k < M - 1; ++k) W->f_hist[k] = W->f_hist[k + 1];
            W->f_hist[M - 1] = W->fv;
            W->f_prev = W->fv;
        }

        // ---- trial point y = x - alpha X g, projection (:311-318)
        W->al = (T)W->alpha;
        W->evals = 0;
        W->lam_proj = (T)0;
        if (pflag) {
            {
                const R3 t = ph_trial_point<T, MK>(ctx, S, W->al);
                double pre[3] = {t.a, t.b, t.c};
                allreduce_fn<0, 3>(ctx, pre);
                W->pre[0] = pre[0]; W->pre[1] = pre[1]; W->pre[2] = pre[2];
                W->have_pre = 1;
            }
            const RfOut rf = rootfind_call<T, MK>(ctx, S, W, P.max_projs);
            ctx.parity = rf.parity;
            const ProjResult pr = rf.pr;
            W->evals = pr.evals;
            W->total_evals += pr.evals;
            if (pr.status != PROJ_OK) { W->status = BSGP_ST_PROJ_NO_BRACKET; break; }
            W->lam_proj = (T)pr.lambda;
        }

        // ---- d = y - x, gd = d.g, d_tf = A(d) with the first line-search trial fused (:318-334)
        {
            double sums[4];   // [0..2] objective terms, [3] gd
            sums[3] = ph_rf_dir<T, MK>(ctx, S, W->al, W->lam_proj);
            conv_middle<T, MK>(ctx, S, S->tf, CONV_TF);
            {
                const R3 o = BSGP_DISPATCH_KIND(W->dk, ph_ri_trial_k, ctx, S, W->dk);
                sums[0] = o.a; sums[1] = o.b; sums[2] = o.c;
            }
            allreduce_fn<0, 4>(ctx, sums);
            W->gd = sums[3];
            refresh_s1();
            W->fv = objective_value(W->dk, sums, W->s1, W->flux, W->npix_d);
            const int M = P.m;
            double f_ref = W->f_hist[0];                                     // fr = max(Fold)
            for (int k = 1; k < M; ++k) f_ref = py_max(f_ref, W->f_hist[k]);
            W->f_ref = f_ref;
        }
        W->lam = 1.0;
        W->trials = 1;
        // ---- backtracking (:328-349 / :776-800): accept iff fv <= fr + gamma*lam*gd or lam < 1e-12
        while (!(W->fv <= nadd(W->f_ref, nmul(nmul(P.gamma, W->lam), W->gd)) || W->lam < 1e-12)) {
            if (is_beta && P.adapt_beta && W->dk.kind == 1) {               // :798-800, den of the rejected trial
                double db = ph_dbeta<T, MK>(ctx, S, (T)W->lam, W->dk.b);
                allreduce_fn<0, 1>(ctx, &db);
                W->beta_p = nsub(W->beta_p, nmul(W->lr, db / W->npix_d));
                W->dk = make_divk<T>(P.divergence, W->beta_p);
                W->s1_valid = 0;
            }
            W->lam = nmul(W->lam, P.ls_beta);
            W->trials += 1;
            double sums[3];
            const R3 o = BSGP_DISPATCH_KIND(W->dk, ph_trial_k, ctx, S, (T)W->lam, W->dk);
            sums[0] = o.a; sums[1] = o.b; sums[2] = o.c;
            allreduce_fn<0, 3>(ctx, sums);
            refresh_s1();
            W->fv = objective_value(W->dk, sums, W->s1, W->flux, W->npix_d);
        }
        W->total_trials += W->trials;

        // ---- accept: x_tf, new gradient through A^T, BB sums (:337-347, 355-365, 402); the new x goes into the d array
        ph_rf_grad<T, MK>(ctx, S, W->dk.kind, (T)W->lam, 0);
        conv_middle<T, MK>(ctx, S, S->tf_at, mode_at);
        R7 bbr;
        if constexpr (ROWS) {
            // pass W->iter forms the iterate after that many passes: a snapshot on every snap_every-th
            if (ra.snap && W->iter % ra.snap_every == 0)
                bbr = ph_ri_bb_snap<T, MK>(ctx, S, (T)W->lam, W->dk.kind, snap_slot(a, ra, img, W->iter / ra.snap_every));
            else bbr = ph_ri_bb<T, MK>(ctx, S, (T)W->lam, W->dk.kind);
        } else {
            bbr = ph_ri_bb<T, MK>(ctx, S, (T)W->lam, W->dk.kind);
        }
        allreduce_fn<0, 7>(ctx, bbr.v);

        // ---- Barzilai-Borwein steps, lr schedule, bookkeeping and stop rules (:366-425)
        const double stop_val = ctl_finish_iteration<T, ROWS>(&P, W, bbr);
        if (leader) {
            const int iter = W->iter;
            const size_t o = toff + (size_t)(iter - 1);
            a.times[o] = ctx.now() - W->t_start;
            a.discr[o] = nmul(W->discr_coeff, W->fv);
            if (a.stop_value) a.stop_value[o] = stop_val;
            if (a.tr_alpha) a.tr_alpha[o] = W->alpha;
            if (a.tr_lambda) a.tr_lambda[o] = W->lam;
            if (a.tr_beta) a.tr_beta[o] = W->beta_p;
            if (a.tr_trials) a.tr_trials[o] = W->trials;
            if (a.tr_evals) a.tr_evals[o] = W->evals;
            if (want_err && iter <= P.maxit + 1) a.err[(size_t)img * (stride + 1) + iter] = sqrt(bbr.v[6] / W->truth_sq);   // :394-396
        }
        ctl_accept_step<T>(ctx, S, W->keep_going);
    }

    // ------------------------------------------------------------------ epilogue (:427-438)
    ph_store_out<T>(ctx, S);
    if (leader) {
        a.iters[img] = W->iter - 1;
        a.status[img] = W->status;
        if (a.beta_final) a.beta_final[img] = W->beta_p;
        if (a.proj_evals) a.proj_evals[img] = W->total_evals;
        if (a.ls_trials) a.ls_trials[img] = W->total_trials;
        if constexpr (ROWS) {
            if (ra.snap && ra.snap_count) ra.snap_count[img] = 1 + (W->iter - 1) / ra.snap_every;   // W->iter - 1 passes made
        }
        if (a.scalars) {
            double* sc = a.scalars + (size_t)img * BSGP_NSCALARS;
            sc[0] = (double)S->scaling; sc[1] = W->flux; sc[2] = W->x_low; sc[3] = W->x_upp; sc[4] = W->tol; sc[5] = W->fv; sc[6] = W->alpha; sc[7] = W->tau;
        }
    }
}

}  // namespace bsgp
