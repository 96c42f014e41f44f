// TEST-ONLY single-thread emulation of the device headers (compiled with g++ -DBSGP_HOST_EMUL).
//
// It lets the CPU test-suite check the index arithmetic of the FFT / convolution phases (including
// the multi-CTA row/column partition, emulated rank by rank) and the solver's controller logic
// against the oracle on machines without a GPU.  It is NOT part of the product: nothing under
// beta-sgp_b200/ loads this library and libbsgp.so does not contain it.
#define BSGP_HOST_EMUL 1
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../beta-sgp_b200/csrc/bsgp_plan.h"
#include "../../beta-sgp_b200/csrc/bsgp_solver.cuh"
#include "../../beta-sgp_b200/csrc/bsgp_wrap.h"

using namespace bsgp;

struct HostCtx {
    static constexpr bool kFrame = false;
    static constexpr bool kSmall = false;
    int tid = 0, nt = 1, rank = 0, G = 1, parity = 0;
    void* wst = nullptr;                       // controller state of the one emulated warp
    template <class S> S* ctl() const { return reinterpret_cast<S*>(wst); }
    void sync() {}
    void cluster_sync() {}
    void allreduce(int, double*, int) {}
    void allreduce_sum(double*, int) {}
    void allreduce_min(double&) {}
    void allreduce_max(double&) {}
    double now() { return 0.0; }
};

struct HostCtxFrame : HostCtx {
    static constexpr bool kFrame = true;      // panel exchange-buffer layout (frame mode)
};

template <typename T, class C = HostCtx> struct HostPlan {
    ConvGeom g;
    size_t ws_bytes;
    std::vector<cplx<T>> twx, twy, spec, tf, tf_adj;
    std::vector<unsigned char> arena;      // emulated dynamic shared memory: [position table][workspace]
    unsigned ws_off = 0, ppx_off = 0;
    void bind() { g_emul_smem = arena.data(); }
    bool init(int ny, int nx, int G, size_t ws_limit, int dft_ny = 0, int dft_nx = 0) {
        if (!make_geom(ny, nx, G, sizeof(cplx<T>), ws_limit, &g, &ws_bytes, dft_ny, dft_nx)) return false;
        make_twiddles<T>(nx, twx, dft_nx);
        make_twiddles<T>(ny, twy, dft_ny);
        spec.assign((size_t)ny * g.hx, cmake<T>(0, 0));
        tf.assign((size_t)(g.hx + 1) * ny, cmake<T>(0, 0));
        ws_off = (unsigned)(((size_t)nx * sizeof(unsigned short) + 127) & ~(size_t)127);
        arena.assign(ws_off + ws_bytes + 256, 0);
        bind();
        HostCtx ctx;
        fill_pos_table(ctx, g.px, smem_at<unsigned short>(ppx_off));
        return true;
    }
    void make_tf(const T* psf, std::vector<cplx<T>>* dst = nullptr) {
        const int ny = g.ny, nx = g.nx;
        std::vector<cplx<T>>& out = dst ? *dst : tf;
        out.assign((size_t)(g.hx + 1) * ny, cmake<T>(0, 0));
        for (int phase = 0; phase < 2; ++phase)
            for (int r = 0; r < g.G; ++r) {
                C ctx; ctx.rank = r; ctx.G = g.G;
                const int r0 = r * g.rows_per_cta;
                auto pf = [&](int i) {
                    const int row = i / nx, c = i % nx;
                    In1<T> q; q.a = ld2(psf + (size_t)((r0 + row + ny / 2) & (ny - 1)) * nx, (c + nx / 2) & (nx - 1)); return q;
                };
                auto pe = [&](int, const In1<T>& in) -> V2<T> { return in.a; };
                if (phase == 0) conv_rows_forward<2, true>(ctx, g, ws_off, twx.data(), kNoSmem, 0, ppx_off, spec.data(), pf, pe);
                else conv_cols<true>(ctx, &g, ws_off, twy.data(), kNoSmem, 0, spec.data(), out.data(), CONV_MAKE_TF);
            }
    }
    void apply(const T* x, T* y, int adjoint) {
        const int nx = g.nx;
        for (int phase = 0; phase < 3; ++phase)
            for (int r = 0; r < g.G; ++r) {
                C ctx; ctx.rank = r; ctx.G = g.G;
                const int r0 = r * g.rows_per_cta;
                const size_t off = (size_t)r0 * nx;
                auto pf = [&](int i) { In1<T> q; q.a = ld2(x + off, i); return q; };
                auto pe = [&](int, const In1<T>& in) -> V2<T> { return in.a; };
                auto cf = [&](int) { In1<T> q; q.a = mk2((T)0, (T)0); return q; };
                auto ca = [&](int i, const In1<T>&, V2<T> v) { st2(y + off, i, v); };
                if (phase == 0) conv_rows_forward<2, true>(ctx, g, ws_off, twx.data(), kNoSmem, 0, ppx_off, spec.data(), pf, pe);
                else if (phase == 1) conv_cols<true>(ctx, &g, ws_off, twy.data(), kNoSmem, 0, spec.data(), tf.data(), adjoint ? CONV_CTF : CONV_TF);
                else conv_rows_inverse<2, true>(ctx, g, ws_off, twx.data(), kNoSmem, 0, ppx_off, spec.data(), cf, ca);
            }
    }
    // wrapped plan (bsgp_wrap.h): grid kernels of A / A^T from the caller's iny x inx PSF, fold widths in the geometry
    void make_tf_wrapped(const T* psf, int iny, int inx) {
        const int ny = g.ny, nx = g.nx;
        std::vector<T> k((size_t)ny * nx);
        for (int adj = 0; adj < 2; ++adj) {
            for (int r = 0; r < ny; ++r)
                for (int c = 0; c < nx; ++c) {
                    int sr, sc;
                    k[(size_t)r * nx + c] = wrap_psf_source(r, c, ny, nx, iny, inx, adj, &sr, &sc) ? psf[(size_t)sr * inx + sc] : (T)0;
                }
            make_tf(k.data(), adj ? &tf_adj : nullptr);
        }
        g.wrap_ny = (ny != iny && !g.py.dft_n) ? iny : 0;
        g.wrap_nx = (nx != inx && !g.px.dft_n) ? inx : 0;
    }
};

template <typename T> static void embed(const T* src, int iny, int inx, T* dst, int ny, int nx) {
    for (int r = 0; r < ny; ++r)
        for (int c = 0; c < nx; ++c) dst[(size_t)r * nx + c] = (r < iny && c < inx) ? src[(size_t)r * inx + c] : (T)0;
}
template <typename T> static void crop(const T* src, int ny, int nx, T* dst, int iny, int inx) {
    for (int r = 0; r < iny; ++r)
        for (int c = 0; c < inx; ++c) dst[(size_t)r * inx + c] = src[(size_t)r * nx + c];
}

extern "C" {

// 1-D transform check: forward then (optionally) inverse of `nfft` rows of length n (complex interleaved)
int emul_fft1d(int n, int nfft, const double* in, double* out, int inverse_after, int split_twiddles) {
    FftPlan pl;
    if (!make_fft_plan(n, &pl)) return 1;
    std::vector<cplx<double>> tw;
    make_twiddles<double>(n, tw);
    const int stride = pl.plen + 1;
    // emulated shared memory: [workspace][two-level twiddle table]
    const size_t ws_elems = (size_t)nfft * stride, tab_elems = 64 + (size_t)(n >> 6);
    std::vector<cplx<double>> arena(ws_elems + tab_elems);
    cplx<double>* ws = arena.data();
    for (size_t k = 0; k < tab_elems; ++k) arena[ws_elems + k] = (k < 64) ? tw[k % n] : tw[((k - 64) << 6) % n];
    for (int f = 0; f < nfft; ++f)
        for (int i = 0; i < n; ++i) ws[(size_t)f * stride + fpad(i, pl.pad_shift)] = cmake<double>(in[2 * ((size_t)f * n + i)], in[2 * ((size_t)f * n + i) + 1]);
    HostCtx ctx;
    g_emul_smem = reinterpret_cast<unsigned char*>(arena.data());
    const unsigned tw_off = split_twiddles ? (unsigned)(ws_elems * sizeof(cplx<double>)) : kNoSmem;
    if (split_twiddles) {
        fft_batch_split<false, HostCtx, double>(ctx, 0u, nfft, stride, pl, tw_off);
        if (inverse_after) fft_batch_split<true, HostCtx, double>(ctx, 0u, nfft, stride, pl, tw_off);
    } else {
        fft_batch<false, false, HostCtx, double>(ctx, 0u, nfft, stride, pl, tw.data(), tw_off);
        if (inverse_after) fft_batch<true, false, HostCtx, double>(ctx, 0u, nfft, stride, pl, tw.data(), tw_off);
    }
    for (int f = 0; f < nfft; ++f)
        for (int k = 0; k < n; ++k) {
            const int p = inverse_after ? k : pos_of_freq(pl, k);
            const cplx<double> z = ws[(size_t)f * stride + fpad(p, pl.pad_shift)];
            out[2 * ((size_t)f * n + k)] = z.re;
            out[2 * ((size_t)f * n + k) + 1] = z.im;
        }
    return 0;
}

// circular PSF convolution of one image with the cluster partition emulated rank by rank
int emul_conv(int ny, int nx, int G, long long ws_limit, const double* x, const double* psf, int adjoint, double* y) {
    HostPlan<double> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit)) return 1;
    pl.make_tf(psf);
    pl.apply(x, y, adjoint);
    return 0;
}

// arbitrary-size circular operator: the host-side steps of a wrapped plan (bsgp_kernels.cu) around the same device code
int emul_conv_wrapped(int iny, int inx, int G, long long ws_limit, const double* x, const double* psf, int adjoint, double* y) {
    const int ny = wrap_grid_side(iny), nx = wrap_grid_side(inx);
    if (ny > kMaxSide || nx > kMaxSide) return 2;
    HostPlan<double> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit, ny != iny ? dense_len(iny) : 0, nx != inx ? dense_len(inx) : 0)) return 1;
    pl.make_tf_wrapped(psf, iny, inx);
    std::vector<double> xe((size_t)ny * nx), ye((size_t)ny * nx);
    embed(x, iny, inx, xe.data(), ny, nx);
    if (adjoint) pl.tf.swap(pl.tf_adj);               // A^T = CONV_TF with the spectrum of h~
    pl.apply(xe.data(), ye.data(), 0);
    crop(ye.data(), ny, nx, y, iny, inx);
    return 0;
}

// the same with the frame-mode (column panel) layout of the exchange buffer
int emul_conv_frame(int ny, int nx, int G, long long ws_limit, const double* x, const double* psf, int adjoint, double* y) {
    HostPlan<double, HostCtxFrame> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit)) return 1;
    pl.make_tf(psf);
    pl.apply(x, y, adjoint);
    return 0;
}

int emul_conv_f32(int ny, int nx, int G, long long ws_limit, const float* x, const float* psf, int adjoint, float* y) {
    HostPlan<float> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit)) return 1;
    pl.make_tf(psf);
    pl.apply(x, y, adjoint);
    return 0;
}

// full solver, one image, one emulated CTA
int emul_solve(int ny, int nx, const bsgp_params* params, const double* gn, const double* psf, const double* psf_adj, const double* bkg,
               int bkg_is_image, const double* flux, const double* beta0, const double* x0, const double* obj,
               double* x_out, int* iters, int* status, double* discr, double* stop_value, double* err, double* beta_final,
               int* proj_evals, int* ls_trials, double* scalars, double* tr_alpha, double* tr_lambda, double* tr_beta,
               int* tr_trials, int* tr_evals) {
    HostPlan<double> pl;
    if (!pl.init(ny, nx, 1, (size_t)1 << 30)) return 1;
    pl.make_tf(psf);
    if (psf_adj) pl.make_tf(psf_adj, &pl.tf_adj);
    const size_t npix = (size_t)ny * nx;
    std::vector<double> work(NBUF * npix, 0.0), times(params->maxit + 1, 0.0);
    double* buf[NBUF];
    for (int b = 0; b < NBUF; ++b) buf[b] = work.data() + b * npix;
    SolveArgs<double> a;
    memset(&a, 0, sizeof(a));
    a.p = *params; a.g = pl.g; a.batch = 1;
    a.gn = gn; a.bkg = bkg; a.bkg_is_image = bkg_is_image; a.flux = flux; a.beta0 = beta0; a.x0 = x0; a.obj = obj;
    a.twx = pl.twx.data(); a.twy = pl.twy.data(); a.tf = pl.tf.data(); a.tf_adj = psf_adj ? pl.tf_adj.data() : nullptr; a.n_psf = 1;
    a.x_out = x_out; a.iters = iters; a.status = status; a.discr = discr; a.times = times.data();
    a.stop_value = stop_value; a.err = err; a.beta_final = beta_final; a.proj_evals = proj_evals; a.ls_trials = ls_trials;
    a.scalars = scalars; a.tr_alpha = tr_alpha; a.tr_lambda = tr_lambda; a.tr_beta = tr_beta; a.tr_trials = tr_trials;
    a.tr_evals = tr_evals;
    HostCtx ctx;
    CtlState<double> ctl_state;
    ctx.wst = &ctl_state;
    ImgState<double> S;
    memset(&S, 0, sizeof(S));
    S.geom = pl.g; S.ws_off = pl.ws_off; S.ppx_off = pl.ppx_off; S.spec = pl.spec.data(); S.twx = pl.twx.data(); S.twy = pl.twy.data(); S.twx_off = kNoSmem; S.twy_off = kNoSmem; S.tw_split = 0;
    pl.bind();
    if (params->region[1] > params->region[0]) solve_image<double, true>(ctx, a, &S, buf, pl.tf.data(), psf_adj ? pl.tf_adj.data() : pl.tf.data(), 0);
    else solve_image<double, false>(ctx, a, &S, buf, pl.tf.data(), psf_adj ? pl.tf_adj.data() : pl.tf.data(), 0);
    return 0;
}

// full solver on a wrapped plan: what solve_t does for plan->embedded (embed, region = image window, both spectra, crop)
int emul_solve_wrapped(int iny, int inx, const bsgp_params* params, const double* gn, const double* psf, const double* bkg,
                       int bkg_is_image, const double* flux, const double* beta0, const double* x0, const double* obj,
                       double* x_out, int* iters, int* status, double* discr, double* stop_value, double* err, double* beta_final,
                       int* proj_evals, int* ls_trials, double* scalars, double* tr_alpha, double* tr_lambda, double* tr_beta,
                       int* tr_trials, int* tr_evals) {
    const int ny = wrap_grid_side(iny), nx = wrap_grid_side(inx);
    if (ny > kMaxSide || nx > kMaxSide) return 2;
    HostPlan<double> pl;
    if (!pl.init(ny, nx, 1, (size_t)1 << 30, ny != iny ? dense_len(iny) : 0, nx != inx ? dense_len(inx) : 0)) return 1;
    pl.make_tf_wrapped(psf, iny, inx);
    const size_t npix = (size_t)ny * nx;
    std::vector<double> work(NBUF * npix, 0.0), times(params->maxit + 1, 0.0), gne(npix), bke(npix), x0e(npix), obe(npix), xe(npix);
    embed(gn, iny, inx, gne.data(), ny, nx);
    if (bkg_is_image) embed(bkg, iny, inx, bke.data(), ny, nx);
    if (x0) embed(x0, iny, inx, x0e.data(), ny, nx);
    if (obj) embed(obj, iny, inx, obe.data(), ny, nx);
    double* buf[NBUF];
    for (int b = 0; b < NBUF; ++b) buf[b] = work.data() + b * npix;
    SolveArgs<double> a;
    memset(&a, 0, sizeof(a));
    a.p = *params;
    a.p.region[0] = 0; a.p.region[1] = iny; a.p.region[2] = 0; a.p.region[3] = inx; a.p.div_a = a.p.div_at = 1.0; a.p.adjoint_second_psf = 1;
    a.g = pl.g; a.batch = 1;
    a.gn = gne.data(); a.bkg = bkg_is_image ? bke.data() : bkg; a.bkg_is_image = bkg_is_image; a.flux = flux; a.beta0 = beta0;
    a.x0 = x0 ? x0e.data() : nullptr; a.obj = obj ? obe.data() : nullptr;
    a.twx = pl.twx.data(); a.twy = pl.twy.data(); a.tf = pl.tf.data(); a.tf_adj = pl.tf_adj.data(); a.n_psf = 1;
    a.x_out = xe.data(); a.iters = iters; a.status = status; a.discr = discr; a.times = times.data();
    a.stop_value = stop_value; a.err = err; a.beta_final = beta_final; a.proj_evals = proj_evals; a.ls_trials = ls_trials;
    a.scalars = scalars; a.tr_alpha = tr_alpha; a.tr_lambda = tr_lambda; a.tr_beta = tr_beta; a.tr_trials = tr_trials;
    a.tr_evals = tr_evals;
    HostCtx ctx;
    CtlState<double> ctl_state;
    ctx.wst = &ctl_state;
    ImgState<double> S;
    memset(&S, 0, sizeof(S));
    S.geom = pl.g; S.ws_off = pl.ws_off; S.ppx_off = pl.ppx_off; S.spec = pl.spec.data(); S.twx = pl.twx.data(); S.twy = pl.twy.data(); S.twx_off = kNoSmem; S.twy_off = kNoSmem; S.tw_split = 0;
    pl.bind();
    solve_image<double, true>(ctx, a, &S, buf, pl.tf.data(), pl.tf_adj.data(), 0);
    crop(xe.data(), ny, nx, x_out, iny, inx);
    return 0;
}

// the library's launch-shape planner (bsgp_plan.h, plan_launch) for an image of iny x inx on the FFT grid bsgp_plan_create
// picks; returns 0 or the BSGP_E_* code.  out: frame, G, threads, minb, resident_mask, smem_bytes, conv_smem, ws_bytes,
// wrap_ny, wrap_nx, grid ny, grid nx
int emul_plan_launch(int iny, int inx, int dtype, int want_G, int want_threads, int num_sms, int max_smem, int smem_per_sm,
                     long long* out) {
    const PlanRequest q{wrap_grid_side(iny), wrap_grid_side(inx), iny, inx, want_G, want_threads, num_sms, max_smem, smem_per_sm};
    LaunchPlan L;
    char err[256];
    const int rc = dtype == BSGP_F64 ? plan_launch<double>(q, &L, err, sizeof err) : plan_launch<float>(q, &L, err, sizeof err);
    if (rc) return rc;
    const long long v[12] = {L.frame, L.g.G, L.threads, L.minb, L.resident_mask, (long long)L.smem_bytes, (long long)L.conv_smem,
                             (long long)L.ws_bytes, L.g.wrap_ny, L.g.wrap_nx, q.ny, q.nx};
    for (int k = 0; k < 12; ++k) out[k] = v[k];
    return 0;
}

// projectDF root-find with the reference's x = (c + lambda) / dia evaluation
int emul_project(const double* c, const double* dia, int n, double b, double sat_cap, int has_cap, int max_projs, int biter, int siter,
                 double* x, int* evals) {
    auto point = [&](int i, double lam) {
        double v = ndiv(nadd(c[i], lam), dia[i]);
        v = (v <= 0.0) ? 0.0 : v;
        if (has_cap) v = (v >= sat_cap) ? sat_cap : v;
        return v;
    };
    auto eval = [&](double lam) -> double {
        double s = 0.0;
        for (int i = 0; i < n; ++i) s += point(i, lam);
        return s - b;
    };
    ProjResult pr = flux_rootfind(eval, b, max_projs, 0.0, 1.0, 1e-11, biter, siter);
    for (int i = 0; i < n; ++i) x[i] = point(i, pr.lambda);
    *evals = pr.evals;
    return pr.status;
}

}  // extern "C"

// pow_inline (bsgp_math.cuh): the call-free pow used by the beta-divergence phases
extern "C" void emul_pow(const double* x, const double* y, double* out, long long n) {
    for (long long i = 0; i < n; ++i) out[i] = pow_inline(x[i], y[i]);
}

extern "C" int emul_sizeof_params() { return (int)sizeof(bsgp_params); }
extern "C" int emul_sizeof_inputs() { return (int)sizeof(bsgp_inputs); }
extern "C" int emul_sizeof_outputs() { return (int)sizeof(bsgp_outputs); }
extern "C" int emul_sizeof_plan_info() { return (int)sizeof(bsgp_plan_info); }
