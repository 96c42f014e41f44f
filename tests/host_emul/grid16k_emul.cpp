// TEST-ONLY: frame-mode pieces of the device headers that the exports of emul.cpp do not reach: the fp32 circular operator
// with the frame (column panel) layout of the exchange buffer, and the split transforms of axes whose single transform does
// not fit the workspace (bsgp_conv.cuh; fp64 16384-point axes on a B200), forced here at small sizes by a small workspace
// limit: the operator, the wrapped operator and a full one-thread solve.  Not part of the product.
#include "emul.cpp"

struct HostCtxSplit : HostCtxFrame {
    static constexpr bool kSplit = true;       // split transforms compiled in (SplitCtx)
};

// a plan with split transforms on the axes `split` (bit 0 rows, bit 1 columns), as plan_launch lays it out
template <typename T> struct SplitPlan : HostPlan<T, HostCtxSplit> {
    bool init_split(int ny, int nx, int G, size_t ws_limit, int split) {
        if (!make_geom(ny, nx, G, sizeof(cplx<T>), ws_limit, &this->g, &this->ws_bytes, 0, 0, split)) return false;
        make_twiddles<T>(this->g.px.n, this->twx);
        make_twiddles<T>(this->g.py.n, this->twy);
        this->spec.assign((size_t)ny * this->g.hx, cmake<T>(0, 0));
        this->tf.assign((size_t)(this->g.hx + 1) * ny, cmake<T>(0, 0));
        this->ws_off = (unsigned)(((size_t)nx * sizeof(unsigned short) + 127) & ~(size_t)127);
        this->arena.assign(this->ws_off + this->ws_bytes + 256, 0);
        this->bind();
        HostCtx ctx;
        fill_pos_table(ctx, this->g.px, smem_at<unsigned short>(this->ppx_off));
        return true;
    }
};

extern "C" {

int emul_conv_frame_f32(int ny, int nx, int G, long long ws_limit, const float* x, const float* psf, int adjoint, float* y) {
    HostPlan<float, HostCtxFrame> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit)) return 1;
    pl.make_tf(psf);
    pl.apply(x, y, adjoint);
    return 0;
}

int emul_conv_wrapped_frame_f32(int iny, int inx, int G, long long ws_limit, const float* x, const float* psf, int adjoint, float* y) {
    const int ny = wrap_grid_side(iny), nx = wrap_grid_side(inx);
    if (ny > kMaxSide || nx > kMaxSide) return 2;
    HostPlan<float, HostCtxFrame> pl;
    if (!pl.init(ny, nx, G, (size_t)ws_limit)) return 1;
    pl.make_tf_wrapped(psf, iny, inx);
    std::vector<float> xe((size_t)ny * nx), ye((size_t)ny * nx);
    embed(x, iny, inx, xe.data(), ny, nx);
    if (adjoint) pl.tf.swap(pl.tf_adj);
    pl.apply(xe.data(), ye.data(), 0);
    crop(ye.data(), ny, nx, y, iny, inx);
    return 0;
}

// the split axes of the plan plan_launch makes for an image of iny x inx (bit 0 rows, bit 1 columns), or -1 if it refuses it
int emul_plan_split(int iny, int inx, int dtype, int num_sms, int max_smem, int smem_per_sm) {
    const PlanRequest q{wrap_grid_side(iny), wrap_grid_side(inx), iny, inx, 0, 0, num_sms, max_smem, smem_per_sm};
    LaunchPlan L;
    char err[256];
    const int rc = dtype == BSGP_F64 ? plan_launch<double>(q, &L, err, sizeof err) : plan_launch<float>(q, &L, err, sizeof err);
    if (rc) return -1;
    return (L.g.px.n != L.g.nx ? 1 : 0) | (L.g.py.n != L.g.ny ? 2 : 0);
}

// the axes plan_launch would split for this workspace limit (0: none)
int emul_split_axes(int ny, int nx, long long ws_limit) { return split_axes(ny, nx, sizeof(cplx<double>), (size_t)ws_limit); }

// fp64 circular operator with split transforms on the axes `split`; wrapped: iny x inx on its wrapped grid
int emul_conv_split(int iny, int inx, int G, long long ws_limit, int split, const double* x, const double* psf, int adjoint, double* y) {
    const int ny = wrap_grid_side(iny), nx = wrap_grid_side(inx);
    if (ny > kMaxSide || nx > kMaxSide || dense_len(iny) || dense_len(inx)) return 2;
    SplitPlan<double> pl;
    if (!pl.init_split(ny, nx, G, (size_t)ws_limit, split)) return 1;
    if (ny == iny && nx == inx) {
        pl.make_tf(psf);
        pl.apply(x, y, adjoint);
        return 0;
    }
    pl.make_tf_wrapped(psf, iny, inx);
    std::vector<double> xe((size_t)ny * nx), ye((size_t)ny * nx);
    embed(x, iny, inx, xe.data(), ny, nx);
    if (adjoint) pl.tf.swap(pl.tf_adj);
    pl.apply(xe.data(), ye.data(), 0);
    crop(ye.data(), ny, nx, y, iny, inx);
    return 0;
}

// full solver, one image on a power-of-two grid, with split transforms on the axes `split` (the G CTAs of the frame run
// as one emulated CTA over the whole image)
int emul_solve_split(int ny, int nx, long long ws_limit, int split, const bsgp_params* params, const double* gn, const double* psf,
                     const double* bkg, int bkg_is_image, const double* flux, const double* beta0, double* x_out, int* iters,
                     int* status, double* discr, double* stop_value, double* err, double* beta_final, int* proj_evals, int* ls_trials,
                     double* scalars, double* tr_alpha, double* tr_lambda, double* tr_beta, int* tr_trials, int* tr_evals) {
    SplitPlan<double> pl;
    if (!pl.init_split(ny, nx, 1, (size_t)ws_limit, split)) return 1;
    pl.make_tf(psf);
    const size_t npix = (size_t)ny * nx;
    std::vector<double> work(NBUF * npix, 0.0), times(params->maxit + 1, 0.0);
    double* buf[NBUF];
    for (int b = 0; b < NBUF; ++b) buf[b] = work.data() + b * npix;
    SolveArgs<double> a;
    memset(&a, 0, sizeof(a));
    a.p = *params; a.g = pl.g; a.batch = 1;
    a.gn = gn; a.bkg = bkg; a.bkg_is_image = bkg_is_image; a.flux = flux; a.beta0 = beta0;
    a.twx = pl.twx.data(); a.twy = pl.twy.data(); a.tf = pl.tf.data(); a.n_psf = 1;
    a.x_out = x_out; a.iters = iters; a.status = status; a.discr = discr; a.times = times.data();
    a.stop_value = stop_value; a.err = err; a.beta_final = beta_final; a.proj_evals = proj_evals; a.ls_trials = ls_trials;
    a.scalars = scalars; a.tr_alpha = tr_alpha; a.tr_lambda = tr_lambda; a.tr_beta = tr_beta; a.tr_trials = tr_trials;
    a.tr_evals = tr_evals;
    HostCtxSplit ctx;
    CtlState<double> ctl_state;
    ctx.wst = &ctl_state;
    ImgState<double> S;
    memset(&S, 0, sizeof(S));
    S.geom = pl.g; S.ws_off = pl.ws_off; S.ppx_off = pl.ppx_off; S.spec = pl.spec.data(); S.twx = pl.twx.data(); S.twy = pl.twy.data(); S.twx_off = kNoSmem; S.twy_off = kNoSmem; S.tw_split = 0;
    pl.bind();
    solve_image<double, false>(ctx, a, &S, buf, pl.tf.data(), pl.tf.data(), 0);
    return 0;
}

}  // extern "C"
