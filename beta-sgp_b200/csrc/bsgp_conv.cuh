// Circular PSF convolution of one real image, split over the G CTAs of a thread-block cluster.
//
// Replaces `afunction` (sgp.py:111-117 / 573-579): out = real(ifftn(TF * fftn(x))) with
// TF = fftn(fftshift(psf)) (sgp.py:109 / 571) or its conjugate for A^T.
//
// Decomposition (real-to-complex / complex-to-real, half spectrum, fused PSF multiply):
//   rows_forward : CTA `rank` owns image rows [rank*ny/G, (rank+1)*ny/G).  Two real rows are
//                  transformed by one complex FFT (row 2p -> real part, row 2p+1 -> imaginary
//                  part) and untangled into two half spectra.  Values come from a producer functor
//                  (so the elementwise step that creates the input is fused in) and the half
//                  spectra go to the cluster's exchange buffer in global memory
//                  spec (ny x hx, hx = nx/2, stored in column panels, see spec_idx); column 0 packs the two real columns kx = 0 and
//                  kx = nx/2 as (re, im).
//   cols         : CTA `rank` owns packed spectrum columns [rank*hx/G, (rank+1)*hx/G): forward
//                  column FFT, multiply by the precomputed PSF spectrum (or its conjugate),
//                  inverse column FFT, back to the exchange buffer.
//   rows_inverse : the mirror of rows_forward; real outputs are handed to a consumer functor (so
//                  the elementwise step that uses the result is fused in).
// A cluster barrier is required between the three phases (the caller issues it).
//
// Scaling: rows_forward stores 2*A[k]; the stored PSF spectrum carries 0.5/(nx*ny) (0.25/(nx*ny)
// for the two packed columns, whose untangle doubles once more), all powers of two, so the result
// equals numpy's normalised ifftn without a separate scaling pass.
//
// Memory-level parallelism.  Per-image state that is not resident in shared memory lives in L2
// (~700 cycles away).  Every loop that touches it works on PAIRS of adjacent pixels (one 16-byte
// load per array and pair) and is written in two phases over a small register tile: first all
// loads of U steps (independent, issued back to back), then the arithmetic and the stores.
// Producers / consumers follow the same protocol: `fetch(i)` only loads (i = even slab pixel index,
// returns a small struct of V2 values), `eval` / `apply` compute, accumulate and store.
#pragma once
#include <type_traits>

#include "bsgp_fft.cuh"

namespace bsgp {

struct ConvGeom {
    int ny, nx, hx;          // hx = nx / 2 packed spectrum columns
    int lg_nx, lg_ny, lg_hx;
    int G;                   // CTAs per image (cluster size)
    int rows_per_cta;        // ny / G (even)
    int cols_per_cta;        // hx / G
    int row_tile_pairs;      // row pairs per workspace tile (divides rows_per_cta / 2), power of two
    int col_tile;            // columns per workspace tile (divides cols_per_cta), power of two
    int lg_col_tile;
    int lg_cp;               // log2 of the panel width of the exchange buffer: cols_per_cta (narrow column tiles) or hx (row-major)
    int rowstride;           // padded complex elements per row pair in the workspace
    int colstride;           // padded complex elements per column in the workspace (odd)
    // Arbitrary-size circular operator (bsgp_kernels.cu, "wrapped plans"): the ny x nx grid holds an image of
    // wrap_ny x wrap_nx pixels at its origin, zero elsewhere, and the kernel's linear convolution with it; the circular
    // result is obtained by folding: out[i] = z[i] + z[i + wrap_n] along each wrapped axis (0 = axis not wrapped).
    int wrap_ny, wrap_nx;
    FftPlan px, py;
};

enum ConvMode { CONV_TF = 0, CONV_CTF = 1, CONV_MAKE_TF = 2 };

// the scalars of ConvGeom the row passes need, copied to registers once per pass (the geometry itself
// lives in shared memory, where every store through another pointer would force a reload)
// Row transform of length n = fft_len(px) (nx itself, or a shorter dense DFT): frequency k pairs with its mirror n - k for
// k = 1 .. kmax = (n - 1) / 2; an even n has a Nyquist frequency nyq = n / 2 whose (real) coefficient shares packed
// column 0 with the DC term (nyq = -1: odd n, no such term).  Packed columns beyond kmax carry zeros.
// GEN (compile time) enables all of this plus the folds of wrapped plans; it is set in the kernels of embedded plans
// only (MK = true: images that are not a power-of-two grid by themselves), so that the power-of-two path, which is
// bound by instruction fetch on small images and by registers on large ones, carries none of it.
struct RowGeom { int nx, hx, lg_nx, lg_hx, lg_ny, lg_cp, rows_per_cta, row_tile_pairs, rowstride, ps, wrap_nx, nmir, kmax, nyq; };
template <bool GEN> BSGP_DEV RowGeom row_geom(const ConvGeom& g) {
    RowGeom r;
    r.nx = g.nx; r.hx = g.hx; r.lg_nx = g.lg_nx; r.lg_hx = g.lg_hx; r.lg_ny = g.lg_ny; r.lg_cp = g.lg_cp; r.rows_per_cta = g.rows_per_cta;
    r.row_tile_pairs = g.row_tile_pairs; r.rowstride = g.rowstride; r.ps = g.px.pad_shift; r.wrap_nx = g.wrap_nx;
    if (GEN) { r.nmir = fft_len(g.px); r.kmax = (r.nmir - 1) >> 1; r.nyq = (r.nmir & 1) ? -1 : (r.nmir >> 1); }
    else { r.nmir = g.nx; r.kmax = g.hx - 1; r.nyq = g.hx; }      // never read: the !GEN code uses nx and hx directly
    return r;
}

// Exchange-buffer layout in frame mode: column panels.  Element (row, k) of the half spectrum lives at
//   ((k >> lg_cp) * ny + row) << lg_cp | (k & (cp - 1)),          cp = 2^lg_cp = cols_per_cta,
// i.e. the cp columns one CTA transforms form one contiguous [ny][cp] panel.  The row passes write / read cp-element
// chunks (>= 256 bytes), and the column pass of a CTA walks its own panel only: a column tile narrower than the
// panel (long columns leave room for a single one in the workspace) still touches every 32-byte sector of the panel
// exactly once per two columns, with the neighbouring column served by L2, instead of one sector per 64 KB row.
// PANEL is a compile-time property of the execution context (Ctx::kFrame): the cluster kernels keep the plain
// row-major buffer (their column tiles are >= 8 columns wide, and they are sensitive to every extra register).
template <bool PANEL> BSGP_DEV size_t spec_idx(int row, int k, int lg_ny, int lg_cp, int hx) {
    if (!PANEL) return (size_t)row * hx + k;
    return ((((size_t)(k >> lg_cp) << lg_ny) + (size_t)row) << lg_cp) | (size_t)(k & ((1 << lg_cp) - 1));
}

// two adjacent pixels
template <typename T> struct alignas(2 * sizeof(T)) V2 {
    T x, y;
};
template <typename T> BSGP_DEV V2<T> mk2(T x, T y) { V2<T> r; r.x = x; r.y = y; return r; }
template <typename T> BSGP_DEV V2<T> ld2(const T* p, int i) { return *reinterpret_cast<const V2<T>*>(p + i); }
template <typename T> BSGP_DEV void st2(T* p, int i, V2<T> v) { *reinterpret_cast<V2<T>*>(p + i) = v; }

// small register tiles returned by the fetch phase of the batched loops
template <typename T> struct In1 { V2<T> a; };
template <typename T> struct In2 { V2<T> a, b; };
template <typename T> struct In3 { V2<T> a, b, c; };
template <typename T> struct In4 { V2<T> a, b, c, d; };
template <typename T> struct In5 { V2<T> a, b, c, d, e; };

// ppx[k] = padded workspace position of frequency k after the forward row stages (a shared-memory table;
// evaluating pos_of_freq per element costs as many instructions as the butterflies themselves).
template <class Ctx> BSGP_DEV void fill_pos_table(Ctx& ctx, const FftPlan& pl, unsigned short* tab) {
    for (int k = ctx.tid; k < pl.n; k += ctx.nt) tab[k] = (unsigned short)fpad(pos_of_freq(pl, k), pl.pad_shift);
}

// ---------------------------------------------------------------------------------------------
// Split transforms (frame mode, an axis of N = 2M points whose single transform does not fit the workspace: fp64 axes of
// 16384 on a B200).  The geometry marks a split axis by an FFT plan of M = N / 2 points (px.n != nx, py.n != ny); the
// execution context compiles the split path in through Ctx::kSplit (SplitCtx, only the kernels of such plans), so that the
// kernels of every other plan carry none of it.
//   rows    : one real row x per transform, packed z[j] = x[2j] + i x[2j+1] (M points); the untangle
//             2X[k] = (Z[k] + conj Z[M-k]) - i W_N^k (Z[k] - conj Z[M-k]), k = 0 .. M, keeps the half-spectrum layout of
//             the row-pair path (2X stored, column 0 = (2X[0], 2X[N/2])).  The inverse feeds
//             Q[k] = (Y[k] + Y[k+M]) + i conj(W_N^k) (Y[k] - Y[k+M]), Y[k+M] = conj Y[M-k], whose unnormalised inverse is
//             y[2j] + i y[2j+1] of the unnormalised N-point inverse.
//   columns : one radix-2 step outside shared memory: u[j] = a[j] + a[j+M] (even frequencies), v[j] = (a[j] - a[j+M]) W_N^j
//             (odd frequencies), each transformed with the M-point machinery and multiplied by its half of the PSF spectrum
//             (tf column = [even frequencies][odd frequencies], each in M-point position order); out[j] = U[j] + W_N^-j V[j],
//             out[j+M] = U[j] - W_N^-j V[j].  Only one half fits the workspace: v waits in the exchange buffer rows [M, N)
//             while u is processed, and the inverse-transformed u waits in rows [0, M) while v is processed (2 N w bytes
//             of extra exchange-buffer traffic per convolution, DESIGN.md section 4).
// ---------------------------------------------------------------------------------------------
template <class C, class = void> struct is_split : std::false_type {};
template <class C> struct is_split<C, std::void_t<decltype(C::kSplit)>> : std::integral_constant<bool, C::kSplit> {};
template <class Ctx> struct SplitCtx : Ctx { static constexpr bool kSplit = true; };

// twiddle W_M^k of the M-point plan's table: two-level in shared memory, full in shared memory, or full in global memory
template <typename T> BSGP_DEV cplx<T> split_tw_m(const cplx<T>* tw, unsigned tw_off, int tw_split, int k) {
    if (tw_split) return twiddle_at<T, true>(smem_at<cplx<T>>(tw_off), k);
    return tw_off != kNoSmem ? smem_at<cplx<T>>(tw_off)[k] : tw[k];
}
// W_N^1, N = 2M
template <typename T> BSGP_DEV cplx<T> split_w1(int M) {
    double s, c;
#ifdef BSGP_HOST_EMUL
    const long double a = 3.141592653589793238462643383279502884L / (long double)M;
    s = (double)sinl(a); c = (double)cosl(a);
#else
    sincospi(1.0 / (double)M, &s, &c);
#endif
    return cmake<T>((T)c, (T)-s);
}
// W_N^k = W_M^(k >> 1) (times W_N^1 for odd k), k < N
template <typename T> BSGP_DEV cplx<T> split_tw_n(const cplx<T>* tw, unsigned tw_off, int tw_split, cplx<T> w1, int k) {
    const cplx<T> w = split_tw_m(tw, tw_off, tw_split, k >> 1);
    return (k & 1) ? cmul(w, w1) : w;
}

template <bool INV, class Ctx, typename T>
BSGP_DEV void split_fft(Ctx& ctx, unsigned ws_off, int nfft, int fstride, const FftPlan& pl, const cplx<T>* tw, unsigned tw_off, int tw_split) {
    if (tw_split) fft_batch_split<INV, Ctx, T>(ctx, ws_off, nfft, fstride, pl, tw_off);
    else fft_batch<INV, false>(ctx, ws_off, nfft, fstride, pl, tw, tw_off);
}

// rows_forward of a split row axis: row_tile_pairs rows (one transform each) per workspace tile
template <class Ctx, typename T, class Fetch, class Eval>
BSGP_DEV void split_rows_forward(Ctx& ctx, const ConvGeom& gg, unsigned ws_off, const cplx<T>* twx, unsigned twx_off, int tw_split, unsigned ppx_off, cplx<T>* spec, Fetch& fetch, Eval& eval) {
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    const unsigned short* ppx = smem_at<unsigned short>(ppx_off);
    const int M = gg.px.n, lgM = gg.px.log2n, ps = gg.px.pad_shift, lg_nx = gg.lg_nx, rs = gg.rowstride, R = gg.row_tile_pairs;
    const int lg_ny = gg.lg_ny, lg_cp = gg.lg_cp, hx = gg.hx;
    const int r0 = ctx.rank * gg.rows_per_cta;
    const cplx<T> w1 = split_w1<T>(M);
    for (int row0 = 0; row0 < gg.rows_per_cta; row0 += R) {
        for (int e = ctx.tid; e < (R << lgM); e += ctx.nt) {
            const int r = e >> lgM, j = e & (M - 1);
            const int i = ((row0 + r) << lg_nx) + 2 * j;
            const auto in = fetch(i);
            const V2<T> v = eval(i, in);
            ws[r * rs + fpad(j, ps)] = cmake<T>(v.x, v.y);
        }
        ctx.sync();
        split_fft<false>(ctx, ws_off, R, rs, gg.px, twx, twx_off, tw_split);
        for (int e = ctx.tid; e < (R << lgM); e += ctx.nt) {
            const int r = e >> lgM, k = e & (M - 1);
            const cplx<T>* a = ws + r * rs;
            const cplx<T> zk = a[ppx[k]];
            cplx<T> X;
            if (k == 0) {
                X = cmake<T>((T)2 * (zk.re + zk.im), (T)2 * (zk.re - zk.im));
            } else {
                const cplx<T> zm = a[ppx[M - k]];
                const cplx<T> S = cmake<T>(zk.re + zm.re, zk.im - zm.im), D = cmake<T>(zk.re - zm.re, zk.im + zm.im);
                const cplx<T> wd = cmul(split_tw_n(twx, twx_off, tw_split, w1, k), D);
                X = cmake<T>(S.re + wd.im, S.im - wd.re);                      // S - i W D
            }
            spec[spec_idx<true>(r0 + row0 + r, k, lg_ny, lg_cp, hx)] = X;
        }
        ctx.sync();
    }
}

// rows_inverse of a split row axis; WRAP: the column fold of a wrapped plan
template <bool WRAP, class Ctx, typename T, class Fetch, class Apply>
BSGP_DEV void split_rows_inverse(Ctx& ctx, const ConvGeom& gg, unsigned ws_off, const cplx<T>* twx, unsigned twx_off, int tw_split, unsigned ppx_off, const cplx<T>* spec, Fetch& fetch, Apply& apply) {
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    const unsigned short* ppx = smem_at<unsigned short>(ppx_off);
    const int M = gg.px.n, lgM = gg.px.log2n, ps = gg.px.pad_shift, lg_nx = gg.lg_nx, rs = gg.rowstride, R = gg.row_tile_pairs;
    const int lg_ny = gg.lg_ny, lg_cp = gg.lg_cp, hx = gg.hx, wn = WRAP ? gg.wrap_nx : 0;
    const int r0 = ctx.rank * gg.rows_per_cta;
    const cplx<T> w1 = split_w1<T>(M);
    for (int row0 = 0; row0 < gg.rows_per_cta; row0 += R) {
        for (int e = ctx.tid; e < (R << lgM); e += ctx.nt) {
            const int r = e >> lgM, k = e & (M - 1);
            const int row = r0 + row0 + r;
            const cplx<T> yk = spec[spec_idx<true>(row, k, lg_ny, lg_cp, hx)];
            cplx<T> q;
            if (k == 0) {
                q = cmake<T>(yk.re + yk.im, yk.re - yk.im);                     // Y[0] = re, Y[M] = im, both real
            } else {
                const cplx<T> ym = spec[spec_idx<true>(row, M - k, lg_ny, lg_cp, hx)];
                const cplx<T> S = cmake<T>(yk.re + ym.re, yk.im - ym.im), D = cmake<T>(yk.re - ym.re, yk.im + ym.im);
                const cplx<T> wd = cmulc(D, split_tw_n(twx, twx_off, tw_split, w1, k));
                q = cmake<T>(S.re - wd.im, S.im + wd.re);                      // S + i conj(W) D
            }
            ws[r * rs + ppx[k]] = q;
        }
        ctx.sync();
        split_fft<true>(ctx, ws_off, R, rs, gg.px, twx, twx_off, tw_split);
        for (int e = ctx.tid; e < (R << lgM); e += ctx.nt) {
            const int r = e >> lgM, j = e & (M - 1);
            const cplx<T>* a = ws + r * rs;
            const cplx<T> z = a[fpad(j, ps)];
            T v0 = z.re, v1 = z.im;
            if (WRAP && 2 * j < wn) {
                auto px = [&](int c) { const cplx<T> t = a[fpad(c >> 1, ps)]; return (c & 1) ? t.im : t.re; };
                v0 += px(2 * j + wn);
                if (2 * j + 1 < wn) v1 += px(2 * j + 1 + wn);
            }
            const int i = ((row0 + r) << lg_nx) + 2 * j;
            const auto in = fetch(i);
            apply(i, in, mk2<T>(v0, v1));
        }
        ctx.sync();
    }
}

// the column pass of a split column axis (see above); GEN: wrapped plans fold the rows
template <bool GEN, class Ctx, typename T>
BSGP_NOINLINE void split_cols(Ctx ctx, const ConvGeom* gp, unsigned ws_off, const cplx<T>* twy, unsigned twy_off, int tw_split, cplx<T>* spec, cplx<T>* tf, int mode) {
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    const int ny = gp->ny, nx = gp->nx, hx = gp->hx, lg_ny = gp->lg_ny, lg_cp = gp->lg_cp;
    const int M = gp->py.n, lgM = gp->py.log2n, ps = gp->py.pad_shift, cs = gp->colstride;
    const int ct = gp->col_tile, lct = gp->lg_col_tile, c0 = ctx.rank * gp->cols_per_cta;
    const FftPlan& py = gp->py;
    const cplx<T> w1 = split_w1<T>(M);
    auto sidx = [&](int row, int col) { return spec_idx<true>(row, col, lg_ny, lg_cp, hx); };
    const int total = ct << lgM;
    for (int cc0 = c0; cc0 < c0 + gp->cols_per_cta; cc0 += ct) {
        for (int e = ctx.tid; e < total; e += ctx.nt) {
            const int j = e >> lct, cl = e & (ct - 1);
            const cplx<T> lo = spec[sidx(j, cc0 + cl)], hi = spec[sidx(j + M, cc0 + cl)];
            ws[cl * cs + fpad(j, ps)] = cadd(lo, hi);
            spec[sidx(j + M, cc0 + cl)] = cmul(csub(lo, hi), split_tw_n(twy, twy_off, tw_split, w1, j));   // v waits here
        }
        ctx.sync();
        for (int h = 0; h < 2; ++h) {
            if (h == 1) {
                for (int e = ctx.tid; e < total; e += ctx.nt) {
                    const int j = e >> lct, cl = e & (ct - 1);
                    ws[cl * cs + fpad(j, ps)] = spec[sidx(j + M, cc0 + cl)];
                }
                ctx.sync();
            }
            split_fft<false>(ctx, ws_off, ct, cs, py, twy, twy_off, tw_split);
            const size_t hoff = (size_t)h * M;
            // column 0 packs kx = 0 and kx = nx/2; frequency ky = 2 k + h pairs with N - ky = 2 k' + h, k' = (M - k - h) mod M
            const int kend = h ? (M >> 1) - 1 : (M >> 1);
            if (mode == CONV_MAKE_TF) {
                const T sc = (T)0.25 / ((T)nx * (T)ny), sp = (T)0.0625 / ((T)nx * (T)ny);
                for (int e = ctx.tid; e < total; e += ctx.nt) {
                    const int cl = e >> lgM, p = e & (M - 1);
                    if (cc0 + cl == 0) continue;
                    tf[(size_t)(cc0 + cl) * ny + hoff + p] = cscale(ws[cl * cs + fpad(p, ps)], sc);
                }
                if (cc0 == 0) {
                    for (int k = ctx.tid; k <= kend; k += ctx.nt) {
                        const int pa = pos_of_freq(py, k), pb = pos_of_freq(py, (M - k - h) & (M - 1));
                        const cplx<T> za = ws[fpad(pa, ps)], zb = ws[fpad(pb, ps)];
                        const cplx<T> c0v = cmake<T>(za.re + zb.re, za.im - zb.im), chv = cmake<T>(za.im + zb.im, zb.re - za.re);
                        tf[hoff + pa] = cscale(c0v, sp);
                        tf[(size_t)hx * ny + hoff + pa] = cscale(chv, sp);
                        tf[hoff + pb] = cscale(cconj(c0v), sp);
                        tf[(size_t)hx * ny + hoff + pb] = cscale(cconj(chv), sp);
                    }
                }
                ctx.sync();
                continue;
            }
            for (int e = ctx.tid; e < total; e += ctx.nt) {
                const int cl = e >> lgM, p = e & (M - 1);
                if (cc0 + cl == 0) continue;
                cplx<T>* z = ws + cl * cs + fpad(p, ps);
                const cplx<T> t = tf[(size_t)(cc0 + cl) * ny + hoff + p];
                *z = (mode == CONV_TF) ? cmul(*z, t) : cmulc(*z, t);
            }
            if (cc0 == 0) {
                for (int k = ctx.tid; k <= kend; k += ctx.nt) {
                    const int pa = pos_of_freq(py, k), pb = pos_of_freq(py, (M - k - h) & (M - 1));
                    cplx<T> t0a = tf[hoff + pa], tha = tf[(size_t)hx * ny + hoff + pa], t0b = tf[hoff + pb], thb = tf[(size_t)hx * ny + hoff + pb];
                    const cplx<T> za = ws[fpad(pa, ps)], zb = ws[fpad(pb, ps)];
                    const cplx<T> c0a = cmake<T>(za.re + zb.re, za.im - zb.im), cha = cmake<T>(za.im + zb.im, zb.re - za.re);
                    if (mode == CONV_CTF) { t0a = cconj(t0a); tha = cconj(tha); t0b = cconj(t0b); thb = cconj(thb); }
                    const cplx<T> ya0 = cmul(t0a, c0a), yah = cmul(tha, cha);
                    const cplx<T> yb0 = cmul(t0b, cconj(c0a)), ybh = cmul(thb, cconj(cha));
                    ws[fpad(pa, ps)] = cmake<T>(ya0.re - yah.im, ya0.im + yah.re);
                    if (pb != pa) ws[fpad(pb, ps)] = cmake<T>(yb0.re - ybh.im, yb0.im + ybh.re);
                }
            }
            ctx.sync();
            split_fft<true>(ctx, ws_off, ct, cs, py, twy, twy_off, tw_split);
            for (int e = ctx.tid; e < total; e += ctx.nt) {
                const int j = e >> lct, cl = e & (ct - 1);
                const cplx<T> z = ws[cl * cs + fpad(j, ps)];
                if (h == 0) {
                    spec[sidx(j, cc0 + cl)] = z;                                  // U waits here
                } else {
                    const cplx<T> u = spec[sidx(j, cc0 + cl)], v = cmulc(z, split_tw_n(twy, twy_off, tw_split, w1, j));
                    spec[sidx(j, cc0 + cl)] = cadd(u, v);
                    spec[sidx(j + M, cc0 + cl)] = csub(u, v);
                }
            }
            ctx.sync();
        }
        if (GEN && mode != CONV_MAKE_TF && gp->wrap_ny > 0) {                    // wrapped plan: z[i] += z[i + n]
            const int wn = gp->wrap_ny;
            for (int e = ctx.tid; e < ct * wn; e += ctx.nt) {
                const int cl = e / wn, row = e - cl * wn;
                spec[sidx(row, cc0 + cl)] = cadd(spec[sidx(row, cc0 + cl)], spec[sidx(row + wn, cc0 + cl)]);
            }
            ctx.sync();
        }
    }
}

// Producer: In fetch(i); V2 eval(i, In) for the slab pixel pair (i, i + 1), i = local_row * nx + col.
template <int U_, bool GEN = false, class Ctx, typename T, class Fetch, class Eval>
BSGP_DEV void conv_rows_forward(Ctx& ctx, const ConvGeom& gg, unsigned ws_off, const cplx<T>* twx, unsigned twx_off, int tw_split, unsigned ppx_off, cplx<T>* spec, Fetch& fetch, Eval& eval) {
    if constexpr (is_split<Ctx>::value) {
        if (gg.px.n != gg.nx) { split_rows_forward(ctx, gg, ws_off, twx, twx_off, tw_split, ppx_off, spec, fetch, eval); return; }
    }
    constexpr int U = Ctx::kSmall ? 1 : U_;                  // small images: a thread has one or two steps per pass, batches would only be code
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    const unsigned short* ppx = smem_at<unsigned short>(ppx_off);
    const RowGeom g = row_geom<GEN>(gg);                     // scalars in registers; the FFT plan stays where it is
    const FftPlan& px = gg.px;
    const int r0 = ctx.rank * g.rows_per_cta;
    const int ps = g.ps;
    const int ntiles = (g.rows_per_cta >> 1) / g.row_tile_pairs;
    for (int tile = 0; tile < ntiles; ++tile) {
        const int pair0 = tile * g.row_tile_pairs;
        const int total = g.row_tile_pairs << g.lg_hx;      // steps: one row pair x one column pair
        // full batches without guards (a guarded assignment would push the register tile into local memory); with U == 1 a
        // batch is exactly one step of the loop below, so the batched copy of the (large, inlined) producer is left out
        int e0 = ctx.tid;
        for (; U > 1 && e0 + (U - 1) * ctx.nt < total; e0 += ctx.nt * U) {
            decltype(fetch(0)) in0[U], in1[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = e0 + u * ctx.nt;
                const int i0 = ((2 * (pair0 + (e >> g.lg_hx))) << g.lg_nx) + 2 * (e & (g.hx - 1));
                in0[u] = fetch(i0);
                in1[u] = fetch(i0 + g.nx);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = e0 + u * ctx.nt;
                const int p = e >> g.lg_hx, c = 2 * (e & (g.hx - 1));
                const int i0 = ((2 * (pair0 + p)) << g.lg_nx) + c;
                const V2<T> v0 = eval(i0, in0[u]);
                const V2<T> v1 = eval(i0 + g.nx, in1[u]);
                cplx<T>* row = ws + p * g.rowstride;
                row[fpad(c, ps)] = cmake<T>(v0.x, v1.x);
                row[fpad(c + 1, ps)] = cmake<T>(v0.y, v1.y);
            }
        }
#pragma unroll 1
        for (; e0 < total; e0 += ctx.nt) {
            const int p = e0 >> g.lg_hx, c = 2 * (e0 & (g.hx - 1));
            const int i0 = ((2 * (pair0 + p)) << g.lg_nx) + c;
            const auto a0 = fetch(i0);
            const auto a1 = fetch(i0 + g.nx);
            const V2<T> v0 = eval(i0, a0);
            const V2<T> v1 = eval(i0 + g.nx, a1);
            cplx<T>* row = ws + p * g.rowstride;
            row[fpad(c, ps)] = cmake<T>(v0.x, v1.x);
            row[fpad(c + 1, ps)] = cmake<T>(v0.y, v1.y);
        }
        ctx.sync();
        if (Ctx::kFrame && tw_split) fft_batch_split<false, Ctx, T>(ctx, ws_off, g.row_tile_pairs, g.rowstride, px, twx_off);
        else fft_batch<false, GEN>(ctx, ws_off, g.row_tile_pairs, g.rowstride, px, twx, twx_off);
        for (int e = ctx.tid; e < total; e += ctx.nt) {
            const int p = e >> g.lg_hx, k = e & (g.hx - 1);
            const cplx<T>* a = ws + p * g.rowstride;
            cplx<T> A, B;
            if (k == 0) {
                const cplx<T> z0 = a[ppx[0]], zh = (!GEN || g.nyq >= 0) ? a[ppx[GEN ? g.nyq : g.hx]] : cmake<T>(0, 0);
                A = cmake<T>(z0.re + z0.re, zh.re + zh.re);
                B = cmake<T>(z0.im + z0.im, zh.im + zh.im);
            } else if (!GEN || k <= g.kmax) {
                const cplx<T> zk = a[ppx[k]], zm = a[ppx[(GEN ? g.nmir : g.nx) - k]];
                A = cmake<T>(zk.re + zm.re, zk.im - zm.im);
                B = cmake<T>(zk.im + zm.im, zm.re - zk.re);
            } else {
                A = B = cmake<T>(0, 0);
            }
            const size_t row = (size_t)(r0 + 2 * (pair0 + p));
            spec[spec_idx<Ctx::kFrame>((int)row, k, g.lg_ny, g.lg_cp, g.hx)] = A;
            spec[spec_idx<Ctx::kFrame>((int)row + 1, k, g.lg_ny, g.lg_cp, g.hx)] = B;
        }
        ctx.sync();
    }
}

// tf: [hx + 1][ny] complex in column-workspace position order (written by CONV_MAKE_TF);
// row 0 = kx 0, rows 1..hx-1 = kx, row hx = kx nx/2.  Not inlined: it does not depend on the
// producer / consumer, so all convolutions of the solver share one copy of the code.
template <bool GEN, class Ctx, typename T>
BSGP_NOINLINE void conv_cols(Ctx ctx, const ConvGeom* gp, unsigned ws_off, const cplx<T>* twy, unsigned twy_off, int tw_split, cplx<T>* spec, cplx<T>* tf, int mode) {
    if constexpr (is_split<Ctx>::value) {
        if (gp->py.n != gp->ny) { split_cols<GEN>(ctx, gp, ws_off, twy, twy_off, tw_split, spec, tf, mode); return; }
    }
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    constexpr int U = Ctx::kSmall ? 1 : 8;
    struct { int ny, nx, hx, lg_ny, lg_col_tile, col_tile, colstride, cols_per_cta, lg_cp; } g;      // register copies
    g.ny = gp->ny; g.nx = gp->nx; g.hx = gp->hx; g.lg_ny = gp->lg_ny; g.lg_col_tile = gp->lg_col_tile; g.col_tile = gp->col_tile; g.lg_cp = gp->lg_cp;
    g.colstride = gp->colstride; g.cols_per_cta = gp->cols_per_cta;
    const FftPlan& py = gp->py;
    // transform lengths (== ny, nx unless an axis is a dense DFT; a split axis has no dense DFT and px.n == nx / 2)
    const int ney = GEN ? fft_len(gp->py) : g.ny, nex = (GEN && !is_split<Ctx>::value) ? fft_len(gp->px) : g.nx;
    const int c0 = ctx.rank * g.cols_per_cta;
    const int ps = gp->py.pad_shift;
    const int ntiles = g.cols_per_cta / g.col_tile;
    const int ct = g.col_tile;
    for (int tile = 0; tile < ntiles; ++tile) {
        const int cc0 = c0 + tile * ct;
        const int total = g.ny << g.lg_col_tile;
        {
            int e0 = ctx.tid;
            for (; U > 1 && e0 + (U - 1) * ctx.nt < total; e0 += ctx.nt * U) {
                cplx<T> v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = e0 + u * ctx.nt;
                    v[u] = spec[spec_idx<Ctx::kFrame>(e >> g.lg_col_tile, cc0 + (e & (ct - 1)), g.lg_ny, g.lg_cp, g.hx)];
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = e0 + u * ctx.nt;
                    ws[(e & (ct - 1)) * g.colstride + fpad(e >> g.lg_col_tile, ps)] = v[u];
                }
            }
#pragma unroll 1
            for (; e0 < total; e0 += ctx.nt)
                ws[(e0 & (ct - 1)) * g.colstride + fpad(e0 >> g.lg_col_tile, ps)] = spec[spec_idx<Ctx::kFrame>(e0 >> g.lg_col_tile, cc0 + (e0 & (ct - 1)), g.lg_ny, g.lg_cp, g.hx)];
        }
        ctx.sync();
        if (Ctx::kFrame && tw_split) fft_batch_split<false, Ctx, T>(ctx, ws_off, ct, g.colstride, py, twy_off);
        else fft_batch<false, GEN>(ctx, ws_off, ct, g.colstride, py, twy, twy_off);
        if (mode == CONV_MAKE_TF) {
            // column FFT of 2*A holds 2*TF; store TF * 0.5/(nx ny)
            const T sc = (T)0.25 / ((T)nex * (T)ney);
            for (int e = ctx.tid; e < (ct << g.lg_ny); e += ctx.nt) {
                const int cl = e >> g.lg_ny, p = e & (g.ny - 1);
                if (cc0 + cl == 0) continue;
                tf[(size_t)(cc0 + cl) * g.ny + p] = cscale(ws[cl * g.colstride + fpad(p, ps)], sc);
            }
            if (cc0 == 0) {
                const T sp = (T)0.0625 / ((T)nex * (T)ney);   // (C0 = 4 TF0) * 0.25/(nx ny)
                for (int ky = ctx.tid; ky <= (ney >> 1); ky += ctx.nt) {
                    const int pa = pos_of_freq(py, ky), pb = pos_of_freq(py, GEN ? (ky ? ney - ky : 0) : ((g.ny - ky) & (g.ny - 1)));
                    const cplx<T> za = ws[fpad(pa, ps)], zb = ws[fpad(pb, ps)];
                    const cplx<T> c0v = cmake<T>(za.re + zb.re, za.im - zb.im);          // za + conj(zb)
                    const cplx<T> chv = cmake<T>(za.im + zb.im, zb.re - za.re);          // -i (za - conj(zb))
                    tf[pa] = cscale(c0v, sp);
                    tf[(size_t)g.hx * g.ny + pa] = cscale(chv, sp);
                    tf[pb] = cscale(cconj(c0v), sp);
                    tf[(size_t)g.hx * g.ny + pb] = cscale(cconj(chv), sp);
                }
            }
            ctx.sync();
            continue;
        }
        const int mtotal = ct << g.lg_ny;
        {
            auto mul_one = [&](int e, const cplx<T>& t) {
                if (cc0 + (e >> g.lg_ny) != 0) {
                    cplx<T>* z = ws + (e >> g.lg_ny) * g.colstride + fpad(e & (g.ny - 1), ps);
                    *z = (mode == CONV_TF) ? cmul(*z, t) : cmulc(*z, t);
                }
            };
            int e0 = ctx.tid;
            for (; U > 1 && e0 + (U - 1) * ctx.nt < mtotal; e0 += ctx.nt * U) {
                cplx<T> t[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = e0 + u * ctx.nt;
                    t[u] = tf[(size_t)(cc0 + (e >> g.lg_ny)) * g.ny + (e & (g.ny - 1))];
                }
#pragma unroll
                for (int u = 0; u < U; ++u) mul_one(e0 + u * ctx.nt, t[u]);
            }
#pragma unroll 1
            for (; e0 < mtotal; e0 += ctx.nt) mul_one(e0, tf[(size_t)(cc0 + (e0 >> g.lg_ny)) * g.ny + (e0 & (g.ny - 1))]);
        }
        if (cc0 == 0) {
            for (int ky = ctx.tid; ky <= (ney >> 1); ky += ctx.nt) {
                const int pa = pos_of_freq(py, ky), pb = pos_of_freq(py, GEN ? (ky ? ney - ky : 0) : ((g.ny - ky) & (g.ny - 1)));
                cplx<T> t0a = tf[pa], tha = tf[(size_t)g.hx * g.ny + pa], t0b = tf[pb], thb = tf[(size_t)g.hx * g.ny + pb];
                const cplx<T> za = ws[fpad(pa, ps)], zb = ws[fpad(pb, ps)];
                const cplx<T> c0a = cmake<T>(za.re + zb.re, za.im - zb.im);
                const cplx<T> cha = cmake<T>(za.im + zb.im, zb.re - za.re);
                if (mode == CONV_CTF) { t0a = cconj(t0a); tha = cconj(tha); t0b = cconj(t0b); thb = cconj(thb); }
                const cplx<T> ya0 = cmul(t0a, c0a), yah = cmul(tha, cha);
                const cplx<T> yb0 = cmul(t0b, cconj(c0a)), ybh = cmul(thb, cconj(cha));
                // Y = Y0 + i Yh
                ws[fpad(pa, ps)] = cmake<T>(ya0.re - yah.im, ya0.im + yah.re);
                if (pb != pa) ws[fpad(pb, ps)] = cmake<T>(yb0.re - ybh.im, yb0.im + ybh.re);
            }
        }
        ctx.sync();
        if (Ctx::kFrame && tw_split) fft_batch_split<true, Ctx, T>(ctx, ws_off, ct, g.colstride, py, twy_off);
        else fft_batch<true, GEN>(ctx, ws_off, ct, g.colstride, py, twy, twy_off);
        if (GEN && gp->wrap_ny > 0) {                            // wrapped plan: fold the linear result along the rows, z[i] += z[i + n]
            const int wn = gp->wrap_ny;
            for (int e = ctx.tid; e < ct * wn; e += ctx.nt) {
                const int cl = e / wn, row = e - cl * wn;
                cplx<T>* col = ws + cl * g.colstride;
                col[fpad(row, ps)] = cadd(col[fpad(row, ps)], col[fpad(row + wn, ps)]);
            }
            ctx.sync();
        }
        for (int e = ctx.tid; e < total; e += ctx.nt) {
            const int row = e >> g.lg_col_tile, cl = e & (ct - 1);
            spec[spec_idx<Ctx::kFrame>(row, cc0 + cl, g.lg_ny, g.lg_cp, g.hx)] = ws[cl * g.colstride + fpad(row, ps)];
        }
        ctx.sync();
    }
}

// Consumer: In fetch(i); void apply(i, In, V2 value) for the slab pixel pair (i, i + 1).
// WRAP: the geometry may ask for the column fold of a wrapped plan (value(c) = z[c] + z[c + wrap_nx] for c < wrap_nx) or
// for a dense row transform (the GEN features of row_geom).
template <int U_, bool WRAP = false, class Ctx, typename T, class Fetch, class Apply>
BSGP_DEV void conv_rows_inverse(Ctx& ctx, const ConvGeom& gg, unsigned ws_off, const cplx<T>* twx, unsigned twx_off, int tw_split, unsigned ppx_off, const cplx<T>* spec, Fetch& fetch, Apply& apply) {
    if constexpr (is_split<Ctx>::value) {
        if (gg.px.n != gg.nx) { split_rows_inverse<WRAP>(ctx, gg, ws_off, twx, twx_off, tw_split, ppx_off, spec, fetch, apply); return; }
    }
    cplx<T>* ws = smem_at<cplx<T>>(ws_off);
    const unsigned short* ppx = smem_at<unsigned short>(ppx_off);
    constexpr int U = Ctx::kSmall ? 1 : U_;
    constexpr int UL = Ctx::kSmall ? 1 : 4;
    const RowGeom g = row_geom<WRAP>(gg);
    const FftPlan& px = gg.px;
    const int r0 = ctx.rank * g.rows_per_cta;
    const int ps = g.ps;
    const int ntiles = (g.rows_per_cta >> 1) / g.row_tile_pairs;
    for (int tile = 0; tile < ntiles; ++tile) {
        const int pair0 = tile * g.row_tile_pairs;
        const int total = g.row_tile_pairs << g.lg_hx;
        {
            auto tangle = [&](int e, const cplx<T>& A, const cplx<T>& B) {
                const int k = e & (g.hx - 1);
                cplx<T>* a = ws + (e >> g.lg_hx) * g.rowstride;
                if (k == 0) {
                    a[ppx[0]] = cmake<T>(A.re, B.re);
                    if (!WRAP || g.nyq >= 0) a[ppx[WRAP ? g.nyq : g.hx]] = cmake<T>(A.im, B.im);
                } else if (!WRAP || k <= g.kmax) {
                    a[ppx[k]] = cmake<T>(A.re - B.im, A.im + B.re);
                    a[ppx[(WRAP ? g.nmir : g.nx) - k]] = cmake<T>(A.re + B.im, B.re - A.im);
                }
            };
            int e0 = ctx.tid;
            for (; UL > 1 && e0 + (UL - 1) * ctx.nt < total; e0 += ctx.nt * UL) {
                cplx<T> A[UL], B[UL];
#pragma unroll
                for (int u = 0; u < UL; ++u) {
                    const int e = e0 + u * ctx.nt;
                    const size_t row = (size_t)(r0 + 2 * (pair0 + (e >> g.lg_hx)));
                    A[u] = spec[spec_idx<Ctx::kFrame>((int)row, e & (g.hx - 1), g.lg_ny, g.lg_cp, g.hx)];
                    B[u] = spec[spec_idx<Ctx::kFrame>((int)row + 1, e & (g.hx - 1), g.lg_ny, g.lg_cp, g.hx)];
                }
#pragma unroll
                for (int u = 0; u < UL; ++u) tangle(e0 + u * ctx.nt, A[u], B[u]);
            }
#pragma unroll 1
            for (; e0 < total; e0 += ctx.nt) {
                const size_t row = (size_t)(r0 + 2 * (pair0 + (e0 >> g.lg_hx)));
                tangle(e0, spec[spec_idx<Ctx::kFrame>((int)row, e0 & (g.hx - 1), g.lg_ny, g.lg_cp, g.hx)], spec[spec_idx<Ctx::kFrame>((int)row + 1, e0 & (g.hx - 1), g.lg_ny, g.lg_cp, g.hx)]);
            }
        }
        ctx.sync();
        if (Ctx::kFrame && tw_split) fft_batch_split<true, Ctx, T>(ctx, ws_off, g.row_tile_pairs, g.rowstride, px, twx_off);
        else fft_batch<true, WRAP>(ctx, ws_off, g.row_tile_pairs, g.rowstride, px, twx, twx_off);
        {
            int e0 = ctx.tid;
            for (; U > 1 && e0 + (U - 1) * ctx.nt < total; e0 += ctx.nt * U) {
                decltype(fetch(0)) in0[U], in1[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = e0 + u * ctx.nt;
                    const int i0 = ((2 * (pair0 + (e >> g.lg_hx))) << g.lg_nx) + 2 * (e & (g.hx - 1));
                    in0[u] = fetch(i0);
                    in1[u] = fetch(i0 + g.nx);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = e0 + u * ctx.nt;
                    const int p = e >> g.lg_hx, c = 2 * (e & (g.hx - 1));
                    const int i0 = ((2 * (pair0 + p)) << g.lg_nx) + c;
                    const cplx<T>* row = ws + p * g.rowstride;
                    cplx<T> z0 = row[fpad(c, ps)], z1 = row[fpad(c + 1, ps)];
                    if (WRAP && c < g.wrap_nx) { z0 = cadd(z0, row[fpad(c + g.wrap_nx, ps)]); z1 = cadd(z1, row[fpad(c + 1 + g.wrap_nx, ps)]); }
                    apply(i0, in0[u], mk2<T>(z0.re, z1.re));
                    apply(i0 + g.nx, in1[u], mk2<T>(z0.im, z1.im));
                }
            }
#pragma unroll 1
            for (; e0 < total; e0 += ctx.nt) {
                const int p = e0 >> g.lg_hx, c = 2 * (e0 & (g.hx - 1));
                const int i0 = ((2 * (pair0 + p)) << g.lg_nx) + c;
                const auto a0 = fetch(i0);
                const auto a1 = fetch(i0 + g.nx);
                const cplx<T>* row = ws + p * g.rowstride;
                cplx<T> z0 = row[fpad(c, ps)], z1 = row[fpad(c + 1, ps)];
                if (WRAP && c < g.wrap_nx) { z0 = cadd(z0, row[fpad(c + g.wrap_nx, ps)]); z1 = cadd(z1, row[fpad(c + 1 + g.wrap_nx, ps)]); }
                apply(i0, a0, mk2<T>(z0.re, z1.re));
                apply(i0 + g.nx, a1, mk2<T>(z0.im, z1.im));
            }
        }
        ctx.sync();
    }
}

// elementwise loop over pixel pairs with batched loads: In fetch(i) (loads only), body(i, In), i even
template <int U_, class Ctx, class Fetch, class Body>
BSGP_DEV void pair_loop(Ctx& ctx, int n, Fetch& fetch, Body& body) {
    constexpr int U = Ctx::kSmall ? 1 : U_;
    const int np = n >> 1;
    int q0 = ctx.tid;
    for (; U > 1 && q0 + (U - 1) * ctx.nt < np; q0 += ctx.nt * U) {  // full batches: no guards, the tile stays in registers (U == 1: the loop below is the same)
        decltype(fetch(0)) in[U];
#pragma unroll
        for (int u = 0; u < U; ++u) in[u] = fetch(2 * (q0 + u * ctx.nt));
#pragma unroll
        for (int u = 0; u < U; ++u) body(2 * (q0 + u * ctx.nt), in[u]);
    }
#pragma unroll 1
    for (; q0 < np; q0 += ctx.nt) {
        const auto in = fetch(2 * q0);
        body(2 * q0, in);
    }
}

}  // namespace bsgp
