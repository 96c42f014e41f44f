// Host-side planning shared by libbsgp (bsgp_kernels.cu) and the test-only emulation
// (tests/host_emul): FFT stage factorisation, twiddle tables, cluster / tile geometry, launch shape.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdio.h>
#include <vector>

#include "bsgp_conv.cuh"
#include "bsgp_smem.h"
#include "bsgp_solver.cuh"
#include "bsgp_wrap.h"

namespace bsgp {

inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }
inline bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

// Stage radices (2, 4 or 8: a radix-8 butterfly of complex doubles fits a 128-register thread): every
// stage has an in-block stride >= 8 (conflict-free 16-byte quarter-warp access) except the last,
// whose radix (8) sets the padding period.
inline bool make_fft_plan(int n, FftPlan* pl, int dft_n = 0) {
    static const int table[16][6] = {
        {0}, {0}, {0},
        {3, 0},              // 8
        {1, 3, 0},           // 16   = 2 x 8
        {2, 3, 0},           // 32   = 4 x 8
        {3, 3, 0},           // 64   = 8 x 8
        {2, 2, 3, 0},        // 128  = 4 x 4 x 8
        {2, 3, 3, 0},        // 256  = 4 x 8 x 8
        {3, 3, 3, 0},        // 512
        {2, 2, 3, 3, 0},     // 1024
        {2, 3, 3, 3, 0},     // 2048
        {3, 3, 3, 3, 0},     // 4096
        {2, 2, 3, 3, 3, 0},  // 8192
        {2, 3, 3, 3, 3, 0},  // 16384
        {3, 3, 3, 3, 3, 0}}; // 32768
    if (!is_pow2(n) || n < 8 || n > 32768) return false;
    if (dft_n < 0 || dft_n > n || dft_n > 64) return false;
    pl->n = n;
    pl->dft_n = dft_n;
    pl->log2n = ilog2(n);
    int ns = 0;
    for (int s = 0; s < 6; ++s) pl->log2r[s] = 0;
    while (table[pl->log2n][ns] != 0) { pl->log2r[ns] = table[pl->log2n][ns]; ++ns; }
    pl->nstages = ns;
    pl->pad_shift = pl->log2r[ns - 1];
    pl->plen = n + (n >> pl->pad_shift);
    // run_stage's constant-stride addressing needs every non-final stage stride to be a multiple of the padding period
    int lgL = pl->log2n;
    for (int s = 0; s + 1 < ns; ++s) {
        lgL -= pl->log2r[s];
        if (lgL < pl->pad_shift) return false;
    }
    return true;
}

// W_n^k = exp(-2 pi i k / n), k in [0, n), computed in long double and rounded once.
// A dense transform of length dft_n < n keeps the table size n (the kernels copy n entries to shared memory) and
// fills its first dft_n entries with W_dft_n^k.
template <typename T> inline void make_twiddles(int n, std::vector<cplx<T>>& tw, int dft_n = 0) {
    if (dft_n) {
        tw.assign(n, cplx<T>{(T)0, (T)0});
        const long double two_pi = 6.283185307179586476925286766559005768L;
        for (int k = 0; k < dft_n; ++k) {
            const long double ang = two_pi * (long double)k / (long double)dft_n;
            tw[k].re = (T)cosl(ang);
            tw[k].im = (T)(-sinl(ang));
        }
        tw[0].re = 1; tw[0].im = 0;
        if (dft_n % 2 == 0) { tw[dft_n / 2].re = -1; tw[dft_n / 2].im = 0; }
        if (dft_n % 4 == 0) { tw[dft_n / 4].re = 0; tw[dft_n / 4].im = -1; tw[3 * dft_n / 4].re = 0; tw[3 * dft_n / 4].im = 1; }
        return;
    }
    tw.resize(n);
    const long double two_pi = 6.283185307179586476925286766559005768L;
    for (int k = 0; k < n; ++k) {
        // reduce to the first octant for accuracy
        int kk = k % n;
        long double ang = two_pi * (long double)kk / (long double)n;
        tw[k].re = (T)cosl(ang);
        tw[k].im = (T)(-sinl(ang));
    }
    // exact values on the axes
    tw[0].re = 1; tw[0].im = 0;
    if (n % 4 == 0) { tw[n / 4].re = 0; tw[n / 4].im = -1; tw[n / 2].re = -1; tw[n / 2].im = 0; tw[3 * n / 4].re = 0; tw[3 * n / 4].im = 1; }
}

// Geometry for a cluster of G CTAs and a shared-memory FFT workspace of at most ws_limit bytes.
// Returns false if the shape cannot be handled.
// dft_ny / dft_nx: 0, or the length of the dense DFT that replaces the radix transform along that axis (bsgp_fft.cuh).
// split: bit 0 / bit 1: the rows / columns run split transforms of nx / 2 / ny / 2 points (bsgp_conv.cuh; frame mode only),
// marked in the geometry by px.n == nx / 2 / py.n == ny / 2.  A split row tile holds row_tile_pairs single rows.
inline bool make_geom(int ny, int nx, int G, size_t elem_bytes /* sizeof(cplx<T>) */, size_t ws_limit, ConvGeom* g,
                      size_t* ws_bytes, int dft_ny = 0, int dft_nx = 0, int split = 0) {
    if (!is_pow2(ny) || !is_pow2(nx) || ny < 16 || nx < 16) return false;
    if (split && (dft_ny || dft_nx)) return false;
    if (!make_fft_plan((split & 1) ? nx / 2 : nx, &g->px, dft_nx) || !make_fft_plan((split & 2) ? ny / 2 : ny, &g->py, dft_ny)) return false;
    if ((dft_ny || dft_nx) && G != 1) return false;          // dense transforms: small images, one CTA each
    g->ny = ny; g->nx = nx; g->hx = nx / 2;
    g->lg_nx = ilog2(nx); g->lg_ny = ilog2(ny); g->lg_hx = g->lg_nx - 1;
    g->G = G;
    g->wrap_ny = g->wrap_nx = 0;
    if (ny % (2 * G) != 0 || (nx / 2) % G != 0) return false;
    g->rows_per_cta = ny / G;
    g->cols_per_cta = g->hx / G;
    g->rowstride = g->px.plen;
    g->colstride = g->py.plen | 1;                   // odd: conflict-free transposing loads
    int rtp = g->rows_per_cta / 2;
    while (rtp > 1 && (size_t)rtp * g->rowstride * elem_bytes > ws_limit) rtp >>= 1;
    int ct = g->cols_per_cta;
    while (ct > 1 && (size_t)ct * g->colstride * elem_bytes > ws_limit) ct >>= 1;
    if ((size_t)rtp * g->rowstride * elem_bytes > ws_limit || (size_t)ct * g->colstride * elem_bytes > ws_limit) return false;
    g->row_tile_pairs = rtp;
    g->col_tile = ct;
    g->lg_col_tile = ilog2(ct);
    g->lg_cp = ilog2(g->cols_per_cta);              // panel width of the exchange buffer in frame mode (bsgp_conv.cuh)
    const size_t a = (size_t)rtp * g->rowstride * elem_bytes, b = (size_t)ct * g->colstride * elem_bytes;
    *ws_bytes = a > b ? a : b;
    return true;
}

// The axes whose single transform does not fit a workspace of ws_limit bytes (bit 0: rows, bit 1: columns), make_geom's split
inline int split_axes(int ny, int nx, size_t elem_bytes, size_t ws_limit) {
    FftPlan px, py;
    if (!make_fft_plan(nx, &px) || !make_fft_plan(ny, &py)) return 0;
    return ((size_t)px.plen * elem_bytes > ws_limit ? 1 : 0) | ((size_t)(py.plen | 1) * elem_bytes > ws_limit ? 2 : 0);
}
inline bool has_split(const ConvGeom& g) { return g.px.n != g.nx || g.py.n != g.ny; }

// A plan's request: the FFT grid, the caller's image shape, the cluster size (0: automatic, -1: frame mode) and threads
// per CTA (0: automatic) asked for, and the device's SM count, opt-in shared memory per block and shared memory per SM.
struct PlanRequest {
    int ny, nx, img_ny, img_nx;
    int want_G, want_threads;
    int num_sms, max_smem, smem_per_sm;
};

// The launch shape of a plan: everything the solve and convolution kernels are launched with except the occupancy.
struct LaunchPlan {
    bool frame = false;          // one image over the whole grid (cooperative launch) instead of one per cluster
    int threads = 0, minb = 1;   // solve kernel: threads per CTA and the CTAs per SM it is compiled for
    ConvGeom g{};                // g.G: CTAs per image
    size_t ws_bytes = 0;         // FFT workspace
    SmemPlan sp{};
    int resident_mask = 0;       // bit b: slab array b (Buf) lives in the solve kernel's shared memory
    size_t smem_bytes = 0;       // the solve kernel's dynamic shared memory
    unsigned conv_off_geom = 0, conv_off_ppx = 0, conv_off_ws = 0;
    size_t conv_smem = 0;        // the convolution kernel's dynamic shared memory
};

inline size_t up128(size_t v) { return (v + 127) & ~(size_t)127; }
inline size_t tw_table_entries(int mode, int n) { return mode == 0 ? 0 : (mode == 1 ? (size_t)n : (size_t)64 + (size_t)(n >> 6)); }

// Residency priority: the two projection buffers (read E times per iteration), then the arrays with
// the most touches per iteration; the background image last (unused when the background is a scalar).
constexpr int kResidencyOrder[NBUF] = {B_D, B_T1, B_G, B_X, B_XTF, B_DTF, B_GN, B_BKG};

// The launch shape of a request for element type T.  Makes no CUDA call.  Returns BSGP_OK, or BSGP_E_ARG / BSGP_E_SHAPE
// with the reason written to err.
template <typename T> inline int plan_launch(const PlanRequest& q, LaunchPlan* out, char* err, size_t errlen) {
    LaunchPlan L;
    const size_t npix = (size_t)q.ny * q.nx;
    // short sides that are not a power of two: dense DFT of the image's own length on the first slots of the grid
    // (bsgp_wrap.h); make_geom refuses them for more than one CTA per image, frame mode included
    const int dny = q.ny != q.img_ny ? dense_len(q.img_ny) : 0, dnx = q.nx != q.img_nx ? dense_len(q.img_nx) : 0;
    if (q.ny > kMaxSide || q.nx > kMaxSide) {
        snprintf(err, errlen, "unsupported image shape %dx%d: power-of-two sides up to %d, other sides up to %d", q.img_ny, q.img_nx,
                 kMaxSide, kMaxSide / 2);
        return BSGP_E_SHAPE;
    }
    // A 16384-point axis: one transform takes (16384 + 2048) complex elements of workspace, 144 KB in fp32.  Only frame mode
    // has a workspace that large with room for the 32 KB position table, and only frame mode runs split transforms (fp64:
    // 288 KB, more than a CTA's shared memory); a dense axis runs one CTA per image.
    const bool long_axis = q.ny > kMaxClusterSide || q.nx > kMaxClusterSide;
    if (long_axis) {
        const char* why = dny || dnx ? "a dense axis (a side of at most 32 that is not a power of two) runs one CTA per image"
                        : q.want_G > 0 ? "it runs in frame mode only (cluster size -1 or 0)"
                        : nullptr;
        if (why) {
            snprintf(err, errlen, "unsupported shape %dx%d (FFT grid %dx%d) with a %d-point axis: %s", q.img_ny, q.img_nx, q.ny, q.nx,
                     kMaxSide, why);
            return BSGP_E_SHAPE;
        }
    }
    // Frame mode (bsgp_device.cuh, GridCtx): images of a megapixel or more, and every grid with a 16384-point axis, get the
    // whole GPU each, one CTA per SM on the largest power of two of SMs that divides the image
    L.frame = q.want_G == -1 || (q.want_G == 0 && (npix >= ((size_t)1 << 20) || long_axis));
    int G = q.want_G > 0 ? q.want_G : 1;
    if (L.frame) {
        while (2 * G <= q.num_sms && q.ny % (4 * G) == 0 && (q.nx / 2) % (2 * G) == 0) G *= 2;
    } else if (q.want_G <= 0) {
        // cluster size: slabs of <= 64 KB, at most 8 CTAs (portable cluster limit)
        while (G < 8 && npix * sizeof(T) / G > 65536 && q.ny % (4 * G) == 0 && (q.nx / 2) % (2 * G) == 0) G *= 2;
    }
    const bool auto_threads = q.want_threads <= 0;
    if (!L.frame && !auto_threads && q.want_threads != 128 && q.want_threads != 256 && q.want_threads != 512) {
        snprintf(err, errlen, "threads must be 128, 256 or 512");
        return BSGP_E_ARG;
    }
    // Threads and CTAs per SM.  The solve is a chain of short phases separated by reductions, so one CTA leaves
    // the SM idle while it waits; several small CTAs of DIFFERENT images per SM fill those gaps (measured on
    // B200, 320 solves of 256x256: 1 x 512 threads 112 ms, 2 x 256 threads 94 ms, 4 x 128 threads 87 ms).
    //   big slabs   : 4 CTAs x 128 threads, 38 KB FFT workspace, per-image state in L2 / HBM
    //   small slabs : (stamps) 3 CTAs x 128 or 2 CTAs x 256 threads, everything resident in shared memory
    //   frame mode  : 1 CTA x 512 threads, 160 KB FFT workspace, nothing resident
    // The small-slab launch shapes compile DeviceCtxSmall, whose all-reduce (allreduce_sum8) sums over ONE CTA: a cluster of
    // several CTAs takes the large-slab shapes whatever its slab size (with DeviceCtxSmall its CTAs would each see their
    // own partial sums, take different control paths and never meet at the next cluster barrier).
    const bool small_slab = !L.frame && G == 1 && npix / G * sizeof(T) <= 16384;
    // Small slabs, automatic configuration: three 128-thread CTAs per SM if everything but the background image stays
    // resident in a third of the SM's shared memory (32 x 32 fp64 stamps: 8192 stamps 19.7 ms against 22.8 ms for two
    // 256-thread CTAs); otherwise (e.g. 31 x 31 cut-outs, whose tensor-core table takes 8 KB) two 256-thread CTAs.
    const int ncand = small_slab && auto_threads ? 2 : 1;
    for (int c = 0; c < ncand; ++c) {
        L.threads = L.frame ? 512 : !auto_threads ? q.want_threads : (small_slab && c == 1 ? 256 : 128);
        L.minb = L.threads >= 512 ? 1 : (L.threads >= 256 ? (small_slab ? 2 : 1) : (small_slab ? 3 : 4));
        const size_t ws_limit = L.frame ? 160 * 1024 : (L.minb >= 4 ? 38 : 76) * 1024;
        bool ok = make_geom(q.ny, q.nx, G, sizeof(cplx<T>), ws_limit, &L.g, &L.ws_bytes, dny, dnx);
        if (!ok && L.frame && !dny && !dnx) {
            // one transform of an axis does not fit the frame workspace (fp64 16384): split transforms along that axis only
            const int split = split_axes(q.ny, q.nx, sizeof(cplx<T>), ws_limit);
            ok = split && make_geom(q.ny, q.nx, G, sizeof(cplx<T>), ws_limit, &L.g, &L.ws_bytes, 0, 0, split);
        }
        if (!ok && !L.frame && auto_threads) {
            // one transform does not fit the small workspace (sides >= 4096): fall back to one big CTA per SM
            L.threads = 512; L.minb = 1;
            ok = make_geom(q.ny, q.nx, G, sizeof(cplx<T>), 160 * 1024, &L.g, &L.ws_bytes, dny, dnx);
        }
        if (!ok) {
            if (L.frame) snprintf(err, errlen, "unsupported shape %dx%d for frame mode (grid of %d CTAs)", q.ny, q.nx, G);
            else snprintf(err, errlen, "unsupported shape %dx%d for cluster size %d (power-of-two sides >= 16 required)", q.ny, q.nx, G);
            return BSGP_E_SHAPE;
        }
        if (L.frame) {
            // Panel width of the exchange buffer (bsgp_conv.cuh, spec_idx).  A column tile narrower than the panel reads 16 bytes
            // of every 32-byte sector per sweep; with panels of max(col_tile, 4) columns the sectors one sweep fetches are the
            // ones the next column's sweep needs, and they are still in L2 (4-column panel x 8192 rows x 128 CTAs = 64 MB), so
            // the column pass reads the buffer once from DRAM instead of twice (8192^2: 121.5 -> 103.4 ms per 10 iterations).
            const int want = L.g.lg_col_tile > 2 ? L.g.lg_col_tile : 2;
            if (want < L.g.lg_cp) L.g.lg_cp = want;
        }
        // the solve kernel: [SharedCtl][ImgState][CtlState x warps][twiddles][position table][workspace][resident slabs]
        SmemPlan& sp = L.sp;
        size_t off = up128(sizeof(SharedCtl));
        sp.off_state = (unsigned)off; off = up128(off + sizeof(ImgState<T>));
        sp.ctl_stride = (unsigned)((sizeof(CtlState<T>) + 15) & ~(size_t)15);
        sp.off_ctl = (unsigned)off; off = up128(off + (size_t)(L.threads / 32) * sp.ctl_stride);
        // full twiddle tables in shared memory when they fit 16 KB; otherwise global memory (cluster mode) or two-level
        // tables of 64 + n/64 entries (frame mode).  A dense axis of an fp64 plan keeps the DMMA fragment table of its
        // transform there instead (bsgp_fft.cuh, fill_dense_table)
        const size_t tw_bytes = ((size_t)q.nx + (q.ny != q.nx ? q.ny : 0)) * sizeof(cplx<T>);
        sp.tw_smem = tw_bytes <= 16384 ? 1 : (L.frame ? 2 : 0);
        auto tw_bytes_of = [&](int n, int dft_n) -> size_t {
            if (dft_n && sizeof(T) == 8) return (size_t)8 * n * n;
            return tw_table_entries(sp.tw_smem, n) * sizeof(cplx<T>);
        };
        sp.off_twx = sp.off_twy = (unsigned)off;
        off = up128(off + tw_bytes_of(q.nx, L.g.px.dft_n));
        if (q.ny != q.nx || L.g.py.dft_n != L.g.px.dft_n) { sp.off_twy = (unsigned)off; off = up128(off + tw_bytes_of(q.ny, L.g.py.dft_n)); }
        sp.off_ppx = (unsigned)off; off = up128(off + (size_t)q.nx * sizeof(unsigned short));
        sp.off_ws = (unsigned)off; off = up128(off + L.ws_bytes);
        sp.off_bufs = (unsigned)off;
        // resident slabs in cluster mode, in priority order, within the per-CTA budget: the opt-in maximum, or an equal
        // share of the SM (1 KB per CTA is reserved by the system)
        size_t budget = (size_t)q.max_smem;
        if (L.minb > 1) {
            const size_t share = ((size_t)q.smem_per_sm - (size_t)L.minb * 1024) / L.minb;
            budget = share < budget ? share : budget;
            budget &= ~(size_t)127;
        }
        const size_t slab_bytes = npix / G * sizeof(T);
        L.smem_bytes = off;
        L.resident_mask = 0;
        for (int k = 0; !L.frame && k < NBUF; ++k) {
            if (L.smem_bytes + slab_bytes <= budget) { L.resident_mask |= 1 << kResidencyOrder[k]; L.smem_bytes += slab_bytes; }
        }
        if ((L.resident_mask | (1 << B_BKG)) == (1 << NBUF) - 1) break;
    }
    if (L.smem_bytes > (size_t)q.max_smem) {
        snprintf(err, errlen, "shape %dx%d needs %zu B of shared memory per CTA (limit %d)", q.ny, q.nx, L.smem_bytes, q.max_smem);
        return BSGP_E_SHAPE;
    }
    // the stand-alone convolution kernel: [SharedCtl][ConvGeom][position table][workspace]
    L.conv_off_geom = (unsigned)up128(sizeof(SharedCtl));
    L.conv_off_ppx = (unsigned)up128(L.conv_off_geom + sizeof(ConvGeom));
    L.conv_off_ws = (unsigned)up128(L.conv_off_ppx + (size_t)q.nx * sizeof(unsigned short));
    L.conv_smem = L.conv_off_ws + up128(L.ws_bytes);
    // fold widths of wrapped axes; a dense axis is circular by itself
    L.g.wrap_ny = (q.ny != q.img_ny && !L.g.py.dft_n) ? q.img_ny : 0;
    L.g.wrap_nx = (q.nx != q.img_nx && !L.g.px.dft_n) ? q.img_nx : 0;
    *out = L;
    return BSGP_OK;
}

}  // namespace bsgp
