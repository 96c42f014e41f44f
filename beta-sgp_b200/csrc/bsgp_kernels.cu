// libbsgp: C ABI (include/bsgp.h), plan management and the small stand-alone kernels of the B200
// (sm_100a) SGP / beta-SGP restoration path.  The persistent cluster solve kernel lives in
// bsgp_solve_kernel.cuh (instantiated by bsgp_solve_f64.cu / bsgp_solve_f32.cu).
//
// Execution model
//   * One thread-block CLUSTER of G CTAs restores one image from start to finish
//     (bsgp_solver.cuh); clusters are persistent and pull image indices from a global queue, so
//     images with very different iteration counts (2..160 observed) never wait for each other and
//     the host is not involved between "inputs resident" and "outputs written".
//   * Scalars travel between the CTAs of a cluster through distributed shared memory
//     (bsgp_device.cuh).
//   * Per-image state that does not fit in shared memory lives in a per-CLUSTER scratch area (not
//     per image) in global memory.  Big slabs run as 4 small CTAs of different images per SM (71 clusters
//     in flight for 256x256), so that scratch streams through L2 / HBM; stamps keep everything in shared
//     memory.  Images of a megapixel or more use frame mode: one image over the whole (cooperative) grid.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "bsgp_device.cuh"
#include "bsgp_launch.h"
#include "bsgp_plan.h"
#include "bsgp_solver.cuh"
#include "bsgp_wrap.h"

using namespace bsgp;

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
template <typename T> struct ConvArgs {
    ConvGeom g;
    int count;
    const T* in; T* out;                // images / PSFs [count][ny][nx]
    const cplx<T>* twx; const cplx<T>* twy; cplx<T>* tf; int n_psf; size_t tf_stride;
    cplx<T>* spec; size_t spec_stride;
    int mode;                           // CONV_TF / CONV_CTF / CONV_MAKE_TF
    int* queue;
};

// mode CONV_MAKE_TF: tf[p] = fftn(fftshift(psf[p])) in workspace order (sgp.py:109); otherwise
// out[i] = A(in[i]) or A^T(in[i]) (sgp.py:111-120).  Dynamic shared memory: [SharedCtl][ConvGeom][position table][workspace].
// `cluster_id` selects this cluster's exchange buffer; next() hands out the items.
template <typename T, class Ctx, class Next>
__device__ __forceinline__ void conv_items(Ctx& ctx, const ConvArgs<T>& a, const unsigned off_geom, const unsigned off_ppx, const unsigned off_ws,
                                           const int cluster_id, Next next) {
    unsigned char* smem = dyn_smem();
    ConvGeom* gs = reinterpret_cast<ConvGeom*>(smem + off_geom);
    unsigned short* ppx = reinterpret_cast<unsigned short*>(smem + off_ppx);
    if (ctx.tid == 0) *gs = a.g;
    fill_pos_table(ctx, a.g.px, ppx);
    __syncthreads();
    const ConvGeom& g = *gs;
    const int ny = a.g.ny, nx = a.g.nx;
    const size_t npix = (size_t)ny * nx;
    cplx<T>* spec = a.spec + (size_t)cluster_id * a.spec_stride;
    const int r0 = ctx.rank * a.g.rows_per_cta;
    for (;;) {
        const int img = next();
        if (img >= a.count) break;
        const T* src = a.in + (size_t)img * npix;
        if (a.mode == CONV_MAKE_TF) {
            const int lg_nx = a.g.lg_nx;
            auto pf = [&](int i) {
                const int row = i >> lg_nx, c = i & (nx - 1);
                In1<T> r; r.a = ld2(src + (size_t)((r0 + row + (ny >> 1)) & (ny - 1)) * nx, (c + (nx >> 1)) & (nx - 1)); return r;
            };
            auto pe = [&](int, const In1<T>& in) -> V2<T> { return in.a; };
            ctx.sync();
            conv_rows_forward<2, true>(ctx, g, off_ws, a.twx, kNoSmem, 0, off_ppx, spec, pf, pe);
            ctx.cluster_sync();
            conv_cols<true>(ctx, gs, off_ws, a.twy, kNoSmem, 0, spec, a.tf + (size_t)img * a.tf_stride, CONV_MAKE_TF);
        } else {
            T* dst = a.out + (size_t)img * npix + (size_t)r0 * nx;
            const T* s0 = src + (size_t)r0 * nx;
            auto pf = [&](int i) { In1<T> r; r.a = ld2(s0, i); return r; };
            auto pe = [&](int, const In1<T>& in) -> V2<T> { return in.a; };
            auto cf = [&](int) { In1<T> r; r.a = mk2((T)0, (T)0); return r; };
            auto ca = [&](int i, const In1<T>&, V2<T> v) { st2(dst, i, v); };
            ctx.sync();
            conv_rows_forward<2, true>(ctx, g, off_ws, a.twx, kNoSmem, 0, off_ppx, spec, pf, pe);
            ctx.cluster_sync();
            conv_cols<true>(ctx, gs, off_ws, a.twy, kNoSmem, 0, spec, a.tf + (a.n_psf > 1 ? (size_t)img * a.tf_stride : 0), a.mode);
            ctx.cluster_sync();
            conv_rows_inverse<2, true>(ctx, g, off_ws, a.twx, kNoSmem, 0, off_ppx, spec, cf, ca);
        }
        ctx.cluster_sync();   // spec is reused by the next item
    }
}

// one cluster per item, from the work queue
template <typename T>
__global__ void __launch_bounds__(512, 1) bsgp_conv_kernel(const ConvArgs<T> a, const unsigned off_geom, const unsigned off_ppx, const unsigned off_ws) {
    DeviceCtx ctx = make_ctx(reinterpret_cast<SharedCtl*>(dyn_smem()), a.g.G);
    conv_items(ctx, a, off_geom, off_ppx, off_ws, blockIdx.x / a.g.G, [&] {
        bool ready_ok;
        return next_item(ctx, a.queue, nullptr, a.count, &ready_ok);
    });
}

// frame mode: every item, one after the other, by the whole (cooperative) grid
template <typename T>
__global__ void __launch_bounds__(512, 1) bsgp_conv_frame_kernel(const ConvArgs<T> a, const unsigned off_geom, const unsigned off_ppx, const unsigned off_ws,
                                                                 double* gpart) {
    GridCtx ctx = make_grid_ctx(reinterpret_cast<SharedCtl*>(dyn_smem()), gpart);
    conv_items(ctx, a, off_geom, off_ppx, off_ws, 0, [img = 0]() mutable { return img++; });
}

// projectDF (flux_conserve_proj.py:7-144): one CTA per problem, x = clamp((c + lambda) / dia).
__global__ void __launch_bounds__(512, 1) bsgp_project_kernel(const double* __restrict__ b, const double* __restrict__ c,
                                                              const double* __restrict__ dia, int n, int batch, double cap, int has_cap,
                                                              double lambda0, double dlambda0, double tol_lam, int max_projs, int biter0, int siter0,
                                                              double* __restrict__ x, int* evals, int* status) {
    __shared__ SharedCtl ctl;
    DeviceCtx ctx = make_ctx(&ctl, 1);
    for (int p = blockIdx.x; p < batch; p += gridDim.x) {
        const double* cp = c + (size_t)p * n;
        const double* dp = dia + (size_t)p * n;
        auto point = [&](int i, double lam) -> double {
            double v = ndiv(nadd(cp[i], lam), dp[i]);
            v = (v <= 0.0) ? 0.0 : v;
            if (has_cap) v = (v >= cap) ? cap : v;
            return v;
        };
        const double target = b[p];
        auto eval = [&](double lam) -> double {
            KSum s; s.clear();
            for (int i = ctx.tid; i < n; i += ctx.nt) s.add(point(i, lam));
            double t = s.value();
            ctx.allreduce_sum(&t, 1);
            return t - target;
        };
        const ProjResult pr = flux_rootfind(eval, target, max_projs, lambda0, dlambda0, tol_lam, biter0, siter0);
        for (int i = ctx.tid; i < n; i += ctx.nt) x[(size_t)p * n + i] = point(i, pr.lambda);
        if (ctx.tid == 0) { if (evals) evals[p] = pr.evals; if (status) status[p] = pr.status; }
        __syncthreads();
    }
}

// betaDiv partial sums + optional betaDivDeriv (sgp.py:441-495).  part[block][3]
__global__ void __launch_bounds__(256) bsgp_betadiv_kernel(const double* __restrict__ y, const double* __restrict__ x, long long n,
                                                           double beta, double* part, double* deriv) {
    __shared__ SharedCtl ctl;
    DeviceCtx ctx = make_ctx(&ctl, 1);
    DivK<double> dk = make_divk<double>(BSGP_DIV_BETA, beta);
    KSum acc[3];
    acc[0].clear(); acc[1].clear(); acc[2].clear();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        objective_pixel<double>(dk, x[i], y[i], 0.0, true, acc);
        if (deriv) deriv[i] = (dk.kind == 1) ? dbeta_pixel<false, double>(x[i], y[i], beta) : 0.0;
    }
    double v[3] = {acc[0].value(), acc[1].value(), acc[2].value()};
    ctx.allreduce_sum(v, 3);
    if (threadIdx.x == 0) { part[blockIdx.x * 3 + 0] = v[0]; part[blockIdx.x * 3 + 1] = v[1]; part[blockIdx.x * 3 + 2] = v[2]; }
}

// the two per-pixel pieces of betaDivDerivwrtY (sgp.py:498-499): p1 = den^(beta-1), u = gn * den^(beta-2)
__global__ void __launch_bounds__(256) bsgp_betagrad_kernel(const double* __restrict__ den, const double* __restrict__ gn, long long n,
                                                            double beta, double* __restrict__ p1, double* __restrict__ u) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double d = den[i];
        const double p = mpow(d, beta - 1.0);
        p1[i] = p;
        u[i] = nmul(gn[i], ndiv(p, d));
    }
}

// ------------------------------------------------------------------------------------------------
// Tiling of a frame into overlapping subdivisions and re-assembly (reference: utils.py:332-389 create_subdivisions /
// calculate_slice_bboxes, utils.py:392-397 reconstruct_full_image_from_patches).  Pure data movement, HBM-bound:
// every thread moves one pixel, consecutive threads consecutive columns (tile origins are arbitrary, so rows are
// not 16-byte aligned in general); grids are sized in multiples of the SM count.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void bsgp_extract_tiles_kernel(const T* __restrict__ frame, int height, int width, const int* __restrict__ origins, int n, int th, int tw, T* __restrict__ tiles) {
    const size_t per = (size_t)th * tw, total = per * n;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int t = (int)(e / per);
        const int r = (int)((e - (size_t)t * per) / tw), c = (int)(e - (size_t)t * per - (size_t)r * tw);
        const int y = origins[2 * t] + r, x = origins[2 * t + 1] + c;
        tiles[e] = (y >= 0 && y < height && x >= 0 && x < width) ? frame[(size_t)y * width + x] : (T)0;
    }
}

// out(y, x) = sum_t w_t tile_t / sum_t w_t over the tiles covering the pixel, in tile order (deterministic), with
// w_t = ramp(dy) * ramp(dx), ramp(d) = min(d + 1, size - d, feather): a linear cross-fade over `feather` pixels at
// tile borders (feather <= 1: plain average of the overlapping tiles).  Pixels covered by no tile get 0.
template <typename T>
__global__ void bsgp_assemble_tiles_kernel(const T* __restrict__ tiles, const int* __restrict__ origins, int n, int th, int tw, int feather, T* __restrict__ frame, int height, int width) {
    const size_t total = (size_t)height * width, per = (size_t)th * tw;
    const int f = feather < 1 ? 1 : feather;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(e / width), x = (int)(e - (size_t)y * width);
        double num = 0.0, den = 0.0;
        for (int t = 0; t < n; ++t) {
            const int dy = y - origins[2 * t], dx = x - origins[2 * t + 1];
            if (dy < 0 || dy >= th || dx < 0 || dx >= tw) continue;
            int wy = dy + 1 < th - dy ? dy + 1 : th - dy; wy = wy < f ? wy : f;
            int wx = dx + 1 < tw - dx ? dx + 1 : tw - dx; wx = wx < f ? wx : f;
            const double w = (double)wy * (double)wx;
            num += w * (double)tiles[(size_t)t * per + (size_t)dy * tw + dx];
            den += w;
        }
        frame[e] = den > 0.0 ? (T)(num / den) : (T)0;
    }
}

// ------------------------------------------------------------------------------------------------
// Embedded plans: image sides that are not a power of two in [16, 8192] (the reference's numpy closure takes any
// size, sgp.py:108-120; its star-stamp application runs it on 31 x 31 cut-outs, application_sgp_star_stamps.py:24,58).
// Per axis (bsgp_wrap.h): a side n <= 32 keeps a grid of 16 or 32 slots and is transformed by a dense DFT of length n
// over the first n slots (the circular operator itself, no fold); any other side is WRAPPED:
// the image sits at the origin of a power-of-two grid of side P >= 2 n - 1 (zeros elsewhere) and the circular
// convolution with h = fftshift(psf) (sgp.py:109: np.roll by n // 2, which for odd n puts the PSF centre at index
// n - 1, not 0) is computed as the LINEAR convolution on the grid followed by the fold out[i] = z[i] + z[i + n]
// (conv_cols / conv_rows_inverse).  A^T = correlation with h = convolution with h~[j] = h[(-j) mod n], so both
// operators are "kernel on [0, n)^2, CONV_TF, fold"; the plan keeps the two spectra (tf, tf_adj).
// The kernels below move user arrays [count][iny][inx] to / from the grid [count][ny][nx]; pure data movement,
// one pixel per thread, consecutive threads consecutive columns, grids sized in multiples of the SM count.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void bsgp_embed_images_kernel(const T* __restrict__ src, int iny, int inx, T* __restrict__ dst, int ny, int nx, size_t count) {
    const size_t per = (size_t)ny * nx, total = per * count;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t b = e / per;
        const int r = (int)((e - b * per) / nx), c = (int)(e - b * per - (size_t)r * nx);
        dst[e] = (r < iny && c < inx) ? src[(b * iny + r) * inx + c] : (T)0;
    }
}

template <typename T>
__global__ void bsgp_crop_images_kernel(const T* __restrict__ src, int ny, int nx, T* __restrict__ dst, int iny, int inx, size_t count) {
    const size_t per = (size_t)iny * inx, total = per * count;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t b = e / per;
        const int r = (int)((e - b * per) / inx), c = (int)(e - b * per - (size_t)r * inx);
        dst[e] = src[(b * ny + r) * nx + c];
    }
}

// the kernel of A (adjoint = 0) or A^T (adjoint = 1) on the grid, in the placement CONV_MAKE_TF expects (bsgp_wrap.h)
template <typename T>
__global__ void bsgp_embed_psf_kernel(const T* __restrict__ psf, int iny, int inx, T* __restrict__ out, int ny, int nx, size_t count, int adjoint) {
    const size_t per = (size_t)ny * nx, total = per * count;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t b = e / per;
        const int r = (int)((e - b * per) / nx), c = (int)(e - b * per - (size_t)r * nx);
        int sr, sc;
        out[e] = wrap_psf_source(r, c, ny, nx, iny, inx, adjoint, &sr, &sc) ? psf[(b * iny + sr) * inx + sc] : (T)0;
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// PSF model evaluation (reference: psf/psf_calculate.py:52-111, PSF.calc_psf_pix / get_psf_mat / normalize_psf_mat): the
// DIAPL model, a sum of `ngauss` elliptical Gaussians (widths in geometric progression) times a local polynomial of degree
// 2 in (x, y).  One CTA evaluates one PSF on its (2 hw + 1)^2 support, sums it and writes it, optionally normalised to
// sum 1, centred at (ny/2, nx/2) of an ny x nx image (zeros elsewhere): the placement the circular operator expects
// (sgp.py:109, fftshift), so per-stamp PSFs are generated where they are used instead of being uploaded.
// params row: cos, sin, ax, ay, sigma_inc, then ngauss * 6 coefficients.  Operand order follows the reference.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double psf_model_pixel(const double* __restrict__ pr, int ngauss, double x, double y) {
    const double x1 = __dsub_rn(__dmul_rn(pr[0], x), __dmul_rn(pr[1], y));
    const double y1 = __dadd_rn(__dmul_rn(pr[1], x), __dmul_rn(pr[0], y));
    double rr = __dadd_rn(__dmul_rn(__dmul_rn(pr[2], x1), x1), __dmul_rn(__dmul_rn(pr[3], y1), y1));
    const double s2 = __dmul_rn(pr[4], pr[4]);
    double v = 0.0;
    int ic = 5;
    for (int ig = 0; ig < ngauss; ++ig) {
        const double f = exp(rr);
        double a1 = 1.0;
        for (int m = 0; m <= 2; ++m) {
            double a2 = 1.0;
            for (int n = 0; n <= 2 - m; ++n) {
                v = __dadd_rn(v, __dmul_rn(__dmul_rn(__dmul_rn(pr[ic], f), a1), a2));
                ++ic;
                a2 = __dmul_rn(a2, y);
            }
            a1 = __dmul_rn(a1, x);
        }
        rr = __dmul_rn(rr, s2);
    }
    return v;
}

template <typename T>
__global__ void bsgp_psf_model_kernel(const double* __restrict__ params, int stride, int ngauss, int hw, int ny, int nx, int normalize, T* __restrict__ out) {
    __shared__ double part[32];
    __shared__ double total;
    const double* pr = params + (size_t)blockIdx.x * stride;
    T* o = out + (size_t)blockIdx.x * ny * nx;
    const int side = 2 * hw + 1, npix = side * side;
    const int cy = ny / 2, cx = nx / 2;
    for (int e = threadIdx.x; e < ny * nx; e += blockDim.x) o[e] = (T)0;
    double s = 0.0;
    for (int e = threadIdx.x; e < npix; e += blockDim.x) {
        const int i = e / side - hw, j = e % side - hw;              // i: row offset (y), j: column offset (x)
        s += psf_model_pixel(pr, ngauss, (double)j, (double)i);
    }
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)((blockDim.x + 31) >> 5); ++w) t += part[w];
        total = t;
    }
    __syncthreads();
    const double scale = normalize ? total : 1.0;
    for (int e = threadIdx.x; e < npix; e += blockDim.x) {
        const int i = e / side - hw, j = e % side - hw;
        const int yy = cy + i, xx = cx + j;
        if (yy < 0 || yy >= ny || xx < 0 || xx >= nx) continue;
        o[(size_t)yy * nx + xx] = (T)__ddiv_rn(psf_model_pixel(pr, ngauss, (double)j, (double)i), scale);
    }
}

static thread_local std::string g_err;
// kernels launched by this library since it was loaded (bsgp_launch_count): what a caller reports as "my kernels ran"
static std::atomic<long long> g_launches{0};
static inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CU(expr)                                                                                          \
    do {                                                                                                  \
        cudaError_t e__ = (expr);                                                                         \
        if (e__ != cudaSuccess) return fail(BSGP_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

// a plan is its launch shape (bsgp_plan.h, plan_launch) and the device state that goes with it
struct bsgp_plan : LaunchPlan {
    int ny = 0, nx = 0, dtype = 0, device = 0;   // ny, nx: the power-of-two FFT grid the kernels work on
    int img_ny = 0, img_nx = 0;                   // the caller's image shape (== grid unless the plan is wrapped)
    bool embedded = false;                        // wrapped plan: user arrays are moved to / from the grid by the library
    void* emb_psf = nullptr; size_t emb_psf_cap = 0;   // grow-only staging: PSFs on the grid
    void* emb_img = nullptr; size_t emb_img_cap = 0;   //                    images on the grid (inputs and restored output)
    cudaEvent_t ev_last = nullptr;                // completion of the plan's most recent launch (cross-stream ordering)
    int num_sms = 0, max_smem = 0, smem_per_sm = 0;
    int want_G = 0, want_threads = 0;
    bool configured = false;
    size_t elem = 8;
    int num_clusters = 0, conv_clusters = 0;
    void* twx = nullptr; void* twy = nullptr;
    void* tf = nullptr; int n_psf = 0; int tf_capacity = 0; size_t tf_stride = 0;
    void* tf_adj = nullptr; int n_psf_adj = 0; int tf_adj_capacity = 0;   // spectra of the second (adjoint) kernel
    void* work = nullptr; size_t work_stride = 0;
    void* spec = nullptr; size_t spec_stride = 0;
    int* queue = nullptr;
    double* gpart = nullptr;     // frame mode: all-reduce partials [2][G][kMaxK]
    size_t workspace_bytes = 0;
    // pipelined host path (bsgp_solve_batch_pinned): grow-only device staging, ready flags, two private streams
    void* stage = nullptr; size_t stage_cap = 0;
    int* ready = nullptr; int* ones_host = nullptr; int ready_cap = 0;
    cudaStream_t s_copy = nullptr, s_run = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_flags = nullptr, ev_copy = nullptr, ev_run = nullptr;
};

template <typename T> static const void* conv_kernel_ptr() { return (const void*)bsgp_conv_kernel<T>; }

static void plan_free_pipeline(bsgp_plan* p) {
    cudaFree(p->stage); cudaFree(p->ready); cudaFreeHost(p->ones_host);
    cudaFree(p->emb_psf); cudaFree(p->emb_img);
    p->emb_psf = p->emb_img = nullptr; p->emb_psf_cap = p->emb_img_cap = 0;
    if (p->ev_last) { cudaEventDestroy(p->ev_last); p->ev_last = nullptr; }
    p->stage = nullptr; p->stage_cap = 0; p->ready = nullptr; p->ones_host = nullptr; p->ready_cap = 0;
    if (p->s_copy) cudaStreamDestroy(p->s_copy);
    if (p->s_run) cudaStreamDestroy(p->s_run);
    p->s_copy = p->s_run = nullptr;
    for (cudaEvent_t* e : {&p->ev_fork, &p->ev_flags, &p->ev_copy, &p->ev_run}) { if (*e) cudaEventDestroy(*e); *e = nullptr; }
}

static void plan_free_buffers(bsgp_plan* p) {
    cudaFree(p->twx); cudaFree(p->twy); cudaFree(p->tf); cudaFree(p->tf_adj); cudaFree(p->work); cudaFree(p->spec); cudaFree(p->queue); cudaFree(p->gpart);
    p->twx = p->twy = p->tf = p->work = p->spec = nullptr; p->queue = nullptr; p->gpart = nullptr;
    p->tf_capacity = 0; p->n_psf = 0; p->tf_adj = nullptr; p->tf_adj_capacity = 0; p->n_psf_adj = 0;
}

template <typename T> static const void* conv_frame_kernel_ptr() { return (const void*)bsgp_conv_frame_kernel<T>; }

template <typename T> static int alloc_tables(bsgp_plan* p) {
    std::vector<cplx<T>> tw;
    make_twiddles<T>(p->nx, tw, p->g.px.dft_n);
    CU(cudaMalloc(&p->twx, tw.size() * sizeof(cplx<T>)));
    CU(cudaMemcpy(p->twx, tw.data(), tw.size() * sizeof(cplx<T>), cudaMemcpyHostToDevice));
    make_twiddles<T>(p->ny, tw, p->g.py.dft_n);
    CU(cudaMalloc(&p->twy, tw.size() * sizeof(cplx<T>)));
    CU(cudaMemcpy(p->twy, tw.data(), tw.size() * sizeof(cplx<T>), cudaMemcpyHostToDevice));
    return BSGP_OK;
}

// The launch shape (plan_launch), how many clusters of it fit the device, and the plan's device buffers.  A frame plan
// is one "cluster" of G CTAs for both kernels.
template <typename T> static int plan_setup_t(bsgp_plan* p) {
    const PlanRequest q{p->ny, p->nx, p->img_ny, p->img_nx, p->want_G, p->want_threads, p->num_sms, p->max_smem, p->smem_per_sm};
    LaunchPlan L;
    char err[256];
    const int code = plan_launch<T>(q, &L, err, sizeof err);
    if (code) return fail(code, "%s", err);
    static_cast<LaunchPlan&>(*p) = L;
    p->elem = sizeof(T);
    const int G = p->g.G;
    if (p->frame) {
        int coop = 0;
        CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, p->device));
        if (!coop) return fail(BSGP_E_CUDA, "device does not support cooperative launches (frame mode)");
        LaunchCfg lc{G, 512, 1, p->smem_bytes, nullptr, 1};
        int per_sm = 0;
        cudaError_t e = query_frame_ctas<T, false>(lc, &per_sm);
        if (e != cudaSuccess) return fail(BSGP_E_CUDA, "occupancy query failed: %s", cudaGetErrorString(e));
        if (per_sm < 1) return fail(BSGP_E_CUDA, "frame kernel does not fit: %zu B shared memory", p->smem_bytes);
        CU(cudaFuncSetAttribute(conv_frame_kernel_ptr<T>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->conv_smem));
        p->num_clusters = p->conv_clusters = 1;
    } else {
        LaunchCfg lc{G * p->num_sms, p->threads, G, p->smem_bytes, nullptr, p->minb};
        int nc = 0;
        cudaError_t e = query_solve_clusters<T, false>(lc, p->num_sms, &nc);
        if (e != cudaSuccess) return fail(BSGP_E_CUDA, "occupancy query failed: %s", cudaGetErrorString(e));
        if (nc <= 0) return fail(BSGP_E_CUDA, "kernel does not fit: cluster %d, %d threads, %zu B shared memory", G, p->threads, p->smem_bytes);
        p->num_clusters = nc;
        LaunchCfg cc{G * p->num_sms, 512, G, p->conv_smem, nullptr};
        e = query_clusters(conv_kernel_ptr<T>(), cc, p->num_sms, &nc);
        if (e != cudaSuccess) return fail(BSGP_E_CUDA, "occupancy query failed: %s", cudaGetErrorString(e));
        if (nc <= 0) return fail(BSGP_E_CUDA, "convolution kernel does not fit: cluster %d, %zu B shared memory", G, p->conv_smem);
        p->conv_clusters = nc;
    }
    { int rc = alloc_tables<T>(p); if (rc) return rc; }
    const int nscratch = p->num_clusters > p->conv_clusters ? p->num_clusters : p->conv_clusters;
    p->work_stride = NBUF * (size_t)p->ny * p->nx;
    p->spec_stride = (size_t)p->ny * p->g.hx;
    p->tf_stride = (size_t)(p->g.hx + 1) * p->ny;
    CU(cudaMalloc(&p->work, (size_t)p->num_clusters * p->work_stride * sizeof(T)));
    CU(cudaMalloc(&p->spec, (size_t)nscratch * p->spec_stride * sizeof(cplx<T>)));
    CU(cudaMalloc((void**)&p->queue, sizeof(int)));
    if (p->frame) CU(cudaMalloc((void**)&p->gpart, (size_t)2 * G * kMaxK * sizeof(double)));
    p->workspace_bytes = (size_t)p->num_clusters * p->work_stride * sizeof(T) + (size_t)nscratch * p->spec_stride * sizeof(cplx<T>);
    p->configured = true;
    return BSGP_OK;
}

static int plan_setup(bsgp_plan* p) {
    if (p->configured) return BSGP_OK;
    CU(cudaSetDevice(p->device));
    return p->dtype == BSGP_F64 ? plan_setup_t<double>(p) : plan_setup_t<float>(p);
}

// Stream ordering of a plan.  A plan owns mutable device state (PSF spectra, per-cluster scratch, the work-queue counter),
// so two launches on the same plan must not overlap.  Every public device entry point makes its stream wait for the
// plan's previous launch and records its own completion: callers may use one plan from several streams, the launches
// are serialised on the device (include/bsgp.h, "Streams").
static int plan_enter(bsgp_plan* p, cudaStream_t st) {
    if (!p->ev_last) { CU(cudaEventCreateWithFlags(&p->ev_last, cudaEventDisableTiming)); return BSGP_OK; }
    CU(cudaStreamWaitEvent(st, p->ev_last, 0));
    return BSGP_OK;
}
static int plan_leave(bsgp_plan* p, cudaStream_t st) {
    CU(cudaEventRecord(p->ev_last, st));
    return BSGP_OK;
}

static int grow(void** buf, size_t* cap, size_t bytes) {
    if (bytes <= *cap) return BSGP_OK;
    cudaFree(*buf); *buf = nullptr; *cap = 0;           // cudaFree waits for the work that may still use the old buffer
    CU(cudaMalloc(buf, bytes));
    *cap = bytes;
    return BSGP_OK;
}

static int data_grid(int device, size_t total, int* blocks) {
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    size_t want = (total + 255) / 256, cap = (size_t)sms * 8;          // 8 CTAs of 256 threads per SM, grid-stride beyond
    *blocks = (int)(want < cap ? (want ? want : 1) : cap);
    return BSGP_OK;
}

// user images [count][img_ny][img_nx] -> grid [count][ny][nx] (zeros in the padding) and back
template <typename T> static int embed_images(bsgp_plan* p, const void* src, void* dst, size_t count, cudaStream_t st) {
    int blocks = 0, rc = data_grid(p->device, count * p->ny * p->nx, &blocks);
    if (rc) return rc;
    count_launch();
    bsgp_embed_images_kernel<T><<<blocks, 256, 0, st>>>((const T*)src, p->img_ny, p->img_nx, (T*)dst, p->ny, p->nx, count);
    CU(cudaGetLastError());
    return BSGP_OK;
}
template <typename T> static int crop_images(bsgp_plan* p, const void* src, void* dst, size_t count, cudaStream_t st) {
    int blocks = 0, rc = data_grid(p->device, count * p->img_ny * p->img_nx, &blocks);
    if (rc) return rc;
    count_launch();
    bsgp_crop_images_kernel<T><<<blocks, 256, 0, st>>>((const T*)src, p->ny, p->nx, (T*)dst, p->img_ny, p->img_nx, count);
    CU(cudaGetLastError());
    return BSGP_OK;
}

template <typename T> static int launch_conv(bsgp_plan* p, ConvArgs<T>& a, int count, cudaStream_t st) {
    if (p->frame) {
        unsigned og = p->conv_off_geom, op = p->conv_off_ppx, ow = p->conv_off_ws;
        double* gp = p->gpart;
        void* args[] = {&a, &og, &op, &ow, &gp};
        count_launch();
        cudaError_t e = cudaLaunchCooperativeKernel(conv_frame_kernel_ptr<T>(), dim3(p->g.G), dim3(512), args, p->conv_smem, st);
        if (e != cudaSuccess) return fail(BSGP_E_CUDA, "convolution kernel launch failed: %s", cudaGetErrorString(e));
        return BSGP_OK;
    }
    CU(cudaMemsetAsync(p->queue, 0, sizeof(int), st));
    const int nclu = count < p->conv_clusters ? count : p->conv_clusters;
    LaunchCfg lc{nclu * p->g.G, 512, p->g.G, p->conv_smem, st};
    unsigned og = p->conv_off_geom, op = p->conv_off_ppx, ow = p->conv_off_ws;
    void* args[] = {&a, &og, &op, &ow};
    count_launch();
    cudaError_t e = launch_clustered(conv_kernel_ptr<T>(), lc, args);
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "convolution kernel launch failed: %s", cudaGetErrorString(e));
    return BSGP_OK;
}

template <typename T> static int set_psf_t(bsgp_plan* p, const void* psf_dev, int n_psf, cudaStream_t st, bool adjoint_kernel = false) {
    void*& tfbuf = adjoint_kernel ? p->tf_adj : p->tf;
    int& cap = adjoint_kernel ? p->tf_adj_capacity : p->tf_capacity;
    if (n_psf > cap) {
        cudaFree(tfbuf); tfbuf = nullptr; cap = 0;
        CU(cudaMalloc(&tfbuf, (size_t)n_psf * p->tf_stride * sizeof(cplx<T>)));
        cap = n_psf;
    }
    (adjoint_kernel ? p->n_psf_adj : p->n_psf) = n_psf;
    ConvArgs<T> a;
    memset(&a, 0, sizeof a);
    a.g = p->g; a.count = n_psf; a.in = (const T*)psf_dev; a.out = nullptr;
    a.twx = (const cplx<T>*)p->twx; a.twy = (const cplx<T>*)p->twy; a.tf = (cplx<T>*)tfbuf; a.n_psf = n_psf; a.tf_stride = p->tf_stride;
    a.spec = (cplx<T>*)p->spec; a.spec_stride = p->spec_stride; a.mode = CONV_MAKE_TF; a.queue = p->queue;
    return launch_conv<T>(p, a, n_psf, st);
}

template <typename T> static int apply_psf_t(bsgp_plan* p, const void* x, void* y, int batch, int adjoint, cudaStream_t st) {
    ConvArgs<T> a;
    memset(&a, 0, sizeof a);
    a.g = p->g; a.count = batch; a.in = (const T*)x; a.out = (T*)y;
    a.twx = (const cplx<T>*)p->twx; a.twy = (const cplx<T>*)p->twy; a.tf = (cplx<T>*)p->tf; a.n_psf = p->n_psf; a.tf_stride = p->tf_stride;
    a.spec = (cplx<T>*)p->spec; a.spec_stride = p->spec_stride; a.mode = adjoint ? CONV_CTF : CONV_TF; a.queue = p->queue;
    if (!p->embedded) return launch_conv<T>(p, a, batch, st);
    // wrapped plan: embed, convolve on the grid with the spectrum of h (A) or of h~ (A^T), fold (in the kernel), crop
    const size_t gb = (size_t)batch * p->ny * p->nx * sizeof(T);
    int rc = grow(&p->emb_img, &p->emb_img_cap, 2 * gb);
    if (rc) return rc;
    T* xe = (T*)p->emb_img; T* ye = (T*)((char*)p->emb_img + gb);
    rc = embed_images<T>(p, x, xe, batch, st);
    if (rc) return rc;
    a.in = xe; a.out = ye; a.mode = CONV_TF;
    if (adjoint) a.tf = (cplx<T>*)p->tf_adj;
    rc = launch_conv<T>(p, a, batch, st);
    if (rc) return rc;
    return crop_images<T>(p, ye, y, batch, st);
}

// bsgp_set_psf on a wrapped plan: both kernels (h for A, h~ for A^T) are built on the grid from the caller's PSFs
template <typename T> static int set_psf_wrapped(bsgp_plan* p, const void* psf_dev, int n_psf, cudaStream_t st) {
    const size_t gb = (size_t)n_psf * p->ny * p->nx * sizeof(T);
    int rc = grow(&p->emb_psf, &p->emb_psf_cap, gb);
    if (rc) return rc;
    int blocks = 0;
    rc = data_grid(p->device, (size_t)n_psf * p->ny * p->nx, &blocks);
    if (rc) return rc;
    for (int adj = 0; adj < 2; ++adj) {
        count_launch();
        bsgp_embed_psf_kernel<T><<<blocks, 256, 0, st>>>((const T*)psf_dev, p->img_ny, p->img_nx, (T*)p->emb_psf, p->ny, p->nx, (size_t)n_psf, adj);
        CU(cudaGetLastError());
        rc = set_psf_t<T>(p, p->emb_psf, n_psf, st, adj != 0);
        if (rc) return rc;
    }
    return BSGP_OK;
}

template <typename T>
static int solve_grid(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, cudaStream_t st, const int* ready);

// wrapped plans: move the caller's arrays onto the grid, solve there with the image window as the valid region (the
// zero-padded operator's masked kernels) and the fold of the geometry, crop the restored images
template <typename T>
static int solve_t(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, cudaStream_t st, const int* ready) {
    if (!p->embedded) return solve_grid<T>(p, prm, batch, in, out, st, ready);
    const size_t gb = (size_t)batch * p->ny * p->nx * sizeof(T);
    const int narr = 2 + (in->bkg_is_image ? 1 : 0) + (in->x0 ? 1 : 0) + (in->obj ? 1 : 0);
    int rc = grow(&p->emb_img, &p->emb_img_cap, (size_t)narr * gb);
    if (rc) return rc;
    char* base = (char*)p->emb_img;
    int k = 0;
    auto up = [&](const void* src, const void** dst) -> int {
        if (!src) { *dst = nullptr; return BSGP_OK; }
        void* d = base + (size_t)(k++) * gb;
        *dst = d;
        return embed_images<T>(p, src, d, (size_t)batch, st);
    };
    bsgp_inputs gi = *in;
    bsgp_outputs go = *out;
    if ((rc = up(in->gn, &gi.gn))) return rc;
    if (in->bkg_is_image && (rc = up(in->bkg, &gi.bkg))) return rc;
    if ((rc = up(in->x0, &gi.x0))) return rc;
    if ((rc = up(in->obj, &gi.obj))) return rc;
    go.x = base + (size_t)(k++) * gb;
    bsgp_params q = *prm;
    q.region[0] = 0; q.region[1] = p->img_ny; q.region[2] = 0; q.region[3] = p->img_nx;
    q.div_a = q.div_at = 1.0;
    q.adjoint_second_psf = 1;
    rc = solve_grid<T>(p, &q, batch, &gi, &go, st, ready);
    if (rc) return rc;
    return crop_images<T>(p, go.x, out->x, (size_t)batch, st);
}

template <typename T>
static int solve_grid(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, cudaStream_t st, const int* ready) {
    SolveArgs<T> a;
    memset(&a, 0, sizeof a);
    a.p = *prm; a.g = p->g; a.batch = batch;
    a.gn = (const T*)in->gn; a.bkg = (const T*)in->bkg; a.bkg_is_image = in->bkg_is_image; a.flux = in->flux; a.beta0 = in->beta0;
    a.x0 = (const T*)in->x0; a.obj = (const T*)in->obj; a.order = in->order;
    a.twx = (const cplx<T>*)p->twx; a.twy = (const cplx<T>*)p->twy; a.tf = (cplx<T>*)p->tf; a.n_psf = p->n_psf;
    a.tf_adj = prm->adjoint_second_psf ? (cplx<T>*)p->tf_adj : nullptr;
    a.work = (T*)p->work; a.work_stride = p->work_stride; a.spec = (cplx<T>*)p->spec; a.spec_stride = p->spec_stride;
    a.resident_mask = p->resident_mask;
    a.x_out = (T*)out->x; a.iters = out->iters; a.status = out->status; a.discr = out->discr; a.times = out->times;
    a.stop_value = out->stop_value; a.err = out->err; a.beta_final = out->beta_final; a.proj_evals = out->proj_evals;
    a.ls_trials = out->ls_trials; a.scalars = out->scalars; a.tr_alpha = out->trace_alpha; a.tr_lambda = out->trace_lambda;
    a.tr_beta = out->trace_beta; a.tr_trials = out->trace_trials; a.tr_evals = out->trace_evals;
    a.queue = p->queue;
    a.ready = p->frame ? nullptr : ready;
    if (p->frame) {
        LaunchCfg fc{p->g.G, 512, 1, p->smem_bytes, st, 1};
        const bool mk = prm->region[1] > prm->region[0];
        count_launch();
        cudaError_t fe = mk ? launch_frame<T, true>(fc, a, p->sp, p->tf_stride, p->gpart) : launch_frame<T, false>(fc, a, p->sp, p->tf_stride, p->gpart);
        if (fe != cudaSuccess) return fail(BSGP_E_CUDA, "frame kernel launch failed: %s", cudaGetErrorString(fe));
        return BSGP_OK;
    }
    CU(cudaMemsetAsync(p->queue, 0, sizeof(int), st));
    const int nclu = batch < p->num_clusters ? batch : p->num_clusters;
    LaunchCfg lc{nclu * p->g.G, p->threads, p->g.G, p->smem_bytes, st, p->minb};
    const bool mk = prm->region[1] > prm->region[0];
    count_launch();
    cudaError_t e = mk ? launch_solve<T, true>(lc, a, p->sp, p->tf_stride) : launch_solve<T, false>(lc, a, p->sp, p->tf_stride);
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "solve kernel launch failed: %s", cudaGetErrorString(e));
    return BSGP_OK;
}

static inline bool misaligned(const void* p) { return ((uintptr_t)p & 15) != 0; }

static int check_params(const bsgp_params* q) {
    if (q->divergence != BSGP_DIV_KL && q->divergence != BSGP_DIV_BETA) return fail(BSGP_E_ARG, "bad divergence");
    if (q->init_recon < 0 || q->init_recon > 3) return fail(BSGP_E_ARG, "init_recon must be 0..3");
    if (q->proj_type < 0 || q->proj_type > 1) return fail(BSGP_E_ARG, "proj_type must be 0 or 1");
    if (q->stop_criterion < 0 || q->stop_criterion > 4) return fail(BSGP_E_ARG, "stop_criterion must be 0..4");
    if (q->maxit < 1) return fail(BSGP_E_ARG, "MAXIT must be >= 1");
    if (q->m < 1 || q->m > kMaxMem || q->m_alpha < 1 || q->m_alpha > kMaxMem) return fail(BSGP_E_ARG, "M and M_alpha must be in 1..%d", kMaxMem);
    return BSGP_OK;
}

static int adjoint_on_wrapped_plan() {
    return fail(BSGP_E_STATE, "bsgp_set_psf_adjoint: a plan whose sides are not powers of two builds both kernels in bsgp_set_psf");
}

// bsgp_set_psf / bsgp_set_psf_adjoint from host memory: the caller's PSFs [n_psf][img_ny][img_nx], staged for the call
static int set_psf_host(bsgp_plan* p, const void* psf_host, int n_psf, bool adjoint) {
    if (!p || !psf_host || n_psf < 1) return fail(BSGP_E_ARG, "bad argument");
    if (adjoint && p->embedded) return adjoint_on_wrapped_plan();
    CU(cudaSetDevice(p->device));
    const size_t bytes = (size_t)n_psf * p->img_ny * p->img_nx * p->elem;
    void* d = nullptr;
    CU(cudaMalloc(&d, bytes));
    cudaError_t e = cudaMemcpy(d, psf_host, bytes, cudaMemcpyHostToDevice);
    int rc = e != cudaSuccess ? fail(BSGP_E_CUDA, "H2D copy failed: %s", cudaGetErrorString(e))
                              : (adjoint ? bsgp_set_psf_adjoint : bsgp_set_psf)(p, d, n_psf, nullptr);
    if (rc == BSGP_OK) { e = cudaDeviceSynchronize(); if (e != cudaSuccess) rc = fail(BSGP_E_CUDA, "PSF spectrum kernel failed: %s", cudaGetErrorString(e)); }
    cudaFree(d);
    return rc;
}

// the caller's device index, made current
static int use_device(int device) {
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(BSGP_E_CUDA, "device %d not available", device);
    CU(cudaSetDevice(device));
    return BSGP_OK;
}

extern "C" {

int bsgp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
const char* bsgp_last_error_string(void) { return g_err.c_str(); }
long long bsgp_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
#ifndef BSGP_SRC_HASH
#define BSGP_SRC_HASH "unknown"
#endif
const char* bsgp_version(void) { return "libbsgp 0.2 (sm_100a) src:" BSGP_SRC_HASH; }

int bsgp_plan_create(int ny, int nx, int dtype, int device, bsgp_plan** plan) {
    if (!plan) return fail(BSGP_E_ARG, "plan is NULL");
    *plan = nullptr;
    if (dtype != BSGP_F64 && dtype != BSGP_F32) return fail(BSGP_E_ARG, "dtype must be BSGP_F64 or BSGP_F32");
    if (ny < 1 || nx < 1) return fail(BSGP_E_SHAPE, "unsupported image shape %dx%d", ny, nx);
    // FFT grid: a power-of-two side in [16, 8192] is used as it is; any other side n runs on a grid of side
    // P = 2^k >= 2 n - 1 (linear convolution + fold, see "Wrapped plans" above)
    const int gy = wrap_grid_side(ny), gx = wrap_grid_side(nx);
    if (gy > 8192 || gx > 8192)
        return fail(BSGP_E_SHAPE, "unsupported image shape %dx%d: sides that are not a power of two are limited to 4096 (FFT grid of 8192)", ny, nx);
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(BSGP_E_CUDA, "device %d not available (%d CUDA devices)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 9) return fail(BSGP_E_CUDA, "thread-block clusters need compute capability >= 9.0 (found %d.%d)", prop.major, prop.minor);
    bsgp_plan* p = new bsgp_plan();
    p->ny = gy; p->nx = gx; p->img_ny = ny; p->img_nx = nx; p->embedded = (gy != ny || gx != nx);
    p->dtype = dtype; p->device = device;
    p->num_sms = prop.multiProcessorCount;
    p->max_smem = (int)prop.sharedMemPerBlockOptin;
    p->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
    int rc = plan_setup(p);
    if (rc) { plan_free_buffers(p); delete p; return rc; }
    *plan = p;
    return BSGP_OK;
}

int bsgp_plan_configure(bsgp_plan* p, int cluster_size, int threads) {
    if (!p) return fail(BSGP_E_ARG, "plan is NULL");
    CU(cudaSetDevice(p->device));
    CU(cudaDeviceSynchronize());
    plan_free_buffers(p);
    p->configured = false;
    p->want_G = cluster_size; p->want_threads = threads;
    return plan_setup(p);
}

int bsgp_plan_destroy(bsgp_plan* p) {
    if (!p) return BSGP_OK;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    plan_free_buffers(p);
    plan_free_pipeline(p);
    delete p;
    return BSGP_OK;
}

int bsgp_plan_get_info(const bsgp_plan* p, bsgp_plan_info* info) {
    if (!p || !info) return fail(BSGP_E_ARG, "NULL argument");
    info->ny = p->img_ny; info->nx = p->img_nx; info->dtype = p->dtype; info->device = p->device;
    info->grid_ny = p->ny; info->grid_nx = p->nx;
    info->cluster_size = p->g.G; info->num_clusters = p->num_clusters; info->threads = p->threads;
    info->smem_bytes = (int)p->smem_bytes; info->num_sms = p->num_sms; info->resident_mask = p->resident_mask;
    info->workspace_bytes = (long long)p->workspace_bytes;
    return BSGP_OK;
}

int bsgp_set_psf(bsgp_plan* p, const void* psf_dev, int n_psf, void* stream) {
    if (!p || !psf_dev || n_psf < 1) return fail(BSGP_E_ARG, "bad argument");
    if (!p->embedded && misaligned(psf_dev)) return fail(BSGP_E_ARG, "image pointers must be 16-byte aligned (vector loads)");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = plan_enter(p, st);
    if (rc) return rc;
    if (p->embedded) rc = p->dtype == BSGP_F64 ? set_psf_wrapped<double>(p, psf_dev, n_psf, st) : set_psf_wrapped<float>(p, psf_dev, n_psf, st);
    else rc = p->dtype == BSGP_F64 ? set_psf_t<double>(p, psf_dev, n_psf, st) : set_psf_t<float>(p, psf_dev, n_psf, st);
    if (rc) return rc;
    return plan_leave(p, st);
}

int bsgp_set_psf_adjoint(bsgp_plan* p, const void* psf_dev, int n_psf, void* stream) {
    if (!p || !psf_dev || n_psf < 1) return fail(BSGP_E_ARG, "bad argument");
    if (p->embedded) return adjoint_on_wrapped_plan();
    if (misaligned(psf_dev)) return fail(BSGP_E_ARG, "image pointers must be 16-byte aligned (vector loads)");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = plan_enter(p, st);
    if (rc) return rc;
    rc = p->dtype == BSGP_F64 ? set_psf_t<double>(p, psf_dev, n_psf, st, true) : set_psf_t<float>(p, psf_dev, n_psf, st, true);
    if (rc) return rc;
    return plan_leave(p, st);
}

int bsgp_set_psf_host(bsgp_plan* p, const void* psf_host, int n_psf) { return set_psf_host(p, psf_host, n_psf, false); }
int bsgp_set_psf_adjoint_host(bsgp_plan* p, const void* psf_host, int n_psf) { return set_psf_host(p, psf_host, n_psf, true); }

// Argument checks of every solve entry point.  The host entry points run them on the caller's pointers before they size
// anything from batch or prm->maxit (the device copies they stage are present exactly where the caller's arrays are),
// and they can read the queue order: the kernel indexes the images with it, so every entry must lie in 0..batch-1.
static int check_solve(const bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, bool host) {
    if (!p || !prm || !in || !out) return fail(BSGP_E_ARG, "NULL argument");
    if (batch < 1) return fail(BSGP_E_ARG, "batch must be >= 1");
    int rc = check_params(prm);
    if (rc) return rc;
    if (p->n_psf != 1 && p->n_psf != batch) return fail(BSGP_E_STATE, "bsgp_set_psf was called with %d PSFs; need 1 or batch (%d)", p->n_psf, batch);
    if (!in->gn || !in->bkg || !out->x || !out->iters || !out->status || !out->discr || !out->times) return fail(BSGP_E_ARG, "required pointer is NULL");
    if (prm->has_flux && !in->flux) return fail(BSGP_E_ARG, "has_flux set but inputs.flux is NULL");
    if (prm->divergence == BSGP_DIV_BETA && !in->beta0) return fail(BSGP_E_ARG, "beta-divergence needs inputs.beta0");
    if (prm->init_recon == 1 && !in->x0) return fail(BSGP_E_ARG, "init_recon = 1 needs inputs.x0");
    if (prm->errflag && (!in->obj || !out->err)) return fail(BSGP_E_ARG, "errflag needs inputs.obj and outputs.err");
    if (p->n_psf < 1) return fail(BSGP_E_STATE, "bsgp_set_psf has not been called");
    if (prm->adjoint_second_psf && (p->tf_adj == nullptr || p->n_psf_adj != p->n_psf))
        return fail(BSGP_E_STATE, "adjoint_second_psf set but bsgp_set_psf_adjoint was not called with the same number of PSFs");
    if (p->embedded && (prm->region[1] > prm->region[0] || prm->region[3] > prm->region[2] || prm->adjoint_second_psf))
        return fail(BSGP_E_ARG, "region / adjoint_second_psf (zero-padded operator) need a plan with power-of-two sides; embed the image into such a grid");
    if (prm->region[1] > prm->region[0] || prm->region[3] > prm->region[2]) {
        const int* r = prm->region;
        if (r[0] < 0 || r[1] > p->ny || r[2] < 0 || r[3] > p->nx || r[1] <= r[0] || r[3] <= r[2])
            return fail(BSGP_E_ARG, "region {%d, %d, %d, %d} does not fit the %dx%d grid", r[0], r[1], r[2], r[3], p->ny, p->nx);
        if (!(prm->div_a > 0.0) || !(prm->div_at > 0.0)) return fail(BSGP_E_ARG, "div_a / div_at must be positive when a region is set");
    }
    if (host && in->order) for (int i = 0; i < batch; ++i) if (in->order[i] < 0 || in->order[i] >= batch) return fail(BSGP_E_ARG, "inputs.order is not a permutation of 0..batch-1");
    return BSGP_OK;
}

// launch on device arrays that passed check_solve; `ready` (device, [batch]) makes the kernel wait for queue item i until ready[i] != 0
static int solve_launch(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, void* stream, const int* ready) {
    if (!p->embedded && (misaligned(in->gn) || misaligned(out->x) || misaligned(in->x0) || misaligned(in->obj) || (in->bkg_is_image && misaligned(in->bkg))))
        return fail(BSGP_E_ARG, "image pointers must be 16-byte aligned (vector loads)");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = plan_enter(p, st);
    if (rc) return rc;
    rc = p->dtype == BSGP_F64 ? solve_t<double>(p, prm, batch, in, out, st, ready) : solve_t<float>(p, prm, batch, in, out, st, ready);
    if (rc) return rc;
    return plan_leave(p, st);
}

int bsgp_solve_batch(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, void* stream) {
    const int rc = check_solve(p, prm, batch, in, out, false);
    return rc ? rc : solve_launch(p, prm, batch, in, out, stream, nullptr);
}

// host staging helpers -----------------------------------------------------------------------
struct DevBuf {
    void* d = nullptr;
    ~DevBuf() { cudaFree(d); }
    int up(const void* h, size_t bytes) {
        if (!h) return BSGP_OK;
        CU(cudaMalloc(&d, bytes));
        CU(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice));
        return BSGP_OK;
    }
    int alloc(bool want, size_t bytes) {
        if (!want) return BSGP_OK;
        CU(cudaMalloc(&d, bytes));
        CU(cudaMemset(d, 0, bytes));
        return BSGP_OK;
    }
    int down(void* h, size_t bytes) {
        if (!h || !d) return BSGP_OK;
        CU(cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost));
        return BSGP_OK;
    }
};
#define TRY(e) do { rc = (e); if (rc) return rc; } while (0)

// The host I/O of one solve, laid out in one device staging area: the caller's pointer of every array (nullptr: absent),
// its size for this batch and its offset in the area, inputs first, then the outputs, which are zero-filled before the
// launch and copied back after it.  The restored images are staged too, unless the kernel stores them straight into
// host memory through `x_mapped`.
struct HostIO {
    enum Slot { GN, BKG, X0, OBJ, FLUX, BETA0, ORDER,                 // inputs, the image-shaped ones first
                X, ITERS, STATUS, DISCR, TIMES, STOP_VALUE, ERR, BETA_FINAL, PROJ_EVALS, LS_TRIALS, SCALARS,
                TRACE_ALPHA, TRACE_LAMBDA, TRACE_BETA, TRACE_TRIALS, TRACE_EVALS, NSLOT };
    const void* host[NSLOT];              // nullptr: not staged
    size_t bytes[NSLOT], off[NSLOT];
    size_t out_begin = 0, size = 0;       // the outputs occupy [out_begin, size)
    size_t img;                           // bytes of one image
    int bkg_is_image;
    void* x_mapped;

    HostIO(const bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, void* x_mapped_)
        : img((size_t)p->img_ny * p->img_nx * p->elem), bkg_is_image(in->bkg_is_image), x_mapped(x_mapped_) {
        const size_t B = (size_t)batch, tr = (size_t)prm->maxit + 1, imgs = B * img, it8 = B * tr * 8, it4 = B * tr * 4;
        const void* const h[NSLOT] = {in->gn, in->bkg, in->x0, in->obj, in->flux, in->beta0, in->order,
                                      x_mapped ? nullptr : out->x, out->iters, out->status, out->discr, out->times, out->stop_value,
                                      out->err, out->beta_final, out->proj_evals, out->ls_trials, out->scalars,
                                      out->trace_alpha, out->trace_lambda, out->trace_beta, out->trace_trials, out->trace_evals};
        const size_t n[NSLOT] = {imgs, bkg_is_image ? imgs : B * p->elem, imgs, imgs, B * 8, B * 8, B * 4,
                                 imgs, B * 4, B * 4, it8, it8, it8,
                                 B * (tr + 1) * 8, B * 8, B * 4, B * 4, B * BSGP_NSCALARS * 8,
                                 it8, it8, it8, it4, it4};
        for (int k = 0; k < NSLOT; ++k) {
            if (k == X) out_begin = size;
            host[k] = h[k]; bytes[k] = n[k]; off[k] = size;
            if (h[k]) size = (size + n[k] + 255) & ~(size_t)255;
        }
    }
    bool image(int k) const { return k <= OBJ && (k != BKG || bkg_is_image); }
    // the solve on the staging area at `base`
    int launch(bsgp_plan* p, const bsgp_params* prm, int batch, char* base, void* stream, const int* ready) const {
        auto dev = [&](int k) -> void* { return host[k] ? base + off[k] : nullptr; };
        const bsgp_inputs in = {dev(GN), dev(BKG), bkg_is_image, (const double*)dev(FLUX), (const double*)dev(BETA0), dev(X0), dev(OBJ),
                                (const int*)dev(ORDER)};
        const bsgp_outputs out = {x_mapped ? x_mapped : dev(X), (int*)dev(ITERS), (int*)dev(STATUS), (double*)dev(DISCR), (double*)dev(TIMES),
                                  (double*)dev(STOP_VALUE), (double*)dev(ERR), (double*)dev(BETA_FINAL), (int*)dev(PROJ_EVALS),
                                  (int*)dev(LS_TRIALS), (double*)dev(SCALARS), (double*)dev(TRACE_ALPHA), (double*)dev(TRACE_LAMBDA),
                                  (double*)dev(TRACE_BETA), (int*)dev(TRACE_TRIALS), (int*)dev(TRACE_EVALS)};
        return solve_launch(p, prm, batch, &in, &out, stream, ready);
    }
    // the staged outputs to the caller's arrays, queued on `st`
    int copy_back(const char* base, cudaStream_t st) const {
        for (int k = X; k < NSLOT; ++k)
            if (host[k]) CU(cudaMemcpyAsync(const_cast<void*>(host[k]), base + off[k], bytes[k], cudaMemcpyDeviceToHost, st));
        return BSGP_OK;
    }
};

// pageable host arrays: one staging allocation per call, freed before returning
int bsgp_solve_batch_host(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out) {
    int rc;
    TRY(check_solve(p, prm, batch, in, out, true));
    CU(cudaSetDevice(p->device));
    const HostIO io(p, prm, batch, in, out, nullptr);
    DevBuf area;
    TRY(area.alloc(true, io.size));
    char* base = (char*)area.d;
    for (int k = 0; k < HostIO::X; ++k)
        if (io.host[k]) CU(cudaMemcpy(base + io.off[k], io.host[k], io.bytes[k], cudaMemcpyHostToDevice));
    TRY(io.launch(p, prm, batch, base, nullptr, nullptr));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "solve kernel failed: %s", cudaGetErrorString(e));
    TRY(io.copy_back(base, nullptr));
    CU(cudaStreamSynchronize(nullptr));
    return BSGP_OK;
}

// ---------------------------------------------------------------------------------------------
// Pipelined host path.  Page-locked image buffers in, page-locked restored images out:
//   * copy stream : the images go up one queue item at a time, in the order the persistent kernel hands them out,
//                   each group followed by a 4-byte-per-item copy that raises the items' ready flags;
//   * run stream  : the solve kernel starts right away and waits per queue item for its flag (wait_ready), so the
//                   upload of image i+1.. overlaps the restoration of image ..i;
//   * results     : the kernel stores every restored image straight into the page-locked output (mapped, zero-copy:
//                   posted writes over PCIe while other images are still being solved); the small per-image outputs
//                   come back with ordinary copies after the kernel.
// Small images (< 64 KB) with a permuted queue would need one tiny copy per image; they are uploaded as whole arrays
// instead (one flag write for everything), still with the zero-copy output.  Frame mode: upload, then launch.
// ---------------------------------------------------------------------------------------------
static bool page_locked(const void* h) {
    if (!h) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, h) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

int bsgp_solve_batch_pinned(bsgp_plan* p, const bsgp_params* prm, int batch, const bsgp_inputs* in, const bsgp_outputs* out, void* stream) {
    int rc;
    TRY(check_solve(p, prm, batch, in, out, true));
    CU(cudaSetDevice(p->device));
    if (!page_locked(in->gn) || !page_locked(out->x) || !page_locked(in->x0) || !page_locked(in->obj) || (in->bkg_is_image && !page_locked(in->bkg)))
        return fail(BSGP_E_ARG, "bsgp_solve_batch_pinned needs page-locked image buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory)");
    void* x_mapped = nullptr;
    CU(cudaHostGetDevicePointer(&x_mapped, out->x, 0));
    const HostIO io(p, prm, batch, in, out, x_mapped);
    const size_t img = io.img, B = (size_t)batch;
    // images in the caller's own shape: a plan whose grid differs from it (sides that are not a power of two) moves them
    // to and from the grid on the device (solve_t), which needs all of them resident first, like frame mode
    const bool resident_first = p->frame || p->embedded;
    TRY(grow(&p->stage, &p->stage_cap, io.size));
    if (batch > p->ready_cap) {
        CU(cudaDeviceSynchronize());
        cudaFree(p->ready); cudaFreeHost(p->ones_host); p->ready = nullptr; p->ones_host = nullptr; p->ready_cap = 0;
        CU(cudaMalloc((void**)&p->ready, B * sizeof(int)));
        CU(cudaHostAlloc((void**)&p->ones_host, B * sizeof(int), cudaHostAllocDefault));
        for (int i = 0; i < batch; ++i) p->ones_host[i] = 1;
        p->ready_cap = batch;
    }
    if (!p->s_copy) {
        CU(cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&p->s_run, cudaStreamNonBlocking));
        for (cudaEvent_t* e : {&p->ev_fork, &p->ev_flags, &p->ev_copy, &p->ev_run}) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    char* S = (char*)p->stage;
    cudaStream_t user = (cudaStream_t)stream, sc = p->s_copy, sr = p->s_run;
    // ---- fork from the caller's stream (the PSF spectra may still be in flight there)
    CU(cudaEventRecord(p->ev_fork, user));
    CU(cudaStreamWaitEvent(sc, p->ev_fork, 0));
    CU(cudaStreamWaitEvent(sr, p->ev_fork, 0));
    // ---- run stream: small inputs, cleared outputs and flags, then the kernel
    for (int k = 0; k < HostIO::X; ++k)
        if (io.host[k] && !io.image(k)) CU(cudaMemcpyAsync(S + io.off[k], io.host[k], io.bytes[k], cudaMemcpyHostToDevice, sr));
    CU(cudaMemsetAsync(S + io.out_begin, 0, io.size - io.out_begin, sr));
    CU(cudaMemsetAsync(p->ready, 0, B * sizeof(int), sr));
    CU(cudaEventRecord(p->ev_flags, sr));
    CU(cudaStreamWaitEvent(sc, p->ev_flags, 0));                   // no flag may be raised before the flags are cleared
    // ---- copy stream: items [first, first + n) of every image-shaped input, then the flags that hand them to the kernel
    auto upload = [&](size_t first, size_t n) -> int {
        for (int k = 0; k < HostIO::X; ++k)
            if (io.host[k] && io.image(k))
                CU(cudaMemcpyAsync(S + io.off[k] + first * img, (const char*)io.host[k] + first * img, n * img, cudaMemcpyHostToDevice, sc));
        return BSGP_OK;
    };
    const bool per_item = !p->frame && (img >= 65536 || in->order == nullptr);
    auto feed = [&]() -> int {
        if (resident_first) {                                      // no per-item hand-over: everything resident first
            TRY(upload(0, B));
            CU(cudaEventRecord(p->ev_copy, sc));
            CU(cudaStreamWaitEvent(sr, p->ev_copy, 0));
        } else if (!per_item) {
            TRY(upload(0, B));
            CU(cudaMemcpyAsync(p->ready, p->ones_host, B * sizeof(int), cudaMemcpyHostToDevice, sc));
        } else {
            // images in queue order, flags behind them; consecutive queue items that are also consecutive in memory
            // travel as one copy of <= ~1 MB per array
            const size_t max_run = img >= ((size_t)1 << 20) ? 1 : (((size_t)1 << 20) / img);
            for (int i0 = 0, n = 0; i0 < batch; i0 += n) {
                const int first = in->order ? in->order[i0] : i0;
                for (n = 1; i0 + n < batch && (size_t)n < max_run && (in->order ? in->order[i0 + n] : i0 + n) == first + n;) ++n;
                TRY(upload((size_t)first, (size_t)n));
                CU(cudaMemcpyAsync(p->ready + i0, p->ones_host, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, sc));
            }
        }
        return BSGP_OK;
    };
    rc = feed();
    if (rc) { cudaGetLastError(); cudaStreamSynchronize(sc); cudaStreamSynchronize(sr); return rc; }
    // ---- run stream: the kernel.  Launched AFTER the copies are queued, so that a launch made synchronous by a tool
    // (ncu, compute-sanitizer, CUDA_LAUNCH_BLOCKING) cannot wait for flags that nobody has been asked to raise yet.
    rc = io.launch(p, prm, batch, S, sr, resident_first ? nullptr : p->ready);
    if (rc) { cudaStreamSynchronize(sc); cudaStreamSynchronize(sr); return rc; }
    // ---- small outputs behind the kernel
    TRY(io.copy_back(S, sr));
    // ---- join: the caller's stream continues after both private streams; results are complete when this returns
    CU(cudaEventRecord(p->ev_copy, sc));
    CU(cudaEventRecord(p->ev_run, sr));
    CU(cudaStreamWaitEvent(user, p->ev_copy, 0));
    CU(cudaStreamWaitEvent(user, p->ev_run, 0));
    cudaError_t e = cudaStreamSynchronize(sc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(sr);
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "pipelined solve failed: %s", cudaGetErrorString(e));
    return BSGP_OK;
}

int bsgp_apply_psf(bsgp_plan* p, const void* x_dev, void* y_dev, int batch, int adjoint, void* stream) {
    if (!p || !x_dev || !y_dev || batch < 1) return fail(BSGP_E_ARG, "bad argument");
    if (p->n_psf < 1) return fail(BSGP_E_STATE, "bsgp_set_psf has not been called");
    if (p->n_psf != 1 && p->n_psf != batch) return fail(BSGP_E_STATE, "%d PSFs set; need 1 or batch (%d)", p->n_psf, batch);
    if (!p->embedded && (misaligned(x_dev) || misaligned(y_dev))) return fail(BSGP_E_ARG, "image pointers must be 16-byte aligned (vector loads)");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = plan_enter(p, st);
    if (rc) return rc;
    rc = p->dtype == BSGP_F64 ? apply_psf_t<double>(p, x_dev, y_dev, batch, adjoint, st) : apply_psf_t<float>(p, x_dev, y_dev, batch, adjoint, st);
    if (rc) return rc;
    return plan_leave(p, st);
}

int bsgp_apply_psf_host(bsgp_plan* p, const void* x_host, void* y_host, int batch, int adjoint) {
    if (!p || !x_host || !y_host) return fail(BSGP_E_ARG, "NULL argument");
    CU(cudaSetDevice(p->device));
    const size_t bytes = (size_t)batch * p->img_ny * p->img_nx * p->elem;
    DevBuf x, y;
    int rc;
    TRY(x.up(x_host, bytes)); TRY(y.alloc(true, bytes));
    TRY(bsgp_apply_psf(p, x.d, y.d, batch, adjoint, nullptr));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "convolution kernel failed: %s", cudaGetErrorString(e));
    return y.down(y_host, bytes);
}

int bsgp_project_df(const double* b, const double* c, const double* dia, int n, int batch, double sat_cap, double lambda0,
                    double dlambda0, double tol_lam, int max_projs, int biter, int siter, double* x, int* evals, int* status, int device, void* stream) {
    if (!b || !c || !dia || !x || n < 1 || batch < 1) return fail(BSGP_E_ARG, "bad argument");
    CU(cudaSetDevice(device));
    const int has_cap = (sat_cap == sat_cap) && sat_cap >= 0.0;
    const int grid = batch < 4096 ? batch : 4096;
    count_launch();
    bsgp_project_kernel<<<grid, 512, 0, (cudaStream_t)stream>>>(b, c, dia, n, batch, sat_cap, has_cap, lambda0, dlambda0, tol_lam,
                                                                max_projs, biter, siter, x, evals, status);
    CU(cudaGetLastError());
    return BSGP_OK;
}

int bsgp_project_df_host(const double* b, const double* c, const double* dia, int n, int batch, double sat_cap, double lambda0,
                         double dlambda0, double tol_lam, int max_projs, int biter, int siter, double* x, int* evals, int* status, int device) {
    if (!b || !c || !dia || !x) return fail(BSGP_E_ARG, "NULL argument");
    int rc;
    TRY(use_device(device));
    const size_t vb = (size_t)n * batch * 8;
    DevBuf db, dc, dd, dx, de, ds;
    TRY(db.up(b, (size_t)batch * 8)); TRY(dc.up(c, vb)); TRY(dd.up(dia, vb)); TRY(dx.alloc(true, vb));
    TRY(de.alloc(true, (size_t)batch * 4)); TRY(ds.alloc(true, (size_t)batch * 4));
    TRY(bsgp_project_df((const double*)db.d, (const double*)dc.d, (const double*)dd.d, n, batch, sat_cap, lambda0, dlambda0, tol_lam,
                        max_projs, biter, siter, (double*)dx.d, (int*)de.d, (int*)ds.d, device, nullptr));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(BSGP_E_CUDA, "projection kernel failed: %s", cudaGetErrorString(e));
    TRY(dx.down(x, vb)); TRY(de.down(evals, (size_t)batch * 4)); TRY(ds.down(status, (size_t)batch * 4));
    return BSGP_OK;
}

int bsgp_beta_div_host(const double* y, const double* x, long long n, double beta, double* value, double* deriv, int device) {
    if (!y || !x || !value || n < 1) return fail(BSGP_E_ARG, "bad argument");
    int rc;
    TRY(use_device(device));
    DevBuf dy, dx, dp, dd;
    long long want = (n + 255) / 256;
    const int grid = (int)(want < 592 ? want : 592);
    TRY(dy.up(y, (size_t)n * 8)); TRY(dx.up(x, (size_t)n * 8)); TRY(dp.alloc(true, (size_t)grid * 3 * 8)); TRY(dd.alloc(deriv != nullptr, (size_t)n * 8));
    count_launch();
    bsgp_betadiv_kernel<<<grid, 256>>>((const double*)dy.d, (const double*)dx.d, n, beta, (double*)dp.d, (double*)dd.d);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    std::vector<double> part((size_t)grid * 3);
    TRY(dp.down(part.data(), part.size() * 8));
    double acc[3] = {0.0, 0.0, 0.0};
    for (int b = 0; b < grid; ++b) for (int k = 0; k < 3; ++k) acc[k] += part[(size_t)b * 3 + k];
    // combine exactly like the solver (sgp.py:452-458); s1 is acc[0] for the generic case
    DivK<double> dk;
    dk.kind = (beta == 0.0) ? 2 : (beta == 1.0 ? 3 : 1);
    if (dk.kind == 1) *value = (acc[0] + acc[1]) - acc[2];
    else if (dk.kind == 2) *value = (acc[0] - acc[1]) - (double)n;
    else *value = (acc[0] - acc[1]) + acc[2];
    TRY(dd.down(deriv, (size_t)n * 8));
    return BSGP_OK;
}
int bsgp_beta_grad_terms_host(const double* den, const double* gn, long long n, double beta, double* p1, double* u, int device) {
    if (!den || !gn || !p1 || !u || n < 1) return fail(BSGP_E_ARG, "bad argument");
    int rc;
    TRY(use_device(device));
    DevBuf dd, dg, dp, du;
    TRY(dd.up(den, (size_t)n * 8)); TRY(dg.up(gn, (size_t)n * 8)); TRY(dp.alloc(true, (size_t)n * 8)); TRY(du.alloc(true, (size_t)n * 8));
    long long want = (n + 255) / 256;
    count_launch();
    bsgp_betagrad_kernel<<<(int)(want < 1184 ? want : 1184), 256>>>((const double*)dd.d, (const double*)dg.d, n, beta, (double*)dp.d, (double*)du.d);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    TRY(dp.down(p1, (size_t)n * 8)); TRY(du.down(u, (size_t)n * 8));
    return BSGP_OK;
}
#undef TRY

// ------------------------------------------------------------------------------------------------
// tiling (utils.py:332-397)
// ------------------------------------------------------------------------------------------------
int bsgp_tile_boxes(int height, int width, int tile_h, int tile_w, double overlap_h_ratio, double overlap_w_ratio, int* boxes_xyxy, int max_boxes, int* n_boxes) {
    if (!n_boxes || height < 1 || width < 1 || tile_h < 1 || tile_w < 1) return fail(BSGP_E_ARG, "bad argument");
    // utils.py:360-375: rows outer, columns inner; step = tile - int(ratio * tile); a tile that would stick out is
    // shifted back inside (clamped at 0 when the image is smaller than the tile)
    const int oy = (int)(overlap_h_ratio * (double)tile_h), ox = (int)(overlap_w_ratio * (double)tile_w);
    if (oy >= tile_h || ox >= tile_w || oy < 0 || ox < 0) return fail(BSGP_E_ARG, "overlap must be smaller than the tile");
    int n = 0;
    for (int y0 = 0;; y0 += tile_h - oy) {
        const int y1 = y0 + tile_h;
        for (int x0 = 0;; x0 += tile_w - ox) {
            const int x1 = x0 + tile_w;
            int bx0 = x0, by0 = y0, bx1 = x1, by1 = y1;
            if (y1 > height || x1 > width) {
                bx1 = x1 < width ? x1 : width; by1 = y1 < height ? y1 : height;
                bx0 = bx1 - tile_w > 0 ? bx1 - tile_w : 0; by0 = by1 - tile_h > 0 ? by1 - tile_h : 0;
            }
            if (boxes_xyxy && n < max_boxes) { int* b = boxes_xyxy + 4 * (size_t)n; b[0] = bx0; b[1] = by0; b[2] = bx1; b[3] = by1; }
            ++n;
            if (x1 >= width) break;
        }
        if (y1 >= height) break;
    }
    *n_boxes = n;
    if (boxes_xyxy && n > max_boxes) return fail(BSGP_E_ARG, "%d boxes needed, room for %d", n, max_boxes);
    return BSGP_OK;
}

int bsgp_extract_tiles(const void* frame_dev, int height, int width, int dtype, const int* origins_dev, int n, int tile_h, int tile_w, void* tiles_dev, int device, void* stream) {
    if (!frame_dev || !origins_dev || !tiles_dev || n < 1 || tile_h < 1 || tile_w < 1 || height < 1 || width < 1) return fail(BSGP_E_ARG, "bad argument");
    if (dtype != BSGP_F64 && dtype != BSGP_F32) return fail(BSGP_E_ARG, "bad dtype");
    CU(cudaSetDevice(device));
    int blocks = 0, rc = data_grid(device, (size_t)n * tile_h * tile_w, &blocks);
    if (rc) return rc;
    count_launch();
    if (dtype == BSGP_F64) bsgp_extract_tiles_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)frame_dev, height, width, origins_dev, n, tile_h, tile_w, (double*)tiles_dev);
    else bsgp_extract_tiles_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)frame_dev, height, width, origins_dev, n, tile_h, tile_w, (float*)tiles_dev);
    CU(cudaGetLastError());
    return BSGP_OK;
}

int bsgp_assemble_tiles(const void* tiles_dev, const int* origins_dev, int n, int tile_h, int tile_w, int dtype, int feather, void* frame_dev, int height, int width, int device, void* stream) {
    if (!frame_dev || !origins_dev || !tiles_dev || n < 1 || tile_h < 1 || tile_w < 1 || height < 1 || width < 1) return fail(BSGP_E_ARG, "bad argument");
    if (dtype != BSGP_F64 && dtype != BSGP_F32) return fail(BSGP_E_ARG, "bad dtype");
    CU(cudaSetDevice(device));
    int blocks = 0, rc = data_grid(device, (size_t)height * width, &blocks);
    if (rc) return rc;
    count_launch();
    if (dtype == BSGP_F64) bsgp_assemble_tiles_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)tiles_dev, origins_dev, n, tile_h, tile_w, feather, (double*)frame_dev, height, width);
    else bsgp_assemble_tiles_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)tiles_dev, origins_dev, n, tile_h, tile_w, feather, (float*)frame_dev, height, width);
    CU(cudaGetLastError());
    return BSGP_OK;
}

// ------------------------------------------------------------------------------------------------
// PSF model (psf/psf_calculate.py:52-111)
// ------------------------------------------------------------------------------------------------
int bsgp_psf_model_eval(const double* params_dev, int n, int ngauss, int hw, int ny, int nx, int normalize, int dtype, void* out_dev, int device, void* stream) {
    if (!params_dev || !out_dev || n < 1 || ngauss < 1 || ngauss > 8 || hw < 0 || ny < 1 || nx < 1) return fail(BSGP_E_ARG, "bad argument");
    if (dtype != BSGP_F64 && dtype != BSGP_F32) return fail(BSGP_E_ARG, "bad dtype");
    CU(cudaSetDevice(device));
    const int stride = 5 + 6 * ngauss;
    count_launch();
    if (dtype == BSGP_F64) bsgp_psf_model_kernel<double><<<n, 256, 0, (cudaStream_t)stream>>>(params_dev, stride, ngauss, hw, ny, nx, normalize, (double*)out_dev);
    else bsgp_psf_model_kernel<float><<<n, 256, 0, (cudaStream_t)stream>>>(params_dev, stride, ngauss, hw, ny, nx, normalize, (float*)out_dev);
    CU(cudaGetLastError());
    return BSGP_OK;
}

}  // extern "C"
