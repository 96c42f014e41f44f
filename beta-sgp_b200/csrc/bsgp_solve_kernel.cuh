// The persistent solve kernel and its launchers.  Included by one translation unit per data type
// and operator kind (bsgp_solve_f64.cu, bsgp_solve_f32.cu, *_padded.cu) so they compile in parallel.  MK = true is the
// zero-padded operator (valid-window masks compiled in); MK = false the circular one (no mask code at all).
#pragma once
#include <string.h>

#include <type_traits>

#include "bsgp_device.cuh"
#include "bsgp_launch.h"
#include "bsgp_solver.cuh"

namespace bsgp {

// shared-memory twiddle table: mode 1 = the full table W_n^k, mode 2 = two-level [W^0 .. W^63][W^(64 m)] (bsgp_fft.cuh)
template <class Ctx, typename T> __device__ __forceinline__ void fill_twiddles(Ctx& ctx, int mode, int n, const cplx<T>* tw, cplx<T>* dst, int dft_n = 0) {
    if (dft_n) {          // dense axis: the DMMA fragment table (fp64), nothing otherwise (the scalar version reads global memory)
        if (sizeof(T) == 8 && mode == 1) fill_dense_table(ctx, n, dft_n, tw, reinterpret_cast<double*>(dst));
        return;
    }
    if (mode == 1) {
        for (int k = ctx.tid; k < n; k += ctx.nt) dst[k] = tw[k];
    } else if (mode == 2) {
        for (int k = ctx.tid; k < 64 + (n >> 6); k += ctx.nt) dst[k] = (k < 64) ? tw[k] : tw[(k - 64) << 6];
    }
}

// Prologue of both persistent kernels: this warp's controller state, the slab arrays (resident in shared memory or in
// this cluster's global scratch), the twiddle and position tables, and the per-image constants in shared memory.  Frame
// plans have no resident arrays, one scratch area and no dense axes (bsgp_plan.h): the constants below keep that code
// out of the frame kernel.
template <typename T, class Ctx>
__device__ __forceinline__ ImgState<T>* solve_prologue(Ctx& ctx, unsigned char* smem, const SolveArgs<T>& a, const SmemPlan& sp, T* (&buf)[NBUF]) {
    ctx.wst = smem + sp.off_ctl + (threadIdx.x >> 5) * sp.ctl_stride;
    ImgState<T>* S = reinterpret_cast<ImgState<T>*>(smem + sp.off_state);
    const int cluster_id = Ctx::kFrame ? 0 : blockIdx.x / a.g.G;
    const int resident = Ctx::kFrame ? 0 : a.resident_mask;
    const size_t npix = (size_t)a.g.ny * a.g.nx;
    const size_t nslab = (size_t)a.g.rows_per_cta * a.g.nx;
    size_t soff = sp.off_bufs;
#pragma unroll
    for (int b = 0; b < NBUF; ++b) {
        if (resident & (1 << b)) { buf[b] = reinterpret_cast<T*>(smem + soff); soff += nslab * sizeof(T); }
        else buf[b] = a.work + (size_t)cluster_id * a.work_stride + (size_t)b * npix + (size_t)ctx.rank * nslab;
    }
    cplx<T>* twx_s = reinterpret_cast<cplx<T>*>(smem + sp.off_twx);
    cplx<T>* twy_s = reinterpret_cast<cplx<T>*>(smem + sp.off_twy);
    fill_twiddles(ctx, sp.tw_smem, a.g.nx, a.twx, twx_s, Ctx::kFrame ? 0 : a.g.px.dft_n);
    if (sp.off_twy != sp.off_twx) fill_twiddles(ctx, sp.tw_smem, a.g.ny, a.twy, twy_s, Ctx::kFrame ? 0 : a.g.py.dft_n);
    fill_pos_table(ctx, a.g.px, reinterpret_cast<unsigned short*>(smem + sp.off_ppx));
    if (ctx.tid == 0) {
        S->geom = a.g;
        S->ppx_off = sp.off_ppx;
        S->ws_off = sp.off_ws;
        // One CTA per image with d_tf resident (stamps): the half-spectrum exchange buffer (ny x nx/2 complex = one image
        // array) BORROWS the d_tf array instead of living in global memory.  With one workspace tile per pass every
        // producer has read all of its inputs before the first spectrum element is written, and every consumer has moved
        // the whole spectrum into the workspace before it stores its first output; d_tf itself is dead across every
        // convolution: it is written by the consumer of A(d) (ph_ri_trial), read by the line search and, for the last
        // time, by the producer of the accepted step's A^T (ph_rf_grad).
        const bool spec_in_dtf = a.g.G == 1 && ((resident >> B_DTF) & 1) && 2 * a.g.row_tile_pairs == a.g.ny && a.g.col_tile == a.g.hx;
        S->spec = spec_in_dtf ? reinterpret_cast<cplx<T>*>(buf[B_DTF]) : a.spec + (size_t)cluster_id * a.spec_stride;
        S->twx = a.twx; S->twy = a.twy;
        S->twx_off = sp.tw_smem ? sp.off_twx : kNoSmem;
        S->twy_off = sp.tw_smem ? sp.off_twy : kNoSmem;
        S->tw_split = sp.tw_smem == 2;
    }
    __syncthreads();
    return S;
}

template <typename T, int NT, int MINB, bool MK>
__global__ void __launch_bounds__(NT, MINB) bsgp_solve_kernel(const SolveArgs<T> a, const SmemPlan sp, const size_t tf_stride) {
    unsigned char* smem = dyn_smem();
    // 2 CTAs x 256 threads and 3 CTAs x 128 threads per SM are the configurations of images that are resident in shared memory
    // (bsgp_plan.h, plan_launch)
    typename std::conditional<(NT == 256 && MINB == 2) || (NT == 128 && MINB == 3), DeviceCtxSmall, DeviceCtx>::type ctx;
    static_cast<DeviceCtx&>(ctx) = make_ctx(reinterpret_cast<SharedCtl*>(smem), a.g.G);
    T* buf[NBUF];
    ImgState<T>* S = solve_prologue(ctx, smem, a, sp, buf);
    for (;;) {
        bool ready_ok;
        const int item = next_item(ctx, a.queue, a.ready, a.batch, &ready_ok);
        if (item >= a.batch) break;
        const int img = a.order ? a.order[item] : item;
        if (!ready_ok) {                                   // upload never arrived: report and skip (cluster-uniform)
            if (ctx.rank == 0 && ctx.tid == 0) { a.status[img] = BSGP_ST_INPUT_TIMEOUT; a.iters[img] = 0; }
            continue;
        }
        cplx<T>* tf = a.tf + (a.n_psf > 1 ? (size_t)img * tf_stride : 0);
        cplx<T>* tfa = a.tf_adj ? a.tf_adj + (a.n_psf > 1 ? (size_t)img * tf_stride : 0) : tf;
        solve_image<T, MK>(ctx, a, S, buf, tf, tfa, img);
    }
}

// Frame mode (GridCtx): the images of the batch are restored one after the other, each by the whole grid.
template <typename T, bool MK>
__global__ void __launch_bounds__(512, 1) bsgp_frame_kernel(const SolveArgs<T> a, const SmemPlan sp, const size_t tf_stride, double* gpart) {
    unsigned char* smem = dyn_smem();
    GridCtx ctx = make_grid_ctx(reinterpret_cast<SharedCtl*>(smem), gpart);
    T* buf[NBUF];
    ImgState<T>* S = solve_prologue(ctx, smem, a, sp, buf);
    for (int img = 0; img < a.batch; ++img) {
        cplx<T>* tf = a.tf + (a.n_psf > 1 ? (size_t)img * tf_stride : 0);
        cplx<T>* tfa = a.tf_adj ? a.tf_adj + (a.n_psf > 1 ? (size_t)img * tf_stride : 0) : tf;
        solve_image<T, MK>(ctx, a, S, buf, tf, tfa, img);
        ctx.cluster_sync();          // the scratch arrays and the exchange buffer are reused by the next image
    }
}

template <typename T, bool MK>
cudaError_t launch_frame(const LaunchCfg& lc, const SolveArgs<T>& a, const SmemPlan& sp, size_t tf_stride, double* gpart) {
    SolveArgs<T> args = a;
    SmemPlan plan = sp;
    size_t tfs = tf_stride;
    double* gp = gpart;
    void* params[] = {&args, &plan, &tfs, &gp};
    const void* fn = (const void*)bsgp_frame_kernel<T, MK>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lc.smem);
    if (e != cudaSuccess) return e;
    return cudaLaunchCooperativeKernel(fn, dim3(lc.grid), dim3(lc.threads), params, lc.smem, lc.stream);
}

template <typename T, bool MK> cudaError_t query_frame_ctas(const LaunchCfg& lc, int* per_sm) {
    const void* fn = (const void*)bsgp_frame_kernel<T, MK>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lc.smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, fn, lc.threads, lc.smem);
}

// register budgets: 512 x 128, 256 x 255 (one CTA per SM), 256 x 128 (two CTAs per SM), 128 x 168 (three), 128 x 128 (four)
template <typename T, bool MK> static const void* solve_kernel_ptr(int threads, int minb) {
    if (threads <= 128) return minb >= 4 ? (const void*)bsgp_solve_kernel<T, 128, 4, MK> : (const void*)bsgp_solve_kernel<T, 128, 3, MK>;
    if (threads <= 256) return minb >= 2 ? (const void*)bsgp_solve_kernel<T, 256, 2, MK> : (const void*)bsgp_solve_kernel<T, 256, 1, MK>;
    return (const void*)bsgp_solve_kernel<T, 512, 1, MK>;
}

template <typename T, bool MK>
cudaError_t launch_solve(const LaunchCfg& lc, const SolveArgs<T>& a, const SmemPlan& sp, size_t tf_stride) {
    SolveArgs<T> args = a;
    SmemPlan plan = sp;
    size_t tfs = tf_stride;
    void* params[] = {&args, &plan, &tfs};
    return launch_clustered(solve_kernel_ptr<T, MK>(lc.threads, lc.minb), lc, params);
}

template <typename T, bool MK> cudaError_t query_solve_clusters(const LaunchCfg& lc, int num_sms, int* out) {
    return query_clusters(solve_kernel_ptr<T, MK>(lc.threads, lc.minb), lc, num_sms, out);
}

}  // namespace bsgp
