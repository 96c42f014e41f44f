// Device-side execution context of libbsgp: one thread-block CLUSTER of G CTAs works on one image.
//
//   * Scalars travel between the CTAs of a cluster through distributed shared memory: every CTA
//     stores its partial sums into every peer's inbox and one hardware cluster barrier publishes
//     them; all CTAs then add the G partials in the same order, so all controllers agree bit for bit.
//   * Clusters are persistent and pull image indices from a global queue, so images with very
//     different iteration counts (2..160 observed) never wait for each other and the host is not
//     involved between "inputs resident" and "outputs written".
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "bsgp_math.cuh"
#include "bsgp_smem.h"

namespace bsgp {

namespace cg = cooperative_groups;

__device__ __forceinline__ double red_combine(int op, double a, double b) {
    if (op == 0) return a + b;
    if (op == 1) return (b < a) ? b : a;
    return (b > a) ? b : a;
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned map_to_rank(unsigned addr, int rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}

struct DeviceCtx {
    static constexpr bool kFrame = false;     // cluster mode: row-major exchange buffer, full twiddle tables
    static constexpr bool kSmall = false;     // see DeviceCtxSmall
    int tid, nt, rank, G;
    SharedCtl* sh;
    int parity;        // bit 0: inbox half in use; bits 1, 2: phase of mbar[0], mbar[1]
    void* wst;         // this warp's copy of the solver's controller state (shared memory), see CtlState in bsgp_solver.cuh
    template <class S> __device__ __forceinline__ S* ctl() const { return reinterpret_cast<S*>(wst); }

    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ void cluster_sync() {
        if (G > 1) cg::this_cluster().sync();
        else __syncthreads();
    }
    __device__ __forceinline__ double now() {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return (double)t * 1e-9;
    }
    // All-reduce of k <= 8 doubles over the whole cluster; every thread of every CTA receives the same
    // bits (the G partials are combined in rank order everywhere).  One block barrier, then the
    // partials travel as asynchronous distributed-shared-memory stores that complete a transaction
    // barrier in the destination CTA (st.async ... mbarrier::complete_tx): no cluster-wide hardware
    // barrier, no GPU-scope fence, no L1 invalidation.  Safe reuse of the two inbox halves: a CTA can
    // be at most one reduction ahead of a peer, because it needs that peer's partials to finish one.
    __device__ __forceinline__ void allreduce(int op, double* v, int k) {
        const int lane = tid & 31, warp = tid >> 5, nwarps = (nt + 31) >> 5;
        const int half = parity & 1;
        for (int j = 0; j < k; ++j) {
            double x = v[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x = red_combine(op, x, __shfl_xor_sync(0xffffffffu, x, o));
            if (lane == 0) sh->warp_part[half][warp][j] = x;
        }
        __syncthreads();
        if (G == 1) {
            // one CTA per image (stamps): every thread adds the warp partials itself, in warp order; the other half of
            // warp_part is free for the next all-reduce (a thread is at most one all-reduce ahead of the slowest one)
            for (int j = 0; j < k; ++j) v[j] = sh->warp_part[half][0][j];
#pragma unroll 1
            for (int w = 1; w < nwarps; ++w) {
                for (int j = 0; j < k; ++j) v[j] = red_combine(op, v[j], sh->warp_part[half][w][j]);
            }
            parity ^= 1;
            return;
        }
        const unsigned bar = smem_u32(&sh->mbar[half]);
        if (tid < G * k) {
            const int dst = tid / k, j = tid - dst * k;
            double s = sh->warp_part[half][0][j];
#pragma unroll 1          // compact code: the all-reduces are real functions now and part of every iteration's instruction footprint
            for (int w = 1; w < nwarps; ++w) s = red_combine(op, s, sh->warp_part[half][w][j]);
            const unsigned slot = map_to_rank(smem_u32(&sh->inbox[half][rank][j]), dst);
            const unsigned rbar = map_to_rank(bar, dst);
            asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                         :: "r"(slot), "l"(__double_as_longlong(s)), "r"(rbar) : "memory");
        }
        {
            if (tid == 0) {
                unsigned long long state;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 %0, [%1], %2;"
                             : "=l"(state) : "r"(bar), "r"((unsigned)(G * k * 8)) : "memory");
                (void)state;
            }
            const unsigned ph = (parity >> (1 + half)) & 1;
            unsigned done = 0;
            while (!done) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                             "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar), "r"(ph) : "memory");
            }
            parity ^= 2 << half;
        }
        for (int j = 0; j < k; ++j) v[j] = sh->inbox[half][0][j];
#pragma unroll 1
        for (int r = 1; r < G; ++r) {
            for (int j = 0; j < k; ++j) v[j] = red_combine(op, v[j], sh->inbox[half][r][j]);
        }
        parity ^= 1;
    }
    __device__ __forceinline__ void allreduce_sum(double* v, int k) { allreduce(0, v, k); }
    __device__ __forceinline__ void allreduce_min(double& v) { allreduce(1, &v, 1); }
    __device__ __forceinline__ void allreduce_max(double& v) { allreduce(2, &v, 1); }
};

// The same context for images that live entirely in one CTA's shared memory (stamps: 32 x 32 pixels over 256 threads).  A
// thread then has one or two steps per pass: the register-tile batches that hide HBM latency on large slabs would only
// be code that is fetched and never looped over, and these kernels are bound by instruction fetch (the per-iteration code
// of a stamp solve is several times the instruction cache).  kSmall compiles every pass as its plain loop.
struct DeviceCtxSmall : DeviceCtx {
    static constexpr bool kSmall = true;
    // Sum all-reduce of EIGHT doubles per thread over the CTA (G = 1), one copy of the code for every call site of the
    // solver (unused slots carry zeros): the per-K variants of the generic all-reduce add up to a fifth of the
    // instructions on an iteration's path.  Within the warp the eight values are reduced together by a transposing
    // butterfly: at distance 16 every lane keeps one half of the values and hands the other half to its partner, at
    // distance 8 a quarter, at distance 4 one value, then two plain steps - 9 shuffle-adds instead of 40, and the same
    // pairing (l, l ^ 16), (l, l ^ 8), ... as the generic version, hence the same bits.  Lane l ends with the warp total
    // of value (l >> 2) & 7; one barrier, then every thread adds the warp partials in warp order.
    __device__ __forceinline__ void allreduce_sum8(double* v) {
        const int lane = tid & 31, warp = tid >> 5, nwarps = (nt + 31) >> 5;
        const int half = parity & 1;
        const bool b16 = lane & 16, b8 = lane & 8, b4 = lane & 4;
        double w[4], u[2], t;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double send = b16 ? v[i] : v[i + 4], keep = b16 ? v[i + 4] : v[i];
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const double send = b8 ? w[i] : w[i + 2], keep = b8 ? w[i + 2] : w[i];
            u[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {
            const double send = b4 ? u[0] : u[1], keep = b4 ? u[1] : u[0];
            t = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        t += __shfl_xor_sync(0xffffffffu, t, 2);
        t += __shfl_xor_sync(0xffffffffu, t, 1);
        if ((lane & 3) == 0) sh->warp_part[half][warp][lane >> 2] = t;
        __syncthreads();
        // second stage, per warp: lane j < 8 adds the partials of value j in warp order, eight shuffles hand the totals to
        // every lane (64 shared-memory loads and adds per thread otherwise)
        double tot = sh->warp_part[half][0][lane & 7];
#pragma unroll 1
        for (int wi = 1; wi < nwarps; ++wi) tot += sh->warp_part[half][wi][lane & 7];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __shfl_sync(0xffffffffu, tot, j);
        parity ^= 1;
    }
};

// every CTA initialises its two transaction barriers (one arrival each: its own expect_tx); the first
// next_item() cluster barrier publishes them before any peer can target them
__device__ __forceinline__ void init_ctx_barriers(const DeviceCtx& c) {
    if (c.tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&c.sh->mbar[0])) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&c.sh->mbar[1])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
}

__device__ __forceinline__ DeviceCtx make_ctx(SharedCtl* sh, int G) {
    DeviceCtx c;
    c.tid = threadIdx.x; c.nt = blockDim.x; c.G = G;
    c.rank = (G > 1) ? (int)cg::this_cluster().block_rank() : 0;
    c.sh = sh; c.parity = 0; c.wst = nullptr;
    init_ctx_barriers(c);
    return c;
}

// -------------------------------------------------------------------------------------------------
// Frame mode: ONE image spread over the whole GPU (sides >= 1024, BASELINE config 5: one 8192 x 8192
// frame).  The same solver code runs with the grid in the role of the cluster: G = gridDim.x CTAs (a
// power of two <= number of SMs, one per SM, cooperative launch), the "cluster barrier" is a grid
// barrier, and the all-reduce goes through a small global buffer: every CTA publishes its k partials,
// grid barrier, every CTA adds the G partials in the same order (warp j handles value j: strided sum
// per lane in rank order, then a fixed shuffle tree), so all controllers agree bit for bit.
// -------------------------------------------------------------------------------------------------
struct GridCtx {
    static constexpr bool kFrame = true;      // frame mode: panel exchange buffer, two-level twiddle tables allowed
    static constexpr bool kSmall = false;
    int tid, nt, rank, G;
    SharedCtl* sh;
    double* gpart;      // [2][G][kMaxK]
    int parity;
    void* wst;          // this warp's copy of the controller state (shared memory)
    template <class S> __device__ __forceinline__ S* ctl() const { return reinterpret_cast<S*>(wst); }

    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ void cluster_sync() { cg::this_grid().sync(); }
    __device__ __forceinline__ double now() {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return (double)t * 1e-9;
    }
    __device__ __forceinline__ void allreduce(int op, double* v, int k) {
        const int lane = tid & 31, warp = tid >> 5, nwarps = (nt + 31) >> 5;
        const int half = parity & 1;
        for (int j = 0; j < k; ++j) {
            double x = v[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x = red_combine(op, x, __shfl_xor_sync(0xffffffffu, x, o));
            if (lane == 0) sh->warp_part[0][warp][j] = x;
        }
        __syncthreads();
        if (tid < k) {
            double s = sh->warp_part[0][0][tid];
            for (int w = 1; w < nwarps; ++w) s = red_combine(op, s, sh->warp_part[0][w][tid]);
            gpart[((size_t)half * G + rank) * kMaxK + tid] = s;
        }
        cg::this_grid().sync();
        if (warp < k) {
            const double ident = (op == 0) ? 0.0 : (op == 1 ? INFINITY : -INFINITY);
            double x = ident;
            for (int r = lane; r < G; r += 32) x = red_combine(op, x, __ldcg(&gpart[((size_t)half * G + r) * kMaxK + warp]));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x = red_combine(op, x, __shfl_xor_sync(0xffffffffu, x, o));
            if (lane == 0) sh->inbox[half][0][warp] = x;
        }
        __syncthreads();
        for (int j = 0; j < k; ++j) v[j] = sh->inbox[half][0][j];
        parity ^= 1;
    }
    __device__ __forceinline__ void allreduce_sum(double* v, int k) { allreduce(0, v, k); }
    __device__ __forceinline__ void allreduce_min(double& v) { allreduce(1, &v, 1); }
    __device__ __forceinline__ void allreduce_max(double& v) { allreduce(2, &v, 1); }
};

__device__ __forceinline__ GridCtx make_grid_ctx(SharedCtl* sh, double* gpart) {
    GridCtx c;
    c.tid = threadIdx.x; c.nt = blockDim.x; c.G = gridDim.x; c.rank = blockIdx.x;
    c.sh = sh; c.gpart = gpart; c.parity = 0; c.wst = nullptr;
    return c;
}

// Pipelined ingest (bsgp_solve_batch_pinned): the copy engine writes an image into the staging buffer and then its
// flag; the cluster leader polls the flag with a system-scope acquire load before anybody reads the image (the cluster
// barrier of next_item passes the acquire on to the other CTAs).  A flag that does not arrive within 20 s (a failed
// upload) makes the cluster skip the image with BSGP_ST_INPUT_TIMEOUT instead of spinning forever.
__device__ __forceinline__ int poll_ready(const int* flag) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    int v;
    for (;;) {
        asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v) break;
        __nanosleep(400);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > 20000000000ull) break;
    }
    return v != 0;
}

// next work item for the whole cluster (leader claims it, waits for its upload if there is one, and pushes the item and
// the verdict into every CTA's shared memory).  *ready_ok = false: the item's inputs never arrived.  The flags belong to
// the queue items, or with a source map (source != NULL, the mixed-batch kernels only) to the observations: item v then
// waits for the flag of the observation its solve order[v] reads.
__device__ __forceinline__ int next_item(DeviceCtx& ctx, int* queue, const int* ready, int batch, bool* ready_ok,
                                         const int* order = nullptr, const int* source = nullptr) {
    if (ctx.rank == 0 && ctx.tid == 0) {
        const int v = atomicAdd(queue, 1);
        const int f = (source && v < batch) ? source[order ? order[v] : v] : v;
        const int ok = (ready && v < batch) ? poll_ready(ready + f) : 1;
        if (ctx.G > 1) {
            cg::cluster_group cl = cg::this_cluster();
            for (int r = 0; r < ctx.G; ++r) { *cl.map_shared_rank(&ctx.sh->next_img, r) = v; *cl.map_shared_rank(&ctx.sh->ready_verdict, r) = ok; }
        } else {
            ctx.sh->next_img = v; ctx.sh->ready_verdict = ok;
        }
    }
    ctx.cluster_sync();
    const int img = ctx.sh->next_img;
    *ready_ok = ctx.sh->ready_verdict != 0;
    ctx.cluster_sync();          // nobody may still be reading when the leader claims the next one
    return img;
}

}  // namespace bsgp
