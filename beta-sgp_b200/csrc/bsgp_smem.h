// Plain-data layouts of the persistent kernels' shared memory, shared by the device code (bsgp_device.cuh) and the
// launch-shape planner (bsgp_plan.h), which g++ also compiles for the test-only host emulation (tests/host_emul).
#pragma once

namespace bsgp {

constexpr int kMaxWarps = 16;      // 512 threads per CTA at most
constexpr int kMaxG = 16;
constexpr int kMaxK = 8;

struct SharedCtl {
    double warp_part[2][kMaxWarps][kMaxK];   // two halves (parity bit 0), so that a single-CTA all-reduce needs one barrier only
    double inbox[2][kMaxG][kMaxK];
    unsigned long long mbar[2];     // transaction barriers of the two inbox halves (cluster all-reduce)
    int next_img;
    int ready_verdict;
    int pad[2];
};

// dynamic shared memory layout of the persistent kernels (byte offsets, computed by the host)
struct SmemPlan {
    unsigned off_state;     // ImgState<T>
    unsigned off_ctl;       // CtlState<T>, one copy per warp (stride ctl_stride bytes)
    unsigned ctl_stride;
    unsigned off_twx;       // twiddles of the row transforms (if tw_smem)
    unsigned off_twy;       // twiddles of the column transforms (if tw_smem; may equal off_twx)
    unsigned off_ppx;       // padded-position table of the row transforms (nx x u16)
    unsigned off_ws;        // FFT workspace
    unsigned off_bufs;      // resident slab buffers
    int tw_smem;            // 0: twiddles stay in global memory, 1: full tables in shared memory, 2: two-level tables
};

}  // namespace bsgp
