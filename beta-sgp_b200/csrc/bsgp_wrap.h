// Wrapped plans: the index arithmetic of the arbitrary-size circular operator, shared by the CUDA library
// (bsgp_kernels.cu) and the test-only host emulation (tests/host_emul).
//
// The reference's numpy closure (sgp.py:108-120 / 570-582) accepts any image size: TF = fftn(fftshift(psf)),
// A(x) = real(ifftn(TF * fftn(x))), A^T with conj(TF).  That is the circular convolution of x with
// h = fftshift(psf), h[j] = psf[(j - n//2) mod n] per axis (np.roll by n//2: for odd n the PSF centre n//2 lands at
// index n - 1, not 0 - the one-pixel offset SURVEY.md 8(a2) lists as a quirk to keep), and for A^T the circular
// correlation with h, i.e. the convolution with h~[j] = h[(-j) mod n].
//
// A side n that is not a power of two in [16, 8192] runs on a power-of-two grid of side P >= 2 n - 1: the image sits at
// the origin (zeros elsewhere), the kernel occupies [0, n) as well, the grid convolution is then the LINEAR convolution
// z of the two (no wrap-around: 2 n - 1 <= P), and the circular result is the fold y[i] = z[i] + z[i + n], i < n.
#pragma once

#if defined(__CUDACC__)
#define BSGP_HD __host__ __device__ inline
#else
#define BSGP_HD inline
#endif

namespace bsgp {

// Largest grid side: power-of-two sides up to kMaxSide run on their own grid; any other side up to kMaxSide / 2 wraps onto
// a grid of at most kMaxSide (2 n - 1 <= kMaxSide - 1).  Grid sides above kMaxClusterSide run in frame mode only
// (bsgp_plan.h, plan_launch).
constexpr int kMaxSide = 16384;
constexpr int kMaxClusterSide = 8192;
constexpr int kMaxDense = 32;

// Short sides that are not a power of two (n <= 32: the reference's 31 x 31 cut-outs) do not wrap: they keep a grid of
// side 16 or 32 >= n and their transform is a dense DFT of length n over the first n slots (bsgp_fft.cuh,
// dense_dft_batch), i.e. the circular operator itself - no fold, and arrays of the image's own size.
// dense_len(n) is that length, 0 for every other side.
BSGP_HD int dense_len(int n) {
    if (n >= 16 && (n & (n - 1)) == 0) return 0;
    return n <= kMaxDense ? n : 0;
}

// FFT grid side for an image side n; > kMaxSide means unsupported
BSGP_HD int wrap_grid_side(int n) {
    if (n >= 16 && n <= kMaxSide && (n & (n - 1)) == 0) return n;
    if (dense_len(n)) return n <= 16 ? 16 : 32;
    int P = 16;
    while (P < 2 * n - 1 && P <= kMaxSide) P *= 2;
    return P;
}

// Kernel image handed to CONV_MAKE_TF for a wrapped plan.  CONV_MAKE_TF computes fftn(fftshift_P(g)) on the grid, so
// g[(j + P/2) mod P] = k[j] puts kernel value k[j] at grid index j: k = h for A, k = h~ for A^T.  Returns false where
// g is zero; otherwise (*sr, *sc) is the pixel of the caller's PSF that belongs at grid position (r, c).  An axis whose
// grid side equals the image side (a power of two) reduces to g = psf (A) or the index-reversed psf (A^T).  A dense axis
// uses the same placement: its transform sees k on slots [0, n) and computes the length-n DFT of it.
BSGP_HD bool wrap_psf_source(int r, int c, int ny, int nx, int iny, int inx, int adjoint, int* sr, int* sc) {
    int jr = (r + ny - (ny >> 1)) % ny, jc = (c + nx - (nx >> 1)) % nx;
    if (jr >= iny || jc >= inx) return false;
    if (adjoint) { jr = (iny - jr) % iny; jc = (inx - jc) % inx; }
    *sr = (jr + iny - (iny >> 1)) % iny;
    *sc = (jc + inx - (inx >> 1)) % inx;
    return true;
}

}  // namespace bsgp
