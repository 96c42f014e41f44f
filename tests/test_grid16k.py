"""16384-point FFT grids on the CPU: the planner's rules for them (power-of-two sides up to 16384, other sides up to 8192
wrapped onto a grid of up to 16384, frame mode on such grids, split transforms where one transform does not fit the frame
workspace), the fp32 frame-mode operator at that length, and the split transforms forced at small sizes by a small workspace
limit (operator, wrapped operator, a one-thread solve against the oracle), through the host emulation of the device headers."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import emul_helper as eh
from test_gpu_variants import FP32_OP_C
from test_host_logic import B200, BSGP_E_SHAPE

SRC = os.path.join(eh.HERE, "host_emul", "grid16k_emul.cpp")
FRAME_WS = 160 * 1024                  # the frame plans' FFT workspace limit (bsgp_plan.h, plan_launch)

# (image shape, FFT grid, CTAs per image) of the fp32 plans with a 16384-point axis, on a B200.  8200 x 900 is the padded
# grid of an 8200 x 900 image with a 31 x 31 kernel (engine.PaddedGeometry: 8200 + 31 > 8192).
LONG_AXIS_PLANS = [
    ((16384, 16384), (16384, 16384), 128),
    ((6000, 6000), (16384, 16384), 128),
    ((8191, 8191), (16384, 16384), 128),
    ((16384, 128), (16384, 128), 64),
    ((128, 16384), (128, 16384), 64),
    ((16384, 16), (16384, 16), 8),
]
REFUSED = [(16384, 20), (20, 16384), (8193, 8193), (16385, 16385), (32768, 32768), (8192, 40000)]


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("grid16k_emul") / "libgrid16k_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility-inlines-hidden",
                           "-fno-gnu-unique", "-Wl,-Bsymbolic", "-o", so, SRC])
    L = C.CDLL(so)
    for f in (L.emul_conv_frame_f32, L.emul_conv_wrapped_frame_f32):
        f.argtypes = [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.emul_plan_split.argtypes = [C.c_int] * 6
    L.emul_split_axes.argtypes = [C.c_int, C.c_int, C.c_longlong]
    L.emul_conv_split.argtypes = [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.emul_solve_split.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_int, C.POINTER(eh.capi.Params)] + [C.c_void_p] * 3 + [C.c_int] + \
        [C.c_void_p] * 17
    return L


@pytest.mark.parametrize("shape,grid,G", LONG_AXIS_PLANS)
def test_long_axis_plans_land_in_frame_mode(shape, grid, G):
    rc, s = eh.plan_launch(shape, "float32", **B200)
    assert rc == 0, rc
    assert s["frame"] and s["cluster_size"] == G and (s["grid_ny"], s["grid_nx"]) == grid
    assert s["threads"] == 512 and s["smem_bytes"] <= B200["max_smem"] and s["conv_smem"] <= B200["max_smem"]
    # a 16384-point transform, (16384 + 2048) complex floats, fits the frame workspace
    assert 147456 <= s["ws_bytes"] <= FRAME_WS
    assert (s["wrap_ny"], s["wrap_nx"]) == tuple(n if n != g else 0 for n, g in zip(shape, grid))


def test_padded_grid_of_8200_by_900_is_16384():
    from beta_sgp_b200 import engine
    geo = engine.PaddedGeometry(8200, 900, 31, 31)
    assert geo.P == 16384
    rc, s = eh.plan_launch((geo.P, geo.P), "float32", **B200)
    assert rc == 0 and s["frame"] and s["cluster_size"] == 128


def _split(lib, shape, dtype):
    return lib.emul_plan_split(shape[0], shape[1], eh.capi.BSGP_F64 if dtype == "float64" else eh.capi.BSGP_F32, B200["num_sms"],
                               B200["max_smem"], B200["smem_per_sm"])


@pytest.mark.parametrize("shape,grid,G", LONG_AXIS_PLANS)
def test_fp64_long_axis_plans_split_where_one_transform_does_not_fit(lib, shape, grid, G):
    """One fp64 transform of 16384 points needs (16384 + 2048) x 16 B = 288 KB, more than the frame workspace: exactly the
    16384-point axes run split transforms of 8192 points, on the same frame grid as fp32; fp32 never splits."""
    rc, s = eh.plan_launch(shape, "float64", **B200)
    assert rc == 0 and s["frame"] and s["cluster_size"] == G and (s["grid_ny"], s["grid_nx"]) == grid
    assert s["smem_bytes"] <= B200["max_smem"] and s["conv_smem"] <= B200["max_smem"] and s["ws_bytes"] <= FRAME_WS
    assert _split(lib, shape, "float64") == (1 if grid[1] == 16384 else 0) | (2 if grid[0] == 16384 else 0)
    assert _split(lib, shape, "float32") == 0


def test_grids_up_to_8192_never_split(lib):
    from test_gpu_variants import VARIANTS
    for v in VARIANTS:
        if not v.kernel:
            assert _split(lib, v.shape, v.dtype) == 0, v.label
    for shape in [(8192, 8192), (4096, 4096), (8192, 16), (16, 8192), (4095, 100), (1024, 1024)]:
        for dtype in ("float32", "float64"):
            assert _split(lib, shape, dtype) == 0, (shape, dtype)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("shape", REFUSED)
def test_refused_shapes(shape, dtype):
    """A 16384 side with a dense axis, sides that are not powers of two above 8192 and sides above 16384."""
    assert eh.plan_launch(shape, dtype, **B200)[0] == BSGP_E_SHAPE


@pytest.mark.parametrize("G", [1, 2, 8])
def test_long_axis_refuses_cluster_mode(G):
    assert eh.plan_launch((16384, 16384), "float32", G, **B200)[0] == BSGP_E_SHAPE
    assert eh.plan_launch((16384, 128), "float32", G, **B200)[0] == BSGP_E_SHAPE


def test_grids_up_to_8192_keep_their_plans():
    """Sides that were supported before keep the planner's result: no side of 8192 or less is forced into frame mode, and
    the largest wrapped sides of before (4096) keep their 8192 grid."""
    for shape, frame in [((8192, 16), False), ((16, 8192), False), ((4096, 4096), True), ((4095, 100), True), ((200, 200), False)]:
        for dtype in ("float32", "float64"):
            rc, s = eh.plan_launch(shape, dtype, **B200)
            assert rc == 0 and bool(s["frame"]) == frame, (shape, dtype, s)
            assert max(s["grid_ny"], s["grid_nx"]) <= 8192


def _circular(x, k, adjoint):
    """numpy's circular convolution with fftshift(k) (A), or the correlation (A^T), in fp64"""
    K = np.fft.fft2(np.fft.fftshift(k.astype(np.float64)))
    X = np.fft.fft2(x.astype(np.float64))
    return np.real(np.fft.ifft2((np.conj(K) if adjoint else K) * X))


def _bar(ref, shape):
    return FP32_OP_C * 2.0 ** -23 * np.log2(shape[0] * shape[1]) * np.abs(ref).max()


def _inputs(shape, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.0, 1000.0, shape).astype(np.float32)
    yy, xx = np.mgrid[0:shape[0], 0:shape[1]]
    cy, cx = shape[0] // 2, shape[1] // 2
    k = np.exp(-(((yy - cy) / 3.0) ** 2 + ((xx - cx) / 2.0) ** 2)).astype(np.float32)
    k /= k.sum()
    return x, k


@pytest.mark.parametrize("shape", [(16384, 32), (32, 16384)])
def test_frame_operator_f32_at_16384(lib, shape):
    """A and A^T of the fp32 frame kernels' code (column panels, the planner's grid of CTAs, 16384-point transforms in the
    frame workspace) against numpy."""
    rc, s = eh.plan_launch(shape, "float32", **B200)
    assert rc == 0 and s["frame"]
    x, k = _inputs(shape, 5)
    for adjoint in (0, 1):
        y = np.zeros(shape, np.float32)
        assert lib.emul_conv_frame_f32(shape[0], shape[1], s["cluster_size"], FRAME_WS, x.ctypes.data, k.ctypes.data, adjoint,
                                       y.ctypes.data) == 0
        ref = _circular(x, k, adjoint)
        assert np.abs(y - ref).max() <= _bar(ref, shape), (adjoint, np.abs(y - ref).max() / _bar(ref, shape))


@pytest.mark.parametrize("shape", [(6000, 40), (40, 6000)])
def test_wrapped_frame_operator_f32_on_16384_grid(lib, shape):
    """A side of 6000 wraps onto a 16384-point axis (2 n - 1 > 8192): A and A^T against numpy's circular operator."""
    grid = tuple(eh.plan_launch(shape, "float32", **B200)[1][k] for k in ("grid_ny", "grid_nx"))
    assert max(grid) == 16384
    rc, s = eh.plan_launch(shape, "float32", **B200)
    x, k = _inputs(shape, 6)
    for adjoint in (0, 1):
        y = np.zeros(shape, np.float32)
        assert lib.emul_conv_wrapped_frame_f32(shape[0], shape[1], s["cluster_size"], FRAME_WS, x.ctypes.data, k.ctypes.data,
                                               adjoint, y.ctypes.data) == 0
        ref = _circular(x, k, adjoint)
        assert np.abs(y - ref).max() <= _bar(ref, grid), (adjoint, np.abs(y - ref).max() / _bar(ref, grid))


# ------------------------------------------------------------------------------------------------
# split transforms forced at small sizes: a workspace limit that holds a transform of N / 2 points but not one of N
# ------------------------------------------------------------------------------------------------
SPLIT_CASES = [((256, 256), 4, 4000), ((512, 64), 8, 8000), ((64, 512), 8, 8000), ((256, 256), 1, 4000)]
WRAPPED_SPLIT_CASES = [((200, 150), 4, 8000), ((100, 60), 2, 2500)]


def _grid_side(n):
    return n if n & (n - 1) == 0 else 1 << int(np.ceil(np.log2(2 * n - 1)))


@pytest.mark.parametrize("shape,G,ws", SPLIT_CASES + WRAPPED_SPLIT_CASES)
def test_split_operator_fp64(lib, shape, G, ws):
    """A and A^T with split transforms (rows, columns or both, CONV_MAKE_TF included) against numpy's circular operator to
    1e-14 of max|ref|; wrapped shapes run on their power-of-two grid with the fold."""
    grid = (_grid_side(shape[0]), _grid_side(shape[1]))
    split = lib.emul_split_axes(grid[0], grid[1], ws)
    assert split != 0
    rng = np.random.default_rng(shape[0] + shape[1])
    x = rng.uniform(0.0, 1000.0, shape)
    k = rng.uniform(0.0, 1.0, shape)
    k /= k.sum()
    for adjoint in (0, 1):
        y = np.zeros(shape)
        assert lib.emul_conv_split(shape[0], shape[1], G, ws, split, x.ctypes.data, k.ctypes.data, adjoint, y.ctypes.data) == 0
        ref = _circular(x, k, adjoint)
        assert np.abs(y - ref).max() <= 1e-14 * np.abs(ref).max(), (adjoint, np.abs(y - ref).max() / np.abs(ref).max())


def test_split_solve_matches_oracle(lib):
    """Six iterations of beta-SGP (flux projection, 2-D background) with split transforms on both axes of a 256^2 grid, one
    emulated thread, against the oracle at the strict fp64 bar."""
    import importlib.util
    from oracle import sgp_oracle as orc
    from test_gpu_variants import RUNS, BETA0
    spec = importlib.util.spec_from_file_location("_grid16k_synth", os.path.join(eh.ROOT, "beta-sgp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    n, ws = 256, 4000
    rng = np.random.default_rng(77)
    psf = synth.moffat_psf(n, n, 3.0, axis_ratio=1.2, theta=0.5)
    psf /= psf.sum()
    truth = np.zeros((n, n))
    truth[rng.integers(0, n, 150), rng.integers(0, n, 150)] = 10 ** rng.uniform(2.5, 4.5, 150)
    blur = orc.CircularPsf(psf).forward(truth.ravel()).reshape(n, n)
    yy, xx = np.mgrid[0:n, 0:n]
    bkg = 300.0 + 20.0 * xx / n - 10.0 * yy / n
    gn = rng.poisson(np.maximum(blur, 0) + bkg).astype(np.float64)
    flux = float((gn - bkg).sum())
    kw = dict(RUNS["beta"])
    kw.pop("divergence")
    o = orc.solve(gn, psf, bkg, divergence="beta", flux=np.float64(flux), betaParam=BETA0, verbose=False, **kw)
    p = eh.capi.make_params(eh.capi.DIV_BETA, has_flux=True, verbose=False, **kw)
    T = p.maxit + 1
    x = np.zeros((n, n)); iters = np.zeros(1, np.int32); status = np.zeros(1, np.int32)
    discr = np.zeros(T); stopv = np.zeros(T); err = np.zeros(T + 1); bfin = np.zeros(1)
    pe = np.zeros(1, np.int32); lt = np.zeros(1, np.int32); sc = np.zeros(8)
    ta = np.zeros(T); tl = np.zeros(T); tb = np.zeros(T); tt = np.zeros(T, np.int32); te = np.zeros(T, np.int32)
    fl = np.array([flux]); b0 = np.array([BETA0])
    gnc, psfc, bkgc = (np.ascontiguousarray(a) for a in (gn, psf, bkg))
    ptr = lambda a: a.ctypes.data  # noqa: E731
    assert lib.emul_solve_split(n, n, ws, 3, C.byref(p), ptr(gnc), ptr(psfc), ptr(bkgc), 1, ptr(fl), ptr(b0), ptr(x), ptr(iters),
                              ptr(status), ptr(discr), ptr(stopv), ptr(err), ptr(bfin), ptr(pe), ptr(lt), ptr(sc), ptr(ta), ptr(tl),
                              ptr(tb), ptr(tt), ptr(te)) == 0
    it = int(iters[0])
    assert int(status[0]) == 0 and it == o.iters == kw["MAXIT"]
    assert np.array_equal(tt[1:it + 1], o.trace.trials) and np.array_equal(te[1:it + 1], o.trace.proj_evals)
    assert np.abs(discr[:it + 1] - o.discr).max() <= 1e-10 * np.abs(o.discr).max()
    assert np.abs(x - o.x).max() <= 1e-8 * np.abs(o.x).max()
    assert abs(x.sum() - o.x.sum()) <= 1e-9 * abs(o.x.sum())

