"""Frame plans on 16384-point FFT grids (run with -m gpu on a B200): power-of-two sides of 16384, and sides up to 8192 that
are not powers of two, wrapped onto a 16384-point axis (6000 x 6000: 2 n - 1 > 8192).  fp64 runs such axes as split
transforms (two 8192-point halves, bsgp_conv.cuh), fp32 as one transform.  The planner's choice on the device, the operator
against numpy, six-iteration solves against the oracle, properties of full 16384^2 solves and a two-iteration one against the
oracle, images beyond a 2^31-byte offset, the page-locked path, the padded operator and the shapes that stay refused."""
import numpy as np
import pytest

import emul_helper as eh
from test_gpu_variants import FP32_DISCR, FP32_FLUX, FP32_IMAGE, FP32_OP_C, RUNS, BETA0, _scene

pytestmark = pytest.mark.gpu
F32, F64 = "float32", "float64"
NP = {F32: np.float32, F64: np.float64}


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    yield b
    b.clear_plans()


def _device_props():
    import torch
    p = torch.cuda.get_device_properties(0)
    return dict(num_sms=p.multi_processor_count, max_smem=p.shared_memory_per_block_optin,
                smem_per_sm=p.shared_memory_per_multiprocessor)


def _op_bar(ref, grid, dtype):
    """fp64: 1e-14 of max|ref|; fp32: the operator bar of test_gpu_variants.py"""
    if dtype == F64:
        return 1e-14 * np.abs(ref).max()
    return FP32_OP_C * 2.0 ** -23 * np.log2(grid[0] * grid[1]) * np.abs(ref).max()


def _circular(x, k, adjoint):
    K = np.fft.fft2(np.fft.fftshift(k.astype(np.float64)))
    X = np.fft.fft2(x.astype(np.float64))
    return np.real(np.fft.ifft2((np.conj(K) if adjoint else K) * X))


@pytest.mark.parametrize("dtype", [F32, F64])
@pytest.mark.parametrize("shape", [(16384, 16384), (6000, 6000), (8191, 8191), (16384, 128), (128, 16384), (16384, 16)])
def test_plan_lands_where_the_planner_says(bs, shape, dtype):
    rc, s = eh.plan_launch(shape, dtype, **_device_props())
    assert rc == 0
    plan = bs.Plan(shape[0], shape[1], dtype)
    info = plan.info()
    plan.close()
    assert (info["grid_ny"], info["grid_nx"]) == (s["grid_ny"], s["grid_nx"])
    assert info["num_clusters"] == 1 and info["cluster_size"] == s["cluster_size"] and info["threads"] == 512
    assert info["smem_bytes"] == s["smem_bytes"]


@pytest.mark.parametrize("shape", [(16384, 20), (8193, 8193), (16385, 16385), (32768, 32768)])
def test_refused_shapes(bs, shape):
    for dtype in (F64, F32):
        with pytest.raises(bs.engine.BsgpError, match="error 2"):
            bs.Plan(shape[0], shape[1], dtype)


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("shape", [(16384, 128), (128, 16384), (6000, 100)])
def test_operator_against_numpy(bs, shape, dtype):
    rng = np.random.default_rng(21)
    x = rng.uniform(0.0, 1000.0, (2,) + shape).astype(NP[dtype])
    k = bs.synth.moffat_psf(shape[0], shape[1], 3.0, axis_ratio=1.3, theta=0.3)
    k = (k / k.sum()).astype(NP[dtype])
    plan = bs.Plan(shape[0], shape[1], dtype)
    grid = (plan.info()["grid_ny"], plan.info()["grid_nx"])
    plan.set_psf(k)
    for adjoint in (False, True):
        y = plan.apply_psf(x, adjoint=adjoint)
        for b in range(2):
            ref = _circular(x[b], k, adjoint)
            err = np.abs(y[b] - ref).max()
            print(f"\n{shape} {dtype} adjoint={adjoint}: {err / np.abs(ref).max():.3e} of max|ref|")
            assert err <= _op_bar(ref, grid, dtype)
    plan.close()


@pytest.mark.parametrize("dtype", [F64, F32])
def test_operator_16384_squared_impulses_linearity_and_sum(bs, dtype):
    n = 16384
    k = np.zeros((n, n), NP[dtype])
    c = n // 2
    k[c - 4:c + 5, c - 3:c + 4] = np.arange(63).reshape(9, 7) + 1.0
    k /= k.sum()
    plan = bs.Plan(n, n, dtype)
    plan.set_psf(k)
    h = np.fft.fftshift(k)                      # the operator is the circular convolution with fftshift(psf)
    tol = 1e-14 if dtype == F64 else 2.0 ** -23 * np.log2(n * n)
    for (r, q) in [(0, 0), (1, 16383), (8191, 12345), (16383, 1)]:
        x = np.zeros((n, n), NP[dtype])
        x[r, q] = 1.0
        y = plan.apply_psf(x)
        ref = np.roll(h, (r, q), axis=(0, 1))
        assert np.abs(y - ref).max() <= tol * ref.max(), (r, q)
    rng = np.random.default_rng(3)
    a = rng.uniform(0.0, 100.0, (n, n)).astype(NP[dtype])
    ya = plan.apply_psf(a)
    y2 = plan.apply_psf(2 * a)
    assert np.array_equal(y2, 2 * ya)                                    # scaling by 2 is exact in every operation
    s, sa = float(a.sum(dtype=np.float64)), float(ya.sum(dtype=np.float64))
    assert abs(sa - s) <= (1e-12 if dtype == F64 else 1e-6) * s
    plan.close()
    bs.clear_plans()


def _check(r, o, dtype, it_expected):
    it = int(r.iters[0])
    assert int(r.status[0]) == 0 and it == o.iters == it_expected
    e_d = np.abs(r.discr[0, :it + 1] - o.discr).max() / np.abs(o.discr).max()
    e_x = np.abs(r.x[0] - o.x).max() / np.abs(o.x).max()
    e_f = abs(float(r.x[0].sum(dtype=np.float64)) - o.x.sum()) / abs(o.x.sum())
    print(f"\n{dtype}: discr {e_d:.3e} image {e_x:.3e} flux {e_f:.3e}")
    if dtype == F64:
        assert np.array_equal(r.trace["evals"][0, 1:it + 1], o.trace.proj_evals)
        assert np.array_equal(r.trace["trials"][0, 1:it + 1], o.trace.trials)
        assert e_d <= 1e-10 and e_x <= 1e-8 and e_f <= 1e-9, (e_d, e_x, e_f)
    else:
        assert e_d <= FP32_DISCR and e_x <= FP32_IMAGE and e_f <= FP32_FLUX, (e_d, e_x, e_f)


@pytest.mark.parametrize("run", ["beta", "kl"])
def test_6000_wrapped_solve_matches_oracle(bs, run):
    """Six iterations on a 6000 x 6000 image (wrapped on the 16384^2 grid) against the oracle: fp64 (split transforms) at
    the strict bar of test_gpu_variants.py, fp32 on the same fp32-exact inputs at its fp32 bars."""
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _scene(bs, (6000, 6000), 0, seed=6000)
    kw = dict(RUNS[run])
    div = kw.pop("divergence")
    if run == "beta":
        o = orc.solve(gn, psf, bkg, divergence=div, flux=np.float64(flux), betaParam=BETA0, verbose=False, **kw)
        args = dict(bkg=bkg[None], flux=[flux], betaParam=BETA0)
    else:
        o = orc.solve(gn, psf, np.float64(300.0), divergence=div, verbose=False, **kw)
        args = dict(bkg=np.array([300.0]), flux=None, betaParam=1.005)
    for dtype in (F64, F32):
        r = bs.solve_batch(gn[None].astype(NP[dtype]), psf.astype(NP[dtype]), divergence=div, dtype=dtype, trace=True, verbose=False,
                           **args, **kw)
        _check(r, o, dtype, kw["MAXIT"])
        bs.clear_plans()


def _frame_16384(bs, seed, dtype):
    n = 16384
    rng = np.random.default_rng(seed)
    psf = bs.synth.moffat_psf(n, n, 3.5).astype(NP[dtype])
    truth = np.zeros((n, n), NP[dtype])
    k = 400_000
    truth[rng.integers(0, n, k), rng.integers(0, n, k)] = 10.0 ** rng.uniform(3.0, 5.0, k)
    plan = bs.get_plan(n, n, dtype)
    plan.set_psf(psf)
    blurred = plan.apply_psf(truth)
    gn = rng.poisson(np.maximum(blurred, 0.0).astype(np.float64) + 300.0).astype(NP[dtype])
    return gn, psf, float((gn.astype(np.float64) - 300.0).sum())


@pytest.mark.parametrize("dtype", [F64, F32])
def test_16384_squared_solve_properties(bs, dtype):
    """beta-SGP with the flux projection on a full 16384^2 frame: status OK, non-negative, flux conserved (fp64 to 1e-9),
    objective decreasing."""
    gn, psf, flux = _frame_16384(bs, 11, dtype)
    kw = dict(bs.synth.TILE_KWARGS, stop_criterion=1, MAXIT=3)
    r = bs.solve_batch(gn[None], psf, np.array([300.0], NP[dtype]), divergence="beta", flux=[flux], betaParam=BETA0,
                       dtype=dtype, **kw)
    assert int(r.status[0]) == 0 and int(r.iters[0]) == 3
    assert r.x.min() >= 0.0 and np.isfinite(r.x).all()
    assert abs(float(r.x[0].sum(dtype=np.float64)) - flux) <= (1e-9 if dtype == F64 else FP32_FLUX) * flux
    assert np.all(np.diff(r.discr[0, :4]) < 0)
    bs.clear_plans()


def test_16384_squared_fp64_two_iterations_match_oracle(bs):
    """Two iterations of beta-SGP (flux projection, 2-D background) on a 16384^2 fp64 frame against the oracle, strict bar."""
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _scene(bs, (16384, 16384), 0, seed=16384)
    kw = dict(RUNS["beta"], MAXIT=2)
    div = kw.pop("divergence")
    o = orc.solve(gn, psf, bkg, divergence=div, flux=np.float64(flux), betaParam=BETA0, verbose=False, **kw)
    r = bs.solve_batch(gn[None], psf, bkg[None], divergence=div, flux=[flux], betaParam=BETA0, dtype=F64, trace=True,
                       verbose=False, **kw)
    _check(r, o, F64, 2)
    bs.clear_plans()


def test_images_beyond_a_2gib_offset_match_their_single_solves(bs):
    """A batch of two 16384^2 fp64 images: one image is exactly 2^31 bytes, so the second starts at byte offset 2^31 of
    every image array (inputs, outputs).  Each image must be bit-identical to its own solve."""
    gn0, psf, f0 = _frame_16384(bs, 12, F64)
    gns = np.stack([gn0, np.roll(gn0, 777, axis=1)])
    assert gns[1].ctypes.data - gns.ctypes.data == 2 ** 31
    fl = [float((g - 300.0).sum()) for g in gns]
    kw = dict(bs.synth.TILE_KWARGS, stop_criterion=1, MAXIT=2)
    common = dict(divergence="beta", betaParam=BETA0, dtype=F64, **kw)
    rb = bs.solve_batch(gns, psf, np.full(2, 300.0), flux=fl, **common)
    for i in (0, 1):
        r1 = bs.solve_batch(gns[i:i + 1], psf, np.array([300.0]), flux=[fl[i]], **common)
        assert int(rb.status[i]) == int(r1.status[0]) == 0
        assert np.array_equal(rb.x[i], r1.x[0]), i
        assert np.array_equal(rb.discr[i], r1.discr[0]), i
    bs.clear_plans()


def test_6000_page_locked_path_matches_numpy(bs):
    import torch
    gn, psf, bkg, flux = _scene(bs, (6000, 6000), 0, seed=6001)
    kw = dict(RUNS["beta"], MAXIT=3)
    div = kw.pop("divergence")
    common = dict(divergence=div, flux=[flux], betaParam=BETA0, dtype=F64, verbose=False, **kw)
    ref = bs.solve_batch(gn[None], psf, bkg[None], **common)
    g_p = torch.from_numpy(np.ascontiguousarray(gn[None])).pin_memory()
    b_p = torch.from_numpy(np.ascontiguousarray(bkg[None])).pin_memory()
    r = bs.solve_batch(g_p, psf, b_p, **common)
    assert int(r.status[0]) == int(ref.status[0]) == 0
    assert np.array_equal(r.x.numpy(), ref.x)
    assert np.array_equal(r.discr, ref.discr)
    bs.clear_plans()


def test_padded_operator_on_a_16384_grid(bs):
    """padded=True on an 8200 x 900 image with a 31 x 31 kernel (padded grid 16384^2, fp64: split transforms): runs,
    conserves the flux, and gives the same result from numpy arrays and from CUDA tensors."""
    import torch
    rng = np.random.default_rng(8)
    psf = bs.synth.moffat_psf(31, 31, 3.0)
    psf /= psf.sum()
    truth = np.zeros((8200, 900))
    truth[rng.integers(5, 8195, 3000), rng.integers(5, 895, 3000)] = 10 ** rng.uniform(3, 4.5, 3000)
    from oracle import sgp_oracle as orc
    blur = orc.PaddedPsf(psf, truth.shape).forward(truth.ravel()).reshape(truth.shape)
    gn = rng.poisson(np.maximum(blur, 0) + 300.0).astype(np.float64)
    flux = float((gn - 300.0).sum())
    kw = dict(bs.synth.TILE_KWARGS, stop_criterion=1, MAXIT=3)
    common = dict(divergence="beta", flux=[flux], betaParam=BETA0, dtype=F64, padded=True, **kw)
    r = bs.solve_batch(gn[None], psf, np.array([300.0]), **common)
    assert int(r.status[0]) == 0 and r.x.shape == (1, 8200, 900)
    assert abs(float(r.x[0].sum()) - flux) <= 1e-9 * flux
    rt = bs.solve_batch(torch.from_numpy(gn[None]).cuda(), psf, torch.tensor(300.0, dtype=torch.float64, device="cuda"), **common)
    assert np.array_equal(rt.x.cpu().numpy(), r.x)
    bs.clear_plans()
