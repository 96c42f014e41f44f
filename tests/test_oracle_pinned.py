"""The oracle (oracle/sgp_oracle.py) against the committed vectors produced by the UNMODIFIED
reference (tests/golden/make_golden.py).  make_golden asserted bit equality when it ran; here a
tight tolerance is used so that a different CPU (other SIMD code paths in numpy's pow/log) cannot
fail the suite spuriously."""
import numpy as np
import pytest

import golden_store
from cases import CASES
from oracle import sgp_oracle as orc

FAST = [n for n in CASES if not n.endswith("_332")]


@pytest.fixture(autouse=True, scope="module")
def golden_blas_threads():
    """np.dot (the reference's, hence the oracle's) runs on OpenBLAS, whose ddot splits vectors of more than 10 000 elements
    over its threads: the thread count fixes the summation order, and the long runs below amplify that last-bit difference
    to 1e-3 within a few hundred iterations.  make_golden.py ran with golden_store.BLAS_THREADS OpenBLAS threads; a machine
    with another core count reproduces its vectors only with the same count."""
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=golden_store.BLAS_THREADS, user_api="blas"):
        yield


@pytest.mark.parametrize("name", FAST)
def test_oracle_reproduces_reference(name, get_case, golden):
    gn, psf, bkg, div, kw = get_case(name)
    r = orc.solve(gn.copy(), psf.copy(), bkg, divergence=div, **kw)
    assert r.iters == int(golden[name + "/iters"])
    np.testing.assert_allclose(r.discr, golden[name + "/discr"], rtol=1e-9)
    np.testing.assert_allclose(r.x[::8, ::8], golden[name + "/x_sub"], rtol=0, atol=1e-7 * np.abs(golden[name + "/x_sub"]).max())
    if name + "/x" in golden.files:
        np.testing.assert_allclose(r.x, golden[name + "/x"], rtol=0, atol=1e-7 * np.abs(golden[name + "/x"]).max())
    assert np.array_equal(np.array(r.trace.proj_evals), golden[name + "/proj_evals"])
    if div == "beta":
        assert r.beta_param == pytest.approx(float(golden[name + "/beta_final"]), rel=1e-12)


def test_oracle_long_run_rel_err(get_case, golden, fixtures):
    """simulation_test_sgp.py:37-54: KL-SGP on the satellite simulation at the SGP-dec-optimal 332 iterations;
    the reference only returns the relative reconstruction error."""
    gn, psf, bkg, div, kw = get_case("sat_kl_332")
    r = orc.solve(gn.copy(), psf.copy(), bkg, divergence=div, **kw)
    obj = fixtures["sat/obj"]
    rel = np.sqrt(np.sum((r.x - obj) ** 2) / np.sum(obj * obj))
    assert r.iters == 332
    assert rel == pytest.approx(float(golden["sat_kl_332/rel_err"]), rel=1e-6)


def test_oracle_projection_known_answers(golden):
    for i in range(12):
        k = f"proj{i:02d}"
        sat = float(golden[k + "/sat"])
        cnt = []
        x = orc.flux_projection(np.float64(golden[k + "/b"]), golden[k + "/c"].copy(), golden[k + "/dia"].copy(),
                                float(golden[k + "/scaling"]), ccd_sat_level=None if np.isnan(sat) else sat, counter=cnt)
        np.testing.assert_allclose(x, golden[k + "/x"], rtol=1e-12, atol=1e-15)
        assert cnt[-1] == int(golden[k + "/evals"])
        assert abs(x.sum() - float(golden[k + "/b"])) <= 1e-9 * float(golden[k + "/b"])


def test_oracle_beta_divergence_helpers(golden):
    """tests.py:9-19 and :54-68 restated without torchnmf: closed form of the beta-divergence and a central
    difference of it in beta."""
    x, y = golden["betadiv/x"], golden["betadiv/y"]
    b = 1.5
    closed = np.sum((x ** b + (b - 1) * y ** b - b * x * y ** (b - 1)) / (b * (b - 1)))
    assert np.isclose(orc.beta_divergence(y, x, b), closed)
    assert np.isclose(orc.beta_divergence(y, x, b), float(golden["betadiv/value_1p5"]))
    h = 1e-6
    fd = (orc.beta_divergence(y, x, 1.7 + h) - orc.beta_divergence(y, x, 1.7 - h)) / (2 * h)
    assert np.isclose(orc.beta_divergence_dbeta(y, x, 1.7).sum(), fd, rtol=1e-6)
    np.testing.assert_allclose(orc.beta_divergence_dbeta(y, x, 1.7), golden["betadiv/deriv_1p7"], rtol=1e-13)
    # KL special case (tests.py:21-52): beta = 1 gradient equals the KL gradient
    op = orc.CircularPsf(np.full((8, 8), 1 / 64.0))
    den = np.random.default_rng(0).uniform(1, 2, 64)
    gnv = np.random.default_rng(1).uniform(1, 2, 64)
    np.testing.assert_allclose(orc.beta_divergence_grad(op.adjoint, den, gnv, 1), 1 - op.adjoint(gnv / den))


def test_oracle_error_behaviour(fixtures):
    gn, psf = fixtures["ngc/gn"], fixtures["ngc/psf"]
    with pytest.raises(ValueError, match="PSF is not normalized"):
        orc.solve(gn, psf * 1.01, np.float64(1.0), MAXIT=2)
    with pytest.raises(ValueError, match="errflag"):
        orc.solve(gn, psf, np.float64(1.0), MAXIT=2, errflag=True)


@pytest.mark.parametrize("shape,kshape", [((31, 31), (31, 31)), ((32, 32), (9, 9)), ((40, 37), (7, 11)), ((37, 40), (8, 8)),
                                           ((64, 48), (10, 7)), ((33, 33), (32, 32))])
def test_padded_operator_against_direct_space_convolution(shape, kshape):
    """Independent check of oracle.PaddedPsf (the restatement of astropy's convolve_fft for sgp.py:138,157, whose parity
    stays UNPINNED because astropy cannot be run here): for finite input, boundary='fill' with fill_value 0 and a
    normalised kernel is the plain zero-fill 'same' convolution with the kernel origin at index n_k // 2, and the
    "adjoint" of the reference is the same with the kernel psf.conj().T.  The comparison uses a DIRECT-SPACE convolution
    (scipy.signal.convolve2d, no FFT), on odd and even image and kernel sizes."""
    from scipy.signal import convolve2d
    rng = np.random.default_rng(shape[0] * 100 + kshape[1])
    x = rng.uniform(0.0, 100.0, shape)
    k = rng.random(kshape) ** 3
    k /= 7.3                                              # not normalised: convolve_fft(normalize_kernel=True) divides by the sum
    op = orc.PaddedPsf(k, shape)
    for kern, apply in ((k, op.forward), (k.conj().T, op.adjoint)):
        kn = kern / kern.sum()
        full = convolve2d(x, kn, mode="full", boundary="fill", fillvalue=0.0)
        oy, ox = kern.shape[0] // 2, kern.shape[1] // 2
        ref = full[oy:oy + shape[0], ox:ox + shape[1]]
        got = apply(x.ravel()).reshape(shape)
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()
