"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol of include/bsgp.h, the
ctypes structs match the C structs, the product fails loudly without a device, and the device headers
— compiled for the host as a one-thread emulation, tests/host_emul — produce the reference's numbers:
FFT stages, the cluster-partitioned convolution, the projection root-find and the solver controller."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import emul_helper as eh
from cases import CASES, SENSITIVE, STRICT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
capi = eh.capi
P = C.POINTER(C.c_double)


def test_library_exports_header_symbols():
    if not os.path.exists(capi.LIB_PATH):
        pytest.skip("libbsgp.so not built (run __graft_entry__.build())")
    hdr = open(os.path.join(ROOT, "include", "bsgp.h")).read()
    declared = set(re.findall(r"\b(bsgp_[a-z_0-9]+)\s*\(", hdr))
    L = capi.lib()
    for sym in declared:
        assert hasattr(L, sym), f"{sym} declared in include/bsgp.h but not exported"
    assert declared == set(capi.EXPORTED)
    assert b"sm_100a" in L.bsgp_version()


def test_ctypes_structs_match_c_layout():
    L = eh.lib()
    assert C.sizeof(capi.Params) == L.emul_sizeof_params()
    assert C.sizeof(capi.Inputs) == L.emul_sizeof_inputs()
    assert C.sizeof(capi.Outputs) == L.emul_sizeof_outputs()
    assert C.sizeof(capi.PlanInfo) == L.emul_sizeof_plan_info()


def test_no_cpu_fallback():
    """Without a CUDA device the product raises; it never computes on the host."""
    if not os.path.exists(capi.LIB_PATH):
        pytest.skip("libbsgp.so not built")
    if capi.lib().bsgp_device_count() > 0:
        pytest.skip("a GPU is present")
    import beta_sgp_b200 as b
    img = np.ones((32, 32))
    with pytest.raises(RuntimeError, match="libbsgp error"):
        b.sgp_betaDiv_batch(img[None], img / img.sum(), 0.1, MAXIT=2)
    with pytest.raises(RuntimeError, match="libbsgp error"):
        b.projectDF(np.float64(1.0), np.ones(8), np.ones(8), 1.0)
    pkg = os.path.join(ROOT, "beta-sgp_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            src = open(os.path.join(pkg, f)).read()
            assert not re.search(r"^\s*(import|from)\s+oracle", src, re.M), f"{f} imports the oracle"
            assert "host_emul" not in src and "libbsgp_emul" not in src, f"{f} reaches the test-only emulation"


@pytest.mark.parametrize("n", [8, 16, 32, 64, 128, 256, 512, 1024, 4096, 8192])
def test_emulated_fft_stages(n):
    L = eh.lib()
    rng = np.random.default_rng(n)
    x = rng.normal(size=(3, n)) + 1j * rng.normal(size=(3, n))
    xin = np.ascontiguousarray(x).view(np.float64).copy()
    for split in ((0, 1) if n >= 64 else (0,)):          # full twiddle table / two-level table (long transforms)
        for inverse_after in (0, 1):
            out = np.zeros_like(xin)
            assert L.emul_fft1d(n, 3, xin.ctypes.data_as(P), out.ctypes.data_as(P), inverse_after, split) == 0
            got = out.view(np.complex128).reshape(3, n)
            ref = np.fft.fft(x, axis=1) if not inverse_after else x * n
            assert np.abs(got - ref).max() <= 2e-15 * np.abs(ref).max() * np.log2(n)


@pytest.mark.parametrize("ny,nx,G,ws", [(32, 32, 1, 1 << 20), (32, 32, 2, 1 << 20), (64, 64, 4, 1 << 20), (256, 256, 8, 72 * 1024),
                                        (256, 256, 16, 72 * 1024), (128, 512, 8, 40 * 1024), (512, 128, 2, 72 * 1024), (64, 32, 2, 4096)])
def test_emulated_cluster_convolution(ny, nx, G, ws):
    """real(ifftn(TF * fftn(x))) with TF = fftn(fftshift(psf)) or conj (sgp.py:109-117), rows/columns
    partitioned over G emulated CTAs and tiled to the workspace limit."""
    L = eh.lib()
    L.emul_conv.argtypes = [C.c_int] * 3 + [C.c_longlong, P, P, C.c_int, P]
    rng = np.random.default_rng(ny * 1000 + nx + G)
    x = rng.normal(size=(ny, nx))
    psf = rng.random((ny, nx))
    psf /= psf.sum()
    L.emul_conv_frame.argtypes = L.emul_conv.argtypes
    for fn in (L.emul_conv, L.emul_conv_frame):            # row-major exchange buffer / column panels (frame mode)
        for adjoint in (0, 1):
            y = np.zeros((ny, nx))
            assert fn(ny, nx, G, ws, x.ctypes.data_as(P), psf.ctypes.data_as(P), adjoint, y.ctypes.data_as(P)) == 0
            tf = np.fft.fftn(np.fft.fftshift(psf))
            ref = np.real(np.fft.ifftn((np.conj(tf) if adjoint else tf) * np.fft.fftn(x)))
            assert np.abs(y - ref).max() <= 5e-15 * np.abs(ref).max()


def _tile_split(ny, nx, G, ws, elem):
    """(row tile pairs, column tile) of make_geom (csrc/bsgp_plan.h) for complex elements of `elem` bytes."""
    def plen(n):
        return n + (n >> 3)                               # the last radix stage is 8 for every side >= 16
    rtp, ct = ny // G // 2, nx // 2 // G
    while rtp > 1 and rtp * plen(nx) * elem > ws:
        rtp >>= 1
    while ct > 1 and ct * (plen(ny) | 1) * elem > ws:
        ct >>= 1
    return rtp, ct


@pytest.mark.parametrize("ny,nx,G,ws", [(32, 32, 1, 1 << 20), (32, 32, 2, 1 << 20), (64, 64, 4, 1 << 20), (256, 256, 8, 72 * 1024),
                                        (256, 256, 16, 72 * 1024), (128, 512, 8, 40 * 1024), (512, 128, 2, 72 * 1024), (64, 32, 2, 4096),
                                        (256, 256, 2, 36 * 1024)])
def test_emulated_cluster_convolution_f32(ny, nx, G, ws):
    """The fp32 sibling of test_emulated_cluster_convolution: make_geom sizes the tiles with sizeof(cplx<float>), so fp32
    runs row / column tile partitions that fp64 never runs (the last case: 16 row-tile pairs and 8 columns per tile in fp32
    against 8 and 4 in fp64).  Against numpy in fp64 on the same fp32 values, within 2^-23 * log2(ny * nx) of the
    largest value (the bar of the device's fp32 operator, tests/test_gpu_variants.py)."""
    if (ny, nx, G, ws) == (256, 256, 2, 36 * 1024):
        assert _tile_split(ny, nx, G, ws, 8) != _tile_split(ny, nx, G, ws, 16)
    L = eh.lib()
    F = C.POINTER(C.c_float)
    L.emul_conv_f32.argtypes = [C.c_int] * 3 + [C.c_longlong, F, F, C.c_int, F]
    rng = np.random.default_rng(ny * 1000 + nx + G)
    x = rng.normal(size=(ny, nx)).astype(np.float32)
    psf = rng.random((ny, nx))
    psf = (psf / psf.sum()).astype(np.float32)
    tf = np.fft.fftn(np.fft.fftshift(psf.astype(np.float64)))
    for adjoint in (0, 1):
        y = np.zeros((ny, nx), np.float32)
        assert L.emul_conv_f32(ny, nx, G, ws, x.ctypes.data_as(F), psf.ctypes.data_as(F), adjoint, y.ctypes.data_as(F)) == 0
        ref = np.real(np.fft.ifftn((np.conj(tf) if adjoint else tf) * np.fft.fftn(x.astype(np.float64))))
        assert np.abs(y - ref).max() <= 2.0 ** -23 * np.log2(ny * nx) * np.abs(ref).max()


def test_emulated_projection_known_answers(golden):
    for i in range(12):
        k = f"proj{i:02d}"
        sat = float(golden[k + "/sat"])
        cap = None if np.isnan(sat) else sat / float(golden[k + "/scaling"]) - np.finfo(float).eps
        x, evals, st = eh.project(golden[k + "/c"], golden[k + "/dia"], float(golden[k + "/b"]), cap)
        assert st == 0
        assert evals == int(golden[k + "/evals"])
        np.testing.assert_allclose(x, golden[k + "/x"], rtol=1e-9, atol=1e-12 * np.abs(golden[k + "/x"]).max())


EMUL_CASES = ["ngc_kl_27", "ngc_beta_p1_stop3", "ngc_kl_p1_stop2", "ngc_kl_stop2_quiet", "ngc_kl_stop4", "ngc_kl_init0",
              "ngc_kl_init1_p1", "ngc_kl_noscale_flux", "ngc_kl_nonmonotone", "sat_kl_default_stop", "ngc_beta_adapt",
              "ngc_beta_is", "ngc_beta_one", "ngc_beta_two", "stamp00", "stamp01", "stamp06", "stamp10", "tile00", "tile07",
              "cutout31_00", "cutout31_04", "cutout31_07", "cutout31_kl_03"]


@pytest.mark.parametrize("name", EMUL_CASES)
def test_emulated_solver_matches_reference(name, get_case, golden):
    """bsgp_solver.cuh run as one emulated CTA: identical iteration counts, projection-evaluation counts
    and stopping decisions; objective trace and image within the north-star tolerances."""
    gn, psf, bkg, div, kw = get_case(name)
    r = eh.solve(gn, psf, bkg, divergence=div, wrapped=name.startswith("cutout31"), **kw)      # 31 x 31: wrapped plan
    assert r["status"] == 0
    assert r["iters"] == int(golden[name + "/iters"])
    ref = golden[name + "/discr"]
    tol_d, tol_x = SENSITIVE.get(name, (1e-10, 1e-8))
    assert np.abs(r["discr"] - ref).max() <= tol_d * np.abs(ref).max()
    xs = golden[name + "/x_sub"]
    assert np.abs(r["x"][::8, ::8] - xs).max() <= tol_x * np.abs(xs).max()
    assert np.array_equal(r["evals"], golden[name + "/proj_evals"])
    assert r["proj_evals"] == int(golden[name + "/proj_evals"].sum() + golden[name + "/init_proj_evals"])
    n = r["iters"]
    # every line search but the (discarded) last one takes the reference's number of trials
    assert np.array_equal(r["trials"][:n - 1], golden[name + "/trials"][:n - 1])
    # step lengths agree wherever the step was not a line-search escape (lam < 1e-12: sk, yk are rounding noise)
    real = golden[name + "/lam"][:n - 1] > 1e-6
    np.testing.assert_allclose(r["alpha"][:n - 1][real], golden[name + "/alpha"][:n - 1][real], rtol=1e-6)
    if div == "beta":
        assert r["beta_final"] == pytest.approx(float(golden[name + "/beta_final"]), rel=1e-9)


def test_emulated_solver_flags_bad_flux(fixtures):
    gn, psf = fixtures["stamp0/gn"], fixtures["stamp0/psf"]
    r = eh.solve(gn, psf, np.float64(1e9), divergence="beta", proj_type=1, init_recon=2, stop_criterion=3, MAXIT=5)
    assert r["status"] == capi.ST_BAD_FLUX and r["iters"] == 0


def test_pow_inline_accuracy():
    """pow_inline (csrc/bsgp_math.cuh) replaces the library pow in the beta-divergence phases: den^(beta-1),
    gn^beta (sgp.py:457-458, 495, 499).  Against 80-bit long-double pow: at most 1.3 ulp (CUDA's own pow is
    documented at 2 ulp), exact special cases through the library fallback."""
    import ctypes as C
    L = eh.lib()
    rng = np.random.default_rng(0)

    def run(x, y):
        out = np.empty_like(x)
        L.emul_pow(x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.c_longlong(x.size))
        return out

    n = 400_000
    for lo, hi, ylo, yhi in [(-8, 0.3, -0.15, 0.15), (-40, 0.3, 0.85, 1.15), (-300, 300, -2.0, 2.0)]:
        x = 10.0 ** rng.uniform(lo, hi, n)
        y = rng.uniform(ylo, yhi, n)
        got = run(x, y)
        with np.errstate(over="ignore"):
            ref = np.power(x.astype(np.longdouble), y.astype(np.longdouble))
            ok = np.isfinite(ref.astype(np.float64)) & (np.abs(ref) > 1e-300)
        ulp = np.spacing(np.abs(ref[ok]).astype(np.float64)).astype(np.longdouble)
        err = np.abs(got[ok].astype(np.longdouble) - ref[ok]) / ulp
        assert float(err.max()) <= 1.3, float(err.max())
    x = np.array([1.0, 2.0, 0.5, 4.0, 1e-310, 0.0, -1.0, np.inf, np.nan, 3.0])
    y = np.array([0.3, 0.5, 2.0, -0.5, 0.5, 0.5, 0.5, 0.5, 0.5, 0.0])
    with np.errstate(invalid="ignore"):
        np.testing.assert_allclose(run(x, y), np.power(x, y), rtol=3e-16, atol=0, equal_nan=True)


def test_queue_order_hint():
    """The work queue hands out the images with beta closest to 1 first (engine._queue_order); KL batches and
    batches with one common beta keep the natural order."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bsgp_pkg_for_test", os.path.join(ROOT, "beta-sgp_b200", "__init__.py"),
                                                  submodule_search_locations=[os.path.join(ROOT, "beta-sgp_b200")])
    pkg = importlib.util.module_from_spec(spec)
    import sys
    sys.modules["bsgp_pkg_for_test"] = pkg
    spec.loader.exec_module(pkg)
    b = np.array([1.0882, 1.0248, 0.9703, 1.0815, 1.0065, 1.0882, 1.0248])
    order = pkg.engine._queue_order("beta", b)
    assert order.dtype == np.int32 and sorted(order.tolist()) == list(range(7))
    assert order[0] == 4 and np.all(np.diff(np.abs(b[order] - 1.0)) >= 0)
    assert pkg.engine._queue_order("kl", b) is None
    assert pkg.engine._queue_order("beta", np.full(5, 1.005)) is None


def _padded_case(ny, nx, k, seed):
    import importlib.util
    import sys
    from oracle import sgp_oracle as orc
    if "bsgp_pkg_for_test" not in sys.modules:
        spec = importlib.util.spec_from_file_location("bsgp_pkg_for_test", os.path.join(ROOT, "beta-sgp_b200", "__init__.py"),
                                                      submodule_search_locations=[os.path.join(ROOT, "beta-sgp_b200")])
        pkg = importlib.util.module_from_spec(spec)
        sys.modules["bsgp_pkg_for_test"] = pkg
        spec.loader.exec_module(pkg)
    pkg = sys.modules["bsgp_pkg_for_test"]
    rng = np.random.default_rng(seed)
    psf = pkg.synth.moffat_psf(k, k, 3.0, axis_ratio=1.2, theta=0.4)
    psf /= psf.sum()
    truth = np.zeros((ny, nx))
    truth[rng.integers(3, ny - 3, 12), rng.integers(3, nx - 3, 12)] = 10 ** rng.uniform(3, 4.5, 12)
    gn = rng.poisson(np.maximum(orc.PaddedPsf(psf, truth.shape).forward(truth.ravel()).reshape(ny, nx), 0) + 100.0).astype(float)
    return pkg, orc, gn, psf


@pytest.mark.parametrize("div,kw", [
    ("beta", dict(proj_type=1, init_recon=2, stop_criterion=3, MAXIT=40, alpha=10.0, ccd_sat_level=65000, adapt_beta=True,
                  schedule_lr=True, betaParam=1.02)),
    ("kl", dict(init_recon=3, stop_criterion=2, MAXIT=25)),
])
def test_emulated_padded_operator_matches_oracle(div, kw):
    """use_original_SGP_Afunction=False (sgp.py:121-161): odd-sized image (41 x 37), 15 x 15 asymmetric kernel, 64 x 64
    grid.  The device headers (host emulation) against the oracle's restatement of convolve_fft (PARITY UNPINNED:
    astropy itself is not available, see oracle.PaddedPsf)."""
    pkg, orc, gn, psf = _padded_case(41, 37, 15, 0)
    kw = dict(kw)
    b0 = kw.pop("betaParam", 1.005)
    flux = float((gn - 100.0).sum())
    o = orc.solve(gn, psf, np.float64(100.0), divergence=div, betaParam=b0, flux=np.float64(flux), use_original_SGP_Afunction=False, **kw)
    geo = pkg.engine.PaddedGeometry(41, 37, 15, 15)
    assert geo.P == 64 and geo.region == (12, 53, 14, 51)
    big, da = geo.kernel(psf, np.float64)
    bigt, dat = geo.kernel(psf.conj().T, np.float64)
    r = eh.solve(geo.embed(gn, np.float64), big, np.float64(100.0), divergence=div, betaParam=b0, flux=flux, psf_adjoint=bigt,
                 region=geo.region, div_a=da, div_at=dat, adjoint_second_psf=True, **kw)
    assert r["status"] == 0 and r["iters"] == o.iters
    assert np.abs(r["discr"] - o.discr).max() <= 1e-10 * np.abs(o.discr).max()
    x = r["x"][geo.rows, geo.cols]
    assert np.abs(x - o.x).max() <= 1e-8 * np.abs(o.x).max()
    pad = r["x"].copy()
    pad[geo.rows, geo.cols] = 0.0
    assert not pad.any()                                      # nothing leaks into the padding


def test_tile_boxes_match_reference_golden():
    """bsgp_tile_boxes (host index arithmetic, no GPU) against the outputs of the reference's calculate_slice_bboxes
    (utils.py:332-375) committed by tests/golden/make_tiles_golden.py."""
    import json
    import beta_sgp_b200 as bs
    cases = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiles_golden.json")))
    assert len(cases) >= 10
    for c in cases:
        assert bs.tiles.calculate_slice_bboxes(*c["args"]) == c["boxes"], c["args"]
    # create_subdivisions' call shape (utils.py:381-384) and the synthetic workload's own enumeration agree
    org = bs.tiles.tile_origins((2048, 2048), (256, 256), 0)
    assert [tuple(o) for o in org.tolist()] == bs.synth.tile_boxes(2048, 2048, 256, 0)
    with pytest.raises(bs._capi.BsgpError):
        bs.tiles.calculate_slice_bboxes(100, 100, 10, 10, 1.0, 0.0)          # the reference would loop forever


def test_psf_model_file_parsing(tmp_path):
    """PSF(txt_file) reads a DIAPL coefficient file like psf_calculate.py:8-46 (host only; the evaluation is a CUDA kernel)."""
    import beta_sgp_b200 as bs
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "psf_golden.npz"))
    txt = tmp_path / "psf.bin.txt"
    txt.write_text("\n".join(repr(float(v)) for v in g["file_values"]) + "\n")
    p = bs.psf_model.PSF(str(txt))
    assert (p.hw, p.ndeg_spat, p.ndeg_local, p.ngauss) == (15, 1, 2, 2)
    assert (p.cos, p.sin, p.ax, p.ay, p.sigma_inc) == tuple(g["file_values"][[5, 6, 7, 8, 9]])
    assert p.ntot == 36 and len(p.coeffs) == 36
    row = p.params()
    assert row.shape == (5 + 12,) and np.array_equal(row[5:], g["file_values"][14:26])


@pytest.mark.parametrize("ny,nx,G,ws", [(31, 31, 1, 1 << 20), (30, 30, 1, 1 << 20), (17, 24, 1, 1 << 20), (9, 12, 1, 1 << 20), (33, 20, 1, 1 << 20), (48, 48, 4, 1 << 20),
                                        (5, 7, 1, 1 << 20), (32, 31, 1, 1 << 20), (31, 64, 1, 40 * 1024), (100, 75, 8, 72 * 1024),
                                        (375, 375, 8, 72 * 1024), (450, 450, 8, 160 * 1024)])
def test_emulated_wrapped_convolution(ny, nx, G, ws):
    """Sides that are not powers of two (sgp.py:108-120 accepts any size; application_sgp_star_stamps.py:24 uses 31):
    linear convolution on a 2^k >= 2n-1 grid + fold == the reference's circular operator, odd-size fftshift offset
    included (SURVEY.md 8 a2)."""
    L = eh.lib()
    L.emul_conv_wrapped.argtypes = [C.c_int] * 3 + [C.c_longlong, P, P, C.c_int, P]
    rng = np.random.default_rng(ny * 1000 + nx + G)
    x = rng.normal(size=(ny, nx))
    psf = rng.random((ny, nx))
    psf /= psf.sum()
    tf = np.fft.fftn(np.fft.fftshift(psf))
    for adjoint in (0, 1):
        y = np.zeros((ny, nx))
        assert L.emul_conv_wrapped(ny, nx, G, ws, x.ctypes.data_as(P), psf.ctypes.data_as(P), adjoint, y.ctypes.data_as(P)) == 0
        ref = np.real(np.fft.ifftn((np.conj(tf) if adjoint else tf) * np.fft.fftn(x)))
        assert np.abs(y - ref).max() <= 1e-14 * np.abs(ref).max()


def _stamp31(seed, n=31):
    """A 31 x 31 cut-out in the shape of application_sgp_star_stamps.py:58-89 (synthetic: one star, Poisson noise, sky)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_synth_t", os.path.join(ROOT, "beta-sgp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    rng = np.random.default_rng(seed)
    psf = synth.moffat_psf(n, n, rng.uniform(2.5, 4.5), 2.5, rng.uniform(1.0, 1.3), rng.uniform(0, np.pi))
    obj = np.zeros((n, n))
    obj[n // 2 + rng.integers(-2, 3), n // 2 + rng.integers(-2, 3)] = 10.0 ** rng.uniform(4.0, 5.5)
    sky = rng.uniform(50.0, 800.0)
    tf = np.fft.fftn(np.fft.fftshift(psf))
    gn = rng.poisson(np.maximum(np.real(np.fft.ifftn(tf * np.fft.fftn(obj))), 0.0) + sky).astype(np.float64)
    return gn, psf, np.float64(sky), np.float64((gn - sky).sum())


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_emulated_wrapped_solver_matches_oracle(seed):
    """beta-SGP with the stamp application's keyword set on a 31 x 31 cut-out: same iteration count, trial and
    projection-evaluation counts, discr <= 1e-10, image <= 1e-8 against the oracle (numpy closure of any size)."""
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _stamp31(seed)
    kw = dict(gamma=1e-4, beta=0.4, alpha_min=1e-5, alpha_max=1e5, alpha=1e1, M_alpha=3, tau=0.5, M=1, proj_type=1, max_projs=1000,
              init_recon=2, stop_criterion=3, verbose=True, ccd_sat_level=65000, scale_data=True, lr=1e-3, lr_exp_param=0.1,
              schedule_lr=True, adapt_beta=True, MAXIT=500)
    b0 = [1.0882026172983832, 1.0248357076505616, 0.9789][seed % 3]
    o = orc.solve(gn, psf, bkg, divergence="beta", flux=flux, betaParam=b0, **kw)
    r = eh.solve(gn, psf, bkg, divergence="beta", flux=flux, betaParam=b0, wrapped=True, **kw)
    assert r["status"] == 0 and r["iters"] == o.iters
    assert list(r["trials"]) == list(o.trace.trials) and list(r["evals"]) == list(o.trace.proj_evals)
    assert np.abs(r["discr"] - o.discr).max() <= 1e-10 * np.abs(o.discr).max()
    assert np.abs(r["x"] - o.x).max() <= 1e-8 * np.abs(o.x).max()


@pytest.mark.parametrize("mp,bi,si", [(1000, 0, 0), (4, 0, 0), (4, 2, 0), (6, 0, 3), (5, 1, 2), (3, 3, 0)])
def test_emulated_projection_counter_arguments(golden, mp, bi, si):
    """projectDF's biter / siter / max_projs keywords (flux_conserve_proj.py:7): the secant budget is max_projs - biter
    with biter still growing during the bracketing (:39,:64,:103), the loop runs while siter < budget (:106)."""
    from oracle import sgp_oracle as orc
    for k in ("proj02", "proj06", "proj10"):              # the cases with the longest secant phases (8-12 evaluations)
        b, c, dia = np.float64(golden[k + "/b"]), golden[k + "/c"], golden[k + "/dia"]
        cnt = []
        xo = orc.flux_projection(b, c.copy(), dia.copy(), 1.0, max_projs=mp, biter=bi, siter=si, counter=cnt)
        xe, ev, st = eh.project(c, dia, float(b), max_projs=mp, biter=bi, siter=si)
        assert st == 0 and ev == cnt[-1]
        np.testing.assert_allclose(xe, xo, rtol=1e-12, atol=1e-15)


# ------------------------------------------------------------------------------------------------
# the launch-shape planner (csrc/bsgp_plan.h, plan_launch) with a B200's properties: 148 SMs, 227 KB of opt-in shared
# memory per block, 228 KB per SM (cudaDevAttrMaxSharedMemoryPerMultiprocessor, read on a B200)
# ------------------------------------------------------------------------------------------------
B200 = dict(num_sms=148, max_smem=232448, smem_per_sm=233472)
BSGP_E_SHAPE = 2                                          # include/bsgp.h


def _planned_cell(v):
    """The cell a row of tests/test_gpu_variants.py lands on by the planner alone.  Padded rows run on the front end's
    P x P grid (engine.PaddedGeometry); the CTAs per SM of a cluster plan are the ones its kernel variant is compiled for."""
    if v.kernel:
        P = int(2 ** np.ceil(np.log2(max(v.shape[0] + v.kernel, v.shape[1] + v.kernel))))
        assert P in (512, 1024)
        rc, s = eh.plan_launch((P, P), v.dtype, **B200)
    else:
        rc, s = eh.plan_launch(v.shape, v.dtype, v.cfg.get("cluster_size", 0), v.cfg.get("threads", 0), **B200)
    assert rc == 0, (v.label, rc)
    mk = bool(v.kernel) or (s["grid_ny"], s["grid_nx"]) != v.shape
    return (v.dtype, mk, "frame" if s["frame"] else (s["threads"], s["minb"]))


def test_planner_lands_every_variant_on_its_cell():
    """Every row of the variant table (padded rows included) lands on its (threads, CTAs per SM) or frame cell."""
    from test_gpu_variants import VARIANTS
    for v in VARIANTS:
        assert _planned_cell(v) == v.cell, v.label


def test_planner_keeps_clusters_off_one_cta_shapes():
    """128 x 3 and 256 x 2 run DeviceCtxSmall, whose all-reduce sums over one CTA: no cluster of 2..16 CTAs gets them, on
    any supported image shape and thread request."""
    sides = [16, 31, 32, 33, 64, 75, 100, 128, 256, 450, 512, 1024, 2048, 4096, 8192]
    checked = 0
    for dtype in ("float64", "float32"):
        for ny in sides:
            for nx in sides:
                for G in (2, 4, 8, 16):
                    for threads in (0, 128, 256, 512):
                        rc, s = eh.plan_launch((ny, nx), dtype, G, threads, **B200)
                        if rc:
                            continue
                        checked += 1
                        assert s["cluster_size"] == G and not s["frame"]
                        assert (s["threads"], s["minb"]) not in ((128, 3), (256, 2)), (dtype, ny, nx, G, threads, s)
    assert checked > 1000


def test_planner_refuses_dense_axes_in_frame_mode():
    """Sides of at most 32 that are not a power of two use a dense DFT of their own length, which needs one CTA per image.
    Forced into frame mode (G = 16 on a 32 x 32 grid) such a plan used to fall back to the radix FFT and fold a 61-long
    linear convolution on a 32-point circle; it is refused.  A wrapped axis in frame mode keeps its fold width."""
    for dtype in ("float64", "float32"):
        assert eh.plan_launch((31, 31), dtype, -1, **B200)[0] == BSGP_E_SHAPE
        assert eh.plan_launch((15, 13), dtype, -1, **B200)[0] == BSGP_E_SHAPE
        rc, s = eh.plan_launch((100, 75), dtype, -1, **B200)
        assert rc == 0 and s["frame"] and (s["grid_ny"], s["grid_nx"], s["wrap_ny"], s["wrap_nx"]) == (256, 256, 100, 75)
        rc, s = eh.plan_launch((31, 31), dtype, **B200)
        assert rc == 0 and not s["frame"] and s["cluster_size"] == 1 and (s["wrap_ny"], s["wrap_nx"]) == (0, 0)


import test_gpu_options as tgo  # noqa: E402  (the option runs of the GPU suite; importing it needs no device)


@pytest.mark.parametrize("run", list(tgo.OPTION_RUNS))
@pytest.mark.parametrize("shape,kernel", tgo._option_cells(), ids=lambda a: "x".join(map(str, a)) if isinstance(a, tuple) else f"k{a}")
def test_option_run_premises(shape, kernel, run):
    """The option runs of tests/test_gpu_options.py, on the oracle alone: every run ends by its own stop rule before
    MAXIT (rules 2 and 3 inside TOL_WINDOW, tol at least TOL_MARGIN apart from the stop values on both sides of the
    firing iteration), and the saturation cap of stop3-cap holds pixels at the cap.  Without this a scene change could
    turn the GPU runs into MAXIT runs unnoticed."""
    info = tgo.option_premises(shape, kernel, run)
    print(f"\n{shape} kernel {kernel} {run}: {info}")
