"""Shared observations on the GPU (run with -m gpu on a B200): solve_batch(source=...) / bsgp_inputs.source, where solve i
reads observation source[i] and the observations exist once.  Every output except the wall-clock `times` must be
bit-identical to the same launch with the observations replicated (gn[source], bkg[source], psf[source], ...), on every
compiled solve-kernel cell, through the numpy, device-tensor and page-locked routes; the beta sweep must equal its
replicated formulation; a malformed map is refused before anything is launched."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_variants import F64, VARIANTS, _plan_cell, _scene

pytestmark = pytest.mark.gpu

SRC = np.array([2, 0, 0, 1, 2, 2, 0], dtype=np.int32)
FIELDS = ("x", "iters", "status", "discr", "stop_value", "err", "beta_final", "proj_evals", "ls_trials", "scalars")
TRACE = ("alpha", "lam", "beta", "trials", "evals")


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    return b


def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def _same(a, b, what):
    """every output but `times`, bit for bit"""
    for k in FIELDS:
        va, vb = getattr(a, k), getattr(b, k)
        assert (va is None) == (vb is None), (what, k)
        if va is not None:
            assert np.array_equal(_np(va), _np(vb)), (what, k)
    if a.trace is not None or b.trace is not None:
        for k in TRACE:
            assert np.array_equal(_np(a.trace[k]), _np(b.trace[k])), (what, "trace", k)


def _observations(bs, shape, kernel, dtype, n=3, scalar_bkg=False):
    """n observations of one shape, each with its own PSF (different widths), background, truth and start image; all values
    exact in fp32."""
    gns, psfs, bkgs, flux, truth = [], [], [], [], []
    for k in range(n):
        gn, psf, bkg, fl, tr = _scene(bs, shape, kernel, seed=shape[0] * 11 + shape[1] + 5 * k, fwhm=2.5 + 0.5 * k, with_truth=True)
        gns.append(gn); psfs.append(psf); bkgs.append(bkg); flux.append(fl); truth.append(tr.astype(np.float32).astype(np.float64))
    npdt = np.float64 if dtype == F64 else np.float32
    gn = np.stack(gns)
    obs = dict(gn=gn, psf=np.stack(psfs), bkg=np.array([300.0, 301.0, 302.0][:n]) if scalar_bkg else np.stack(bkgs),
               x0=np.round(0.5 * gn) + 1.0, obj=np.stack(truth))
    return {k: v.astype(npdt) for k, v in obs.items()}, np.array(flux)


def _rows(source, flux_obs):
    """KL rows with errflag (obj) on every third solve; beta-SGP rows with their own beta and flux, one from x0."""
    rows = []
    for i, s in enumerate(source):
        if i % 3 == 0:
            rows.append(dict(divergence="kl", errflag=True, flux=None))
        else:
            rows.append(dict(divergence="beta", betaParam=0.95 + 0.02 * i, flux=float(flux_obs[s]) * (1.0 + 0.01 * i), proj_type=1,
                             init_recon=1 if i == 4 else 2))
    return rows


def _replicated(obs, source):
    """the observations copied once per solve: image stacks, and a background of one value per observation"""
    return {k: (v[source] if v.ndim == 3 or (k == "bkg" and v.ndim == 1) else v) for k, v in obs.items()}


def _solve(bs, obs, rows, source=None, route="numpy", **where):
    import torch
    a = dict(obs)
    if route == "device":
        a = {k: torch.as_tensor(v, device="cuda:0") for k, v in a.items()}
    elif route == "pinned":
        a = {k: (torch.from_numpy(np.ascontiguousarray(v)).pin_memory() if v.ndim == 3 and k != "psf" else v) for k, v in a.items()}
    r = bs.solve_batch(a["gn"], a["psf"], a["bkg"], x0=a["x0"], obj=a["obj"], per_image=rows, source=source, trace=True, MAXIT=8,
                       **where)
    if route != "numpy":
        torch.cuda.synchronize()
    return r


# ------------------------------------------------------------------------------------------------
# every solve-kernel cell: 7 solves of 3 observations, per-observation PSFs
# ------------------------------------------------------------------------------------------------
CELLS = list({v.cell: v for v in reversed(VARIANTS)}.values())[::-1]          # the first row of each cell


def test_cells_cover_every_kernel():
    assert len({v.cell for v in CELLS}) == 24 == len(CELLS)


@pytest.mark.parametrize("v", CELLS, ids=lambda v: v.label)
def test_every_cell_shared_equals_replicated(bs, v):
    """source = [2, 0, 0, 1, 2, 2, 0] with one PSF per observation (n_psf = 3) against the replicated launch (n_psf = 7):
    KL and beta-SGP rows with different flux and beta, errflag, a start image; a 2-D or a scalar background per
    observation.  The padded rows build both kernels per observation (bsgp_set_psf_adjoint with 3 kernels)."""
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    obs, flux = _observations(bs, v.shape, v.kernel, v.dtype, scalar_bkg=CELLS.index(v) % 2 == 1)
    rows = _rows(SRC, flux)
    where = dict(padded=True, dtype=v.dtype) if padded else dict(plan=plan, dtype=v.dtype)
    s = _solve(bs, obs, rows, SRC, **where)
    r = _solve(bs, _replicated(obs, SRC), rows, **where)
    assert list(s.status) == [0] * 7 and s.x.shape == (7,) + v.shape
    # errflag on the KL row 0 only: err[0] is the start image's error, err[iter] the error after iteration iter - 1
    # (the reference's counter starts at 1 and is raised before the store, so entry 1 is never written)
    assert s.err[0, 0] > 0 and s.err[0, 2] > 0 and not s.err[1].any()
    _same(s, r, v.label)
    print(f"\n{v.label}: iters {list(s.iters)}")
    if not padded:
        plan.close()


def test_shared_psf_and_unused_observation(bs):
    """One PSF for all solves, and an observation no solve reads (n_sources = 4, index 3 unused)."""
    obs, flux = _observations(bs, (32, 32), 0, F64, n=3)
    obs["gn"] = np.concatenate([obs["gn"], obs["gn"][:1] + 1.0])
    for k in ("bkg", "x0", "obj"):
        obs[k] = np.concatenate([obs[k], obs[k][:1]])
    obs["psf"] = obs["psf"][0]
    rows = _rows(SRC, flux)
    s = _solve(bs, obs, rows, SRC)
    r = _solve(bs, _replicated(obs, SRC), rows)
    _same(s, r, "shared psf")


# ------------------------------------------------------------------------------------------------
# the three routes and the upload paths of the page-locked entry point
# ------------------------------------------------------------------------------------------------
ROUTE_CASES = {
    # 128 KB images: per-observation uploads in the order of first use, flags by observation, permuted queue
    "per-item-128": ((128, 128), {}, SRC),
    # 8 KB images with a permuted queue: whole arrays, one flag write
    "whole-array-32": ((32, 32), {}, SRC),
    # 8 KB images whose first uses come in order (shared keywords, expanded into equal rows; natural queue): per-observation
    # uploads
    "in-order-32": ((32, 32), {}, np.array([0, 0, 1, 1, 2, 2], np.int32)),
    "wrapped-31": ((31, 31), {}, SRC),
    "wrapped-100x75": ((100, 75), {}, SRC),
    "frame-256": ((256, 256), dict(cluster_size=-1), SRC),
}


@pytest.mark.parametrize("name", list(ROUTE_CASES))
def test_routes_agree(bs, name):
    shape, cfg, source = ROUTE_CASES[name]
    plan = bs.Plan(shape[0], shape[1], F64, **cfg)
    obs, flux = _observations(bs, shape, 0, F64)
    rows = _rows(source, flux)
    if name == "in-order-32":
        rows = None
    ref = _solve(bs, _replicated(obs, source), rows, plan=plan)
    for route in ("numpy", "device", "pinned"):
        s = _solve(bs, obs, rows, source, route, plan=plan)
        _same(s, ref, (name, route))
    plan.close()


def test_pinned_output_buffer_is_per_solve(bs):
    import torch
    obs, flux = _observations(bs, (32, 32), 0, F64)
    rows = _rows(SRC, flux)
    pin = {k: (torch.from_numpy(v).pin_memory() if k != "psf" else v) for k, v in obs.items()}
    x = torch.empty((7, 32, 32), dtype=torch.float64, pin_memory=True)
    r = bs.solve_batch(pin["gn"], pin["psf"], pin["bkg"], x0=pin["x0"], obj=pin["obj"], per_image=rows, source=SRC, MAXIT=8, x_out=x)
    assert r.x is x
    ref = _solve(bs, _replicated(obs, SRC), rows)
    assert np.array_equal(x.numpy(), ref.x)
    with pytest.raises(ValueError, match="one image per solve"):
        bs.solve_batch(pin["gn"], pin["psf"], pin["bkg"], x0=pin["x0"], obj=pin["obj"], per_image=rows, source=SRC, MAXIT=8,
                       x_out=torch.empty((3, 32, 32), dtype=torch.float64, pin_memory=True))


# ------------------------------------------------------------------------------------------------
# the beta sweep
# ------------------------------------------------------------------------------------------------
def test_beta_sweep_equals_the_replicated_formulation(bs):
    """sgp_betaDiv_sweep restores every stamp five times from one copy of it; the solves equal the replicated batch of the
    previous formulation (repeat_interleave of gn, psf, bkg) bit for bit, and so does the selection."""
    import torch
    st = bs.synth.star_stamps(6, 32, seed=21)
    kw = dict(bs.synth.STAMP_KWARGS)
    best, best_beta, best_idx, metric, sweep = bs.sgp_betaDiv_sweep(st["gn"], st["psf"], st["bkg"], flux=st["flux"], **kw)
    dev = torch.device("cuda", 0)
    betas = np.array(bs.synth.beta_inits())
    rep = lambda a: torch.as_tensor(np.repeat(a, 5, axis=0), device=dev)    # noqa: E731
    gb, bb = rep(st["gn"]), rep(st["bkg"])
    r = bs.solve_batch(gb, rep(st["psf"]), bb, divergence="beta", flux=rep(st["flux"]), betaParam=torch.as_tensor(np.tile(betas, 6), device=dev),
                       **kw)
    for k in ("x", "iters", "status", "discr", "stop_value", "beta_final", "proj_evals", "ls_trials", "scalars"):
        assert torch.equal(getattr(sweep, k), getattr(r, k)), k
    m = (1.0 - bs.sweep.aperture_flux(r.x, bb) / bs.sweep.aperture_flux(gb, bb)).reshape(6, 5).cpu().numpy()
    # the original flux is now measured once per stamp: the same sums, possibly reduced in another order by torch
    assert np.allclose(metric, m, rtol=1e-12, atol=1e-13)
    assert np.array_equal(best_idx, bs.sweep.select_best(m)) and np.array_equal(best_beta, betas[best_idx])
    assert torch.equal(best.x, r.x[torch.as_tensor(np.arange(6) * 5 + best_idx, device=dev)])


# ------------------------------------------------------------------------------------------------
# refusals: before any launch
# ------------------------------------------------------------------------------------------------
def test_bad_maps_are_refused_before_launch(bs):
    import torch
    capi, L = bs._capi, bs._capi.lib()
    plan = bs.Plan(32, 32)
    rng = np.random.default_rng(3)
    gn = rng.poisson(100.0, (3, 32, 32)).astype(np.float64)
    psf = np.zeros((32, 32)); psf[16, 16] = 1.0
    bkg, flux, b0 = np.full(3, 10.0), np.full(4, 1e5), np.full(4, 1.005)
    x = np.zeros((4, 32, 32))
    i32, f64 = (lambda *s: np.zeros(s, np.int32)), (lambda *s: np.zeros(s))
    outs = [x, i32(4), i32(4), f64(4, 11), f64(4, 11)]
    kl = capi.make_params(capi.DIV_KL, MAXIT=10)
    rows = (capi.Params * 4)(*([kl] * 4))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(entry, source, n_sources):
        m = np.ascontiguousarray(source, dtype=np.int32)
        ci = capi.Inputs(gn.ctypes.data, bkg.ctypes.data, 0, flux.ctypes.data, b0.ctypes.data, None, None, None, m.ctypes.data, n_sources)
        co = capi.Outputs(*(a.ctypes.data for a in outs))
        before = L.bsgp_launch_count()
        args = {"host": (L.bsgp_solve_batch_host, C.byref(kl)), "pinned": (L.bsgp_solve_batch_pinned, C.byref(kl)),
                "device": (L.bsgp_solve_batch, C.byref(kl)), "rows_host": (L.bsgp_solve_batch_rows_host, rows)}[entry]
        extra = () if entry.endswith("host") else (stream,)
        rc = args[0](plan.handle, args[1], 4, C.byref(ci), C.byref(co), *extra)
        return rc, L.bsgp_last_error_string().decode(), L.bsgp_launch_count() - before

    plan.set_psf(np.stack([psf] * 4))                      # 4 PSFs: neither 1 nor n_sources = 3
    for entry in ("host", "pinned", "device", "rows_host"):
        rc, msg, launched = call(entry, [0, 1, 5, 2], 3)
        assert (rc, launched) == (1, 0) and msg == "solve 2: source 5 is outside 0..2", (entry, msg)
        rc, msg, launched = call(entry, [0, 1, -1, 2], 3)
        assert (rc, launched) == (1, 0) and msg.startswith("solve 2: source -1"), (entry, msg)
        rc, msg, launched = call(entry, [0, 0, 0, 0], 0)
        assert (rc, launched) == (1, 0) and "n_sources must be >= 1" in msg, (entry, msg)
        rc, msg, launched = call(entry, [0, 1, 1, 2], 3)
        assert (rc, launched) == (5, 0) and "need 1 or n_sources (3)" in msg, (entry, msg)          # BSGP_E_STATE
    plan.set_psf(np.stack([psf] * 3))
    rc, msg, launched = call("host", [0, 1, 1, 2], 3)
    assert rc == 0 and launched >= 1, msg
    assert np.array_equal(x[1], x[2]) and not np.array_equal(x[0], x[1])
    plan.close()
