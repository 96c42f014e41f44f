"""The solver's options on every compiled solve-kernel variant against the oracle (run with -m gpu on a B200).

test_gpu_variants runs every row of its VARIANTS table (24 kernels: T x MK x launch shape) with stop rule 1 only.  The
options below have code of their own inside the kernels, and each run here takes every row through a set of them:

- stop2-err: KL, x0 = gn with the flux projection, stop rule 2 with verbose (tol squared), errflag with the true image
  as obj, M = M_alpha = 16 (the full histories of the per-warp controller state);
- stop3-cap: beta-SGP with the adaptive beta and the lr schedule, the constant start image (x_const = flux / the window's
  pixel count), the flux projection, stop rule 3, a 2-D background, and a saturation cap of max(gn) / 2 that binds;
- stop4-x0: KL from x0 = randn (seed 42, as the reference draws it), no projection, stop rule 4 (tol = 1 + 1 / mean(gn)),
  scale_data=False (scaling = 1), M = 4, a scalar background of 300.

Every run ends by its own rule before MAXIT, so each row takes the exit on which the accepted step is not swapped in,
at an iteration the data chooses.  The tol of rules 2 and 3 is set from one oracle run to MAXIT: the first iteration k
of TOL_WINDOW whose stop value is TOL_MARGIN below the smallest earlier one, tol the geometric mean of the two (11 % on
either side, more than any rounding of either dtype).  Rule 4's tol is fixed by the data; the margin of the scene is
reported, and fp32 must stop with the oracle where it is at least RULE4_F32_MARGIN.  option_premises() checks all of
this on the oracle alone and runs without a GPU (tests/test_host_logic.py), so a scene change that stops a rule from
firing fails there instead of turning these runs into MAXIT runs.

fp64 is held to the suite's strict bar; fp32 is compared with the fp64 oracle on the same inputs, to the FP32_* bars of
test_gpu_variants.  The inputs are exact in fp32 except x0 of stop4-x0 (randn, rounded to fp32 for the fp32 rows) and
obj (rounded to fp32 for both).  The worst values measured on a B200 (1000 W) over all 36 rows stand beside each bar
below, and the module prints its own worst values and slowest row at the end (pytest -s).
"""
import time
from dataclasses import dataclass
from functools import lru_cache

import numpy as np
import pytest

from test_gpu_variants import BETA0, F32, F64, FP32_DISCR, FP32_FLUX, FP32_IMAGE, VARIANTS, _plan_cell, _scene

pytestmark = pytest.mark.gpu

_KL = dict(divergence="kl", betaParam=1.005)
_BETA = dict(divergence="beta", betaParam=BETA0, gamma=1e-4, beta=0.4, alpha=10.0, M_alpha=3, tau=0.5, M=1, lr=1e-3,
             lr_exp_param=0.1, schedule_lr=True, adapt_beta=True)
OPTION_RUNS = {
    "stop2-err": dict(_KL, init_recon=2, proj_type=1, stop_criterion=2, verbose=True, errflag=True, M=16, M_alpha=16, MAXIT=24),
    "stop3-cap": dict(_BETA, init_recon=3, proj_type=1, stop_criterion=3, MAXIT=24),
    "stop4-x0": dict(_KL, init_recon=1, proj_type=0, stop_criterion=4, scale_data=False, M=4, MAXIT=45),
}
TOL_WINDOW = (4, 20)           # iterations in which rules 2 and 3 are set to fire
TOL_MARGIN = 1.25              # stop value at the firing iteration <= smallest earlier one / TOL_MARGIN
SAT_FRACTION = 0.5             # stop3-cap: ccd_sat_level = SAT_FRACTION * max(gn)
# run-specific scenes: on the variant scene of pad375, rule 4's value is still 1e-2 above tol after 60 iterations
SCENE_SEEDS = {((375, 375), 31, "stop4-x0"): 1}
# fp32 image and flux of stop4-x0, relative to the oracle's largest value.  KL without the flux projection runs 15-28
# iterations from a random start; near convergence its gradient 1 - A^T(gn / den) cancels to ~1e-3 of its terms and fp32
# keeps three digits of it (DESIGN.md section 2, fp32 mode: 9e-4 on the 27-iteration reference simulations).  The error is
# the same on every launch shape of one input, so it is the arithmetic's, not a kernel's.  Measured on a B200 (1000 W):
# image 4.6e-3 (33 x 20, 26 iterations), flux 1.7e-3.  discr stays within FP32_DISCR.
FP32_LONG_IMAGE, FP32_LONG_FLUX = 1e-2, 5e-3
RULE4_F32_MARGIN = 1e-3        # rule 4: fp32 stops with the oracle when tol is this far (relative) from both sides

# fp64 bars beyond the strict ones of test_gpu_variants (discr 1e-10, image 1e-8 of the largest value), each relative to
# the largest value of the run.  Measured worst on a B200 (1000 W) beside each.
STOP_VALUE_BAR = 1e-8          # rules 2 and 3 cancel (sk = lam * d, f_prev - f); rule 4 is discr.  Measured 3.0e-12
SCALAR_BAR = 1e-12             # flux, x_low, x_upp, tol (scaling exactly).  Measured 1.9e-15
# alpha, lambda, beta per iteration and beta_final.  alpha is a ratio of Barzilai-Borwein sums over y_k = g_new - g, which
# cancels near convergence like the stop values: measured 3.3e-10 on stop4-x0 (24 iterations; pad375), 1e-14 on the short
# beta-SGP runs, while the image agrees to 3e-11
TRACE_BAR = 1e-8


@dataclass
class Case:
    gn: np.ndarray
    psf: np.ndarray
    bkg: object                # 2-D image or a float
    flux: object               # None: the solver takes sum(gn - bkg)
    x0: object
    obj: object
    kw: dict                   # solver keywords (divergence and betaParam included)
    o: object                  # the oracle's OracleResult
    tol: float                 # the tol the solver compares with
    fire: int                  # iteration at which the rule fires
    margin: float              # relative distance of tol from the stop values on either side of the firing iteration
    sat: float = None


def _oracle(c, kw, kernel, **over):
    from oracle import sgp_oracle as orc
    kw = dict(kw, **over)
    obj = kw.pop("obj", None)
    return orc.solve(c["gn"], c["psf"], c["bkg"], flux=None if c["flux"] is None else np.float64(c["flux"]), obj=obj,
                     use_original_SGP_Afunction=not kernel, **kw)


def _pick_tol(values):
    """(k, tol): the first iteration k of TOL_WINDOW whose stop value is TOL_MARGIN below every earlier one, tol their
    geometric mean; None if there is none."""
    for k in range(TOL_WINDOW[0], min(TOL_WINDOW[1], len(values)) + 1):
        v, prev = values[k - 1], min(values[:k - 1])
        if v > 0 and prev >= TOL_MARGIN * v:
            return k, float(np.sqrt(v * prev))
    return None


def _margin(values, k, tol):
    """Relative distance of tol from the stop value of iteration k and from the smallest of the earlier ones."""
    return float(min(min(values[:k - 1]) / tol - 1.0, 1.0 - values[k - 1] / tol)) if k > 1 else 0.0


@lru_cache(maxsize=None)
def option_case(shape, kernel, run):
    """Inputs, solver keywords and oracle result of one (image shape, operator, run); shared by the fp64 and fp32 rows.
    Raises AssertionError if the run's rule cannot be set to fire (see option_premises)."""
    import beta_sgp_b200 as bs
    seed = SCENE_SEEDS.get((shape, kernel, run), shape[0] * 7 + shape[1] + kernel)
    gn, psf, bkg, flux, truth = _scene(bs, shape, kernel, seed=seed, with_truth=True)
    kw = dict(OPTION_RUNS[run])
    c = dict(gn=gn, psf=psf, bkg=bkg, flux=None, x0=None, obj=None)
    sat = None
    if run == "stop2-err":
        c["obj"] = truth.astype(np.float32).astype(np.float64)
    elif run == "stop3-cap":
        c["flux"] = flux
        sat = SAT_FRACTION * float(gn.max())
        kw["ccd_sat_level"] = sat
    else:
        c["bkg"] = np.float64(300.0)
        np.random.seed(42)
        c["x0"] = np.random.randn(*shape)                        # the oracle draws the same (sgp.py:168-170)
    rule = kw["stop_criterion"]
    if rule in (2, 3):
        probe = _oracle(c, dict(kw, errflag=False), kernel, tol_convergence=0.0)
        pick = _pick_tol(probe.trace.stop_value)
        assert pick is not None, (shape, kernel, run, probe.trace.stop_value)
        tol = pick[1]
        kw["tol_convergence"] = float(np.sqrt(tol)) if (rule == 2 and kw.get("verbose")) else tol
    if c["obj"] is not None:
        kw["obj"] = c["obj"]
    o = _oracle(c, kw, kernel)
    kw.pop("obj", None)
    if rule == 4:
        tol = 1.0 + 1.0 / np.mean(gn)
    elif rule == 2:
        tol = kw["tol_convergence"] ** 2
    else:
        tol = kw["tol_convergence"]
    fire = o.iters if rule == 4 else pick[0]
    return Case(gn, psf, c["bkg"], c["flux"], c["x0"], c["obj"], kw, o, float(tol), fire,
                _margin(o.trace.stop_value, fire, tol), sat)


def _option_cells():
    """(shape, kernel) of every row of VARIANTS, once each."""
    return sorted({(v.shape, v.kernel) for v in VARIANTS})


def option_premises(shape, kernel, run):
    """The oracle-only premises of one (shape, operator, run), as a dict; asserts them."""
    c = option_case(shape, kernel, run)
    o, maxit = c.o, c.kw["MAXIT"]
    info = dict(fire=c.fire, iters=o.iters, margin=c.margin, tol=c.tol)
    assert o.iters == c.fire < maxit, info                                   # the rule ends the run, not MAXIT
    if c.kw["stop_criterion"] in (2, 3):
        assert TOL_WINDOW[0] <= c.fire <= TOL_WINDOW[1], info
        assert c.margin >= 1.0 - 1.0 / np.sqrt(TOL_MARGIN) - 1e-9, info
    sv = np.asarray(o.trace.stop_value)
    assert np.all(sv[:c.fire - 1] > c.tol) and sv[c.fire - 1] <= c.tol, info
    if c.sat is not None:
        at_cap = int(np.count_nonzero(o.x >= c.sat * (1 - 1e-9)))
        info["at_cap"] = at_cap
        assert at_cap >= 1 and o.x.max() <= c.sat * (1 + 1e-12), info
    return info


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    return b


@pytest.fixture(scope="module")
def worst():
    """Worst measured value per (dtype, bar) and the slowest row, printed at the end of the module."""
    w = {}
    yield w
    print("\n\noption runs, worst measured:")
    for k in sorted(k for k in w if k != "slowest"):
        print(f"  {k[0]} {k[1]}: {w[k][0]:.3e} ({w[k][1]})")
    if "slowest" in w:
        print(f"  slowest row: {w['slowest'][1]} {w['slowest'][0]:.1f} s (oracle included)")


def _note(worst, dtype, bar, value, where):
    if value > worst.get((dtype, bar), (-1.0, ""))[0]:
        worst[(dtype, bar)] = (float(value), where)


def _solve(bs, v, c, plan, padded, route="numpy"):
    """The row's solve of case c; route 'pinned' hands page-locked tensors to bsgp_solve_batch_pinned."""
    npdt = np.float64 if v.dtype == F64 else np.float32
    kw = dict(c.kw)
    div, b0 = kw.pop("divergence"), kw.pop("betaParam")
    gn = c.gn[None].astype(npdt)
    bkg = c.bkg[None].astype(npdt) if np.ndim(c.bkg) == 2 else np.array([float(c.bkg)])
    x0 = None if c.x0 is None else c.x0[None].astype(npdt)
    obj = None if c.obj is None else c.obj[None].astype(npdt)
    psf = c.psf.astype(npdt)
    flux = None if c.flux is None else [c.flux]
    where = dict(plan=plan)
    if padded:
        geo = bs.engine.PaddedGeometry(v.shape[0], v.shape[1], v.kernel, v.kernel)
        if route == "numpy":
            where = dict(padded=True)
        else:                      # the padded operator's own route takes numpy; its grid-sized arrays go pinned here
            big, div_a = geo.kernel(c.psf, npdt)
            bigt, div_at = geo.kernel(c.psf.conj().T, npdt)
            plan.set_psf(big)
            plan.set_psf_adjoint(bigt)
            where = dict(plan=plan, psf_is_set=True, region=geo.region, div_a=div_a, div_at=div_at, adjoint_second_psf=True)
            gn, x0, obj = (None if a is None else geo.embed(a, npdt) for a in (gn, x0, obj))
            if bkg.ndim == 3:
                bkg = geo.embed(bkg, npdt)
            psf = None
    if route == "pinned":
        import torch

        def pin(a):
            return None if a is None or np.ndim(a) < 3 else torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        gn, x0, obj = pin(gn), pin(x0), pin(obj)
        bkg = pin(bkg) if bkg.ndim == 3 else bkg
    r = bs.solve_batch(gn, psf, bkg, divergence=div, flux=flux, betaParam=b0, x0=x0, obj=obj, dtype=v.dtype, trace=True,
                       **where, **kw)
    if route == "pinned":
        r.x = r.x.numpy()
        if padded:
            r.x = r.x[:, geo.rows, geo.cols]
    return r


def _rel(a, b, scale=None):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() if scale is None else scale))


@pytest.mark.parametrize("run", list(OPTION_RUNS))
@pytest.mark.parametrize("v", VARIANTS, ids=lambda v: v.label)
def test_option_run_matches_oracle(bs, worst, v, run):
    """One option run on one kernel variant against the oracle: the rule ends the run before MAXIT, with status OK.
    fp64: identical iteration count, trials and projection evaluations; discr, image, err, stop values, the scalars,
    the alpha / lambda / beta trace and beta_final at the strict bars.  fp32: the oracle's iteration count (rule 4:
    where its margin is at least RULE4_F32_MARGIN, else within one, printed); discr, image, flux and err within the
    FP32_* bars; the cap bound."""
    t0 = time.perf_counter()
    c = option_case(v.shape, v.kernel, run)
    o = c.o
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    r = _solve(bs, v, c, plan, padded)
    if not padded:
        plan.close()
    it, maxit = int(r.iters[0]), c.kw["MAXIT"]
    assert int(r.status[0]) == 0 and it < maxit, (int(r.status[0]), it)
    n = min(it, o.iters)
    e_d = _rel(r.discr[0, :n + 1], o.discr[:n + 1])
    e_x = _rel(r.x[0], o.x)
    e_f = abs(float(r.x[0].sum(dtype=np.float64)) - o.x.sum()) / abs(o.x.sum())
    sv, osv = r.stop_value[0, 1:n + 1], np.asarray(o.trace.stop_value[:n])
    e_s = _rel(sv, osv)
    msg = f"{v.label} {run} fire {c.fire} (margin {c.margin:.2e}) iters {it} oracle {o.iters}"
    print(f"\n{msg} discr {e_d:.2e} image {e_x:.2e} flux {e_f:.2e} stop value {e_s:.2e}")
    where = f"{v.label} {run}"
    if v.dtype == F64 or run != "stop4-x0" or c.margin >= RULE4_F32_MARGIN:
        assert it == o.iters, msg
    else:
        assert abs(it - o.iters) <= 1, msg
    same = it == o.iters
    if c.obj is not None:
        assert r.err[0, 1] == 0.0                                        # the index quirk of sgp.py:394-396
        e_err = _rel(r.err[0, :n + 1], o.err[:n + 1])
    if c.sat is not None:
        at_cap = int(np.count_nonzero(r.x[0] >= c.sat * (1 - (1e-9 if v.dtype == F64 else 1e-6))))
        print(f"  cap {c.sat}: {at_cap} pixels at the cap, max {float(r.x[0].max())!r}")
    if v.dtype == F64:
        assert np.array_equal(r.trace["trials"][0, 1:it + 1], o.trace.trials)
        assert np.array_equal(r.trace["evals"][0, 1:it + 1], o.trace.proj_evals)
        assert int(r.proj_evals[0]) == sum(o.trace.proj_evals) + o.trace.init_proj_evals
        assert e_d <= 1e-10 and e_x <= 1e-8, (e_d, e_x)
        assert e_s <= STOP_VALUE_BAR, e_s
        if c.obj is not None:
            np.testing.assert_allclose(r.err[0, :it + 1], o.err, rtol=1e-9, atol=1e-14)
        sc = r.scalars[0]
        assert sc[0] == o.trace.scaling
        e_sc = max(_rel(sc[1], o.trace.flux), _rel(sc[2], o.trace.x_low), _rel(sc[3], o.trace.x_upp), _rel(sc[4], c.tol))
        assert e_sc <= SCALAR_BAR, (list(sc[:5]), o.trace.flux, o.trace.x_low, o.trace.x_upp, c.tol)
        e_tr = max(_rel(r.trace["alpha"][0, 1:it + 1], o.trace.alpha), _rel(r.trace["lam"][0, 1:it + 1], o.trace.lam))
        if c.kw["divergence"] == "beta":    # KL reports beta = 1, the divergence it minimises; the oracle keeps betaParam
            e_tr = max(e_tr, _rel(r.trace["beta"][0, 1:it + 1], o.trace.beta_param), _rel(r.beta_final[0], o.beta_param))
        else:
            assert np.all(r.trace["beta"][0, 1:it + 1] == 1.0) and r.beta_final[0] == 1.0
        assert e_tr <= TRACE_BAR, e_tr
        if c.sat is not None:
            assert float(r.x[0].max()) <= c.sat * (1 + 1e-12) and at_cap >= 1
        for bar, val in (("discr", e_d), ("image", e_x), ("stop value", e_s), ("scalars", e_sc), ("trace", e_tr)):
            _note(worst, F64, bar, val, where)
    else:
        assert e_d <= FP32_DISCR, e_d
        _note(worst, F32, "discr", e_d, where)
        if same:
            long_run = run == "stop4-x0"
            bar_x, bar_f = (FP32_LONG_IMAGE, FP32_LONG_FLUX) if long_run else (FP32_IMAGE, FP32_FLUX)
            assert e_x <= bar_x and e_f <= bar_f, (e_x, e_f)
            _note(worst, F32, "image" + (" (stop4-x0)" if long_run else ""), e_x, where)
            _note(worst, F32, "flux" + (" (stop4-x0)" if long_run else ""), e_f, where)
        if c.obj is not None:
            assert e_err <= FP32_IMAGE, e_err
            _note(worst, F32, "err", e_err, where)
        if c.sat is not None:
            assert float(r.x[0].max()) <= np.float32(c.sat) * (1 + 2.0 ** -22) and at_cap >= 1
    dt = time.perf_counter() - t0
    if dt > worst.get("slowest", (0.0, ""))[0]:
        worst["slowest"] = (dt, where)


PINNED_ROWS = [v for v in VARIANTS if v.label.rsplit("-", 1)[0] in ("33x20", "pad375", "100x75-frame")]


@pytest.mark.parametrize("run", ["stop2-err", "stop4-x0"])
@pytest.mark.parametrize("v", PINNED_ROWS, ids=lambda v: v.label)
def test_option_run_pinned_path(bs, v, run):
    """The page-locked path stages x0 and obj like gn: on the wrapped and frame rows it embeds them through its staging
    arena into the plan's larger grid (bsgp_solve_batch_pinned), on the padded row it takes the embedded grid arrays.
    Bit-identical to the plain host path."""
    c = option_case(v.shape, v.kernel, run)
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    a = _solve(bs, v, c, plan, padded)
    p = _solve(bs, v, c, plan, padded, route="pinned")
    if not padded:
        plan.close()
    assert int(a.status[0]) == 0 and int(a.iters[0]) < c.kw["MAXIT"]
    assert np.array_equal(p.iters, a.iters) and np.array_equal(p.status, a.status)
    for k in ("x", "discr", "stop_value") + (("err",) if c.obj is not None else ()):
        assert np.array_equal(np.asarray(getattr(p, k)), np.asarray(getattr(a, k))), k
