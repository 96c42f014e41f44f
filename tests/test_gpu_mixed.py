"""Mixed batches on the GPU (run with -m gpu on a B200): one launch for images that each carry their own keywords
(solve_batch(per_image=...), bsgp_solve_batch_rows*).  Every image of a mixed launch must be bit-identical to the same
image solved alone with its own keywords through the shared-keyword entry points, on every compiled kernel variant and
on all three residencies; rows that are all equal give what the shared keywords give; the queue order does not matter;
malformed rows are refused before anything is launched."""
import ctypes as C

import numpy as np
import pytest

from cases import CASES, CUTOUT_CASES, SENSITIVE, STRICT
from test_gpu_options import OPTION_RUNS
from test_gpu_variants import F64, VARIANTS, _plan_cell, _scene

pytestmark = pytest.mark.gpu

# outputs compared bit for bit: whole arrays, or per image up to its own iteration count
WHOLE = ("x", "iters", "status", "proj_evals", "ls_trials", "scalars", "beta_final")
TRACED = ("discr", "stop_value")
TRACE = ("alpha", "lam", "beta", "trials", "evals")


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    return b


def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def _same_image(m, i, s, what="", j=0):
    """Image i of mixed result m against image j of result s: bit-identical outputs and traces up to its own iteration
    count; the mixed traces are untouched (zero) beyond it."""
    it = int(_np(m.iters)[i])
    assert it == int(_np(s.iters)[j]), (what, "iters")
    for k in WHOLE:
        assert np.array_equal(_np(getattr(m, k))[i], _np(getattr(s, k))[j]), (what, k)
    for k in TRACED + (("err",) if m.err is not None and s.err is not None else ()):
        a, b = _np(getattr(m, k))[i], _np(getattr(s, k))[j]
        assert np.array_equal(a[:it + 1], b[:it + 1]), (what, k)
        if k != "err":
            assert not a[it + 1:].any(), (what, k, "written past iters")
    if m.trace is not None and s.trace is not None:
        for k in TRACE:
            assert np.array_equal(_np(m.trace[k])[i, :it + 1], _np(s.trace[k])[j, :it + 1]), (what, "trace", k)


# ------------------------------------------------------------------------------------------------
# the golden cases in mixed launches
# ------------------------------------------------------------------------------------------------
def _golden_batch(names, get_case, bkg_image=False):
    """Stacked inputs and one keyword row per case (divergence, betaParam, flux and the case's own keywords)."""
    gns, psfs, bkgs, x0s, rows = [], [], [], [], []
    for n in names:
        gn, psf, bkg, div, kw = get_case(n)
        row = dict(kw, divergence=div)
        row.setdefault("betaParam", 1.005)
        row["flux"] = None if row.get("flux") is None else float(row["flux"])
        x0 = np.zeros_like(gn)
        if kw.get("init_recon", 0) == 1:
            np.random.seed(42)
            x0 = np.random.randn(*gn.shape)
        gns.append(gn); psfs.append(psf); x0s.append(x0); rows.append(row)
        bkgs.append(np.full(gn.shape, float(bkg)) if bkg_image and np.ndim(bkg) == 0 else bkg)
    bkg = np.stack(bkgs) if np.ndim(bkgs[0]) == 2 else np.array([float(b) for b in bkgs])
    return np.stack(gns), np.stack(psfs), bkg, np.stack(x0s), rows


def _alone(bs, gn, psf, bkg, x0, row, **where):
    kw = dict(row)
    div, b0, flux = kw.pop("divergence"), kw.pop("betaParam"), kw.pop("flux")
    return bs.solve_batch(gn[None], psf, bkg[None] if np.ndim(bkg) == 2 else np.array([float(bkg)]), divergence=div,
                          flux=None if flux is None else [flux], betaParam=b0, x0=x0[None] if kw.get("init_recon", 0) == 1 else None,
                          trace=True, **where, **kw)


def _oracle_bar(name, r, i, golden):
    """DESIGN section 2: the reference's iteration count everywhere; the strict bar (cases.SENSITIVE where the reference
    itself is not reproducible to it) on STRICT and the cut-outs; the stop-rule runs' head bar on the others."""
    it = int(golden[name + "/iters"])
    assert int(r.iters[i]) == it and int(r.status[i]) == 0, name
    ref = golden[name + "/discr"]
    xs = golden[name + "/x_sub"] if name + "/x_sub" in golden.files else None
    if name in STRICT or name in CUTOUT_CASES or name.startswith("stamp"):
        tol_d, tol_x = SENSITIVE.get(name, (1e-10, 1e-8))
        assert np.abs(r.discr[i, :it + 1] - ref).max() <= tol_d * np.abs(ref).max(), name
        if xs is not None:
            assert np.abs(r.x[i][::8, ::8] - xs).max() <= tol_x * np.abs(xs).max(), name
        if name + "/x" in golden.files:
            assert np.abs(r.x[i] - golden[name + "/x"]).max() <= tol_x * np.abs(golden[name + "/x"]).max(), name
        assert np.array_equal(r.trace["evals"][i, 1:it + 1], golden[name + "/proj_evals"]), name
    else:                                        # stop rule 3 after up to 74 iterations, or 332-iteration runs
        rel = np.abs(r.discr[i, :it + 1] - ref) / np.abs(ref)
        assert rel[:41].max() <= (2e-8 if "sat" in name else 1e-10), name


NGC_SAT = [n for n, (d, _, kw, _) in CASES.items() if d in ("ngc", "sat") and "flux" not in kw]
WITH_FLUX = [f"tile{i:02d}" for i in range(10)] + [n for n, (d, _, kw, _) in CASES.items() if d in ("ngc", "sat") and "flux" in kw]


@pytest.mark.parametrize("names,bkg_image", [(NGC_SAT, False), (WITH_FLUX, True), (CUTOUT_CASES, False)],
                         ids=["ngc-sat", "tiles-flux", "cutouts31"])
def test_golden_cases_in_one_launch(bs, get_case, golden, names, bkg_image):
    """The 256 x 256 golden cases (NGC and satellite, KL and beta, each with its own MAXIT, stop rule, projection, start
    image and flags; the tiles and the flux-given case with 2-D backgrounds), and the 31 x 31 cut-outs with their KL
    twins, each set in one launch: every image bit-identical to its own solve, and at the oracle bar."""
    gn, psf, bkg, x0, rows = _golden_batch(names, get_case, bkg_image)
    m = bs.solve_batch(gn, psf, bkg, x0=x0, trace=True, per_image=rows)
    assert m.discr.shape[1] == max(r.get("MAXIT", 500) for r in rows) + 1
    for i, n in enumerate(names):
        s = _alone(bs, gn[i], psf[i], bkg[i], x0[i], rows[i])
        _same_image(m, i, s, n)
        _oracle_bar(n, m, i, golden)


def test_uniform_rows_equal_the_shared_keywords(bs, get_case):
    """Rows that are all equal give what the shared-keyword entry point gives, bit for bit (cut-outs, whole batch)."""
    names = [f"cutout31_{i:02d}" for i in range(10)]
    gn, psf, bkg, x0, rows = _golden_batch(names, get_case)
    kw = dict(rows[0])
    kw.pop("divergence"); kw.pop("betaParam"); kw.pop("flux")
    flux = np.array([r["flux"] for r in rows]); b0 = np.array([r["betaParam"] for r in rows])
    a = bs.solve_batch(gn, psf[0], bkg, flux=flux, betaParam=b0, trace=True, **kw)
    m = bs.solve_batch(gn, psf[0], bkg, flux=flux, betaParam=b0, trace=True, per_image=[{}] * len(names), **kw)
    for i in range(len(names)):
        _same_image(m, i, a, i, j=i)
    assert np.array_equal(m.discr, a.discr)


def test_reversed_queue_order(bs, get_case, monkeypatch):
    """The work queue's order only decides which cluster solves which image when: a reversed order is bit-identical."""
    names = CUTOUT_CASES
    gn, psf, bkg, x0, rows = _golden_batch(names, get_case)
    a = bs.solve_batch(gn, psf, bkg, trace=True, per_image=rows)
    rev = np.ascontiguousarray(np.arange(len(names))[::-1].astype(np.int32))
    monkeypatch.setattr(bs.engine, "_queue_order", lambda *args: rev)
    b = bs.solve_batch(gn, psf, bkg, trace=True, per_image=rows)
    for k in WHOLE + TRACED:
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    for k in TRACE:
        assert np.array_equal(a.trace[k], b.trace[k]), k


# ------------------------------------------------------------------------------------------------
# every kernel variant and every residency: the stop2-err and stop3-cap option sets in one launch
# ------------------------------------------------------------------------------------------------
# tol of rules 2 and 3 fixed here (bit-identity needs no oracle): 24 iterations at most
_TOL = {"stop2-err": 3e-2, "stop3-cap": 1e-4}


def _option_rows(v):
    """(gn [2], psf, bkg [2] images, obj [2], rows): stop2-err (KL, x0 = gn, projection, rule 2, errflag with the truth,
    M = M_alpha = 16) and stop3-cap (beta-SGP, flux given, constant start, rule 3, a binding saturation cap)."""
    import beta_sgp_b200 as bs
    gn, psf, bkg, flux, truth = _scene(bs, v.shape, v.kernel, seed=v.shape[0] * 7 + v.shape[1] + v.kernel, with_truth=True)
    r2 = dict(OPTION_RUNS["stop2-err"], tol_convergence=_TOL["stop2-err"], flux=None)
    r3 = dict(OPTION_RUNS["stop3-cap"], tol_convergence=_TOL["stop3-cap"], flux=flux, ccd_sat_level=0.5 * float(gn.max()))
    obj = np.stack([truth.astype(np.float32).astype(np.float64), np.zeros_like(truth)])
    return np.stack([gn, gn]), psf, np.stack([bkg, bkg]), obj, [r2, r3]


def _run(bs, v, plan, padded, gn, psf, bkg, obj, rows, route="numpy"):
    """One solve of images gn with rows (a mixed batch if len(rows) > 1, else the shared keywords of rows[0]) on the row's
    plan, through the numpy, device-tensor or pinned-tensor route."""
    import torch
    npdt = np.float64 if v.dtype == F64 else np.float32
    gn, bkg, obj, psf = gn.astype(npdt), bkg.astype(npdt), obj.astype(npdt), psf.astype(npdt)
    if len(rows) > 1:
        call = dict(divergence="kl", per_image=rows)
    else:
        call = dict(rows[0])
        call["flux"] = None if call["flux"] is None else [call["flux"]]
    where = dict(plan=plan)
    if padded:
        geo = bs.engine.PaddedGeometry(v.shape[0], v.shape[1], v.kernel, v.kernel)
        if route == "pinned":            # the padded route takes host arrays as numpy: hand it the embedded grid instead
            big, div_a = geo.kernel(psf, npdt)
            bigt, div_at = geo.kernel(psf.conj().T, npdt)
            plan.set_psf(big)
            plan.set_psf_adjoint(bigt)
            where = dict(plan=plan, psf_is_set=True, region=geo.region, div_a=div_a, div_at=div_at, adjoint_second_psf=True)
            gn, bkg, obj = (geo.embed(a, npdt) for a in (gn, bkg, obj))
            psf = None
        else:
            where = dict(padded=True)
    if route == "device":
        dev = torch.device("cuda", 0)
        gn, bkg, obj = (torch.as_tensor(a, device=dev) for a in (gn, bkg, obj))
        psf = None if psf is None else torch.as_tensor(psf, device=dev)
    elif route == "pinned":
        gn, bkg, obj = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (gn, bkg, obj))
    r = bs.solve_batch(gn, psf, bkg, obj=obj, dtype=v.dtype, trace=True, **where, **call)
    if route != "numpy":
        for k in WHOLE + TRACED + ("err",):
            setattr(r, k, _np(getattr(r, k)))
        r.trace = {k: _np(t) for k, t in r.trace.items()}
        if padded and route == "pinned":
            r.x = r.x[:, geo.rows, geo.cols]
    return r


@pytest.mark.parametrize("v", VARIANTS, ids=lambda v: v.label)
def test_every_variant_two_option_sets_in_one_launch(bs, v):
    """stop2-err and stop3-cap (tests/test_gpu_options.py) as the two rows of one launch on every kernel variant: each
    row bit-identical to its single-option launch on the same cell (landing cell checked from bsgp_plan_info)."""
    gn, psf, bkg, obj, rows = _option_rows(v)
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    m = _run(bs, v, plan, padded, gn, psf, bkg, obj, rows)
    assert list(m.status) == [0, 0]
    for i in range(2):
        s = _run(bs, v, plan, padded, gn[i:i + 1], psf, bkg[i:i + 1], obj[i:i + 1], [rows[i]])
        _same_image(m, i, s, (v.label, i))
    assert m.err[0, 0] > 0 and not m.err[1].any()                 # errflag on row 0 only
    print(f"\n{v.label}: iters {list(m.iters)} (MAXIT 24)")
    if not padded:
        plan.close()


RESIDENCY_ROWS = [v for v in VARIANTS if v.dtype == F64 and v.label.rsplit("-", 1)[0] in ("33x20", "pad375", "100x75-frame")]


@pytest.mark.parametrize("v", RESIDENCY_ROWS, ids=lambda v: v.label)
def test_three_residencies_agree(bs, v):
    """The mixed launch of a wrapped, a padded and a frame row through bsgp_solve_batch_rows (device tensors),
    bsgp_solve_batch_rows_host (numpy) and bsgp_solve_batch_rows_pinned (page-locked tensors): bit-identical."""
    gn, psf, bkg, obj, rows = _option_rows(v)
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    a = _run(bs, v, plan, padded, gn, psf, bkg, obj, rows)
    for route in ("device", "pinned"):
        b = _run(bs, v, plan, padded, gn, psf, bkg, obj, rows, route)
        for i in range(2):
            _same_image(b, i, a, (route, i), j=i)
        assert np.array_equal(b.err, a.err), route
    if not padded:
        plan.close()


# ------------------------------------------------------------------------------------------------
# rejections: BSGP_E_ARG before any launch
# ------------------------------------------------------------------------------------------------
def test_malformed_rows_are_refused_before_launch(bs):
    capi, L = bs._capi, bs._capi.lib()
    plan = bs.Plan(64, 64)
    rng = np.random.default_rng(5)
    gn = rng.poisson(100.0, (2, 64, 64)).astype(np.float64)
    psf = np.zeros((64, 64)); psf[32, 32] = 1.0
    plan.set_psf(psf)
    plan.set_psf_adjoint(psf)
    bkg, b0, flux = np.full(2, 10.0), np.full(2, 1.005), np.full(2, gn[0].sum())
    x0, obj = np.ones_like(gn), np.ones_like(gn)
    x = np.zeros_like(gn)
    i32, f64 = (lambda *s: np.zeros(s, np.int32)), (lambda *s: np.zeros(s))
    outs = [x, i32(2), i32(2), f64(2, 40), f64(2, 40), f64(2, 40), f64(2, 41)]

    def solve(rows, with_x0=True, with_obj=True, refused=True):
        ci = capi.Inputs(gn.ctypes.data, bkg.ctypes.data, 0, flux.ctypes.data, b0.ctypes.data,
                         x0.ctypes.data if with_x0 else None, obj.ctypes.data if with_obj else None, None)
        co = capi.Outputs(*(a.ctypes.data for a in outs))
        arr = (capi.Params * 2)(*rows)
        before = L.bsgp_launch_count()
        rc = L.bsgp_solve_batch_rows_host(plan.handle, arr, 2, C.byref(ci), C.byref(co))
        assert not refused or L.bsgp_launch_count() == before, "a refused call launched a kernel"
        return rc, L.bsgp_last_error_string().decode()

    def kl(**kw):
        return capi.make_params(capi.DIV_KL, **dict(dict(MAXIT=39), **kw))

    win = dict(region=(8, 56, 8, 56), div_a=1.0, div_at=1.0)
    cases = [
        ([kl(**win), kl(region=(8, 56, 8, 55), div_a=1.0, div_at=1.0)], {}, "operator"),
        ([kl(**win), kl(region=(8, 56, 8, 56), div_a=2.0, div_at=1.0)], {}, "operator"),
        ([kl(**win), kl(region=(8, 56, 8, 56), div_a=1.0, div_at=0.5)], {}, "operator"),
        ([kl(), kl(adjoint_second_psf=True)], {}, "operator"),
        ([kl(), kl(errflag=True)], dict(with_obj=False), "errflag"),
        ([kl(), kl(init_recon=1)], dict(with_x0=False), "init_recon = 1"),
        ([kl(), kl(MAXIT=0)], {}, "MAXIT"),
        ([kl(), kl(M=17)], {}, "M and M_alpha"),
    ]
    for rows, io, text in cases:
        rc, msg = solve(rows, **io)
        assert rc == 1, (rc, msg)                                          # BSGP_E_ARG
        assert msg.startswith("row 1: ") and text in msg, msg
    rc, msg = solve([kl(), capi.make_params(capi.DIV_BETA, MAXIT=12, stop_criterion=3)], refused=False)
    assert rc == 0, msg
    plan.close()
