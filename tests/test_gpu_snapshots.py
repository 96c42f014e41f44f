"""Iterate snapshots on the GPU (run with -m gpu on a B200): solve_batch(snapshot_every=k) / bsgp_outputs.snap_x.

The rule every test holds: slot j of a solve is bit-identical to the image x that the same solve returns when run with
MAXIT = j * k + 1 and stop rule 1, snapshot_count is 1 + (passes made) // k, and the slots after it keep the NaN the
front end fills them with.  Taking snapshots changes nothing else: every output but the wall-clock times is
bit-identical to the same launch without them."""
import dataclasses

import numpy as np
import pytest

import test_gpu_options as tgo
from test_gpu_shared import _observations
from test_gpu_variants import F64, FP32_IMAGE, VARIANTS, _inputs_and_oracle, _plan_cell

pytestmark = pytest.mark.gpu

FIELDS = ("x", "iters", "status", "discr", "stop_value", "err", "beta_final", "proj_evals", "ls_trials", "scalars")
TRACE = ("alpha", "lam", "beta", "trials", "evals")
MAXIT = 7


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    return b


def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def _same(a, b, what):
    for k in FIELDS:
        va, vb = getattr(a, k), getattr(b, k)
        assert (va is None) == (vb is None), (what, k)
        if va is not None:
            assert np.array_equal(_np(va), _np(vb)), (what, k)
    for k in TRACE:
        assert np.array_equal(_np(a.trace[k]), _np(b.trace[k])), (what, "trace", k)


def _check_slots(r, k, refs, what):
    """r: a result with snapshots; refs[m]: x of the same solves with MAXIT = m + 1, stop rule 1 ([B, ny, nx])."""
    sn, cnt, iters = _np(r.snapshots), _np(r.snapshot_count), _np(r.iters)
    assert sn.shape[2:] == _np(r.x).shape[1:], (what, sn.shape)
    for b in range(sn.shape[0]):
        assert cnt[b] == 1 + iters[b] // k, (what, b, cnt[b], iters[b])
        for j in range(sn.shape[1]):
            if j < cnt[b]:
                assert np.array_equal(sn[b, j], refs[j * k][b]), (what, b, j)
            else:
                assert np.isnan(sn[b, j]).all(), (what, b, j)


# ------------------------------------------------------------------------------------------------
# every row of the variant table: KL and beta-SGP, k = 1 and 3
# ------------------------------------------------------------------------------------------------
def _variant_solve(bs, v, run, **over):
    gn, psf, args, kw, div, _ = _inputs_and_oracle(v.shape, v.kernel, run)
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    npdt = np.float64 if v.dtype == F64 else np.float32
    where = dict(padded=True) if padded else dict(plan=plan)
    bkg = args["bkg"]
    bkg = bkg[None].astype(npdt) if np.ndim(bkg) == 2 else bkg
    kw = dict(kw, **over)
    return bs.solve_batch(gn[None].astype(npdt), psf.astype(npdt), bkg, divergence=div, flux=None if args["flux"] is None else [args["flux"]],
                          betaParam=args["betaParam"], dtype=v.dtype, trace=True, **where, **kw)


@pytest.mark.parametrize("run", ["beta", "kl"])
@pytest.mark.parametrize("v", VARIANTS, ids=lambda v: v.label)
def test_every_variant_slots_follow_the_rule(bs, v, run):
    plain = _variant_solve(bs, v, run, MAXIT=MAXIT)
    assert plain.snapshots is None and plain.snapshot_count is None
    refs = {m: _np(_variant_solve(bs, v, run, MAXIT=m + 1).x) for m in range(MAXIT + 1)}
    for k in (1, 3):
        r = _variant_solve(bs, v, run, MAXIT=MAXIT, snapshot_every=k)
        _same(r, plain, (v.label, run, k))
        assert r.snapshots.shape == (1, MAXIT // k + 1) + v.shape and r.snapshots.dtype == r.x.dtype
        assert int(r.iters[0]) == MAXIT and int(r.snapshot_count[0]) == MAXIT // k + 1
        _check_slots(r, k, refs, (v.label, run, k))


# ------------------------------------------------------------------------------------------------
# against the oracle: slot j = the oracle's x with MAXIT = j * k + 1
# ------------------------------------------------------------------------------------------------
ORACLE_ROWS = [v for v in VARIANTS if v.label.rsplit("-", 1)[0] in ("32", "31", "100x75", "256-frame")]


@pytest.mark.parametrize("run", ["beta", "kl"])
@pytest.mark.parametrize("v", ORACLE_ROWS, ids=lambda v: v.label)
def test_slots_match_the_oracle(bs, v, run):
    """fp64 at the suite's strict image bar (1e-8 of the largest value), fp32 at FP32_IMAGE."""
    from oracle import sgp_oracle as orc
    gn, psf, args, kw, div, _ = _inputs_and_oracle(v.shape, v.kernel, run)
    k = 2
    r = _variant_solve(bs, v, run, MAXIT=6, snapshot_every=k)
    sn = _np(r.snapshots)[0]
    bar = 1e-8 if v.dtype == F64 else FP32_IMAGE
    for j in range(sn.shape[0]):
        okw = dict(kw, MAXIT=j * k + 1)
        if run == "beta":
            o = orc.solve(gn, psf, args["bkg"], divergence=div, flux=np.float64(args["flux"]), betaParam=args["betaParam"],
                          use_original_SGP_Afunction=True, verbose=False, **okw)
        else:
            o = orc.solve(gn, psf, args["bkg"], divergence=div, use_original_SGP_Afunction=True, verbose=False, **okw)
        scale = float(np.abs(o.x).max()) or 1.0                         # KL from x = 0: slot 0 is all zeros
        err = float(np.abs(sn[j].astype(np.float64) - o.x).max()) / scale
        assert err <= bar, (v.label, run, j, err)


# ------------------------------------------------------------------------------------------------
# early stops (rules 2-4): the count is the passes made, the later slots keep their NaN
# ------------------------------------------------------------------------------------------------
STOP_ROWS = [v for v in VARIANTS if v.label in ("32-64", "33x20-32", "100x75-64", "256-frame-32", "pad375-64")]


@pytest.mark.parametrize("run", sorted(tgo.OPTION_RUNS))
@pytest.mark.parametrize("v", STOP_ROWS, ids=lambda v: v.label)
def test_early_stop_counts_the_passes(bs, v, run):
    c = tgo.option_case(v.shape, v.kernel, run)
    plan, padded, _ = _plan_cell(bs, v)
    k = 2
    plain = tgo._solve(bs, v, c, plan, padded)
    r = tgo._solve(bs, v, dataclasses.replace(c, kw=dict(c.kw, snapshot_every=k)), plan, padded)
    _same(r, plain, (v.label, run))
    n = int(r.iters[0])
    assert n < c.kw["MAXIT"] and r.snapshots.shape[1] == c.kw["MAXIT"] // k + 1
    refs = {}
    for m in range(0, n + 1, k):
        rc = dataclasses.replace(c, kw=dict(c.kw, MAXIT=m + 1, stop_criterion=1))
        refs[m] = _np(tgo._solve(bs, v, rc, plan, padded).x)
    _check_slots(r, k, refs, (v.label, run))
    assert int(r.snapshot_count[0]) < r.snapshots.shape[1]               # at least one slot was never reached


# ------------------------------------------------------------------------------------------------
# mixed batches and shared observations
# ------------------------------------------------------------------------------------------------
MIX_ROWS = [v for v in VARIANTS if v.label in ("32-32", "100x75-64", "256-frame-64", "pad375-32")]


@pytest.mark.parametrize("v", MIX_ROWS, ids=lambda v: v.label)
def test_mixed_batch_and_source_map(bs, v):
    """Five solves of two observations with their own divergence, beta, flux and MAXIT (4, 9, 6, 7, 3), k = 2: the slot
    stride is max MAXIT // k + 1 = 5, and each solve's slots follow the rule for its own MAXIT."""
    plan, padded, _ = _plan_cell(bs, v)
    obs, flux = _observations(bs, v.shape, v.kernel, v.dtype, n=2)
    src = np.array([0, 1, 1, 0, 1], dtype=np.int32)
    maxits = [4, 9, 6, 7, 3]
    rows = []
    for i, s in enumerate(src):
        if i % 3 == 1:
            rows.append(dict(divergence="kl", MAXIT=maxits[i], flux=None))
        else:
            rows.append(dict(divergence="beta", betaParam=0.97 + 0.02 * i, flux=float(flux[s]), proj_type=1, init_recon=2,
                             adapt_beta=True, schedule_lr=True, MAXIT=maxits[i]))
    where = dict(padded=True, dtype=v.dtype) if padded else dict(plan=plan, dtype=v.dtype)
    k = 2
    r = bs.solve_batch(obs["gn"], obs["psf"], obs["bkg"], x0=obs["x0"], per_image=rows, source=src, snapshot_every=k, trace=True,
                       **where)
    plain = bs.solve_batch(obs["gn"], obs["psf"], obs["bkg"], x0=obs["x0"], per_image=rows, source=src, trace=True, **where)
    _same(r, plain, v.label)
    assert r.snapshots.shape == (5, max(maxits) // k + 1) + v.shape
    # the reference of slot j: the same launch (the same PSF stack and, on the padded route, the same operator divisors)
    # with every row's MAXIT = j * k + 1
    refs = {}
    for j in range(r.snapshots.shape[1]):
        short = [dict(row, MAXIT=j * k + 1) for row in rows]
        refs[j * k] = bs.solve_batch(obs["gn"], obs["psf"], obs["bkg"], x0=obs["x0"], per_image=short, source=src, **where).x
    for i in range(len(rows)):
        assert int(r.iters[i]) == maxits[i]
    _check_slots(r, k, refs, v.label)


def test_row_subsets_are_not_empty():
    assert (len(ORACLE_ROWS), len(STOP_ROWS), len(MIX_ROWS), len(ROUTE_ROWS)) == (8, 5, 4, 4)


# ------------------------------------------------------------------------------------------------
# routes
# ------------------------------------------------------------------------------------------------
ROUTE_ROWS = [v for v in VARIANTS if v.label in ("100x75-64", "31-32", "pad375-64", "450-32")]


@pytest.mark.parametrize("v", ROUTE_ROWS, ids=lambda v: v.label)
def test_device_route_equals_host_route(bs, v):
    """CUDA tensors in, CUDA tensors out (bsgp_solve_batch_rows): bit-identical to the numpy route (the _host entry
    point), snapshots included, in the caller's image shape on wrapped, dense, padded and frame plans."""
    import torch
    gn, psf, args, kw, div, _ = _inputs_and_oracle(v.shape, v.kernel, "beta")
    plan, padded, _ = _plan_cell(bs, v)
    npdt = np.float64 if v.dtype == F64 else np.float32
    g = np.stack([gn, gn]).astype(npdt)
    bkg = np.stack([args["bkg"]] * 2).astype(npdt)
    where = dict(padded=True) if padded else dict(plan=plan)
    common = dict(divergence=div, flux=[args["flux"]] * 2, betaParam=np.array([args["betaParam"], 1.01]), trace=True,
                  snapshot_every=3, **where, **dict(kw, MAXIT=8))
    h = bs.solve_batch(g, psf.astype(npdt), bkg, dtype=v.dtype, **common)
    d = bs.solve_batch(torch.as_tensor(g, device="cuda"), torch.as_tensor(psf.astype(npdt), device="cuda"),
                       torch.as_tensor(bkg, device="cuda"), **common)
    torch.cuda.synchronize()
    assert isinstance(d.snapshots, torch.Tensor) and d.snapshots.is_cuda and d.snapshots.dtype == d.x.dtype
    assert h.snapshots.shape == (2, 3) + v.shape
    _same(d, h, v.label)
    assert np.array_equal(_np(d.snapshots), h.snapshots) and np.array_equal(_np(d.snapshot_count), h.snapshot_count)


def test_split_axis_plan(bs):
    """An fp64 (16384, 128) plan runs split 16384-point transforms (SplitCtx): its snapshots follow the rule too."""
    from test_gpu_variants import _scene
    shape = (16384, 128)
    gn, psf, bkg, flux = _scene(bs, shape, 0, seed=3)
    plan = bs.Plan(*shape, "float64")
    kw = dict(divergence="beta", flux=[flux], betaParam=1.02, plan=plan, proj_type=1, init_recon=2, alpha=10.0)
    r = bs.solve_batch(gn[None], psf, bkg[None], MAXIT=4, snapshot_every=1, **kw)
    refs = {m: bs.solve_batch(gn[None], psf, bkg[None], MAXIT=m + 1, **kw).x for m in range(5)}
    _check_slots(r, 1, refs, "split")
    plan.close()


def test_refusals(bs):
    import torch
    gn, psf, args, kw, div, _ = _inputs_and_oracle((32, 32), 0, "kl")
    pinned = torch.from_numpy(gn[None].copy()).pin_memory()
    with pytest.raises(ValueError, match="pinned"):
        bs.solve_batch(pinned, psf, 300.0, divergence="kl", snapshot_every=2)
    with pytest.raises(ValueError, match="snapshot_every must be"):
        bs.solve_batch(gn[None], psf, 300.0, divergence="kl", snapshot_every=-1)
    # the library itself: a negative interval, and the page-locked entry points
    plan = bs.Plan(32, 32)
    e = bs.engine
    args = e._Args(gn[None], psf, 300.0, "kl", None, 1.005, None, None, False, plan, False, dict(MAXIT=4), psf_arg=lambda a: a,
                   image=lambda a, n: np.ascontiguousarray(a), vector=e._host_vector, alloc=np.zeros, snapshot_every=1,
                   snap_alloc=lambda s: np.full(s, np.nan))
    x = np.empty((1, 32, 32))
    ci, co = args.structs(x, None)
    co.snap_every = -1
    with pytest.raises(bs._capi.BsgpError, match="snap_every must be >= 0"):
        args.solve(plan, "_host", ci, co)
    co.snap_every, co.snap_x = 1, None
    with pytest.raises(bs._capi.BsgpError, match="needs outputs.snap_x"):
        args.solve(plan, "_host", ci, co)
    co.snap_x = args.snapshots.ctypes.data
    with pytest.raises(bs._capi.BsgpError, match="not supported by bsgp_solve_batch_pinned"):
        args.solve(plan, "_pinned", ci, co, None)
    assert np.isnan(args.snapshots).all()                              # nothing ran
    plan.close()
