"""Iterate snapshots on the CPU (no GPU): the oracle premise the slot rule rests on, the library's snapshot checks
(csrc/bsgp_rows.h, built for the host), and the front end of solve_batch(snapshot_every=...) with the library out of
reach.

The slot rule: slot j of a solve is bit-identical to the image the same solve returns with MAXIT = j * k + 1.  It holds
because a run with a smaller MAXIT follows the same trajectory as a longer one up to its last pass: nothing but the stop
test reads MAXIT (the beta twin's `epoch == MAXIT` break fires on the same pass as `iter > MAXIT`)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import emul_helper as eh

capi = eh.capi
SRC = os.path.join(eh.HERE, "host_emul", "snapshots_emul.cpp")
BSGP_OK, BSGP_E_ARG = 0, 1


# ------------------------------------------------------------------------------------------------
# the oracle: a MAXIT = m + 1 run is a prefix of a longer run
# ------------------------------------------------------------------------------------------------
def _scene(seed=5, shape=(32, 32)):
    from oracle import sgp_oracle as orc
    rng = np.random.default_rng(seed)
    ny, nx = shape
    yy, xx = np.mgrid[0:ny, 0:nx]
    psf = np.exp(-((yy - ny // 2) ** 2 + (xx - nx // 2) ** 2) / (2 * 1.6 ** 2))
    psf /= psf.sum()
    truth = np.zeros(shape)
    truth[rng.integers(0, ny, 6), rng.integers(0, nx, 6)] = 10 ** rng.uniform(3, 4.5, 6)
    blur = orc.CircularPsf(psf).forward(truth.ravel()).reshape(shape)
    bkg = 200.0
    gn = rng.poisson(np.maximum(blur, 0) + bkg).astype(np.float64)
    return gn, psf, bkg, float((gn - bkg).sum())


RUNS = {
    "kl": dict(divergence="kl", init_recon=0, proj_type=0),
    "beta": dict(divergence="beta", init_recon=2, proj_type=1, alpha=10.0, adapt_beta=True, schedule_lr=True, betaParam=1.02,
                 ccd_sat_level=65000),
}


@pytest.mark.parametrize("run", sorted(RUNS))
def test_oracle_shorter_run_is_a_prefix(run):
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _scene()
    kw = dict(RUNS[run], verbose=False, stop_criterion=1)
    if run == "beta":
        kw["flux"] = np.float64(flux)
    L = 20
    full = orc.solve(gn, psf, bkg, MAXIT=L, **kw)
    assert full.iters == L
    for m in (0, 1, 2, 5, 9, 14, L - 1):
        r = orc.solve(gn, psf, bkg, MAXIT=m + 1, **kw)
        assert r.iters == m + 1
        assert np.array_equal(r.discr, full.discr[:m + 2]), m
        for k in ("alpha", "lam", "beta_param", "trials", "proj_evals"):
            assert getattr(r.trace, k) == getattr(full.trace, k)[:m + 1], (m, k)
        assert r.beta_param == full.trace.beta_param[m]


def test_oracle_beta_epoch_break_is_the_maxit_stop():
    """The beta twin's `if epoch == MAXIT: break` (sgp.py:881-882) fires on the pass where iter > MAXIT already stopped the
    loop, so it never shortens a run: the returned image is the one before the last pass for every MAXIT."""
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _scene(seed=9)
    kw = dict(RUNS["beta"], verbose=False, stop_criterion=1, flux=np.float64(flux))
    for maxit in (1, 2, 3, 7):
        r = orc.solve(gn, psf, bkg, MAXIT=maxit, **kw)
        assert r.iters == maxit and len(r.trace.alpha) == maxit


# ------------------------------------------------------------------------------------------------
# the library's checks (host build of bsgp_rows.h)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def snap_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("snapshots_emul") / "libsnapshots_emul.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    L = C.CDLL(so)
    L.emul_check_snapshots.argtypes = [C.POINTER(capi.Outputs), C.c_char_p, C.c_int]
    return L


def _check(L, snap_x, every):
    co = capi.Outputs()
    co.snap_x, co.snap_every = snap_x, every
    msg = C.create_string_buffer(256)
    return L.emul_check_snapshots(C.byref(co), msg, 256), msg.value.decode()


def test_snapshot_checks(snap_lib):
    buf = np.zeros(4)
    assert _check(snap_lib, None, 0) == (BSGP_OK, "")                      # no snapshots: today's behaviour
    assert _check(snap_lib, buf.ctypes.data, 0) == (BSGP_OK, "")
    assert _check(snap_lib, buf.ctypes.data, 3) == (BSGP_OK, "")
    assert _check(snap_lib, None, -1) == (BSGP_E_ARG, "snap_every must be >= 0 (got -1)")
    assert _check(snap_lib, buf.ctypes.data, -5) == (BSGP_E_ARG, "snap_every must be >= 0 (got -5)")
    assert _check(snap_lib, None, 2) == (BSGP_E_ARG, "snap_every = 2 needs outputs.snap_x")


def test_snapshot_slots(snap_lib):
    # trace stride = largest maxit + 1
    for maxit, k, n in ((6, 1, 7), (6, 3, 3), (7, 3, 3), (8, 3, 3), (9, 3, 4), (1, 5, 1), (500, 10, 51)):
        assert snap_lib.emul_snapshot_slots(maxit + 1, k) == n, (maxit, k)


def test_outputs_struct_layout(snap_lib):
    """bsgp_outputs gained snap_x, snap_every and snap_count at its end: the fields before them keep their offsets."""
    assert capi.Outputs.trace_evals.offset == 15 * 8
    assert snap_lib.emul_sizeof_outputs() == C.sizeof(capi.Outputs)
    for i, f in enumerate(("snap_x", "snap_every", "snap_count")):
        assert snap_lib.emul_offsetof_snap(i) == getattr(capi.Outputs, f).offset, f


# ------------------------------------------------------------------------------------------------
# the front end, with the library out of reach
# ------------------------------------------------------------------------------------------------
@pytest.fixture
def bs(monkeypatch):
    import beta_sgp_b200 as b
    monkeypatch.setattr(b.engine, "lib", lambda: pytest.fail("the library was reached"))
    monkeypatch.setattr(b.engine, "get_plan", lambda *a, **k: pytest.fail("a plan was made"))
    return b


def _gn(B=3, shape=(16, 16)):
    return np.random.default_rng(1).poisson(100.0, (B,) + shape).astype(np.float64)


@pytest.mark.parametrize("k", [-1, -10, 1.5, "2", True, None])
def test_bad_interval_is_refused(bs, k):
    gn = _gn()
    with pytest.raises(ValueError, match="snapshot_every must be an integer >= 0"):
        bs.solve_batch(gn, gn[0] / gn[0].sum(), 10.0, snapshot_every=k)


def test_pinned_tensors_are_refused(bs, monkeypatch):
    import torch
    gn = torch.from_numpy(_gn())
    monkeypatch.setattr(torch.Tensor, "is_pinned", lambda self: True)        # no CUDA runtime here to pin memory
    with pytest.raises(ValueError, match="not supported with pinned CPU tensors"):
        bs.solve_batch(gn, gn[0] / gn[0].sum(), 10.0, snapshot_every=2)


def test_sharded_is_refused(bs):
    gn = _gn()
    with pytest.raises(ValueError, match="snapshot_every"):
        bs.solve_batch_sharded(gn, gn[0] / gn[0].sum(), 10.0, snapshot_every=1)


class _Plan:
    """stands in for a plan: the shape and dtype _Args needs, a PSF count"""
    ny = nx = 16
    dtype = "float64"
    device = 0

    def set_psf(self, psf):
        return 1


def _args(bs, per_image=None, k=3, MAXIT=8, alloc=np.zeros):
    gn = _gn(len(per_image) if per_image else 3)
    return bs.engine._Args(gn, gn[0] / gn[0].sum(), 10.0, "beta", None, 1.005, None, None, False, _Plan(), False, dict(MAXIT=MAXIT),
                           psf_arg=lambda a: a, image=lambda a, n: a, vector=bs.engine._host_vector, alloc=alloc,
                           per_image=per_image, snapshot_every=k, snap_alloc=lambda shape: np.full(shape, np.nan))


def test_slot_count_of_a_mixed_batch(bs):
    """n_snap = max MAXIT // k + 1 for every image of a per_image batch with mixed MAXIT"""
    rows = [dict(MAXIT=4), dict(MAXIT=11, divergence="kl"), dict(MAXIT=7)]
    a = _args(bs, rows, k=3)
    assert a.snapshots.shape == (3, 11 // 3 + 1, 16, 16) and np.isnan(a.snapshots).all()
    assert a.snap_count.shape == (3,) and a.snap_count.dtype == np.int32
    assert bs.engine.snapshot_slots(11, 3) == 4 and bs.engine.snapshot_slots(6, 1) == 7 and bs.engine.snapshot_slots(5, 10) == 1


def test_struct_fields(bs):
    a = _args(bs, k=2, MAXIT=6)
    x = np.empty((3, 16, 16))
    _, co = a.structs(x, None)
    assert co.snap_every == 2 and co.snap_x == a.snapshots.ctypes.data and co.snap_count == a.snap_count.ctypes.data
    assert a.snapshots.shape == (3, 4, 16, 16)
    r = a.result(x)
    assert r.snapshots is a.snapshots and r.snapshot_count is a.snap_count
    # without snapshots: the fields stay zero / NULL and the result carries None
    b = _args(bs, k=0)
    _, co = b.structs(x, None)
    assert co.snap_every == 0 and not co.snap_x and not co.snap_count
    r = b.result(x)
    assert r.snapshots is None and r.snapshot_count is None
