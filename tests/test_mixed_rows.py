"""Mixed batches on the CPU (no GPU): the library's keyword checks of one row per image (csrc/bsgp_rows.h, built for the
host), the front end's per_image handling and queue order, and the sharded front end dealing the rows with their images
over gloo, with the CUDA solve replaced by a stand-in."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import emul_helper as eh
from test_sharding import _fake_result, _inputs

capi = eh.capi
SRC = os.path.join(eh.HERE, "host_emul", "rows_emul.cpp")
BSGP_E_ARG = 1


@pytest.fixture(scope="module")
def rows_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("rows_emul") / "librows_emul.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    L = C.CDLL(so)
    L.emul_check_batch_params.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Params), C.c_int, C.POINTER(capi.Inputs),
                                          C.POINTER(capi.Outputs), C.POINTER(C.c_int), C.c_char_p, C.c_int]
    return L


def _io(obj=True, x0=True, flux=True, beta0=True, err=True):
    """Inputs / outputs with the optional arrays present or absent (the checks only look at which pointers are set)."""
    p = C.c_void_p(16)
    ci = capi.Inputs(p, p, 0, p if flux else None, p if beta0 else None, p if x0 else None, p if obj else None, None)
    co = capi.Outputs(p, p, p, p, p, None, p if err else None)
    return ci, co


def _check(L, rows, shared=None, **io):
    ci, co = _io(**io)
    stride = C.c_int(-1)
    msg = C.create_string_buffer(256)
    if rows is None:
        rc = L.emul_check_batch_params(C.byref(shared), None, 1, C.byref(ci), C.byref(co), C.byref(stride), msg, 256)
    else:
        arr = (capi.Params * len(rows))(*rows)
        rc = L.emul_check_batch_params(None, arr, len(rows), C.byref(ci), C.byref(co), C.byref(stride), msg, 256)
    return rc, stride.value, msg.value.decode()


def _kl(**kw):
    return capi.make_params(capi.DIV_KL, **kw)


def _beta(**kw):
    return capi.make_params(capi.DIV_BETA, **kw)


def test_trace_stride_is_the_largest_maxit(rows_lib):
    assert _check(rows_lib, None, shared=_kl(MAXIT=27)) == (0, 28, "")
    assert _check(rows_lib, [_kl(MAXIT=5), _beta(MAXIT=332, stop_criterion=3), _kl(MAXIT=40)]) == (0, 333, "")
    assert _check(rows_lib, [_beta(MAXIT=1)]) == (0, 2, "")


def test_rows_must_share_the_operator(rows_lib):
    geo = dict(region=(64, 439, 64, 439), div_a=1.0, div_at=1.0, adjoint_second_psf=True)
    assert _check(rows_lib, [_kl(**geo), _beta(MAXIT=9, **geo)])[0] == 0
    for k, v in (("region", (64, 439, 65, 440)), ("div_a", 0.5), ("div_at", 2.0), ("adjoint_second_psf", False)):
        rc, _, msg = _check(rows_lib, [_kl(**geo), _kl(**geo), _beta(**dict(geo, **{k: v}))])
        assert rc == BSGP_E_ARG and msg.startswith("row 2: ") and "operator" in msg, (k, msg)


@pytest.mark.parametrize("bad,needs,text", [
    (dict(errflag=True), dict(obj=False), "errflag"),
    (dict(errflag=True), dict(err=False), "errflag"),
    (dict(init_recon=1), dict(x0=False), "init_recon = 1"),
    (dict(has_flux=True), dict(flux=False), "has_flux"),
    (dict(MAXIT=0), {}, "MAXIT"),
    (dict(M=17), {}, "M and M_alpha"),
    (dict(M_alpha=0), {}, "M and M_alpha"),
    (dict(stop_criterion=5), {}, "stop_criterion"),
])
def test_one_bad_row_is_refused_by_index(rows_lib, bad, needs, text):
    """Every row is checked as the shared keywords are; the first bad one is named.  An input that only a bad row needs
    may be absent while no row needs it."""
    rows = [_kl(MAXIT=10), _beta(MAXIT=20), _kl(**dict(dict(MAXIT=30), **bad)), _kl()]
    assert _check(rows_lib, [r for i, r in enumerate(rows) if i != 2], **needs)[0] == 0
    rc, _, msg = _check(rows_lib, rows, **needs)
    assert rc == BSGP_E_ARG and msg.startswith("row 2: ") and text in msg, msg
    rc, _, msg = _check(rows_lib, None, shared=rows[2], **needs)          # the shared keywords: the same check, no row
    assert rc == BSGP_E_ARG and msg.startswith(text.split()[0]), msg


def test_beta_rows_need_beta0(rows_lib):
    assert _check(rows_lib, [_kl(), _kl()], beta0=False)[0] == 0
    rc, _, msg = _check(rows_lib, [_kl(), _beta()], beta0=False)
    assert rc == BSGP_E_ARG and msg.startswith("row 1: beta-divergence")


# ------------------------------------------------------------------------------------------------
# the front end
# ------------------------------------------------------------------------------------------------
def test_per_image_keywords_are_checked_before_the_library(monkeypatch):
    import beta_sgp_b200 as bs
    monkeypatch.setattr(bs.engine, "lib", lambda: pytest.fail("the library was reached"))
    gn = np.ones((2, 16, 16))
    with pytest.raises(TypeError, match="per_image\\[1\\].*MAXITER"):
        bs.solve_batch(gn, gn[0], 0.0, per_image=[{}, {"MAXITER": 3}])
    with pytest.raises(ValueError, match="2 dicts"):
        bs.solve_batch(gn, gn[0], 0.0, per_image=[{}])
    with pytest.raises(ValueError, match="divergence"):
        bs.solve_batch(gn, gn[0], 0.0, per_image=[{}, {"divergence": "is"}])
    with pytest.raises(ValueError, match="padded"):
        bs.solve_batch(gn, gn[0][:5, :5], 0.0, padded=True, per_image=[{}, {"region": (0, 1, 0, 1)}])


def test_row_betas_override_the_call():
    import beta_sgp_b200 as bs
    b = bs.engine._row_betas(1.005, [{}, {"betaParam": 0.95}, {"divergence": "kl"}], 3)
    assert b.tolist() == [1.005, 0.95, 1.005]
    same = np.array([1.1, 1.2])
    assert bs.engine._row_betas(same, [{}, {"MAXIT": 3}], 2) is same


def test_queue_order_of_a_mixed_batch():
    """beta-SGP images by |beta - 1| first, then the KL images, each group in batch order; a batch without any beta-SGP
    image keeps the natural order."""
    import beta_sgp_b200 as bs
    q = bs.engine._queue_order
    beta0 = np.array([1.05, 1.005, 1.005, 0.99, 1.2])
    is_beta = np.array([True, False, True, True, False])
    assert q("beta", beta0, is_beta).tolist() == [2, 3, 0, 1, 4]
    assert q("kl", beta0, is_beta).tolist() == [2, 3, 0, 1, 4]
    assert q("beta", beta0, np.zeros(5, bool)) is None
    assert q("kl", beta0, np.ones(5, bool)).tolist() == [1, 2, 3, 0, 4]
    assert q("beta", beta0).tolist() == q("beta", beta0, np.ones(5, bool)).tolist()


# ------------------------------------------------------------------------------------------------
# the sharded front end deals the rows with their images
# ------------------------------------------------------------------------------------------------
def _rows(n):
    return [dict(MAXIT=3 + (i * 5) % 7, betaParam=1.0 + 0.01 * i) if i % 3 else dict(divergence="kl", MAXIT=4 + i) for i in range(n)]


def _fake_mixed(bs, gn, psf, bkg, flux, betaParam, x0, obj, per_image, kw):
    """_fake_result with the rows folded in: the image depends on the row's MAXIT and divergence, the traces have the
    stride of the largest MAXIT of the rows the call received."""
    maxit = [int(r.get("MAXIT", kw["MAXIT"])) for r in per_image]
    r = _fake_result(bs, gn, psf, bkg, flux, betaParam, x0, obj, max(maxit))
    r.x = r.x + np.array([m + (100 if row.get("divergence", "beta") == "kl" else 0) for m, row in zip(maxit, per_image)])[:, None, None]
    r.iters = np.array(maxit, np.int32)
    for i, m in enumerate(maxit):
        r.discr[i, m + 1:] = 0.0
        r.times[i, m + 1:] = 0.0
    return r


def _mixed_worker(rank, world, n, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, eh.ROOT)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import beta_sgp_b200 as bs
    seen = {}

    def fake_solve(gn, psf, bkg, divergence="beta", flux=None, betaParam=1.005, x0=None, obj=None, per_image=None, **kw):
        seen["rows"] = per_image
        return _fake_mixed(bs, gn, psf, bkg, flux, betaParam, x0, obj, per_image, kw)

    bs.engine.solve_batch = fake_solve
    a, rows = _inputs(n), _rows(n)
    kw = dict(a)
    full = bs.solve_batch_sharded(kw.pop("gn"), kw.pop("psf"), kw.pop("bkg"), MAXIT=5, width=None, per_image=rows, **kw)
    betas = bs.engine._row_betas(a["betaParam"], rows, n)
    want = _fake_mixed(bs, a["gn"], a["psf"], a["bkg"], a["flux"], betas, a["x0"], a["obj"], rows, dict(MAXIT=5))
    ok = True
    for k in ("x", "iters", "status", "discr", "times", "beta_final", "proj_evals", "ls_trials"):
        ok = ok and np.array_equal(full[k], getattr(want, k))
    cr = bs.shard.expected_cost_rank(n, betas, [r.get("divergence", "beta") for r in rows])
    ok = ok and all(rows[int(i)].get("divergence") == "kl" for i in cr[n - sum(r.get("divergence") == "kl" for r in rows):])
    mine = bs.shard.shard_indices(n, rank, world, cr)
    ok = ok and (seen.get("rows") or []) == [rows[int(i)] for i in mine]
    ret[rank] = ok
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 11), (3, 7), (3, 2)])
def test_sharded_front_end_deals_the_rows(world, n):
    """solve_batch_sharded with per_image on `world` CPU processes (gloo): every rank's stand-in solve receives the rows
    of exactly its images (betaParam overrides included in the dealing), shards whose largest MAXIT is below the batch's
    are padded to its trace stride, and the gathered result equals the stand-in run on the whole batch."""
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = 33500 + (os.getpid() + world * 17 + n) % 2000
    procs = [ctx.Process(target=_mixed_worker, args=(r, world, n, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    assert all(ret[r] for r in range(world))
