"""Shared observations on the CPU (no GPU): the library's source-map checks (csrc/bsgp_rows.h, built for the host), the
front end's shape, broadcasting and error rules for solve_batch(source=...), and the sharded front end dealing each rank
only the observations its solves read, over gloo with the CUDA solve replaced by a stand-in."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import emul_helper as eh
from test_sharding import _fake_result, _inputs

capi = eh.capi
SRC = os.path.join(eh.HERE, "host_emul", "sources_emul.cpp")
BSGP_OK, BSGP_E_ARG, BSGP_E_STATE = 0, 1, 5


@pytest.fixture(scope="module")
def src_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sources_emul") / "libsources_emul.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, SRC])
    L = C.CDLL(so)
    L.emul_check_sources.argtypes = [C.POINTER(capi.Inputs), C.c_int, C.c_int, C.c_char_p, C.c_int]
    return L


def _check(L, source, n_sources, batch, n_psf):
    m = None if source is None else np.ascontiguousarray(source, dtype=np.int32)
    ci = capi.Inputs(None, None, 0, None, None, None, None, None, None if m is None else m.ctypes.data, n_sources)
    msg = C.create_string_buffer(256)
    rc = L.emul_check_sources(C.byref(ci), batch, n_psf, msg, 256)
    return rc, msg.value.decode()


def test_source_map_indices(src_lib):
    assert _check(src_lib, [2, 0, 0, 1, 2, 2, 0], 3, 7, 1) == (BSGP_OK, "")
    assert _check(src_lib, [0, 0, 0], 5, 3, 1) == (BSGP_OK, "")            # observations no solve reads are allowed
    rc, msg = _check(src_lib, [2, 0, 0, 3, 2], 3, 5, 1)
    assert rc == BSGP_E_ARG and msg == "solve 3: source 3 is outside 0..2", msg
    rc, msg = _check(src_lib, [0, -1], 3, 2, 1)
    assert rc == BSGP_E_ARG and msg.startswith("solve 1: source -1"), msg
    for n in (0, -4):
        rc, msg = _check(src_lib, [0, 0], n, 2, 1)
        assert rc == BSGP_E_ARG and "n_sources must be >= 1" in msg, msg


def test_psf_count_follows_the_observations(src_lib):
    assert _check(src_lib, [1, 0, 1, 2], 3, 4, 3)[0] == BSGP_OK
    rc, msg = _check(src_lib, [1, 0, 1, 2], 3, 4, 4)                      # one PSF per solve is not one per observation
    assert rc == BSGP_E_STATE and "need 1 or n_sources (3)" in msg, msg
    rc, msg = _check(src_lib, [1, 0, 1, 2], 3, 4, 0)
    assert rc == BSGP_E_STATE, msg
    # without a map: one per image, as before
    assert _check(src_lib, None, 0, 4, 4)[0] == BSGP_OK
    assert _check(src_lib, None, 0, 4, 1)[0] == BSGP_OK
    rc, msg = _check(src_lib, None, 7, 4, 3)
    assert rc == BSGP_E_STATE and msg == "bsgp_set_psf was called with 3 PSFs; need 1 or batch (4)", msg


def test_inputs_struct_layout():
    """bsgp_inputs gained source and n_sources at its end: the fields before them keep their offsets."""
    assert capi.Inputs.order.offset == 7 * 8 and capi.Inputs.source.offset == 8 * 8 and capi.Inputs.n_sources.offset == 9 * 8
    L = eh.lib()
    assert C.sizeof(capi.Inputs) == L.emul_sizeof_inputs()


# ------------------------------------------------------------------------------------------------
# the front end
# ------------------------------------------------------------------------------------------------
SRC_MAP = [2, 0, 0, 1, 2, 2, 0]


def _obs(n=3, shape=(16, 16)):
    rng = np.random.default_rng(1)
    return rng.poisson(100.0, (n,) + shape).astype(np.float64)


BAD_CALLS = [
    (dict(source=[0, 3, 1]), "source\\[1\\] = 3 is outside 0..2"),
    (dict(source=[0, -1]), "source\\[1\\] = -1"),
    (dict(source=[[0, 1]]), "1-D integer"),
    (dict(source=[0.0, 1.0]), "1-D integer"),
    (dict(source=[]), "1-D integer"),
    (dict(psf="per_solve"), "one per observation \\(3\\)"),
    (dict(bkg=np.ones(7)), "bkg must be"),
    (dict(bkg=np.ones((7, 16, 16))), "bkg must be"),
    (dict(x0=np.ones((7, 16, 16))), "x0 must be \\[3, ny, nx\\]"),
    (dict(obj=np.ones((2, 16, 16))), "obj must be \\[3, ny, nx\\]"),
    (dict(flux=np.ones(3)), "flux is per solve"),
    (dict(betaParam=np.ones(3)), "betaParam is per solve"),
]


def _call(bs, route, source=SRC_MAP, psf=None, bkg=10.0, **kw):
    gn = _obs()
    if psf is None:
        psf = gn[0] / gn[0].sum()
    elif isinstance(psf, str):
        psf = np.stack([gn[0] / gn[0].sum()] * len(source))
    if route == "tensor":                               # pageable CPU tensors take the numpy route
        gn, psf = torch.from_numpy(gn), torch.from_numpy(np.asarray(psf))
    extra = dict(padded=True) if route == "padded" else {}
    if route == "padded":
        psf = np.asarray(psf)[..., 5:10, 5:10]
    return bs.solve_batch(gn, psf, bkg, source=source, **extra, **kw)


@pytest.mark.parametrize("route", ["numpy", "tensor", "padded"])
@pytest.mark.parametrize("call,text", BAD_CALLS, ids=[str(i) for i in range(len(BAD_CALLS))])
def test_shape_rules_are_checked_before_the_library(monkeypatch, route, call, text):
    import beta_sgp_b200 as bs
    monkeypatch.setattr(bs.engine, "lib", lambda: pytest.fail("the library was reached"))
    monkeypatch.setattr(bs.engine, "get_plan", lambda *a, **k: pytest.fail("a plan was made"))
    with pytest.raises(ValueError, match=text):
        _call(bs, route, **call)


def test_per_image_rows_are_per_solve(monkeypatch):
    import beta_sgp_b200 as bs
    monkeypatch.setattr(bs.engine, "lib", lambda: pytest.fail("the library was reached"))
    with pytest.raises(ValueError, match="list of 7 dicts"):
        _call(bs, "numpy", per_image=[{}] * 3)


class _FakePlan:
    """What _Args needs of a plan, without a device: shape, dtype and the PSF count it was given."""

    def __init__(self, ny, nx):
        self.ny, self.nx, self.dtype, self.device, self.n_psf = ny, nx, "float64", 0, None

    def set_psf(self, psf):
        self.n_psf = 1 if np.ndim(psf) == 2 else int(np.shape(psf)[0])
        return self.n_psf


@pytest.mark.parametrize("bkg,psf_per_obs", [(10.0, False), ("per_obs", True), ("image", False)])
def test_broadcasting_on_the_host_route(monkeypatch, bkg, psf_per_obs):
    """What the host route hands the library: the observation arrays once each (a scalar background broadcast to one value
    per observation), flux and betaParam per solve, the map as int32 with n_sources, and B outputs."""
    import beta_sgp_b200 as bs
    seen = {}

    def fake_solve(self, plan, entry, ci, co, *stream):
        seen.update(args=self, ci=ci, co=co, entry=entry)

    monkeypatch.setattr(bs.engine._Args, "solve", fake_solve)
    gn = _obs()
    psf = np.stack([g / g.sum() for g in gn]) if psf_per_obs else gn[0] / gn[0].sum()
    b = {10.0: 10.0, "per_obs": np.array([5.0, 6.0, 7.0]), "image": np.full(gn.shape, 3.0)}[bkg if isinstance(bkg, str) else 10.0]
    plan = _FakePlan(16, 16)
    per_image = [dict(divergence="kl") if i % 3 == 0 else {} for i in range(7)]
    res = bs.solve_batch(gn, psf, b, source=SRC_MAP, plan=plan, flux=np.arange(7) + 100.0, betaParam=np.linspace(0.9, 1.1, 7),
                         per_image=per_image, MAXIT=9)
    a, ci = seen["args"], seen["ci"]
    assert seen["entry"] == "_host" and plan.n_psf == (3 if psf_per_obs else 1)
    assert a.B == 7 and a.n_sources == 3 and ci.n_sources == 3
    assert a.source.dtype == np.int32 and a.source.tolist() == SRC_MAP and ci.source == a.source.ctypes.data
    assert a.gn.shape == (3, 16, 16) and ci.gn == a.gn.ctypes.data
    if bkg == "image":
        assert a.bkg_img == 1 and a.bkg.shape == (3, 16, 16)
    else:
        assert a.bkg_img == 0 and a.bkg.shape == (3,)
        assert a.bkg.tolist() == ([10.0] * 3 if bkg == 10.0 else [5.0, 6.0, 7.0])
    assert a.flux.tolist() == list(np.arange(7) + 100.0) and a.beta0.shape == (7,)
    assert len(a.rows) == 7 and [r.divergence for r in a.rows] == [0, 1, 1, 0, 1, 1, 0]
    assert res.x.shape == (7, 16, 16) and res.iters.shape == (7,) and res.discr.shape == (7, 10)
    # the queue order is per solve: beta rows by |beta - 1|, then the KL rows
    assert sorted(a.order.tolist()) == list(range(7)) and set(a.order[-3:].tolist()) == {0, 3, 6}


def test_without_a_map_nothing_changes(monkeypatch):
    import beta_sgp_b200 as bs
    seen = {}
    monkeypatch.setattr(bs.engine._Args, "solve", lambda self, plan, entry, ci, co, *s: seen.update(ci=ci, args=self))
    gn = _obs()
    bs.solve_batch(gn, gn[0] / gn[0].sum(), 10.0, plan=_FakePlan(16, 16), MAXIT=4)
    assert seen["ci"].source is None and seen["ci"].n_sources == 0 and seen["args"].B == 3


# ------------------------------------------------------------------------------------------------
# the sharded front end: each rank gets the observations of its solves, renumbered
# ------------------------------------------------------------------------------------------------
SHARD_MAP = np.array([3, 0, 0, 1, 3, 3, 0, 2, 1, 3, 0])


def _fake_shared(bs, gn, psf, bkg, flux, betaParam, x0, obj, source, maxit):
    """_fake_result on the observations replicated through the map: what the shared solve must equal."""
    def rep(a):
        return a[source] if a is not None and np.ndim(a) >= 1 and np.shape(a)[0] == gn.shape[0] and np.size(a) > 1 else a
    return _fake_result(bs, gn[source], rep(psf) if np.ndim(psf) == 3 else psf, rep(bkg), flux, betaParam, rep(x0), rep(obj), maxit)


def _shared_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, eh.ROOT)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import beta_sgp_b200 as bs
    seen = {}

    def fake_solve(gn, psf, bkg, divergence="beta", flux=None, betaParam=1.005, x0=None, obj=None, source=None, **kw):
        seen.update(gn=gn, source=source, psf=psf, bkg=bkg, x0=x0)
        return _fake_shared(bs, gn, psf, bkg, flux, betaParam, x0, obj, source, kw["MAXIT"])

    bs.engine.solve_batch = fake_solve
    n_obs, B = 4, SHARD_MAP.size
    a = _inputs(n_obs)
    rng = np.random.default_rng(9)
    flux, beta = np.arange(B) + 5.0, rng.normal(1.0, 0.05, B)
    ok = True
    for variant in range(2):
        bkg = a["bkg"] if variant == 0 else a["bkg"][:, 0, 0].copy()
        psf = a["psf"] if variant == 0 else a["psf"][0]
        full = bs.solve_batch_sharded(a["gn"], psf, bkg, flux=flux, betaParam=beta, x0=a["x0"], obj=a["obj"], source=SHARD_MAP,
                                      MAXIT=5, width=None)
        want = _fake_shared(bs, a["gn"], psf, bkg, flux, beta, a["x0"], a["obj"], SHARD_MAP, 5)
        for k in ("x", "iters", "status", "discr", "times", "beta_final", "proj_evals", "ls_trials"):
            ok = ok and np.array_equal(full[k], getattr(want, k))
        mine = bs.shard.shard_indices(B, rank, world, bs.shard.expected_cost_rank(B, beta))
        used = np.unique(SHARD_MAP[mine])
        ok = ok and np.array_equal(seen["gn"], a["gn"][used]) and np.array_equal(seen["x0"], a["x0"][used])
        ok = ok and seen["source"].dtype == np.int32 and np.array_equal(used[seen["source"]], SHARD_MAP[mine])
        ok = ok and (np.array_equal(seen["psf"], a["psf"][used]) if variant == 0 else np.array_equal(seen["psf"], psf))
        ok = ok and np.array_equal(seen["bkg"], bkg[used])
        seen.clear()
    ret[rank] = ok
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_front_end_deals_the_observations():
    """solve_batch_sharded with a source map on two CPU processes (gloo): each rank's stand-in solve receives exactly the
    observations its solves read (gn, psf, bkg, x0 indexed by observation, flux and betaParam by solve) and the map
    renumbered to them, and the gather restores the batch order of the solves."""
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = 35500 + os.getpid() % 2000
    procs = [ctx.Process(target=_shared_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    assert all(ret[r] for r in range(2))
