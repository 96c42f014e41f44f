"""Build and call the TEST-ONLY host emulation of the device headers (tests/host_emul/emul.cpp)."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "host_emul", "emul.cpp")
SO = os.path.join(HERE, "host_emul", "libbsgp_emul.so")
CSRC = os.path.join(ROOT, "beta-sgp_b200", "csrc")


def _capi():
    spec = importlib.util.spec_from_file_location("_bsgp_capi_for_tests", os.path.join(ROOT, "beta-sgp_b200", "_capi.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


capi = _capi()


def build(force=False):
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(ROOT, "include", "bsgp.h"))
    if not force and os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in deps):
        return SO
    # inline functions and their local statics stay private to this library: the product library (loaded by other tests in
    # the same process) defines the same bsgp:: inline symbols, possibly from an older build
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility-inlines-hidden",
                           "-fno-gnu-unique", "-Wl,-Bsymbolic", "-o", SO, SRC])
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def solve(gn, psf, bkg, divergence="kl", flux=None, betaParam=1.005, obj=None, x0=None, psf_adjoint=None, wrapped=False, **kw):
    """Emulated solve of one image; keyword arguments as sgp()/sgp_betaDiv() (+ region / div_a / div_at /
    adjoint_second_psf with psf_adjoint for the zero-padded operator: inputs already embedded in the grid).
    wrapped=True: any image size through the wrapped-plan steps of the library (bsgp_wrap.h)."""
    L = lib()
    ny, nx = gn.shape
    gn = np.ascontiguousarray(gn, dtype=np.float64)
    psf = np.ascontiguousarray(psf, dtype=np.float64)
    bkg = np.asarray(bkg, dtype=np.float64)
    bkg_is_image = int(bkg.ndim == 2)
    bkg = np.ascontiguousarray(bkg.reshape(-1))
    p = capi.make_params(capi.DIV_KL if divergence == "kl" else capi.DIV_BETA, has_flux=flux is not None, **kw)
    if p.init_recon == 1 and x0 is None:
        np.random.seed(42)
        x0 = np.random.randn(ny, nx)
    maxit = p.maxit
    fl = np.array([0.0 if flux is None else float(flux)])
    b0 = np.array([float(betaParam)])
    x = np.zeros((ny, nx)); iters = np.zeros(1, np.int32); status = np.zeros(1, np.int32)
    discr = np.zeros(maxit + 1); stopv = np.zeros(maxit + 1); err = np.zeros(maxit + 2); bfin = np.zeros(1)
    pe = np.zeros(1, np.int32); lt = np.zeros(1, np.int32); sc = np.zeros(8)
    ta = np.zeros(maxit + 1); tl = np.zeros(maxit + 1); tb = np.zeros(maxit + 1)
    tt = np.zeros(maxit + 1, np.int32); te = np.zeros(maxit + 1, np.int32)
    objc = None if obj is None else np.ascontiguousarray(obj, dtype=np.float64)
    x0c = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
    pa = None if psf_adjoint is None else np.ascontiguousarray(psf_adjoint, dtype=np.float64)
    if wrapped:
        L.emul_solve_wrapped.argtypes = [C.c_int, C.c_int, C.POINTER(capi.Params)] + [C.c_void_p] * 2 + [C.c_void_p, C.c_int] + [C.c_void_p] * 19
        rc = L.emul_solve_wrapped(ny, nx, C.byref(p), _p(gn), _p(psf), _p(bkg), bkg_is_image, _p(fl), _p(b0), _p(x0c), _p(objc),
                                  _p(x), _p(iters), _p(status), _p(discr), _p(stopv), _p(err), _p(bfin), _p(pe), _p(lt), _p(sc),
                                  _p(ta), _p(tl), _p(tb), _p(tt), _p(te))
    else:
        L.emul_solve.argtypes = [C.c_int, C.c_int, C.POINTER(capi.Params)] + [C.c_void_p] * 3 + [C.c_void_p, C.c_int] + [C.c_void_p] * 19
        rc = L.emul_solve(ny, nx, C.byref(p), _p(gn), _p(psf), _p(pa), _p(bkg), bkg_is_image, _p(fl), _p(b0), _p(x0c), _p(objc),
                          _p(x), _p(iters), _p(status), _p(discr), _p(stopv), _p(err), _p(bfin), _p(pe), _p(lt), _p(sc),
                          _p(ta), _p(tl), _p(tb), _p(tt), _p(te))
    assert rc == 0
    n = int(iters[0])
    return dict(x=x, iters=n, status=int(status[0]), discr=discr[:n + 1], stop_value=stopv[:n + 1], err=err,
                beta_final=float(bfin[0]), proj_evals=int(pe[0]), ls_trials=int(lt[0]), scalars=sc,
                alpha=ta[1:n + 1], lam=tl[1:n + 1], beta_trace=tb[1:n + 1], trials=tt[1:n + 1], evals=te[1:n + 1])


PLAN_FIELDS = ("frame", "cluster_size", "threads", "minb", "resident_mask", "smem_bytes", "conv_smem", "ws_bytes", "wrap_ny",
               "wrap_nx", "grid_ny", "grid_nx")


def plan_launch(shape, dtype, cluster_size=0, threads=0, *, num_sms, max_smem, smem_per_sm):
    """The library's launch-shape planner (csrc/bsgp_plan.h, plan_launch) for an image of `shape` on the device described by
    the keywords: (0, dict of PLAN_FIELDS) or (BSGP_E_* code, None)."""
    L = lib()
    out = (C.c_longlong * len(PLAN_FIELDS))()
    L.emul_plan_launch.argtypes = [C.c_int] * 8 + [C.POINTER(C.c_longlong)]
    rc = L.emul_plan_launch(shape[0], shape[1], capi.BSGP_F64 if dtype == "float64" else capi.BSGP_F32, cluster_size, threads,
                            num_sms, max_smem, smem_per_sm, out)
    return rc, (dict(zip(PLAN_FIELDS, out)) if rc == 0 else None)


def project(c, dia, b, sat_cap=None, max_projs=1000, biter=0, siter=0):
    L = lib()
    c = np.ascontiguousarray(c, dtype=np.float64); dia = np.ascontiguousarray(dia, dtype=np.float64)
    x = np.zeros_like(c); ev = C.c_int(0)
    L.emul_project.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                               C.POINTER(C.c_int)]
    st = L.emul_project(_p(c), _p(dia), c.size, float(b), 0.0 if sat_cap is None else float(sat_cap),
                        int(sat_cap is not None), max_projs, int(biter), int(siter), _p(x), C.byref(ev))
    return x, ev.value, st


if __name__ == "__main__":
    build(force=True)
    print("built", SO)
