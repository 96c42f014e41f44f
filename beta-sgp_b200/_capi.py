"""ctypes binding of libbsgp.so (include/bsgp.h).

This is the only place the Python package touches native code.  The library is built in-tree by
``__graft_entry__.build()`` / ``beta-sgp_b200/csrc/build.sh`` for sm_100a; there is no CPU fallback:
if the library or a CUDA device is missing, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSGP_LIB") or os.path.join(_HERE, "csrc", "libbsgp.so")   # BSGP_LIB: kernel experiments only

BSGP_F64, BSGP_F32 = 0, 1
DIV_KL, DIV_BETA = 0, 1
ST_OK, ST_BAD_FLUX, ST_EMPTY_BOUNDS, ST_PROJ_NO_BRACKET, ST_INPUT_TIMEOUT = 0, 1, 2, 3, 4
NSCALARS = 8
STATUS_TEXT = {
    ST_BAD_FLUX: "non-positive or non-finite flux with proj_type=1",
    ST_EMPTY_BOUNDS: "no positive entry in flux/(flux+bkg)*AT(gn): scaling-matrix bounds undefined",
    ST_PROJ_NO_BRACKET: "flux-conserving projection could not bracket the multiplier",
    ST_INPUT_TIMEOUT: "pipelined upload of the image did not arrive (bsgp_solve_batch_pinned)",
}


class Params(C.Structure):
    """struct bsgp_params — keyword arguments of sgp()/sgp_betaDiv() (sgp.py:41-47, 506-513)."""
    _fields_ = [
        ("divergence", C.c_int), ("init_recon", C.c_int), ("proj_type", C.c_int), ("stop_criterion", C.c_int),
        ("maxit", C.c_int), ("gamma", C.c_double), ("ls_beta", C.c_double), ("alpha", C.c_double),
        ("alpha_min", C.c_double), ("alpha_max", C.c_double), ("m_alpha", C.c_int), ("tau", C.c_double),
        ("m", C.c_int), ("max_projs", C.c_int), ("verbose", C.c_int), ("has_flux", C.c_int), ("has_sat", C.c_int),
        ("ccd_sat_level", C.c_double), ("scale_data", C.c_int), ("errflag", C.c_int),
        ("tol_convergence", C.c_double), ("adapt_beta", C.c_int), ("lr", C.c_double), ("lr_exp_param", C.c_double),
        ("schedule_lr", C.c_int), ("region", C.c_int * 4), ("div_a", C.c_double), ("div_at", C.c_double),
        ("adjoint_second_psf", C.c_int),
    ]


class Inputs(C.Structure):
    _fields_ = [("gn", C.c_void_p), ("bkg", C.c_void_p), ("bkg_is_image", C.c_int), ("flux", C.c_void_p),
                ("beta0", C.c_void_p), ("x0", C.c_void_p), ("obj", C.c_void_p), ("order", C.c_void_p),
                ("source", C.c_void_p), ("n_sources", C.c_int)]


class Outputs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("iters", C.c_void_p), ("status", C.c_void_p), ("discr", C.c_void_p),
                ("times", C.c_void_p), ("stop_value", C.c_void_p), ("err", C.c_void_p), ("beta_final", C.c_void_p),
                ("proj_evals", C.c_void_p), ("ls_trials", C.c_void_p), ("scalars", C.c_void_p),
                ("trace_alpha", C.c_void_p), ("trace_lambda", C.c_void_p), ("trace_beta", C.c_void_p),
                ("trace_trials", C.c_void_p), ("trace_evals", C.c_void_p),
                ("snap_x", C.c_void_p), ("snap_every", C.c_int), ("snap_count", C.c_void_p)]


class PlanInfo(C.Structure):
    _fields_ = [("ny", C.c_int), ("nx", C.c_int), ("dtype", C.c_int), ("device", C.c_int), ("cluster_size", C.c_int),
                ("num_clusters", C.c_int), ("threads", C.c_int), ("smem_bytes", C.c_int), ("num_sms", C.c_int),
                ("resident_mask", C.c_int), ("workspace_bytes", C.c_longlong), ("grid_ny", C.c_int), ("grid_nx", C.c_int)]


def make_params(divergence, *, init_recon=0, proj_type=0, stop_criterion=0, MAXIT=500, gamma=1e-4, beta=0.4, alpha=1.3,
                alpha_min=1e-5, alpha_max=1e5, M_alpha=3, tau=0.5, M=1, max_projs=1000, verbose=True, has_flux=False,
                ccd_sat_level=None, scale_data=True, errflag=False, tol_convergence=1e-4, adapt_beta=True, lr=1e-3,
                lr_exp_param=0.1, schedule_lr=False, region=None, div_a=1.0, div_at=1.0, adjoint_second_psf=False):
    p = Params()
    p.divergence = divergence
    p.init_recon, p.proj_type, p.stop_criterion, p.maxit = int(init_recon), int(proj_type), int(stop_criterion), int(MAXIT)
    p.gamma, p.ls_beta, p.alpha, p.alpha_min, p.alpha_max = float(gamma), float(beta), float(alpha), float(alpha_min), float(alpha_max)
    p.m_alpha, p.tau, p.m, p.max_projs = int(M_alpha), float(tau), int(M), int(max_projs)
    p.verbose, p.has_flux = int(bool(verbose)), int(bool(has_flux))
    p.has_sat = int(ccd_sat_level is not None)
    p.ccd_sat_level = float(ccd_sat_level) if ccd_sat_level is not None else 0.0
    p.scale_data, p.errflag, p.tol_convergence = int(bool(scale_data)), int(bool(errflag)), float(tol_convergence)
    p.adapt_beta, p.lr, p.lr_exp_param, p.schedule_lr = int(bool(adapt_beta)), float(lr), float(lr_exp_param), int(bool(schedule_lr))
    if region is not None:
        p.region[0], p.region[1], p.region[2], p.region[3] = (int(v) for v in region)
    p.div_a, p.div_at, p.adjoint_second_psf = float(div_a), float(div_at), int(bool(adjoint_second_psf))
    return p


_lib = None


class BsgpError(RuntimeError):
    pass


def lib():
    """Load libbsgp.so (once).  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BsgpError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  beta-sgp_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, ip, dp = C.c_void_p, C.c_int, C.c_double
    L.bsgp_plan_create.argtypes = [ip, ip, ip, ip, C.POINTER(vp)]
    L.bsgp_plan_destroy.argtypes = [vp]
    L.bsgp_plan_get_info.argtypes = [vp, C.POINTER(PlanInfo)]
    L.bsgp_plan_configure.argtypes = [vp, ip, ip]
    L.bsgp_set_psf.argtypes = [vp, vp, ip, vp]
    L.bsgp_set_psf_host.argtypes = [vp, vp, ip]
    L.bsgp_set_psf_adjoint.argtypes = [vp, vp, ip, vp]
    L.bsgp_set_psf_adjoint_host.argtypes = [vp, vp, ip]
    L.bsgp_solve_batch.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs), vp]
    L.bsgp_solve_batch_host.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs)]
    L.bsgp_solve_batch_pinned.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs), vp]
    L.bsgp_solve_batch_rows.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs), vp]
    L.bsgp_solve_batch_rows_host.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs)]
    L.bsgp_solve_batch_rows_pinned.argtypes = [vp, C.POINTER(Params), ip, C.POINTER(Inputs), C.POINTER(Outputs), vp]
    L.bsgp_apply_psf.argtypes = [vp, vp, vp, ip, ip, vp]
    L.bsgp_apply_psf_host.argtypes = [vp, vp, vp, ip, ip]
    L.bsgp_project_df.argtypes = [vp, vp, vp, ip, ip, dp, dp, dp, dp, ip, ip, ip, vp, vp, vp, ip, vp]
    L.bsgp_project_df_host.argtypes = [vp, vp, vp, ip, ip, dp, dp, dp, dp, ip, ip, ip, vp, vp, vp, ip]
    L.bsgp_beta_div_host.argtypes = [vp, vp, C.c_longlong, dp, vp, vp, ip]
    L.bsgp_beta_grad_terms_host.argtypes = [vp, vp, C.c_longlong, dp, vp, vp, ip]
    L.bsgp_tile_boxes.argtypes = [ip, ip, ip, ip, dp, dp, vp, ip, C.POINTER(ip)]
    L.bsgp_extract_tiles.argtypes = [vp, ip, ip, ip, vp, ip, ip, ip, vp, ip, vp]
    L.bsgp_assemble_tiles.argtypes = [vp, vp, ip, ip, ip, ip, ip, vp, ip, ip, ip, vp]
    L.bsgp_psf_model_eval.argtypes = [vp, ip, ip, ip, ip, ip, ip, ip, vp, ip, vp]
    L.bsgp_device_count.restype = ip
    L.bsgp_launch_count.restype = C.c_longlong
    L.bsgp_last_error_string.restype = C.c_char_p
    L.bsgp_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = lib().bsgp_last_error_string().decode(errors="replace")
        raise BsgpError(f"libbsgp error {rc}: {msg}")


EXPORTED = ["bsgp_plan_create", "bsgp_plan_destroy", "bsgp_plan_get_info", "bsgp_plan_configure", "bsgp_set_psf",
            "bsgp_set_psf_host", "bsgp_set_psf_adjoint", "bsgp_set_psf_adjoint_host", "bsgp_solve_batch", "bsgp_solve_batch_host", "bsgp_solve_batch_pinned",
            "bsgp_solve_batch_rows", "bsgp_solve_batch_rows_host", "bsgp_solve_batch_rows_pinned", "bsgp_apply_psf", "bsgp_apply_psf_host",
            "bsgp_project_df", "bsgp_project_df_host", "bsgp_tile_boxes", "bsgp_extract_tiles", "bsgp_assemble_tiles", "bsgp_psf_model_eval", "bsgp_beta_div_host", "bsgp_beta_grad_terms_host", "bsgp_device_count", "bsgp_launch_count",
            "bsgp_last_error_string", "bsgp_version"]
