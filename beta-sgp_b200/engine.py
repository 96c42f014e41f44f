"""Batched front end of libbsgp: plans, buffers and the `solve_batch` call.

Host arrays (numpy) go through the library's ``*_host`` entry points; CUDA tensors (torch, used
only as device-memory handles) go through the asynchronous device entry points on torch's current
stream.  Nothing here computes: all arithmetic of the restoration loop runs in the CUDA kernels
of csrc/bsgp_kernels.cu, and there is no CPU fallback.

Mirrors the call shape of the reference's batched callers, which loop over images one at a time:
application_sgp_star_stamps.py:56-105 and application_sgp_subdivisions.py:83-107.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _capi
from ._capi import BsgpError, DIV_BETA, DIV_KL, check, lib

_NP = {"float64": np.float64, "float32": np.float32}
_DT = {"float64": _capi.BSGP_F64, "float32": _capi.BSGP_F32}

_SOLVER_KEYS = ("region", "div_a", "div_at", "adjoint_second_psf", "init_recon", "proj_type", "stop_criterion", "MAXIT", "gamma", "beta", "alpha", "alpha_min", "alpha_max",
                "M_alpha", "tau", "M", "max_projs", "verbose", "ccd_sat_level", "scale_data", "errflag",
                "tol_convergence", "adapt_beta", "lr", "lr_exp_param", "schedule_lr")
_ROW_KEYS = ("divergence", "betaParam", "flux") + _SOLVER_KEYS         # what one entry of solve_batch(per_image=...) may set
_OPERATOR_KEYS = ("region", "div_a", "div_at", "adjoint_second_psf")


class Plan:
    """One bsgp_plan: (ny, nx, dtype, device) -> twiddles, per-cluster scratch, PSF spectra."""

    def __init__(self, ny, nx, dtype="float64", device=0, cluster_size=0, threads=0):
        self.ny, self.nx, self.dtype, self.device = int(ny), int(nx), str(dtype), int(device)
        if self.dtype not in _DT:
            raise ValueError("dtype must be 'float64' or 'float32'")
        self._h = C.c_void_p()
        check(lib().bsgp_plan_create(self.ny, self.nx, _DT[self.dtype], self.device, C.byref(self._h)))
        if cluster_size or threads:
            check(lib().bsgp_plan_configure(self._h, int(cluster_size), int(threads)))
        self._psf_keepalive = {}

    @property
    def handle(self):
        return self._h

    def info(self):
        i = _capi.PlanInfo()
        check(lib().bsgp_plan_get_info(self._h, C.byref(i)))
        return {f: getattr(i, f) for f, _ in i._fields_}

    def _image_tensor(self, t, name, lead=None):
        """Validate a CUDA tensor handed to the library as raw memory: [ny,nx] or [n,ny,nx] with the plan's image shape,
        on the plan's device; converted to the plan's dtype and made contiguous.  `lead`: allowed leading sizes."""
        import torch
        if not t.is_cuda:
            raise ValueError(f"{name} must be a CUDA tensor (or a numpy array)")
        if (t.device.index or 0) != self.device:
            raise ValueError(f"{name} lives on {t.device}, the plan on cuda:{self.device}")
        if t.dim() not in (2, 3) or tuple(t.shape[-2:]) != (self.ny, self.nx):
            raise ValueError(f"{name} has shape {tuple(t.shape)}; expected [{self.ny},{self.nx}] or [n,{self.ny},{self.nx}]")
        n = 1 if t.dim() == 2 else int(t.shape[0])
        if lead is not None and n not in lead:
            raise ValueError(f"{name} has {n} images; expected one of {sorted(set(lead))}")
        want = torch.float64 if self.dtype == "float64" else torch.float32
        return t.to(want).contiguous(), n

    def set_psf(self, psf):
        """psf: numpy [ny,nx] / [n,ny,nx] or a CUDA tensor of the same shapes."""
        return self._set_psf(psf, adjoint=False)

    def set_psf_adjoint(self, psf):
        """Second kernel, used for A^T by the zero-padded operator (sgp.py:157); numpy or CUDA tensor, [ny,nx] / [n,ny,nx]."""
        return self._set_psf(psf, adjoint=True)

    def _set_psf(self, psf, adjoint):
        L, name = lib(), "adjoint psf" if adjoint else "psf"
        if _is_tensor(psf):
            t, n = self._image_tensor(psf, name)
            check((L.bsgp_set_psf_adjoint if adjoint else L.bsgp_set_psf)(self._h, t.data_ptr(), n, _stream_ptr()))
            self._psf_keepalive[adjoint] = t            # read by the library on the stream, after this call returns
            return n
        a = np.ascontiguousarray(psf, dtype=_NP[self.dtype])
        n = 1 if a.ndim == 2 else a.shape[0]
        if a.shape[-2:] != (self.ny, self.nx):
            raise ValueError(f"{name} shape {a.shape[-2:]} must equal the image shape {(self.ny, self.nx)} "
                             "(the reference's numpy A/AT closure has the same requirement, sgp.py:108-120)")
        check((L.bsgp_set_psf_adjoint_host if adjoint else L.bsgp_set_psf_host)(self._h, a.ctypes.data, n))
        return n

    def apply_psf(self, x, adjoint=False):
        """A(x) / AT(x) for numpy [ny,nx] or [n,ny,nx] (sgp.py:111-120)."""
        a = np.ascontiguousarray(x, dtype=_NP[self.dtype])
        if a.ndim not in (2, 3) or a.shape[-2:] != (self.ny, self.nx):
            raise ValueError(f"x has shape {a.shape}; expected [{self.ny},{self.nx}] or [n,{self.ny},{self.nx}]")
        n = 1 if a.ndim == 2 else a.shape[0]
        y = np.empty_like(a)
        check(lib().bsgp_apply_psf_host(self._h, a.ctypes.data, y.ctypes.data, n, int(bool(adjoint))))
        return y

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().bsgp_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_plans = {}


def get_plan(ny, nx, dtype="float64", device=0, cluster_size=0, threads=0):
    """Process-wide plan cache, one plan per (shape, dtype, device, tuning).  A plan holds mutable device state (PSF
    spectra, scratch, work queue); the library serialises the launches of one plan on the device (an event chained
    through every entry point, include/bsgp.h "Streams"), so sharing a cached plan between CUDA streams is safe but
    not concurrent: callers that want overlap create their own `Plan` per stream."""
    key = (int(ny), int(nx), str(dtype), int(device), int(cluster_size), int(threads))
    p = _plans.get(key)
    if p is None:
        p = Plan(*key)
        _plans[key] = p
    return p


# Width of the CTA configuration as a function of the number of images a GPU holds (measured on B200, 256 x 256 beta-SGP,
# tools/latency_probe.py): the default (clusters of 8 CTAs x 128 threads, 4 CTAs of different images per SM, 71 images in
# flight) has the best throughput but 200 us per iteration of ONE image; 16 x 128 reaches 118 us with 31 images in flight,
# 8 x 256 112 us with 15, 16 x 256 74 us with 7.  A GPU that holds fewer images than slots is bounded by its longest solve,
# so it trades slots for latency.  Thresholds from tools/width_probe.py (one GPU plays every rank of a world of W on the
# 320-tile field; slowest rank in ms for default / 16 x 128 / 8 x 256 / 16 x 256): 160 images per rank 38.8 / 42.7 / 54.7 /
# 73.6; 80: 28.8 / 24.5 / 28.8 / 38.0; 40: 23.3 / 16.2 / 17.7 / 20.8; 20: 20.4 / 13.1 / 13.1 / 11.6; 10: 19.8 / 11.8 / 13.0 /
# 8.4.  8 x 256 never wins.  (threshold on images per default slot, (cluster_size, threads)); first match wins.
_WIDTH_RULES = ((1.7, (0, 0)), (0.42, (16, 128)), (0.0, (16, 256)))


def auto_config(ny, nx, batch, dtype="float64"):
    """(cluster_size, threads) for `batch` images of ny x nx on one GPU; (0, 0) = the library's default."""
    npix = int(ny) * int(nx)
    pow2 = all(v >= 16 and v & (v - 1) == 0 for v in (int(ny), int(nx)))
    if not pow2 or npix * (8 if dtype == "float64" else 4) <= 64 * 1024 or npix >= (1 << 20):
        return (0, 0)                                   # stamps (one CTA each), embedded (dense / wrapped) plans and frame mode: one configuration
    slots = 71.0                                        # images in flight of the default configuration on 148 SMs
    for thr, cfg in _WIDTH_RULES:
        if batch >= thr * slots:
            if cfg[0] == 16 and not (ny % 64 == 0 and (nx // 2) % 32 == 0):
                continue
            return cfg
    return (0, 0)


def clear_plans():
    for p in _plans.values():
        p.close()
    _plans.clear()


def _is_tensor(a):
    return type(a).__module__.startswith("torch") and hasattr(a, "data_ptr")


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class BatchResult:
    x: object                 # [B,ny,nx] restored images
    iters: object             # [B]
    status: object            # [B] 0 = ok
    discr: object             # [B,MAXIT+1]
    times: object             # [B,MAXIT+1]
    stop_value: object
    err: object
    beta_final: object
    proj_evals: object        # [B] total projection evaluations
    ls_trials: object         # [B] total line-search evaluations
    scalars: object           # [B,8]
    trace: dict | None = None
    snapshots: object = None       # [B,n_snap,ny,nx]: slot j is the iterate after j * snapshot_every passes (solve_batch)
    snapshot_count: object = None  # [B] slots each solve wrote


def _queue_order(divergence, beta0, is_beta=None):
    """Order in which the persistent clusters pull images from the work queue.  Iteration counts of beta-SGP
    grow as beta approaches 1 (28..162 iterations over the reference's five beta initialisations,
    application_sgp_subdivisions.py:69-107), so the images with the smallest |beta - 1| go first: the long
    solves do not end up alone at the tail of the queue.  A mixed batch (is_beta: per image) hands out its beta-SGP
    images in that order, then its KL images.  Results do not depend on the order."""
    if is_beta is not None and not is_beta.all():
        if not is_beta.any():
            return None
        key = np.where(is_beta, np.abs(beta0 - 1.0), np.inf)
        return np.ascontiguousarray(np.argsort(key, kind="stable").astype(np.int32))
    if (divergence != "beta" and is_beta is None) or beta0.size < 2 or np.all(beta0 == beta0[0]):
        return None
    return np.ascontiguousarray(np.argsort(np.abs(beta0 - 1.0), kind="stable").astype(np.int32))


class PaddedGeometry:
    """Placement of an ny x nx image and a ky x kx kernel on the square power-of-two grid that
    astropy.convolution.convolve_fft uses with boundary='fill' (fft_pad = psf_pad = True): side
    2^ceil(log2(max(image + kernel shape))), both centred (sgp.py:138,157 call it with the defaults)."""

    def __init__(self, ny, nx, ky, kx):
        self.ny, self.nx, self.ky, self.kx = ny, nx, ky, kx
        self.P = int(2 ** np.ceil(np.log2(max(ny + ky, nx + kx))))
        c = self.P - (self.P + 1) // 2
        self.rows = slice(c - ny // 2, c + (ny + 1) // 2)
        self.cols = slice(c - nx // 2, c + (nx + 1) // 2)
        self.c = c
        self.region = (self.rows.start, self.rows.stop, self.cols.start, self.cols.stop)

    def embed(self, a, dtype):
        """[B,ny,nx] -> [B,P,P] of `dtype`, zeros in the padding: numpy in, numpy out; a tensor in, a tensor on its device out."""
        shape = tuple(a.shape[:-2]) + (self.P, self.P)
        if _is_tensor(a):
            import torch
            out = torch.zeros(shape, dtype=dtype, device=a.device)
        else:
            out = np.zeros(shape, dtype=dtype)
        out[..., self.rows, self.cols] = a
        return out

    def kernel(self, k, dtype):
        """Normalised kernel(s) [.., kh, kw] centred on the grid; returns (grid array, weight constant)."""
        k = np.asarray(k, dtype=np.float64)
        kh, kw = k.shape[-2:]
        k = k / k.sum(axis=(-2, -1), keepdims=True)
        out = np.zeros(k.shape[:-2] + (self.P, self.P), dtype=dtype)
        out[..., self.c - kh // 2:self.c + (kh + 1) // 2, self.c - kw // 2:self.c + (kw + 1) // 2] = k
        return out, float(out.reshape(-1, self.P * self.P)[0].sum())


def _params(divergence, kw, has_flux):
    unknown = set(kw) - set(_SOLVER_KEYS)
    if unknown:
        raise TypeError(f"unexpected keyword argument(s): {sorted(unknown)}")
    return _capi.make_params(DIV_KL if divergence == "kl" else DIV_BETA, has_flux=has_flux, **kw)


def _check_per_image(per_image, B):
    """per_image: B dicts of divergence / betaParam / flux / solver keywords (see solve_batch)."""
    if not isinstance(per_image, (list, tuple)) or len(per_image) != B:
        raise ValueError(f"per_image must be a list of {B} dicts, one per image")
    for i, row in enumerate(per_image):
        if not isinstance(row, dict):
            raise ValueError(f"per_image[{i}] must be a dict of keyword arguments")
        unknown = set(row) - set(_ROW_KEYS)
        if unknown:
            raise TypeError(f"per_image[{i}]: unexpected keyword argument(s): {sorted(unknown)}")
        if row.get("divergence", "kl") not in ("kl", "beta"):
            raise ValueError(f"per_image[{i}]: divergence must be 'kl' or 'beta'")


def _size(a):
    return int(a.numel()) if _is_tensor(a) else int(np.size(a))


def _source_map(source, gn, psf, bkg, flux, betaParam, x0, obj):
    """solve_batch(source=...): the map as a contiguous host int32 array, after the shape rules of shared observations.
    gn, bkg, x0, obj and the PSF hold one entry per observation (gn.shape[0] of them); flux and betaParam one per solve."""
    s = source.detach().cpu().numpy() if _is_tensor(source) else np.asarray(source)
    if s.ndim != 1 or s.size < 1 or not np.issubdtype(s.dtype, np.integer):
        raise ValueError("source must be a non-empty 1-D integer array: one observation index per solve")
    if _ndim(gn) != 3:
        raise ValueError("gn must be [n_sources, ny, nx] with a source map")
    n, B = int(gn.shape[0]), int(s.size)
    bad = np.nonzero((s < 0) | (s >= n))[0]
    if bad.size:
        i = int(bad[0])
        raise ValueError(f"source[{i}] = {int(s[i])} is outside 0..{n - 1}: gn holds {n} observations")
    if psf is not None and _ndim(psf) == 3 and int(psf.shape[0]) not in (1, n):
        raise ValueError(f"psf has {int(psf.shape[0])} images; with a source map it is one image or one per observation ({n})")
    nb = _ndim(bkg)
    if (nb == 3 and int(bkg.shape[0]) != n) or nb == 2 or (nb == 1 and _size(bkg) not in (1, n)):
        raise ValueError(f"bkg must be a scalar, [{n}] or [{n}, ny, nx] (one per observation) with a source map; got shape "
                         f"{tuple(bkg.shape)}")
    for name, a in (("x0", x0), ("obj", obj)):
        if a is not None and (_ndim(a) != 3 or int(a.shape[0]) != n):
            raise ValueError(f"{name} must be [{n}, ny, nx] (one per observation) with a source map; got shape {tuple(a.shape)}")
    for name, a in (("flux", flux), ("betaParam", betaParam)):
        if a is not None and _size(a) not in (1, B):
            raise ValueError(f"{name} is per solve: a scalar or [{B}] with a source map of {B} solves; got {_size(a)} values")
    return np.ascontiguousarray(s, dtype=np.int32)


def _row_betas(betaParam, per_image, B):
    """The call's betaParam with the per-image overrides of per_image, as a host [B] array; betaParam itself if no row
    sets one (a device tensor then stays on the device)."""
    if not any("betaParam" in row for row in per_image):
        return betaParam
    base = betaParam.detach().cpu().numpy() if _is_tensor(betaParam) else betaParam
    b = np.array(np.broadcast_to(np.asarray(base, dtype=np.float64).reshape(-1), (B,)))
    for i, row in enumerate(per_image):
        if "betaParam" in row:
            b[i] = float(row["betaParam"])
    return b


def _row_flux(flux, per_image, B):
    """(flux, per_image) with the per-image overrides of per_image: a row's "flux" (a number, or None for
    sum(gn - bkg)) replaces the call's for that image.  If any row sets one, the flux comes back as a host [B] array and
    every row carries its own "flux" entry; otherwise both come back unchanged."""
    if not any("flux" in row for row in per_image):
        return flux, per_image
    base = None if flux is None else np.broadcast_to(np.asarray(flux.detach().cpu().numpy() if _is_tensor(flux) else flux,
                                                                 dtype=np.float64).reshape(-1), (B,))
    rows = [dict(row) if "flux" in row else dict(row, flux=None if base is None else float(base[i])) for i, row in enumerate(per_image)]
    return np.array([0.0 if row["flux"] is None else float(row["flux"]) for row in rows]), rows


# The solve's outputs besides the restored images, in the order of struct bsgp_outputs: (field, shape for B images and
# T = MAXIT + 1, dtype, present only with).  The trace_* arrays come back as BatchResult.trace under _TRACE_KEYS.
_OUTPUTS = (
    ("iters", lambda B, T: (B,), np.int32, None),
    ("status", lambda B, T: (B,), np.int32, None),
    ("discr", lambda B, T: (B, T), np.float64, None),
    ("times", lambda B, T: (B, T), np.float64, None),
    ("stop_value", lambda B, T: (B, T), np.float64, None),
    ("err", lambda B, T: (B, T + 1), np.float64, "errflag"),
    ("beta_final", lambda B, T: (B,), np.float64, None),
    ("proj_evals", lambda B, T: (B,), np.int32, None),
    ("ls_trials", lambda B, T: (B,), np.int32, None),
    ("scalars", lambda B, T: (B, _capi.NSCALARS), np.float64, None),
    ("trace_alpha", lambda B, T: (B, T), np.float64, "trace"),
    ("trace_lambda", lambda B, T: (B, T), np.float64, "trace"),
    ("trace_beta", lambda B, T: (B, T), np.float64, "trace"),
    ("trace_trials", lambda B, T: (B, T), np.int32, "trace"),
    ("trace_evals", lambda B, T: (B, T), np.int32, "trace"),
)
_TRACE_KEYS = {"trace_alpha": "alpha", "trace_lambda": "lam", "trace_beta": "beta", "trace_trials": "trials", "trace_evals": "evals"}


def _ptr(a):
    return None if a is None else (a.data_ptr() if _is_tensor(a) else a.ctypes.data)


def _ndim(a):
    return a.dim() if _is_tensor(a) else np.ndim(a)


def _torch_dtype(dt):
    import torch
    return {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32, np.dtype(np.int32): torch.int32}[np.dtype(dt)]


def _host_vector(a, B, dtype):
    """A scalar or [B] array -> contiguous numpy [B] of `dtype` (the numpy and pinned routes)."""
    return np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=dtype).reshape(-1), (B,)))


def _plan_for(plan, gn, dtype, device, same_device=False):
    """The caller's plan, or the cached one for gn; it must fit gn's shape and dtype (and device, for device tensors)."""
    if gn.ndim != 3:
        raise ValueError("gn must be [batch, ny, nx]")
    _, ny, nx = gn.shape
    plan = plan or get_plan(ny, nx, dtype, device)
    if (plan.ny, plan.nx, plan.dtype) != (ny, nx, dtype) or (same_device and plan.device != device):
        raise ValueError(f"plan is for {plan.ny}x{plan.nx} {plan.dtype} images on cuda:{plan.device}, gn is {ny}x{nx} {dtype}")
    return plan


class _Args:
    """The arguments of one solve, normalised the same way on every route: the parameters, the PSF on the plan, bkg (an
    image stack, or one value per image), flux and betaParam per image, x0 / obj, and the outputs of _OUTPUTS.  The route
    supplies `psf_arg` (the PSF as it hands it to the plan), `image(a, name)` (a [B,ny,nx] array converted and checked),
    `vector(a, B, dtype)` (a scalar or [B] array as a contiguous [B] array of a numpy dtype) and `alloc(shape, dtype)`."""

    def __init__(self, gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, kw, *, psf_arg, image,
                 vector, alloc, per_image=None, source=None, snapshot_every=0, snap_alloc=None):
        # B solves of n_obs observations: one each, or solve i of observation source[i] (_source_map)
        n_obs = int(gn.shape[0])
        B = self.B = n_obs if source is None else int(source.size)
        self.source, self.n_sources = source, (0 if source is None else n_obs)
        self.params = p = _params(divergence, kw, flux is not None)
        # a mixed batch: one bsgp_params per image, its own keywords merged over the call's (betaParam: see _row_betas)
        self.rows, self.is_beta, rows = None, None, [p]
        if per_image is not None:
            rows = [_params(r.get("divergence", divergence), {**kw, **{k: v for k, v in r.items() if k not in ("divergence", "betaParam", "flux")}},
                            r["flux"] is not None if "flux" in r else flux is not None) for r in per_image]
            self.rows = (_capi.Params * B)(*rows)
            self.is_beta = np.array([r.divergence == DIV_BETA for r in rows])
        if not psf_is_set and plan.set_psf(psf_arg(psf)) not in (1, n_obs):
            raise ValueError("psf must be one image or one per batch entry" if source is None else "psf must be one image or one per observation")
        self.gn, self.bkg_img, self.trace = gn, int(_ndim(bkg) == 3), trace
        self.bkg = image(bkg, "bkg") if self.bkg_img else vector(bkg, n_obs, _NP[plan.dtype])
        self.flux = None if flux is None else vector(flux, B, np.float64)
        self.beta0 = vector(betaParam, B, np.float64)
        self.x0 = None if x0 is None else image(x0, "x0")
        self.obj = None if obj is None else image(obj, "obj")
        if any(r.init_recon == 1 for r in rows) and self.x0 is None:
            raise ValueError("init_recon=1 needs x0 (the sgp()/sgp_betaDiv() wrappers draw it with seed 42)")
        present = {None: True, "errflag": any(r.errflag for r in rows), "trace": bool(trace)}
        stride = max(r.maxit for r in rows) + 1                 # the library's trace stride (include/bsgp.h, bsgp_outputs)
        self.out = {f: alloc(shape(B, stride), dt) if present[when] else None for f, shape, dt, when in _OUTPUTS}
        # iterate snapshots: n_snap slots per solve, NaN until the kernel writes them (include/bsgp.h, bsgp_outputs.snap_x)
        self.snap_every = int(snapshot_every)
        self.snapshots = self.snap_count = None
        if self.snap_every:
            self.snapshots = snap_alloc((B, snapshot_slots(stride - 1, self.snap_every)) + tuple(gn.shape[1:]))
            self.snap_count = alloc((B,), np.int32)

    def structs(self, x, order):
        """_capi.Inputs / _capi.Outputs for restored images `x` and the work-queue order (None: natural order).  The
        structs hold raw addresses, so the order is kept here, with the other arrays, for as long as the arguments live."""
        self.order = order
        ci = _capi.Inputs(_ptr(self.gn), _ptr(self.bkg), self.bkg_img, _ptr(self.flux), _ptr(self.beta0), _ptr(self.x0),
                          _ptr(self.obj), _ptr(order), _ptr(self.source), self.n_sources)
        return ci, _capi.Outputs(_ptr(x), *(_ptr(a) for a in self.out.values()), _ptr(self.snapshots), self.snap_every,
                                 _ptr(self.snap_count))

    def solve(self, plan, entry, ci, co, *stream):
        """bsgp_solve_batch<entry> with the shared keywords, or its bsgp_solve_batch_rows<entry> twin for a mixed batch."""
        L = lib()
        if self.rows is None:
            fn, prm = getattr(L, "bsgp_solve_batch" + entry), C.byref(self.params)
        else:
            fn, prm = getattr(L, "bsgp_solve_batch_rows" + entry), self.rows
        check(fn(plan.handle, prm, self.B, C.byref(ci), C.byref(co), *stream))

    def result(self, x):
        out = dict(self.out)
        trace = {key: out.pop(f) for f, key in _TRACE_KEYS.items()}
        return BatchResult(x=x, trace=trace if self.trace else None, snapshots=self.snapshots, snapshot_count=self.snap_count, **out)


def snapshot_slots(maxit, every):
    """Snapshot slots per solve: the iterates after 0, every, 2 * every, ... <= maxit passes (maxit: the largest MAXIT of
    the batch)."""
    return maxit // every + 1


def _check_snapshot_every(k):
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 0:
        raise ValueError(f"snapshot_every must be an integer >= 0 (0: no snapshots); got {k!r}")
    return int(k)


def solve_batch(gn, psf, bkg, divergence="beta", flux=None, betaParam=1.005, x0=None, obj=None, dtype="float64",
                device=0, trace=False, plan=None, psf_is_set=False, padded=False, x_out=None, per_image=None, source=None,
                snapshot_every=0, **kw):
    """Restore a batch of independent images in one persistent kernel launch.

    gn [B,ny,nx]; psf [ny,nx] (shared) or [B,ny,nx]; bkg scalar, [B] or [B,ny,nx]; flux None or [B];
    betaParam scalar or [B].  Keyword arguments are those of sgp()/sgp_betaDiv() (sgp.py:41-47,
    506-513).  numpy in -> numpy out; CUDA tensors in -> CUDA tensors out (asynchronous on the
    current stream); PINNED CPU tensors in -> pinned CPU tensors out through the pipelined host path
    (upload, solve and download overlap; see bsgp_solve_batch_pinned in include/bsgp.h; ``x_out`` may name a
    pinned tensor that receives the restored images, so that a caller in a loop reuses its buffer); pageable CPU tensors
    are treated like numpy arrays.  ``padded=True`` selects the zero-padded operator of
    use_original_SGP_Afunction=False (sgp.py:121-161): images of any size, kernel of any (smaller or equal) size.

    ``per_image``: a list of B dicts, one per image, of ``divergence``, ``betaParam``, ``flux`` and any solver keyword, each merged
    over the call's own: images with different keywords (KL and beta-SGP, stop rule, MAXIT, projection, saturation, ...)
    share one launch, and image i is exactly the solve of that image alone with its merged keywords.  The trace outputs
    are then [B, max MAXIT + 1]; entries past an image's own iteration count stay zero.  Keywords that describe the
    operator (region, div_a, div_at, adjoint_second_psf) must be the same in every row.

    ``source``: shared observations.  A [B] integer array (host memory): solve i restores observation source[i], so
    several solves of one image (a beta sweep, KL and beta-SGP runs of one sub-frame) carry its pixels and its PSF once.
    gn is then [n_sources, ny, nx]; bkg a scalar, [n_sources] or [n_sources, ny, nx]; psf one image or [n_sources, ...];
    x0 and obj [n_sources, ...].  flux, betaParam and per_image stay per solve, and the result has B entries, each
    bit-identical to the same solve with its observation replicated (gn[source], ...).

    ``snapshot_every``: k >= 1 keeps every k-th iterate of each solve, stored by the kernel as it runs, so that picking
    the iteration to keep (the restored image starts to amplify noise past some iteration) costs one launch.
    ``BatchResult.snapshots`` is [B, n_snap, ny, nx] in the dtype of x (numpy or tensor like x), n_snap = max MAXIT // k
    + 1.  Slot j belongs to iteration j * k: it is the image x of the same solve run with MAXIT = j * k + 1 (stop rule
    1), bit for bit, and slot 0 is the start image after the initial projection.  ``BatchResult.snapshot_count`` [B]
    says how many slots each solve wrote (1 + passes // k); the slots after them are NaN.  Memory: B * n_snap * ny * nx
    values.  Not supported with pinned CPU tensors (ValueError)."""
    if divergence not in ("kl", "beta"):
        raise ValueError("divergence must be 'kl' or 'beta'")
    snapshot_every = _check_snapshot_every(snapshot_every)
    if snapshot_every and _is_tensor(gn) and not gn.is_cuda and gn.is_pinned() and not padded:
        raise ValueError("snapshot_every is not supported with pinned CPU tensors (the pipelined host path); pass CUDA "
                         "tensors or numpy arrays")
    if source is not None:
        source = _source_map(source, gn, psf, bkg, flux, betaParam, x0, obj)
    B = int(gn.shape[0]) if source is None else int(source.size)
    if per_image is not None:
        _check_per_image(per_image, B)
        betaParam = _row_betas(betaParam, per_image, B)
        flux, per_image = _row_flux(flux, per_image, B)
    if padded:
        if _is_tensor(gn) and not gn.is_cuda:             # CPU tensors (pinned or not) take the numpy route of the padded operator
            def host(a):
                return a.numpy() if _is_tensor(a) and not a.is_cuda else a
            gn, psf, bkg, flux, betaParam, x0, obj = (host(a) for a in (gn, psf, bkg, flux, betaParam, x0, obj))
            x_out = None
        if per_image is not None and any(k in row for row in per_image for k in _OPERATOR_KEYS):
            raise ValueError("per_image rows of the padded operator share its geometry: region, div_a, div_at and "
                             "adjoint_second_psf are set by padded=True")
        return _solve_batch_padded(gn, psf, bkg, divergence, flux, betaParam, x0, obj, dtype, device, trace, per_image, source,
                                   snapshot_every, kw)
    if x_out is not None and not (_is_tensor(gn) and not gn.is_cuda and gn.is_pinned()):
        raise ValueError("x_out is only supported with pinned CPU tensor inputs")
    if _is_tensor(gn) and not gn.is_cuda and gn.is_pinned():
        return _solve_batch_pinned(gn, psf, bkg, divergence, flux, betaParam, x0, obj, device, trace, plan, psf_is_set, x_out, per_image,
                                   source, kw)
    if _is_tensor(gn) and gn.is_cuda:
        return _solve_batch_device(gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, per_image, source,
                                   snapshot_every, kw)
    if _is_tensor(gn):                                    # pageable CPU tensor: the plain host path
        gn = gn.numpy()
        psf, bkg, flux, betaParam, x0, obj = (a.numpy() if _is_tensor(a) and not a.is_cuda else a for a in (psf, bkg, flux, betaParam, x0, obj))
    return _solve_batch_host(gn, psf, bkg, divergence, flux, betaParam, x0, obj, dtype, device, trace, plan, psf_is_set, per_image, source,
                             snapshot_every, kw)


def _solve_batch_padded(gn, psf, bkg, divergence, flux, betaParam, x0, obj, dtype, device, trace, per_image, source, snapshot_every, kw):
    """Embed into the padded grid, solve there with the window mask, crop (see PaddedGeometry).  numpy inputs give
    numpy outputs; CUDA-tensor images stay on the device (the small kernels may be numpy or tensors).  With a source map
    the observations and their kernels are embedded once each."""
    on_dev = _is_tensor(gn)
    if on_dev:
        import torch
        dtype = {torch.float64: "float64", torch.float32: "float32"}[gn.dtype]
        device = gn.device.index or 0
    npdt = _NP[dtype]
    if not on_dev:
        gn = np.asarray(gn, dtype=npdt)
    if gn.ndim != 3:
        raise ValueError("gn must be [batch, ny, nx]")
    B, ny, nx = gn.shape
    psf_h = psf.detach().cpu().numpy() if _is_tensor(psf) else np.asarray(psf)
    psf_h = np.asarray(psf_h, dtype=np.float64)
    geo = PaddedGeometry(ny, nx, psf_h.shape[-2], psf_h.shape[-1])
    if geo.P > 16384:
        raise ValueError(f"padded grid {geo.P} exceeds the largest supported side (16384)")
    plan = get_plan(geo.P, geo.P, dtype, device)
    big, div_a = geo.kernel(psf_h, npdt)
    bigt, div_at = geo.kernel(np.conj(np.swapaxes(psf_h, -1, -2)), npdt)          # psf.conj().T, sgp.py:157
    extra = dict(region=geo.region, div_a=div_a, div_at=div_at, adjoint_second_psf=True)
    dt = gn.dtype if on_dev else npdt
    with torch.cuda.device(gn.device) if on_dev else contextlib.nullcontext():
        if on_dev:
            big, bigt = torch.as_tensor(big, device=gn.device), torch.as_tensor(bigt, device=gn.device)
        if plan.set_psf(big) not in (1, B) or plan.set_psf_adjoint(bigt) not in (1, B):
            raise ValueError("psf must be one kernel or one per batch entry" if source is None else "psf must be one kernel or one per observation")
        res = solve_batch(geo.embed(gn, dt), None, geo.embed(bkg, dt) if _ndim(bkg) == 3 else bkg, divergence=divergence,
                          flux=flux, betaParam=betaParam, x0=None if x0 is None else geo.embed(x0, dt),
                          obj=None if obj is None else geo.embed(obj, dt), dtype=dtype, device=device, trace=trace, plan=plan,
                          psf_is_set=True, per_image=per_image, source=source, snapshot_every=snapshot_every, **extra, **kw)
    x = res.x[:, geo.rows, geo.cols]
    res.x = x.contiguous() if on_dev else np.ascontiguousarray(x)
    if res.snapshots is not None:                          # grid-sized like x: cropped the same way
        sn = res.snapshots[..., geo.rows, geo.cols]
        res.snapshots = sn.contiguous() if on_dev else np.ascontiguousarray(sn)
    return res


def _solve_batch_host(gn, psf, bkg, divergence, flux, betaParam, x0, obj, dtype, device, trace, plan, psf_is_set, per_image, source,
                      snapshot_every, kw):
    """numpy arrays -> numpy arrays; one call of bsgp_solve_batch_host."""
    npdt = _NP[dtype]
    gn = np.ascontiguousarray(gn, dtype=npdt)
    plan = _plan_for(plan, gn, dtype, device)

    def image(a, name):
        a = np.ascontiguousarray(a, dtype=npdt)
        if a.shape != gn.shape:
            raise ValueError(f"{name} has shape {a.shape}; expected the shape of gn {gn.shape}")
        return a

    args = _Args(gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, kw,
                 psf_arg=lambda a: a, image=image, vector=_host_vector, alloc=np.zeros, per_image=per_image, source=source,
                 snapshot_every=snapshot_every, snap_alloc=lambda shape: np.full(shape, np.nan, npdt))
    x = np.empty((args.B,) + gn.shape[1:], npdt)
    ci, co = args.structs(x, _queue_order(divergence, args.beta0, args.is_beta))
    args.solve(plan, "_host", ci, co)
    return args.result(x)


def _solve_batch_device(gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, per_image, source, snapshot_every,
                        kw):
    """CUDA tensors -> CUDA tensors, asynchronous on the current stream: no host synchronisation, no host copies."""
    import torch
    if not gn.is_cuda:
        raise BsgpError("tensor inputs must live on a CUDA device (there is no CPU path)")
    dev = gn.device
    if gn.dtype not in (torch.float64, torch.float32):
        raise ValueError("gn must be float64 or float32")
    dtype = {torch.float64: "float64", torch.float32: "float32"}[gn.dtype]
    plan = _plan_for(plan, gn, dtype, dev.index or 0, same_device=True)
    gn = gn.contiguous()

    def image(t, name):
        """[B,ny,nx] tensor of gn's dtype on gn's device (raw pointers go to the library: a short or foreign array would be read out of bounds)"""
        if not _is_tensor(t):
            t = torch.as_tensor(np.ascontiguousarray(t), device=dev)
        if t.device != dev or tuple(t.shape) != tuple(gn.shape):
            raise ValueError(f"{name} must have the shape {tuple(gn.shape)} of gn and live on {dev}; got {tuple(t.shape)} on {t.device}")
        return t.to(gn.dtype).contiguous()

    def vector(a, B, dt):
        t = (a if _is_tensor(a) else torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev)).to(_torch_dtype(dt))
        if t.device != dev:
            raise ValueError(f"bkg, flux and betaParam must live on gn's device {dev}; got {t.device}")
        return t.reshape(-1).expand(B).contiguous()

    def psf_arg(a):
        return a if _is_tensor(a) else torch.as_tensor(np.ascontiguousarray(a), dtype=gn.dtype, device=dev)

    with torch.cuda.device(dev):
        args = _Args(gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, kw, psf_arg=psf_arg,
                     image=image, vector=vector, alloc=lambda shape, dt: torch.zeros(shape, dtype=_torch_dtype(dt), device=dev),
                     per_image=per_image, source=source, snapshot_every=snapshot_every,
                     snap_alloc=lambda shape: torch.full(shape, float("nan"), dtype=gn.dtype, device=dev))
        x = torch.empty((args.B,) + tuple(gn.shape[1:]), dtype=gn.dtype, device=dev)
        order = None
        if args.is_beta is not None and args.is_beta.any() and args.B > 1:
            # mixed batch: beta-SGP images by |beta - 1|, then the KL images (see _queue_order)
            kl = torch.as_tensor(~args.is_beta, device=dev)
            key = torch.where(kl, torch.full_like(args.beta0, float("inf")), (args.beta0 - 1.0).abs())
            order = torch.argsort(key, stable=True).to(torch.int32)
        elif args.is_beta is None and divergence == "beta" and args.B > 1:
            # longest expected solve first (see _queue_order); computed on the device, no host sync
            order = torch.argsort((args.beta0 - 1.0).abs(), stable=True).to(torch.int32)
        ci, co = args.structs(x, order)
        args.solve(plan, "", ci, co, _stream_ptr())
        res = args.result(x)
        res._keepalive = (gn, args.bkg, args.flux, args.beta0, args.x0, args.obj, args.order)
    return res


def _solve_batch_pinned(gn, psf, bkg, divergence, flux, betaParam, x0, obj, device, trace, plan, psf_is_set, x_out, per_image, source, kw):
    """Page-locked CPU tensors -> page-locked CPU tensors; one call of bsgp_solve_batch_pinned (returns when the results
    are in host memory).  `device` selects the GPU.  Image-shaped arguments (bkg stack, x0, obj) must be pinned too."""
    import torch
    dtype = {torch.float64: "float64", torch.float32: "float32"}[gn.dtype]
    gn = gn.contiguous()
    plan = _plan_for(plan, gn, dtype, device)

    def pinned(t, name):
        if not (_is_tensor(t) and not t.is_cuda and t.is_pinned() and t.dtype == gn.dtype and tuple(t.shape) == tuple(gn.shape)):
            raise ValueError(f"{name} must be a pinned CPU tensor of the shape and dtype of gn")
        return t.contiguous()

    def psf_arg(a):
        return (a if _is_tensor(a) else torch.as_tensor(np.ascontiguousarray(a))).to(device=f"cuda:{plan.device}", dtype=gn.dtype, non_blocking=True)

    # the small outputs are page-locked as well (torch's caching host allocator makes repeated calls cheap), handed
    # back as numpy views: the copies behind the kernel run at full PCIe speed and never block on a staging buffer
    def hbuf(shape, dt):
        return torch.empty(shape, dtype=_torch_dtype(dt), pin_memory=True).numpy()

    with torch.cuda.device(plan.device):
        args = _Args(gn, psf, bkg, divergence, flux, betaParam, x0, obj, trace, plan, psf_is_set, kw, psf_arg=psf_arg,
                     image=pinned, vector=_host_vector, alloc=hbuf, per_image=per_image, source=source)
        xshape = (args.B,) + tuple(gn.shape[1:])
        if x_out is None:
            x = torch.empty(xshape, dtype=gn.dtype, pin_memory=True)
        else:
            x = x_out
            if not (_is_tensor(x) and not x.is_cuda and x.is_pinned() and x.dtype == gn.dtype and tuple(x.shape) == xshape and x.is_contiguous()):
                raise ValueError("x_out must be a contiguous pinned CPU tensor of the dtype of gn, one image per solve")
        ci, co = args.structs(x, _queue_order(divergence, args.beta0, args.is_beta))
        args.solve(plan, "_pinned", ci, co, _stream_ptr())
    res = args.result(x)
    for i in np.nonzero(res.status == _capi.ST_INPUT_TIMEOUT)[0]:      # skipped images: defined (zero) pixels, status says why
        x[int(i)].zero_()
    return res


def project_batch(b, c, dia, sat_cap=None, lambda_=0.0, dlambda_=1.0, tol_lam=1e-11, max_projs=1000, biter=0, siter=0, device=0):
    """projectDF for a batch of problems: c, dia [B,n]; b [B] (flux_conserve_proj.py:7-144)."""
    c = np.ascontiguousarray(c, dtype=np.float64)
    dia = np.ascontiguousarray(dia, dtype=np.float64)
    if c.ndim == 1:
        c, dia = c[None], dia[None]
    if c.ndim != 2 or dia.shape != c.shape:
        raise ValueError(f"c and dia must both be [B, n]; got {c.shape} and {dia.shape}")
    B, n = c.shape
    b = np.ascontiguousarray(np.broadcast_to(np.asarray(b, dtype=np.float64).reshape(-1), (B,)))
    x = np.empty_like(c)
    ev = np.zeros(B, np.int32)
    st = np.zeros(B, np.int32)
    cap = float("nan") if sat_cap is None else float(sat_cap)
    check(lib().bsgp_project_df_host(b.ctypes.data, c.ctypes.data, dia.ctypes.data, n, B, cap, float(lambda_), float(dlambda_),
                                     float(tol_lam), int(max_projs), int(biter), int(siter), x.ctypes.data, ev.ctypes.data, st.ctypes.data,
                                     int(device)))
    return x, ev, st
