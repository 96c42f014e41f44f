"""beta-initialisation sweep as ONE batched call (application_sgp_star_stamps.py:69-105, application_sgp_subdivisions.py:69-115).

The reference restores every stamp five times, with betaParam drawn from N(1, 0.05) under five fixed seeds, measures the
restored source with photutils, keeps the beta whose ``flux_fractional_difference = 1 - restored_flux / original_flux``
is smallest (signed comparison, first minimum wins, :91-95) and then runs that beta a sixth time (:96-104).  Here the
S x 5 solves are one persistent-kernel launch, and the sixth run is not needed: the solver is deterministic, so the
selected run IS the re-run (tests/test_gpu_parity.py::test_beta_sweep_selection checks this bit for bit).

The selection metric of the reference needs photutils segmentation (absent offline); ``aperture_flux`` stands in for
``segment_flux``: background-subtracted sum inside a circular aperture around the brightest pixel.  It is an
APPROXIMATION of the reference's measurement — pass ``measure=`` to use another one.
"""
from __future__ import annotations

import numpy as np

from .engine import BatchResult, solve_batch
from .synth import beta_inits


def aperture_flux(images, bkg, radius=6.0):
    """images [B,ny,nx] (CUDA tensor), bkg [B] or [B,ny,nx] -> [B] background-subtracted aperture sums (fp64)."""
    import torch
    B, ny, nx = images.shape
    flat = images.reshape(B, -1)
    peak = flat.argmax(dim=1)
    py, px = (peak // nx).to(torch.float64), (peak % nx).to(torch.float64)
    yy = torch.arange(ny, device=images.device, dtype=torch.float64)[None, :, None]
    xx = torch.arange(nx, device=images.device, dtype=torch.float64)[None, None, :]
    mask = ((yy - py[:, None, None]) ** 2 + (xx - px[:, None, None]) ** 2) <= radius * radius
    b = bkg if bkg.dim() == 3 else bkg.reshape(B, 1, 1)
    return ((images.to(torch.float64) - b.to(torch.float64)) * mask).sum(dim=(1, 2))


def select_best(metric):
    """[S, nb] -> index of the selected beta per stamp: smallest value, first one on ties (strict '<' scan, :93-95)."""
    m = np.asarray(metric, dtype=np.float64)
    best = np.zeros(m.shape[0], dtype=np.int64)
    for s in range(m.shape[0]):
        cur = np.inf
        for k in range(m.shape[1]):
            if m[s, k] < cur:
                cur, best[s] = m[s, k], k
    return best


def sgp_betaDiv_sweep(gn, psf, bkg, flux=None, betas=None, measure=None, device=0, **kw):
    """gn [S,ny,nx]; psf [ny,nx] or [S,ny,nx]; bkg scalar / [S] / [S,ny,nx]; flux None or [S] (numpy or CUDA tensors).
    Returns (best: BatchResult of the selected runs [S], best_beta [S], best_index [S], metric [S,nb], sweep: BatchResult
    of all S x nb runs, stamp-major)."""
    import torch
    betas = np.asarray(beta_inits() if betas is None else betas, dtype=np.float64)
    nb = betas.size
    dev = torch.device("cuda", device)

    def dev_t(a, dtype=torch.float64):
        return (a if type(a).__module__.startswith("torch") else torch.as_tensor(np.ascontiguousarray(a))).to(dev, dtype)

    g = dev_t(gn)
    S, ny, nx = g.shape
    rep = lambda t: t.repeat_interleave(nb, dim=0)                      # noqa: E731  stamp-major: (s, k) -> s * nb + k
    source = np.repeat(np.arange(S, dtype=np.int32), nb)                # solve s * nb + k restores stamp s: one copy of each
    pt = dev_t(psf)
    bt = dev_t(bkg) if np.ndim(bkg) > 0 or type(bkg).__module__.startswith("torch") else torch.full((S,), float(bkg), dtype=torch.float64, device=dev)
    bt = bt.reshape(S) if bt.numel() == S else bt
    fb = None if flux is None else rep(dev_t(flux).reshape(S))
    b0 = torch.as_tensor(np.tile(betas, S), device=dev)
    kw.setdefault("proj_type", 1)
    res = solve_batch(g, pt, bt, divergence="beta", flux=fb, betaParam=b0, source=source, **kw)
    measure = measure or aperture_flux
    orig = rep(measure(g, bt))                                          # the original flux, measured once per stamp
    restored = measure(res.x, rep(bt))
    metric = (1.0 - restored / orig).reshape(S, nb).cpu().numpy()          # flux_fractional_difference, :90
    best = select_best(metric)
    idx = torch.as_tensor(np.arange(S) * nb + best, device=dev)
    pick = {}
    for f in ("x", "iters", "status", "discr", "times", "stop_value", "err", "beta_final", "proj_evals", "ls_trials", "scalars"):
        v = getattr(res, f)
        pick[f] = None if v is None else v.index_select(0, idx)
    return BatchResult(**pick), betas[best], best, metric, res
