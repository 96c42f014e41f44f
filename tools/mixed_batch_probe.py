"""One mixed launch against one launch per option set, on the subdivisions call set (application_sgp_subdivisions.py:69-115):
every 256 x 256 sub-frame of a synthetic crowded field restored five times with beta-SGP (the five beta initialisations,
adapt_beta=False, tol_convergence=1e-5, flux-conserving projection, synth.TILE_KWARGS) and once with KL-SGP (the same
keywords without the beta-only ones).  Reports the solve-kernel time of both ways by CUDA events (PSF spectra set outside
the timed region), the card's name and power limit, and checks that the mixed launch returns exactly what the two
launches return.  Needs a GPU.  Usage: python tools/mixed_batch_probe.py [--tiles 8 16 32 64] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import beta_sgp_b200 as bs  # noqa: E402

BETA_ONLY = ("lr", "lr_exp_param", "schedule_lr", "adapt_beta")


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, reps):
    """fn() once to warm up, then the median of `reps` event-timed calls (ms) and the last result."""
    fn()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), ms, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tiles", type=int, nargs="+", default=[8, 16, 32, 64])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    w = bs.synth.field_tiles(size=2048, tile=256, seed=2024, n_beta=5)
    kb = dict(bs.synth.TILE_KWARGS)
    kk = {k: v for k, v in kb.items() if k not in BETA_ONLY}
    plan = bs.get_plan(256, 256, "float64", 0)
    plan.set_psf(torch.as_tensor(w["psf"], device=dev))
    rows_out = []
    for S in args.tiles:
        nb = 5 * S                                          # field_tiles: five beta inits per tile, tile-major
        t = {k: torch.as_tensor(np.ascontiguousarray(w[k][:nb]), device=dev) for k in ("gn", "bkg", "flux", "beta0")}
        kl = {k: t[k][0:nb:5] for k in ("gn", "bkg", "flux")}          # one KL run per tile
        gn_m = torch.cat([t["gn"], kl["gn"]]); bkg_m = torch.cat([t["bkg"], kl["bkg"]]); flux_m = torch.cat([t["flux"], kl["flux"]])
        beta_m = torch.cat([t["beta0"], torch.full((S,), 1.005, dtype=torch.float64, device=dev)])
        per_image = [dict(divergence="beta")] * nb + [dict(divergence="kl")] * S       # the beta-only keywords do nothing in KL-SGP
        common = dict(plan=plan, psf_is_set=True)

        def two():
            rb = bs.solve_batch(t["gn"], None, t["bkg"], divergence="beta", flux=t["flux"], betaParam=t["beta0"], **common, **kb)
            rk = bs.solve_batch(kl["gn"], None, kl["bkg"], divergence="kl", flux=kl["flux"], **common, **kk)
            return rb, rk

        def mixed():
            return bs.solve_batch(gn_m, None, bkg_m, divergence="beta", flux=flux_m, betaParam=beta_m, per_image=per_image, **common, **kb)

        t2, t2_all, (rb, rk) = timed(two, args.reps)
        t1, t1_all, rm = timed(mixed, args.reps)
        same = bool(torch.equal(rm.x[:nb], rb.x) and torch.equal(rm.x[nb:], rk.x) and torch.equal(rm.iters[:nb], rb.iters)
                    and torch.equal(rm.iters[nb:], rk.iters))
        it_b, it_k = rb.iters.cpu().numpy(), rk.iters.cpu().numpy()
        row = dict(tiles=S, images=nb + S, two_launches_ms=t2, mixed_ms=t1, speedup=t2 / t1, two_all=t2_all, mixed_all=t1_all,
                   beta_iters=[int(it_b.min()), int(it_b.max()), int(it_b.sum())], kl_iters=[int(it_k.min()), int(it_k.max()), int(it_k.sum())],
                   bit_identical=same)
        print(json.dumps(row), flush=True)
        rows_out.append(row)
        if not same:
            raise SystemExit("the mixed launch differs from the two launches")
    res = dict(card=card(), slots=plan.info()["num_clusters"], rows=rows_out)
    print(json.dumps(dict(card=res["card"], slots=res["slots"])))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
