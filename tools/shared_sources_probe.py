"""Shared observations (solve_batch(source=...)) against replicated observations, on the reference's two call sets that
restore every observation several times, from page-locked host memory:

  stamps        S cut-outs of 31 x 31, each with its own PSF, times the five beta initialisations of synth.beta_inits()
                (application_sgp_star_stamps.py:69-105; synth.STAMP_KWARGS);
  subdivisions  the call set of tools/mixed_batch_probe.py: every 256 x 256 sub-frame restored five times with beta-SGP and
                once with KL-SGP in one mixed launch (application_sgp_subdivisions.py:69-115; synth.TILE_KWARGS).

Both formulations run on plans of their own, alternating, `--reps` times each after one warm-up.  Per run: the end-to-end
time (host clock from page-locked inputs to results in page-locked memory: PSF upload, bsgp_set_psf and the pipelined
solve), the bsgp_set_psf time alone (CUDA events), the bytes uploaded (computed from the shapes: observations, backgrounds
and PSFs), the PSF spectra and staged inputs the library holds (computed from the shapes), and torch's peak device memory
(torch.cuda.max_memory_allocated: the PSF tensors and torch's own buffers; the library's buffers are cudaMalloc'd and are
not in it).  Checks that both formulations return the same bits.  Prints the card's name and power limit and writes a JSON
record with --out.  Needs a GPU.  Usage: python tools/shared_sources_probe.py [--stamps 8192] [--tiles 64] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import beta_sgp_b200 as bs  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def stamps_call_set(S):
    """(observations, solves) of the star-stamp sweep: S stamps with per-stamp PSFs, five betas each (stamp-major)."""
    st = bs.synth.star_stamps(S, 31, seed=2031)
    betas = np.array(bs.synth.beta_inits())
    nb = betas.size
    obs = dict(gn=st["gn"], psf=st["psf"], bkg=st["bkg"])
    solves = dict(source=np.repeat(np.arange(S, dtype=np.int32), nb), flux=np.repeat(st["flux"], nb), betaParam=np.tile(betas, S),
                  per_image=None, kw=dict(bs.synth.STAMP_KWARGS))
    return obs, solves


def subdivisions_call_set(S):
    """(observations, solves) of the subdivisions call set: S sub-frames, five beta-SGP solves and one KL solve each."""
    w = bs.synth.field_tiles(size=2048, tile=256, seed=2024, n_beta=5, max_tiles=S)
    S = w["gn"].shape[0] // 5
    first = np.arange(S) * 5
    obs = dict(gn=w["gn"][first], psf=w["psf"], bkg=w["bkg"][first])
    src = np.concatenate([np.repeat(np.arange(S), 5), np.arange(S)]).astype(np.int32)
    kb = dict(bs.synth.TILE_KWARGS)
    per_image = [dict(divergence="beta")] * (5 * S) + [dict(divergence="kl")] * S     # the beta-only keywords do nothing in KL-SGP
    solves = dict(source=src, flux=np.concatenate([w["flux"], w["flux"][first]]), betaParam=np.concatenate([w["beta0"], np.full(S, 1.005)]),
                  per_image=per_image, kw=kb)
    return obs, solves


def run(plan, obs, solves, shared):
    """One end-to-end solve from page-locked memory; the PSFs go up and through bsgp_set_psf inside the timed region."""
    src = solves["source"]
    o = obs if shared else {k: (v[src] if v.ndim == 3 or k == "bkg" else v) for k, v in obs.items()}
    gn = pinned(o["gn"])
    bkg = pinned(o["bkg"]) if o["bkg"].ndim == 3 else o["bkg"]
    psf_h = pinned(o["psf"])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    psf_d = psf_h.to("cuda:0", non_blocking=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    plan.set_psf(psf_d)
    e1.record()
    r = bs.solve_batch(gn, None, bkg, divergence="beta", flux=solves["flux"], betaParam=solves["betaParam"], plan=plan, psf_is_set=True,
                       per_image=solves["per_image"], source=src if shared else None, **solves["kw"])
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    info = plan.info()
    n_psf = 1 if o["psf"].ndim == 2 else o["psf"].shape[0]
    img = gn[0].numel() * 8
    spectrum = (info["grid_nx"] // 2 + 1) * info["grid_ny"] * 16
    up = gn.numel() * 8 + (bkg.numel() * 8 if o["bkg"].ndim == 3 else np.size(o["bkg"]) * 8) + psf_h.numel() * 8
    row = dict(end_to_end_ms=1e3 * (t1 - t0), set_psf_ms=e0.elapsed_time(e1), bytes_uploaded=int(up), observations=int(gn.shape[0]),
               solves=int(src.size), psf_spectra_bytes=int(n_psf * spectrum),
               staged_input_bytes=int(gn.shape[0] * img * (2 if o["bkg"].ndim == 3 else 1)),
               torch_peak_bytes=int(torch.cuda.max_memory_allocated()))
    return row, r


def workload(name, obs, solves, reps):
    plans = {k: bs.Plan(obs["gn"].shape[1], obs["gn"].shape[2], "float64") for k in ("replicated", "shared")}
    out = {k: [] for k in plans}
    last = {}
    for rep in range(reps + 1):                                     # the first round warms both up
        for k in ("replicated", "shared"):
            row, last[k] = run(plans[k], obs, solves, k == "shared")
            if rep:
                out[k].append(row)
    a, b = last["replicated"], last["shared"]
    same = all(np.array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f))) for f in ("iters", "status", "discr", "beta_final")) \
        and torch.equal(a.x, b.x)
    res = dict(workload=name, bit_identical=bool(same), iters=[int(a.iters.min()), int(a.iters.max()), int(a.iters.sum())])
    for k, rows in out.items():
        res[k] = {f: (float(np.median([r[f] for r in rows])) if f.endswith("_ms") else rows[-1][f]) for f in rows[0]}
        res[k]["end_to_end_all_ms"] = [r["end_to_end_ms"] for r in rows]
    for p in plans.values():
        p.close()
    print(json.dumps(res), flush=True)
    if not same:
        raise SystemExit(f"{name}: shared and replicated observations gave different results")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stamps", type=int, default=8192)
    ap.add_argument("--tiles", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    c = card()
    print(json.dumps(dict(card=c)), flush=True)
    res = dict(card=c, workloads=[workload("stamps31x5", *stamps_call_set(args.stamps), args.reps),
                                  workload("subdivisions", *subdivisions_call_set(args.tiles), args.reps)])
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
