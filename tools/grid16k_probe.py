"""Frame plans on 16384-point grids against the 8192^2 frame: ms per iteration by CUDA events, algorithmic bytes per
iteration (the SURVEY.md §8(d) model of bench.py, on the FFT grid's pixel count, plus 2 N w bytes per convolution for the
split transforms of fp64 16384-point columns: DESIGN.md section 4), and the fraction of the HBM bandwidth measured in the same
call (a device-to-device copy of 4 GiB).  Cases: 16384^2 and 6000^2 (wrapped on 16384^2) in fp64 and fp32, and 8192^2 fp64 /
fp32, run in alternation, so that the 8192^2 times are taken under the same conditions as the new ones.
Inputs are resident in HBM and far larger than L2.  Per iteration = the difference of a MAXIT = 8 and a MAXIT = 3 solve over
5 iterations, so the set-up passes cancel.  Records the card's name and power limit.  Needs a GPU.
Usage: python tools/grid16k_probe.py [--rounds 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import beta_sgp_b200 as bs  # noqa: E402
from bench import algorithmic_bytes  # noqa: E402

CASES = [("8192^2 fp64", (8192, 8192), "float64"), ("16384^2 fp64", (16384, 16384), "float64"), ("6000^2 fp64", (6000, 6000), "float64"),
         ("16384^2 fp32", (16384, 16384), "float32"), ("6000^2 fp32", (6000, 6000), "float32"), ("8192^2 fp32", (8192, 8192), "float32")]
CONVS_PER_ITER = 2          # A(d) of the search direction and A^T of the new gradient (bsgp_solver.cuh, solve_image)
SHORT, LONG = 3, 8


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def hbm_gbs(dev, reps=10):
    """device-to-device copy of 4 GiB: 2 x 4 GiB of HBM traffic per copy"""
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * a.numel() * 4 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def inputs(shape, dtype, dev, seed):
    """a star field (0.1 % of the pixels) over a sky of 300, Poisson noise, and a Gaussian PSF (FWHM 3.5), on the device"""
    g = torch.Generator(device=dev).manual_seed(seed)
    tdt = torch.float64 if dtype == "float64" else torch.float32
    lam = torch.full(shape, 300.0, dtype=torch.float64, device=dev)
    k = shape[0] * shape[1] // 1000
    idx = torch.randint(0, shape[0] * shape[1], (k,), generator=g, device=dev)
    lam.view(-1)[idx] += 10.0 ** (3.0 + 2.0 * torch.rand(k, generator=g, device=dev, dtype=torch.float64))
    gn = torch.poisson(lam, generator=g).to(tdt)
    yy = torch.arange(shape[0], device=dev, dtype=torch.float64)[:, None] - shape[0] // 2
    xx = torch.arange(shape[1], device=dev, dtype=torch.float64)[None, :] - shape[1] // 2
    s = 3.5 / 2.3548
    psf = torch.exp(-(yy ** 2 + xx ** 2) / (2 * s * s))
    psf = (psf / psf.sum()).to(tdt)
    flux = float((gn.double() - 300.0).sum())
    return gn[None].contiguous(), psf, flux


def solve(w, maxit):
    gn, psf, flux, dtype = w
    kw = dict(bs.synth.TILE_KWARGS, stop_criterion=1, MAXIT=maxit)
    bkg = torch.tensor(300.0, dtype=gn.dtype, device=gn.device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = bs.solve_batch(gn, psf, bkg, divergence="beta", flux=[flux], betaParam=1.0248357, trace=True, **kw)
    e1.record()
    torch.cuda.synchronize()
    assert int(r.status[0]) == 0 and int(r.iters[0]) == maxit, (int(r.status[0]), int(r.iters[0]))
    return e0.elapsed_time(e1), r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    out = {"card": card(), "hbm_copy_gbs": hbm_gbs(dev), "cases": {}}
    work = {}
    for name, shape, dtype in CASES:
        gn, psf, flux = inputs(shape, dtype, dev, seed=shape[0] + len(dtype))
        work[name] = (gn, psf, flux, dtype)
        solve(work[name], SHORT)                                           # plan set-up, module load
        info = bs.get_plan(shape[0], shape[1], dtype, 0).info()
        out["cases"][name] = {"shape": shape, "dtype": dtype, "grid": [info["grid_ny"], info["grid_nx"]], "ctas": info["cluster_size"],
                              "workspace_bytes": info["workspace_bytes"], "ms_per_iter": []}
    for rnd in range(args.rounds):
        for name, shape, dtype in CASES:
            t_s, _ = solve(work[name], SHORT)
            t_l, r = solve(work[name], LONG)
            c = out["cases"][name]
            c["ms_per_iter"].append((t_l - t_s) / (LONG - SHORT))
            if rnd == args.rounds - 1:
                tr = r.trace
                iters = np.arange(SHORT + 1, LONG + 1)
                host = {k: (v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in tr.items()}
                evals = host["evals"][0, SHORT + 1:LONG + 1].astype(np.float64)
                trials = host["trials"][0, SHORT + 1:LONG + 1].astype(np.float64)
                npix = c["grid"][0] * c["grid"][1]
                w = 8 if dtype == "float64" else 4
                split_cols = dtype == "float64" and c["grid"][0] == 16384
                c["algorithmic_bytes_per_iter"] = algorithmic_bytes(npix, w, np.ones_like(iters, dtype=np.float64), evals, trials,
                                                                    True, False) / (LONG - SHORT) + \
                    (2.0 * npix * w * CONVS_PER_ITER if split_cols else 0.0)
                c["split_extra_bytes_per_iter"] = 2.0 * npix * w * CONVS_PER_ITER if split_cols else 0.0
            print(name, f"round {rnd}: {c['ms_per_iter'][-1]:.2f} ms per iteration", flush=True)
    for c in out["cases"].values():
        c["ms_per_iter_median"] = float(np.median(c["ms_per_iter"]))
        c["achieved_gbs"] = c["algorithmic_bytes_per_iter"] / (c["ms_per_iter_median"] * 1e-3) / 1e9
        c["frac_of_measured_hbm"] = c["achieved_gbs"] / out["hbm_copy_gbs"]
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
