"""Cost of iterate snapshots (solve_batch(snapshot_every=k)) on the reference's subdivision call set: 64 sub-frames of
256 x 256 from a 2048 x 2048 field, five beta initialisations each (320 beta-SGP solves, synth.TILE_KWARGS: stop rule 3,
MAXIT = 500), fp64 CUDA tensors, one plan.

Four launches of the same solves, alternating, `--reps` times each after one warm-up:
  plain    the launch without rows (the kernels compiled without them);
  rows     the same keywords as equal per_image rows (the mixed-batch kernels, no snapshots);
  snap10   snapshot_every = 10;
  snap1    snapshot_every = 1.
Per launch: the call time (CUDA events around solve_batch on its stream: for the snapshot launches this includes filling
the snapshot array with NaN) and, in a separate profiled pass, the solve kernel's own time (torch.profiler, CUDA
activities).  Medians are reported.  The snapshot bytes are computed from the shapes: allocated (B * n_snap * N * 8) and
written (sum over solves of snapshot_count * N * 8).  Checks that x, iters and discr are bit-identical across the four
launches.  Prints the card's name and power limit and writes a JSON record with --out.  Needs a GPU.
Usage: python tools/snapshot_probe.py [--reps 3] [--variants plain,rows,snap10,snap1] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import beta_sgp_b200 as bs  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--variants", default="plain,rows,snap10,snap1", help="a subset, e.g. plain,rows against an older library")
    args = ap.parse_args()
    w = bs.synth.field_tiles(size=2048, tile=256, seed=2024, n_beta=5)
    dev = torch.device("cuda:0")
    gn, bkg = (torch.as_tensor(w[k], device=dev) for k in ("gn", "bkg"))
    psf = torch.as_tensor(w["psf"], device=dev)
    flux, beta0 = (torch.as_tensor(w[k], device=dev) for k in ("flux", "beta0"))
    B, N = int(gn.shape[0]), int(gn.shape[1] * gn.shape[2])
    kw = dict(bs.synth.TILE_KWARGS)
    plan = bs.Plan(256, 256, "float64")
    plan.set_psf(psf)
    variants = {"plain": {}, "rows": dict(per_image=[{}] * B), "snap10": dict(snapshot_every=10), "snap1": dict(snapshot_every=1)}
    variants = {k: variants[k] for k in args.variants.split(",")}

    def run(name):
        return bs.solve_batch(gn, None, bkg, divergence="beta", flux=flux, betaParam=beta0, plan=plan, psf_is_set=True,
                              **variants[name], **kw)

    call_ms, kern_ms, snaps = {k: [] for k in variants}, {k: [] for k in variants}, {}
    ref = run("plain")                                                  # warm-up, and the bits every launch must give
    for name in variants:
        run(name)
    torch.cuda.synchronize()

    def check(name, r):
        for f in ("x", "iters", "discr"):
            assert torch.equal(getattr(r, f), getattr(ref, f)), (name, f)
        if r.snapshots is not None:
            snaps[name] = (int(r.snapshots.shape[1]), int(r.snapshot_count.sum()))

    for _ in range(args.reps):
        for name in variants:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = run(name)
            e1.record()
            torch.cuda.synchronize()
            call_ms[name].append(e0.elapsed_time(e1))
            check(name, r)
            del r                                                       # snap1 holds B * 501 images: one at a time
    # the solve kernel alone, in a profiled pass of its own
    from torch.profiler import ProfilerActivity, profile
    for _ in range(args.reps):
        for name in variants:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                r = run(name)
                torch.cuda.synchronize()
            del r
            kern_ms[name].append(sum(e.time_range.elapsed_us() for e in prof.events() if "bsgp_solve_kernel" in e.name) / 1e3)
    rec = dict(card=card(), call_set="subdivisions: 64 sub-frames of 256 x 256, five beta each (synth.TILE_KWARGS), fp64",
               solves=B, iterations=int(ref.iters.sum()), reps=args.reps, bit_identical=True,
               call_ms_median={k: float(np.median(v)) for k, v in call_ms.items()}, call_ms=call_ms,
               kernel_ms_median={k: float(np.median(v)) for k, v in kern_ms.items()}, kernel_ms=kern_ms)
    for name, (n_snap, written) in snaps.items():
        rec[f"{name}_slots"] = n_snap
        rec[f"{name}_bytes_allocated"] = B * n_snap * N * 8
        rec[f"{name}_bytes_written"] = written * N * 8
    print(json.dumps(rec, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
    plan.close()


if __name__ == "__main__":
    main()
