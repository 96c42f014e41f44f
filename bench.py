#!/usr/bin/env python
"""Benchmark of the beta-SGP restoration path (BASELINE.json metric: restored images/s and ms/iteration,
fraction of the HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload tiles256|stamps32|frame|ngc|sat]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE config 4 — a synthetic 2048x2048 crowded field split into 64
256x256 subdivisions, each solved for the 5 beta initialisations of the reference's application script
(application_sgp_subdivisions.py:69-107), i.e. 320 independent beta-SGP restorations with the
flux-conserving projection, a 2-D background map and one shared PSF.  One "step" = one pass of the hot
path over that batch (PSF spectrum + 320 solves + the gather of the results).

Multi-GPU (BASELINE: "sharded over 1/2/4/8 GPUs"): STRONG scaling.  Every rank holds the same 320-solve field,
restores its share through the product's multi-GPU entry point (solve_batch_sharded: cost-ranked dealing, CTA
width chosen from the local batch size) and the timed region ends when the NCCL all-gather has put all 320
restored images on every rank.  N = 1 is the same call without a process group.  The weak-scaling number of
independent replicas (round 1's SCALE) is kept under "replicas".

Extra key "workloads": the other BASELINE configs in brief (1: KL-SGP on NGC7027, 2: beta-SGP + projection on the
satellite simulation - single-image latency; 3: 8192 stamps; 5: one 8192^2 frame), each with value, ms per
iteration, roofline, cpu_baseline and e2e; at N > 1 the sharded stamp batch.

`--impl reference` times the reference's own CPU algorithm (the oracle port, oracle/sgp_oracle.py: numpy,
same FFT calls and operand order as restoration/sgp.py; the Python reference itself cannot travel to the
GPU box) on all host cores over a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:
    # the CPU arm runs one single-threaded numpy process per core; stop BLAS / OpenMP from oversubscribing them
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.setdefault(_v, "1")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tiles256", choices=["tiles256", "stamps32", "cutouts31", "frame", "ngc", "sat"])
    ap.add_argument("--no-extra", action="store_true", help="skip the brief runs of the other BASELINE configs (key 'workloads')")
    ap.add_argument("--width", default="auto", help="CTA configuration of the sharded solve: auto or cluster,threads")
    ap.add_argument("--field", type=int, default=2048, help="side of the synthetic field (tiles256)")
    ap.add_argument("--stamps", type=int, default=8192, help="number of stamps (stamps32)")
    ap.add_argument("--frame", type=int, default=8192, help="side of the single frame (workload frame, BASELINE config 5)")
    ap.add_argument("--maxit", type=int, default=10, help="iterations of the frame workload (stop_criterion=1)")
    ap.add_argument("--dtype", default="float64", choices=["float64", "float32"])
    ap.add_argument("--cluster", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="experiments: do not sample clocks during the timed region")
    ap.add_argument("--cpu-sample", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def make_workload(args, rank):
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bsgp_synth", os.path.join(ROOT, "beta-sgp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    if args.workload == "tiles256":
        w = synth.field_tiles(size=args.field, tile=256, seed=2024, n_beta=5)
        kw = dict(synth.TILE_KWARGS)
        name = (f"config4: {args.field}x{args.field} synthetic crowded field -> {len(w['gn']) // 5} subdivisions of 256x256 "
                f"(reference tiler utils.py:332-375, overlap 0) x 5 beta inits = {len(w['gn'])} beta-SGP solves, "
                "proj_type=1, 2-D bkg, shared PSF")
        return w, kw, name, True
    if args.workload == "frame":
        f = synth.single_frame(args.frame, seed=77)
        w = dict(gn=f["gn"][None], bkg=f["bkg"][None], psf=f["psf"], flux=np.array([f["flux"]]), beta0=np.array([1.0248357076505616]))
        kw = dict(synth.TILE_KWARGS, stop_criterion=1, MAXIT=args.maxit)
        name = (f"config5: one synthetic {args.frame}x{args.frame} crowded frame, beta-SGP, proj_type=1, 2-D bkg, frame-sized PSF, "
                f"{args.maxit} iterations (stop_criterion=1), frame mode (one image over the whole GPU)")
        return w, kw, name, True
    if args.workload in ("ngc", "sat"):
        # the two SGP-dec simulations the reference bundles (simulated_test/data/*.mat), read from the committed fixtures
        spec = importlib.util.spec_from_file_location("_bsgp_golden_store", os.path.join(ROOT, "tests", "golden", "golden_store.py"))
        store = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(store)
        fx = store.load("fixtures")
        gn, psf, bg = fx[args.workload + "/gn"].astype(np.float64), fx[args.workload + "/psf"].astype(np.float64), float(fx[args.workload + "/bkg"])
        if args.workload == "ngc":
            w = dict(gn=gn[None], bkg=np.array([bg]), psf=psf, flux=None, beta0=np.array([1.0]), divergence="kl")
            kw = dict(init_recon=3, stop_criterion=1, MAXIT=27)
            name = "config1: KL-SGP on NGC7027_255.mat (256x256), init_recon=3, 27 iterations (simulation_test_sgp.py:25), single image"
        else:
            w = dict(gn=gn[None], bkg=np.array([bg]), psf=psf, flux=None, beta0=np.array([1.0001]), divergence="beta")
            kw = dict(init_recon=3, proj_type=1, stop_criterion=1, MAXIT=332, adapt_beta=False)
            name = ("config2: beta-SGP with the flux-conserving projection on satellite_25500.mat (256x256), beta=1.0001, 332 iterations "
                    "(simulation_test_sgp.py:154), single image")
        return w, kw, name, True
    if args.workload == "cutouts31":
        # the literal shape of application_sgp_star_stamps.py:24,58,82-89: 31 x 31 cut-outs restored with the 31 x 31 PSF image the
        # reference ships (psf/psfccfbrd210048_1_1_img.fits; its pixels are committed in tests/golden/psf_golden.npz), one PSF for all
        psf31 = np.load(os.path.join(ROOT, "tests", "golden", "psf_golden.npz"))["shipped"].astype(np.float64)
        w = synth.star_cutouts(args.stamps, psf31, seed=31)
        kw = dict(synth.STAMP_KWARGS)
        name = (f"config3b: {args.stamps} synthetic 31x31 star cut-outs with the 31x31 PSF image shipped by the reference (shared), the call of "
                "application_sgp_star_stamps.py:82-89; odd side -> wrapped plan (64x64 FFT grid, fold)")
        return w, kw, name, True
    w = synth.star_stamps(args.stamps, 32, seed=12345)
    kw = dict(synth.STAMP_KWARGS)
    name = f"config3: {args.stamps} synthetic 32x32 star stamps, per-stamp PSF, adapt_beta, proj_type=1"
    return w, kw, name, False


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def _nvml_loop(self):
        import pynvml as nv
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.nvml_rows.append((float(sm), [n for n, b in bits.items() if r & b]))
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def start(self):
        # NVML in-process (a sample every 20 ms: a 5-step timed region of 0.4 s gets ~20); nvidia-smi -lms as the fallback
        self.nvml_rows, self.h = [], None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.stop_flag = threading.Event()
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.h = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if getattr(self, "h", None) is not None:
            self.stop_flag.set()
            self.t.join(1.0)
            sm = [r[0] for r in self.nvml_rows]
            reasons = sorted({n for r in self.nvml_rows for n in r[1]})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.sm_max, "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(npix, wbytes, iters, evals, trials, shared_psf, bkg_image):
    """SURVEY.md §8(d): B_iter = [26 + 2E + 3(T-1)] N w; shared TF: -2 N w; full-image bkg: +(3 + (T-1)) N w.
    Summed over the iterations of every image with the counted E (projection evaluations; 0 with proj_type=0) and T (trials)."""
    per_iter = 26.0 - (2.0 if shared_psf else 0.0) + (3.0 if bkg_image else 0.0)
    extra_trials = np.maximum(trials - iters, 0)
    units = per_iter * iters + 2.0 * evals + (4.0 if bkg_image else 3.0) * extra_trials
    return float(units.sum()) * npix * wbytes


def _oracle_solve(job):
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux, b0, kw = job
    kw = dict(kw)
    div = kw.pop("divergence", "beta")
    r = orc.solve(gn, psf, bkg, divergence=div, flux=None if flux is None else np.float64(flux), betaParam=float(b0), **kw)
    return r.iters


def cpu_jobs(w, kw, shared_psf, idx):
    jobs = []
    for i in idx:
        psf = w["psf"] if shared_psf else w["psf"][i]
        bkg = w["bkg"][i] if np.ndim(w["bkg"][i]) == 2 else np.float64(w["bkg"][i])
        jobs.append((w["gn"][i], psf, bkg, None if w["flux"] is None else float(w["flux"][i]), float(w["beta0"][i]),
                     dict(kw, divergence=w.get("divergence", "beta"))))
    return jobs


def frame_cpu_baseline(w, kw, side):
    """The oracle needs ~40 s per iteration at 8192^2; time a 2048^2 crop for 3 iterations and scale by the pixel
    ratio (the loop is O(N log N): the scaled figure flatters the CPU slightly)."""
    from oracle import sgp_oracle as orc
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bsgp_synth2", os.path.join(ROOT, "beta-sgp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    c = min(2048, side)
    gn = np.ascontiguousarray(w["gn"][0][:c, :c]); bkg = np.ascontiguousarray(w["bkg"][0][:c, :c])
    psf = synth.moffat_psf(c, c, 3.5)
    k = dict(kw, MAXIT=3)
    t0 = time.perf_counter()
    orc.solve(gn, psf, bkg, divergence="beta", flux=np.float64((gn - bkg).sum()), betaParam=float(w["beta0"][0]), **k)
    per_iter = (time.perf_counter() - t0) / 3.0 * (side * side) / float(c * c)
    return {"value": 1.0 / (per_iter * kw["MAXIT"]), "unit": "images/s", "cores": 1, "kind": "port",
            "sample": f"{c}x{c} crop, 3 iterations of the oracle port on 1 thread, scaled by the pixel ratio to {side}x{side} and {kw['MAXIT']} iterations"}


def run_reference(args, rank):
    """CPU arm: oracle port on all host cores, bounded sample per step."""
    if rank != 0:
        return
    import multiprocessing as mp
    w, kw, name, shared = make_workload(args, 0)
    if args.workload == "frame":
        cb = frame_cpu_baseline(w, kw, w["gn"].shape[-1])
        print(json.dumps({"impl": "reference", "metric": "beta-SGP restored images/s", "value": cb["value"], "unit": "images/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / cb["value"],
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": name}, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    procs = max(1, min(cores, 64))
    if args.workload in ("ngc", "sat"):
        procs = 1                                          # one image: the reference solves it on one core (numpy does not thread)
    n = len(w["gn"])
    per_step = procs if args.workload == "tiles256" else procs * 16
    rng = np.random.default_rng(0)
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        def step():
            idx = rng.choice(n, per_step, replace=per_step > n)
            return sum(pool.map(_oracle_solve, cpu_jobs(w, kw, shared, idx), chunksize=1 if args.workload == "tiles256" else 16))
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        iters = 0
        for _ in range(args.steps):
            iters += step()
        dt = time.perf_counter() - t0
    images = per_step * args.steps
    val = images / dt
    line = {"impl": "reference", "metric": "beta-SGP restored images/s", "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": name, "sample_per_step": per_step},
            "ms_per_image_iteration": 1e3 * dt * procs / max(iters, 1) / procs,
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": procs, "kind": "port",
                             "sample": f"{per_step} random solves of the workload per step on {procs} processes (1 numpy thread each)"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(res, out_dir):
    """--dump-outputs: the arrays the last timed step returned (solve_batch_sharded), one float32 / float64 .npy per field, so
    that two builds can be compared output for output on the same seeded inputs.  Integer fields are written as float64
    (exact).  "times" (device clock stamps of every iteration) is left out: it differs from run to run by nature.  The
    restored images "x" get what the 64 MB budget leaves; when they do not fit, a fixed seeded sample of whole images is
    written (of image rows when not even one image fits), and "x_index" holds the sampled batch indices (row indices
    b * ny + y for rows)."""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.cpu().numpy() for k, v in res.items() if k != "times"}
    out = {k: (v if v.dtype in (np.float32, np.float64) else v.astype(np.float64)) for k, v in host.items() if k != "x"}
    x = host["x"]
    room = DUMP_LIMIT_BYTES - 4096 - sum(v.nbytes for v in out.values())        # 4096: the .npy headers
    units = x if x[0].nbytes + 8 <= room else x.reshape(-1, x.shape[-1])
    keep = min(len(units), room // (units[0].nbytes + 8))
    if keep < len(units):
        idx = np.sort(np.random.default_rng(0).choice(len(units), keep, replace=False))
        out["x_index"] = idx.astype(np.float64)
        units = units[idx]
    out["x"] = units
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measure(args, ctx, workload, steps, warmup, with_cpu, sharded=True, with_clocks=True, dump_dir=None):
    """One workload through the product: `value` with inputs resident in HBM (sharded over the ranks of ctx, gather inside
    the timed region), `e2e` from page-locked host memory, roofline of the solve kernel from CUDA events inside the timed
    region.  dump_dir: rank 0 writes the outputs of the last timed step there (dump_outputs).  Returns the JSON-able dict
    (rank 0) or None."""
    import torch
    import torch.distributed as dist
    bs, dev, rank, local_rank, world = ctx["bs"], ctx["dev"], ctx["rank"], ctx["local_rank"], ctx["world"]
    a = argparse.Namespace(**dict(vars(args), workload=workload))
    w, kw, wname, shared_psf = make_workload(a, rank)
    divergence = w.get("divergence", "beta")
    tdt = torch.float64 if args.dtype == "float64" else torch.float32
    B, ny, nx = w["gn"].shape
    wbytes = 8 if args.dtype == "float64" else 4
    bkg_image = np.ndim(w["bkg"]) == 3
    frame_mode = ny * nx >= (1 << 20)
    keys = [k for k in ("gn", "psf", "bkg", "flux", "beta0") if w.get(k) is not None]
    host = {k: torch.as_tensor(np.ascontiguousarray(w[k])).to(tdt if k in ("gn", "psf", "bkg") else torch.float64).pin_memory() for k in keys}
    devt = {k: v.to(dev) for k, v in host.items()}
    flux_d = devt.get("flux")
    beta_np = np.ascontiguousarray(w["beta0"], dtype=np.float64)
    cost_rank = bs.shard.expected_cost_rank(B, beta_np, divergence)  # the dealing is host logic: computed once, no device sync in the step
    width = "auto" if args.width == "auto" else tuple(int(v) for v in args.width.split(","))
    if args.cluster or args.threads:
        width = (args.cluster, args.threads)
    L = bs._capi.lib()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    timings = []

    def step(record):
        t = {} if record else None
        r = bs.solve_batch_sharded(devt["gn"], devt["psf"], devt["bkg"], flux=flux_d, betaParam=devt["beta0"], divergence=divergence, width=width,
                                   timing=t, cost_rank=cost_rank, **kw)
        if record:
            timings.append(t)
        return r

    # ---------------- value: inputs resident in HBM, sharded solve + gather ----------------
    if world > 1:
        # NCCL's first collectives of a given size are several times slower (connection setup, buffer registration): warm the
        # all-gather up on buffers of the sizes the step uses, so that W warm-up STEPS are enough whatever W the caller picks
        cap = max(bs.shard.shard_counts(B, world, snake=True))
        for shape, dt in (((cap, ny, nx), tdt), ((cap, 2 * (kw.get("MAXIT", 500) + 1) + 6), torch.float64)):
            src = torch.zeros(shape, dtype=dt, device=dev); dst = torch.empty((world * shape[0],) + shape[1:], dtype=dt, device=dev)
            for _ in range(8):
                dist.all_gather_into_tensor(dst, src)
        del src, dst
    for _ in range(warmup):
        res = step(False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0 and with_clocks:
        sampler.start()
    n0 = L.bsgp_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        res = step(True)
    e1.record()
    barrier()
    launches = int(L.bsgp_launch_count() - n0)
    clocks = sampler.stop() if (rank == 0 and with_clocks) else None
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    have_local = all("solve" in t for t in timings)
    kernel_ms = float(np.mean([t["solve"][0].elapsed_time(t["solve"][1]) for t in timings])) if have_local else 0.0
    info = timings[0].get("plan") if have_local else bs.get_plan(ny, nx, args.dtype, local_rank).info()
    iters = res["iters"].cpu().numpy().astype(np.float64)
    evals = res["proj_evals"].cpu().numpy().astype(np.float64)
    trials = res["ls_trials"].cpu().numpy().astype(np.float64)
    assert (res["status"].cpu().numpy() == 0).all(), "solver reported a failure status"
    if kw.get("proj_type", 0) == 1 and args.dtype == "float64":
        fl = w["flux"] if w.get("flux") is not None else (w["gn"] - (w["bkg"] if bkg_image else np.asarray(w["bkg"]).reshape(-1, 1, 1))).sum(axis=(1, 2))
        x_sum = res["x"].sum(dim=(1, 2)).cpu().numpy()
        assert np.abs(x_sum - fl).max() <= 1e-8 * np.abs(fl).max(), "flux not conserved"
    # this rank's share (what its solve kernel processed)
    mine = bs.shard.shard_indices(B, rank, world, cost_rank)
    # share of (clusters in flight x kernel time) spent inside solves: 1 - this is queue tail + launch overhead
    t_img = res["times"].cpu().numpy()[mine, iters[mine].astype(int)]
    slot_util = float(t_img.sum() / (max(1, min(info["num_clusters"], len(mine))) * max(kernel_ms, 1e-9) * 1e-3))
    abytes_mine = algorithmic_bytes(ny * nx, wbytes, iters[mine], evals[mine], trials[mine], shared_psf, bkg_image)

    # ---------------- e2e: page-locked host buffers in, page-locked host results out, everything inside the timed region ----------------
    # The public call for host data: solve_batch with pinned CPU tensors -> bsgp_solve_batch_pinned (upload in queue order on a copy
    # stream behind per-item ready flags, restored images stored zero-copy into the pinned output, small outputs copied back).
    # N > 1: every rank owns its share of the batch in page-locked host memory (dealt before the timed region, as a sharded
    # application would hold it) and restores it into its own page-locked output; the per-image scalars are all-gathered.
    idx_t = torch.as_tensor(mine, dtype=torch.long)
    hl = {k: (host[k].index_select(0, idx_t).pin_memory() if (host[k].dim() >= 1 and host[k].shape[0] == B and (k != "psf" or not shared_psf)) else host[k])
          for k in keys}
    nl = len(mine)
    x_host = torch.empty((max(nl, 1), ny, nx), dtype=tdt).pin_memory()
    cs, th = bs.engine.auto_config(ny, nx, nl, args.dtype) if width == "auto" else width
    plan_e = bs.get_plan(ny, nx, args.dtype, local_rank, cs, th)

    def step_e2e():
        if nl:
            plan_e.set_psf(hl["psf"].to(dev, non_blocking=True))
            r = bs.solve_batch(hl["gn"], None, hl["bkg"] if bkg_image else hl["bkg"].numpy(), divergence=divergence,
                               flux=None if "flux" not in hl else hl["flux"].numpy(), betaParam=hl["beta0"].numpy(), plan=plan_e, psf_is_set=True,
                               device=local_rank, x_out=x_host[:nl], **kw)
            it = torch.as_tensor(np.asarray(r.iters), device=dev)
        else:
            r, it = None, torch.zeros(0, dtype=torch.int32, device=dev)
        if world > 1:
            cap = max(bs.shard.shard_counts(B, world, snake=True))
            pad = torch.zeros(cap, dtype=torch.int32, device=dev); pad[:nl] = it
            allr = torch.empty(world * cap, dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(allr, pad)
        return r

    for _ in range(min(warmup, 3)):
        r_e2e = step_e2e()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(steps):
        r_e2e = step_e2e()
    f1.record()
    barrier()
    ms_e2e = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
    if nl:
        assert np.array_equal(np.asarray(r_e2e.iters), iters[mine].astype(np.int32)) and torch.equal(r_e2e.x, res["x"][idx_t.to(dev)].cpu()), \
            "host path and resident path disagree"
    h2d = sum(v.numel() * v.element_size() for v in hl.values())
    d2h = 0 if not nl else (r_e2e.x.numel() * r_e2e.x.element_size() + sum(getattr(r_e2e, k).nbytes for k in
                            ("iters", "status", "discr", "times", "stop_value", "beta_final", "proj_evals", "ls_trials", "scalars")))
    stats = torch.tensor([kernel_ms, abytes_mine, float(h2d), float(d2h)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
        allst = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
        allst = torch.stack(allst).cpu().numpy()
    else:
        allst = stats.cpu().numpy()[None]
    ms, ms_e2e = float(ms.item()), float(ms_e2e.item())
    if rank != 0:
        return None
    if dump_dir:
        dump_outputs(res, dump_dir)
    images = B * steps
    value = images / (ms * 1e-3)
    peak, peak_src = hbm_peak()
    # roofline of the dominant kernel: the rank whose solve kernel ran longest (it bounds the step), its own bytes / its own time
    slow = int(np.argmax(allst[:, 0]))
    k_ms, k_bytes = float(allst[slow, 0]), float(allst[slow, 1])
    achieved = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get(workload), tj.get("source")
    total_iters = float(iters.sum())
    # every per-image array the solve touches lives in shared memory (bit 1 = the background image, unused with a scalar background)
    on_chip = ((info["resident_mask"] | (0 if bkg_image else 0x02)) & 0xFF) == 0xFF
    line = {
        "metric": "beta-SGP restored images/s", "value": value, "unit": "images/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64" if args.dtype == "float64" else "f32", "data": "synthetic" if workload not in ("ngc", "sat") else "reference fixture (.mat simulation)",
        "config": {"workload": wname, "images_per_step": B, "images_per_gpu_per_step": [len(bs.shard.shard_indices(B, r, world, cost_rank)) for r in range(world)],
                   "sharding": "one batch dealt over the ranks by expected cost (|beta - 1|), NCCL all-gather of the results inside the timed region" if world > 1
                               else "single GPU (same entry point, no process group)",
                   "cluster_size": info["cluster_size"], "clusters_in_flight": info["num_clusters"], "threads": info["threads"], "smem_bytes": info["smem_bytes"],
                   "l2": f"inputs {sum(v.numel() * v.element_size() for v in host.values()) / 1e6:.0f} MB per step > 126 MB L2, no flush needed; per-cluster scratch "
                         f"{info['workspace_bytes'] / 1e6:.0f} MB " + ("streams through L2/HBM" if info['workspace_bytes'] > 100e6 else "fits L2")
                         if B * ny * nx * wbytes > 126e6 else
                         f"working set {B * ny * nx * wbytes * 9 / 1e6:.0f} MB fits the 126 MB L2: an L2-resident (single-image / small-batch latency) configuration, no flush",
                   "mean_iterations": float(iters.mean()), "mean_proj_evals_per_iter": float(evals.sum() / iters.sum()),
                   "mean_trials_per_iter": float(trials.sum() / iters.sum()), "max_iterations": int(iters.max()),
                   "cluster_slot_utilisation": slot_util},
        "ms_per_image_iteration": ms / (total_iters * steps) if total_iters else None,
        "ms_per_iteration_longest_solve": ms / steps / float(iters.max()),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src,
                     "kernel": "bsgp_frame_kernel" if frame_mode else "bsgp_solve_kernel", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": k_bytes,
                     "peak_source": peak_src,
                     "note": ("on-chip workload: the stamp's arrays never leave shared memory (DRAM traffic = inputs + outputs only), the binding limits are "
                              "instruction delivery / issue and the fp64 pipe - see profiles/ for the issue-slot, shared-memory and pipe metrics; the HBM fraction of the "
                              "algorithmic-byte model is reported for uniformity") if on_chip else
                             ("kernel of the slowest rank (it bounds the step)" if world > 1 else None)},
        "e2e": {"value": images / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": int(allst[:, 2].sum()), "d2h_bytes_per_step": int(allst[:, 3].sum())},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if world > 1:
        # the longest solve bounds a rank that holds fewer images than cluster slots: state the bound next to the number
        line["longest_solve_bound"] = {"max_iterations": int(iters.max()), "kernel_ms_per_rank": [float(v) for v in allst[:, 0]],
                                       "note": "a rank's step cannot end before its longest solve does: max_iterations x per-iteration latency of one image"}
    if with_cpu and world == 1:
        sys.path.insert(0, ROOT)
        if workload == "frame":
            line["cpu_baseline"] = frame_cpu_baseline(w, kw, ny)
        else:
            n = min(args.cpu_sample, B) if ny * nx >= 65536 else min(args.cpu_sample * 64, B)
            idx = np.linspace(0, B - 1, n).astype(int)
            jobs = cpu_jobs(w, kw, shared_psf, idx)
            _oracle_solve(jobs[0])
            t0 = time.perf_counter()
            for j in jobs:
                _oracle_solve(j)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n / dt, "unit": "images/s", "cores": 1, "kind": "port",
                                    "sample": f"{n} of the {B} solves (evenly spaced indices), oracle port, 1 thread, after one warm-up solve"}
    return line


def measure_replicas(args, ctx, steps, warmup):
    """Round 1's multi-GPU number: every rank restores the WHOLE field on its own (independent replicas, no gather).  Weak scaling."""
    import torch
    import torch.distributed as dist
    bs, dev, rank, world = ctx["bs"], ctx["dev"], ctx["rank"], ctx["world"]
    w, kw, wname, shared_psf = make_workload(args, rank)
    tdt = torch.float64 if args.dtype == "float64" else torch.float32
    t = {k: torch.as_tensor(np.ascontiguousarray(w[k])).to(tdt if k in ("gn", "psf", "bkg") else torch.float64).to(dev) for k in ("gn", "psf", "bkg", "flux", "beta0")}
    for _ in range(warmup):
        bs.solve_batch(t["gn"], t["psf"], t["bkg"], divergence="beta", flux=t["flux"], betaParam=t["beta0"], **kw)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        bs.solve_batch(t["gn"], t["psf"], t["bkg"], divergence="beta", flux=t["flux"], betaParam=t["beta0"], **kw)
    e1.record()
    torch.cuda.synchronize(); dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return {"value": len(w["gn"]) * world * steps / (float(ms.item()) * 1e-3), "unit": "images/s", "scaling": "weak",
            "what": "every rank restores the whole field on its own (independent replicas, nothing gathered)"}


def brief(line):
    """the part of a workload's record that goes under "workloads" """
    keep = ("value", "unit", "ms_per_step", "ms_per_image_iteration", "ms_per_iteration_longest_solve", "roofline", "e2e", "cpu_baseline", "gpu_launches", "steps",
            "warmup", "scaling", "n_gpus", "longest_solve_bound")
    out = {k: line[k] for k in keep if k in line}
    out["workload"] = line["config"]["workload"]
    for k in ("mean_iterations", "max_iterations", "cluster_size", "threads", "clusters_in_flight", "images_per_gpu_per_step"):
        out[k] = line["config"][k]
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    import torch.distributed as dist
    import beta_sgp_b200 as bs

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = dict(bs=bs, dev=dev, rank=rank, local_rank=local_rank, world=world)
    line = measure(args, ctx, args.workload, args.steps, args.warmup, with_cpu=not args.no_cpu_baseline, with_clocks=not args.no_clocks,
                   dump_dir=args.dump_outputs)
    if args.workload == "tiles256" and not args.no_extra:
        extra = {}
        if world == 1:
            # the other BASELINE configs, briefly (each: W >= 3 warm-up steps; inputs of 3 and 5 exceed L2, 1 and 2 are single-image latency)
            for name, wl, st in (("config1_kl_ngc7027", "ngc", 5), ("config2_beta_proj_satellite", "sat", 3), ("config3_stamps_8192", "stamps32", 5),
                                 ("config3b_cutouts31_8192", "cutouts31", 3), ("config5_frame_8192", "frame", 2)):
                try:
                    extra[name] = brief(measure(args, ctx, wl, st, 3, with_cpu=not args.no_cpu_baseline, with_clocks=False))
                except Exception as e:                    # a failing side workload must not take the headline line with it
                    extra[name] = {"error": f"{type(e).__name__}: {e}"}
                bs.clear_plans()
                torch.cuda.empty_cache()
        else:
            r = measure(args, ctx, "stamps32", 5, 3, with_cpu=False, with_clocks=False)
            if rank == 0:
                extra["config3_stamps_8192"] = brief(r)
            rep = measure_replicas(args, ctx, args.steps, args.warmup)
            if rank == 0:
                line["replicas"] = rep
        if rank == 0:
            line["workloads"] = extra
    if rank == 0:
        print(json.dumps(line), flush=True)
    bs.clear_plans()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
