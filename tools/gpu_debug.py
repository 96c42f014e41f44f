"""Scratch GPU check: prints differences instead of asserting (used during bring-up via gpurun)."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import numpy as np
import beta_sgp_b200 as bs
from cases import CASES
from conftest import case_inputs
import golden_store
fx = golden_store.load("fixtures"); gd = golden_store.load("golden_ref")

def conv_check(shape, G=0):
    rng = np.random.default_rng(1)
    x = rng.normal(size=(3,) + shape); psf = rng.random(shape); psf /= psf.sum()
    plan = bs.Plan(shape[0], shape[1], cluster_size=G)
    print("plan", shape, plan.info(), flush=True)
    plan.set_psf(psf)
    y = plan.apply_psf(x)
    tf = np.fft.fftn(np.fft.fftshift(psf))
    ref = np.real(np.fft.ifftn(tf * np.fft.fftn(x, axes=(1, 2)), axes=(1, 2)))
    print("conv", shape, G, "err", np.abs(y - ref).max() / np.abs(ref).max(), flush=True)
    plan.close()

which = sys.argv[1] if len(sys.argv) > 1 else "all"
if which in ("conv", "all"):
    for shape, G in [((32, 32), 0), ((64, 64), 0), ((256, 256), 1), ((256, 256), 2), ((256, 256), 8), ((512, 512), 0)]:
        conv_check(shape, G)
if which in ("solve", "all"):
    names = sys.argv[2:] or ["stamp00", "stamp01", "ngc_kl_27", "ngc_beta_p1_stop3", "tile00", "sat_beta_p1_stop3", "ngc_beta_adapt", "ngc_beta_is"]
    for name in names:
        gn, psf, bkg, div, kw = case_inputs(name, fx, gd)
        kw = dict(kw); flux = kw.pop("flux", None); b0 = kw.pop("betaParam", 1.005)
        bkg_a = np.asarray(bkg, dtype=np.float64); bkg_a = bkg_a[None] if bkg_a.ndim == 2 else bkg_a.reshape(1)
        x0 = None
        if kw.get("init_recon", 0) == 1:
            np.random.seed(42); x0 = np.random.randn(*gn.shape)[None]
        t = time.time()
        r = bs.solve_batch(gn[None], psf, bkg_a, divergence=div, flux=None if flux is None else [float(flux)], betaParam=b0, x0=x0, trace=True, **kw)
        dt = time.time() - t
        it = int(gd[name + "/iters"]); ref = gd[name + "/discr"]; n = min(it, int(r.iters[0])) + 1
        rel = np.abs(r.discr[0, :n] - ref[:n]) / np.abs(ref[:n])
        xs = gd[name + "/x_sub"]
        print(f"{name:20s} it {int(r.iters[0])}/{it} st {int(r.status[0])} discr {rel.max():.2e} x {np.abs(r.x[0][::8, ::8] - xs).max() / np.abs(xs).max():.2e} "
              f"E {int(r.proj_evals[0])} T {int(r.ls_trials[0])}/{int(gd[name + '/trials'].sum())} gpu_time {r.times[0, int(r.iters[0])]*1e3:.2f} ms wall {dt:.2f}s", flush=True)
