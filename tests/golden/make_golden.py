"""Generate the committed golden vectors by running the UNMODIFIED reference in this container.

    python tests/golden/make_golden.py        (from the repository root)

Writes the golden archives "fixtures" (inputs) and "golden_ref" (reference outputs plus the oracle's
controller trace) as tests/golden/<name>.<part>.npz (golden_store.py).  For every case the oracle
(oracle/sgp_oracle.py) is run on the same inputs and must agree BIT FOR BIT with the reference (image,
iteration count, objective trace) — that is the oracle's pin; the script aborts otherwise.  The tests
never need the reference: they only read the committed archives.
"""
import contextlib
import io
import os
import re
import sys
import tempfile

import numpy as np
from scipy.io import loadmat

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "beta-sgp_b200"))

import golden_store  # noqa: E402
import reference_loader  # noqa: E402
from cases import CASES, N_CUTOUTS31, N_STAMPS, N_TILES  # noqa: E402
import synth  # noqa: E402
from oracle import sgp_oracle as orc  # noqa: E402


def build_inputs():
    data = {}
    base = os.path.join(reference_loader.REFERENCE_DIR, "simulated_test", "data")
    for key, fn in (("ngc", "NGC7027_255.mat"), ("sat", "satellite_25500.mat")):
        m = loadmat(os.path.join(base, fn))
        data[key] = dict(gn=np.ascontiguousarray(m["gn"]), psf=np.ascontiguousarray(m["psf"]),
                         obj=np.ascontiguousarray(m["obj"]), bkg=np.float64(m["bg"][0][0]))
    st = synth.star_stamps(N_STAMPS, 32, seed=12345)
    for i in range(N_STAMPS):
        data[f"stamp{i}"] = dict(gn=st["gn"][i], psf=st["psf"][i], bkg=np.float64(st["bkg"][i]),
                                 flux=float(st["flux"][i]), betaParam=float(st["beta0"][i]))
    # 31 x 31 cut-outs with the PSF image the reference ships (read by make_psf_golden.py into psf_golden.npz)
    sys.path.insert(0, HERE)
    from make_psf_golden import read_fits_f64
    psf31 = read_fits_f64("/root/reference/psf/psfccfbrd210048_1_1_img.fits")
    assert psf31.shape == (31, 31)
    co = synth.star_cutouts(N_CUTOUTS31, psf31, seed=31)
    for i in range(N_CUTOUTS31):
        data[f"cutout31_{i}"] = dict(gn=co["gn"][i], psf=psf31, bkg=np.float64(co["bkg"][i]),
                                     flux=float(co["flux"][i]), betaParam=float(co["beta0"][i]))
    tl = synth.field_tiles(size=1024, tile=256, seed=2024, n_beta=5, max_tiles=N_TILES)
    for i in range(N_TILES * 5):
        data[f"tile{i}"] = dict(gn=tl["gn"][i], psf=tl["psf"], bkg=tl["bkg"][i], flux=float(tl["flux"][i]),
                                betaParam=float(tl["beta0"][i]))
    return data


def main():
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=golden_store.BLAS_THREADS, user_api="blas")
    ref_sgp, ref_proj = reference_loader.load()
    data = build_inputs()
    fixtures, golden = {}, {}
    for key, d in data.items():
        if key.startswith("tile") and int(key[4:]) % 5 != 0:
            continue                       # the 5 beta inits of a tile share gn / bkg / psf
        for f in ("gn", "psf", "obj", "bkg"):
            if f in d:
                if f == "psf" and key.startswith("tile") and key != "tile0":
                    continue               # one shared PSF for all tiles
                if f == "psf" and key.startswith("cutout31_") and key != "cutout31_0":
                    continue               # ... and for all cut-outs
                fixtures[f"{key}/{f}"] = np.asarray(d[f])
    scratch = tempfile.mkdtemp()
    os.chdir(scratch)                      # the reference writes ./sgp.log
    for name, (dkey, div, kw, full) in CASES.items():
        d = data[dkey]
        kw = dict(kw)
        if "flux" in d:
            kw["flux"] = np.float64(d["flux"])
            if div == "beta":
                kw["betaParam"] = d["betaParam"]
        fn = ref_sgp.sgp if div == "kl" else ref_sgp.sgp_betaDiv
        out = io.StringIO()
        with contextlib.redirect_stdout(out):
            x, iters, discr, times, _ = fn(d["gn"].copy(), d["psf"].copy(), d["bkg"], **dict(kw))
        o = orc.solve(d["gn"].copy(), d["psf"].copy(), d["bkg"], divergence=div, **dict(kw))
        assert iters == o.iters and np.array_equal(x, o.x) and np.array_equal(discr, o.discr), \
            f"oracle is not bit-identical to the reference on {name}"
        g = {"iters": iters, "discr": discr, "sum_x": np.sum(x), "x_sub": x[::8, ::8].copy(),
             "trials": np.array(o.trace.trials), "proj_evals": np.array(o.trace.proj_evals),
             "alpha": np.array(o.trace.alpha), "lam": np.array(o.trace.lam),
             "beta_trace": np.array(o.trace.beta_param), "init_proj_evals": o.trace.init_proj_evals,
             "x_low": o.trace.x_low, "x_upp": o.trace.x_upp}
        if "flux" in kw:
            g["flux_in"] = float(kw["flux"])
        if "betaParam" in kw:
            g["beta0"] = float(kw["betaParam"])
        if div == "beta":
            m = re.search(r"final value\): (\S+)", out.getvalue())
            g["beta_final"] = float(m.group(1))
            assert g["beta_final"] == o.beta_param
        if "obj" in d:
            e = x - d["obj"]
            g["rel_err"] = np.sqrt(np.sum(e * e) / np.sum(d["obj"] * d["obj"]))
        if full:
            g["x"] = x
        for k, v in g.items():
            golden[f"{name}/{k}"] = np.asarray(v)
        print(f"{name:24s} iters={iters:4d} discr[-1]={discr[-1]:.15g} sum_x={np.sum(x):.15g}"
              f" E={np.mean(o.trace.proj_evals):.2f} T={np.mean(o.trace.trials):.2f}", flush=True)

    # projectDF standalone known answers (flux_conserve_proj.py:7-144) on seeded random inputs
    rng = np.random.default_rng(99)
    for i in range(12):
        n = [7, 100, 1000, 4096][i % 4]
        c = rng.normal(0.0, 1.0, n) * 10.0 ** rng.uniform(-3, 2)
        dia = rng.uniform(0.2, 5.0, n) if i % 3 else np.ones(n)
        b = np.float64(rng.uniform(0.1, 50.0) * (n if i % 2 else 1))
        sat = None if i % 4 != 3 else 4.0 * float(b) / n * 300.0
        scaling = 300.0 if sat is not None else 1.0
        xr = ref_proj.projectDF(b, c.copy(), dia.copy(), scaling, ccd_sat_level=sat)
        cnt = []
        xo = orc.flux_projection(b, c.copy(), dia.copy(), scaling, ccd_sat_level=sat, counter=cnt)
        assert np.array_equal(xr, xo), f"projection oracle mismatch in case {i}"
        golden[f"proj{i:02d}/c"] = c
        golden[f"proj{i:02d}/dia"] = dia
        golden[f"proj{i:02d}/b"] = np.asarray(b)
        golden[f"proj{i:02d}/sat"] = np.asarray(np.nan if sat is None else sat)
        golden[f"proj{i:02d}/scaling"] = np.asarray(scaling)
        golden[f"proj{i:02d}/x"] = xr
        golden[f"proj{i:02d}/evals"] = np.asarray(cnt[-1])
        print(f"proj{i:02d} n={n} evals={cnt[-1]} sum={xr.sum():.15g} b={float(b):.15g}")

    # beta-divergence helper known answers (tests.py:9-19,54-68 restated without torchnmf)
    import torch
    torch.manual_seed(101); x1 = torch.rand(20).numpy().astype(np.float64)
    torch.manual_seed(1001); y1 = torch.rand(20).numpy().astype(np.float64)
    golden["betadiv/x"] = x1
    golden["betadiv/y"] = y1
    golden["betadiv/value_1p5"] = np.asarray(ref_sgp.betaDiv(y1, x1, 1.5))
    golden["betadiv/deriv_1p7"] = np.asarray(ref_sgp.betaDivDeriv(y1, x1, 1.7))

    for name, arrays in (("fixtures", fixtures), ("golden_ref", golden)):
        for path in golden_store.save(name, arrays):
            print(os.path.basename(path), os.path.getsize(path) / 1e6, "MB")


if __name__ == "__main__":
    main()
