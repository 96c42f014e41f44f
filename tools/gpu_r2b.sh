#!/bin/bash
# round 2, second GPU session: parity suite, the new bench (with the workloads key), fp32 errors against the golden images
mkdir -p gpurun_out
python -m pytest tests -m gpu -q -x > gpurun_out/pytest_gpu_r2b.log 2>&1; echo "pytest rc=$?" | tee -a gpurun_out/pytest_gpu_r2b.log
tail -8 gpurun_out/pytest_gpu_r2b.log
( time python bench.py ) > gpurun_out/bench_default_r2b.json 2> gpurun_out/bench_default_r2b.err; echo "bench rc=$?"
tail -4 gpurun_out/bench_default_r2b.err
python - <<PY
import json
d = json.loads(open("gpurun_out/bench_default_r2b.json").read().strip().splitlines()[-1])
print("main", round(d["value"],1), "e2e", round(d["e2e"]["value"],1), "frac", round(d["roofline"]["frac"],3), "launches", d["gpu_launches"], "cpu", d.get("cpu_baseline",{}).get("value"))
for k, v in d.get("workloads", {}).items():
    if "error" in v: print(k, v); continue
    print(k, "value", round(v["value"],2), "ms/step", round(v["ms_per_step"],3), "ms/it(longest)", round(v["ms_per_iteration_longest_solve"],4), "frac", round(v["roofline"]["frac"],3), "e2e", round(v["e2e"]["value"],2), "cpu", v.get("cpu_baseline",{}).get("value"), "cfg", v["cluster_size"], v["threads"])
PY
python - <<PY
# fp32 mode: actual errors against the fp64 golden images
import sys, os, numpy as np
sys.path.insert(0, os.getcwd()); sys.path.insert(0, "tests"); sys.path.insert(0, "tests/golden")
import beta_sgp_b200 as bs
from conftest import case_inputs
import golden_store
fx = golden_store.load("fixtures"); gd = golden_store.load("golden_ref")
for name in ("ngc_kl_27", "ngc_beta_p1_27", "sat_kl_40", "ngc_beta_p1_stop3", "stamp00", "stamp05", "tile00", "tile07", "cutout31_02"):
    gn, psf, bkg, div, kw = case_inputs(name, fx, gd)
    kw = dict(kw); flux = kw.pop("flux", None); b0 = kw.pop("betaParam", 1.005)
    bk = np.asarray(bkg, dtype=np.float64); bk = bk[None] if bk.ndim == 2 else bk.reshape(1)
    r = bs.solve_batch(gn[None], psf, bk, divergence=div, flux=None if flux is None else [float(flux)], betaParam=b0, dtype="float32", **kw)
    xr = gd[name + "/x"]
    print("fp32", name, "iters", int(r.iters[0]), "vs", int(gd[name + "/iters"]), "image err", float(np.abs(r.x[0] - xr).max() / np.abs(xr).max()),
          "l2 err", float(np.sqrt(((r.x[0] - xr) ** 2).sum() / (xr ** 2).sum())), "flux err", abs(float(r.x[0].sum()) - xr.sum()) / xr.sum())
PY
