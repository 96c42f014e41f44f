"""Every compiled solve-kernel variant against the oracle, and fp32 held to per-operation bounds (run with -m gpu on a B200).

The library instantiates the persistent solve kernel for five launch shapes (128 threads x 4 or x 3 CTAs per SM, 256 x 2,
256 x 1, 512 x 1) plus the grid-wide frame kernel, each for T in {double, float} and MK in {false, true} (MK: the
valid-window masks of wrapped plans and of the zero-padded operator): 24 kernels (bsgp_solve_kernel.cuh).  VARIANTS names
an input for each of them and the cell it must land on; every row runs two short solves against the oracle.  fp32 is
compared with the oracle run in fp64 on the same inputs: the inputs here are exactly representable in fp32 (Poisson
counts, fp32-rounded backgrounds, PSFs on a dyadic grid that sum to exactly 1), so input rounding is not counted as
kernel error.  Further: the fp32 operator at every transform kind, batches across images in frame mode and with mixed
statuses, and the device pow / beta-divergence helpers against long double.
"""
import math
from dataclasses import dataclass, field
from functools import lru_cache

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F64, F32 = "float64", "float32"
FRAME = "frame"
LAUNCH_SHAPES = ((128, 4), (128, 3), (256, 2), (256, 1), (512, 1), FRAME)
ALL_CELLS = {(t, mk, s) for t in (F64, F32) for mk in (False, True) for s in LAUNCH_SHAPES}


@dataclass(frozen=True)
class Variant:
    label: str
    shape: tuple             # image shape
    dtype: str
    cell: tuple              # (dtype, MK, (threads, CTAs per SM) or FRAME) the row must land on
    cfg: dict = field(default_factory=dict)     # Plan(..., cluster_size=, threads=); unused for padded rows
    kernel: int = 0          # > 0: the zero-padded operator with a kernel x kernel PSF (the front end picks the plan)


def _v(label, shape, dtype, nt, per_sm, mk, kernel=0, **cfg):
    return Variant(f"{label}-{dtype[5:]}", shape, dtype, (dtype, mk, FRAME if nt == FRAME else (nt, per_sm)), cfg, kernel)


VARIANTS = [
    # small images: one CTA each, everything resident in shared memory
    _v("32", (32, 32), F64, 128, 3, False),
    _v("32", (32, 32), F32, 128, 3, False),
    _v("32-t256", (32, 32), F64, 256, 2, False, threads=256),
    _v("32-t256", (32, 32), F32, 256, 2, False, threads=256),
    _v("31", (31, 31), F64, 256, 2, True),                   # the DMMA table of the dense 31-point DFT does not fit 128 x 3
    _v("31", (31, 31), F32, 128, 3, True),                   # fp32 has no DMMA table
    _v("31-t256", (31, 31), F32, 256, 2, True, threads=256),
    _v("15x13", (15, 13), F64, 128, 3, True),
    _v("15x13", (15, 13), F32, 128, 3, True),
    _v("33x20", (33, 20), F64, 128, 4, True),                # 128 x 32 grid: a wrapped axis next to a dense one
    _v("33x20", (33, 20), F32, 256, 2, True),
    # tiles: multi-CTA clusters
    _v("256", (256, 256), F64, 128, 4, False),
    _v("256", (256, 256), F32, 128, 4, False),
    _v("256-t512", (256, 256), F64, 512, 1, False, threads=512),
    _v("256-t512", (256, 256), F32, 512, 1, False, threads=512),
    _v("256-g16t256", (256, 256), F64, 256, 1, False, cluster_size=16, threads=256),
    # slabs of <= 16 KB in clusters of several CTAs take the large-slab shapes: the one-CTA contexts of 128 x 3 and
    # 256 x 2 sum over their own CTA only, a cluster on them never finishes its solve
    _v("256-g16t256", (256, 256), F32, 256, 1, False, cluster_size=16, threads=256),
    _v("256-g16t128", (256, 256), F32, 128, 4, False, cluster_size=16, threads=128),   # engine.auto_config's choice for 30-120 tiles
    _v("64-g4", (64, 64), F64, 128, 4, False, cluster_size=4),
    _v("100x75", (100, 75), F64, 128, 4, True),
    _v("100x75", (100, 75), F32, 128, 4, True),
    _v("100x75-t512", (100, 75), F64, 512, 1, True, threads=512),
    _v("100x75-t512", (100, 75), F32, 512, 1, True, threads=512),
    _v("100x75-g16t256", (100, 75), F64, 256, 1, True, cluster_size=16, threads=256),
    _v("100x75-g8t256", (100, 75), F32, 256, 1, True, cluster_size=8, threads=256),
    _v("pad375", (375, 375), F64, 128, 4, True, kernel=31),           # P = 512
    _v("pad375", (375, 375), F32, 128, 4, True, kernel=31),
    # frame mode: one image over the whole GPU
    _v("256-frame", (256, 256), F64, FRAME, 0, False, cluster_size=-1),
    _v("256-frame", (256, 256), F32, FRAME, 0, False, cluster_size=-1),
    _v("100x75-frame", (100, 75), F64, FRAME, 0, True, cluster_size=-1),
    _v("100x75-frame", (100, 75), F32, FRAME, 0, True, cluster_size=-1),
    _v("450", (450, 450), F64, FRAME, 0, True),                       # 1024 x 1024 grid: frame mode automatically
    _v("450", (450, 450), F32, FRAME, 0, True),
    _v("pad500", (500, 500), F64, FRAME, 0, True, kernel=31),         # P = 1024
    _v("pad500", (500, 500), F32, FRAME, 0, True, kernel=31),
]

# cells no input can reach, with the reason
UNREACHABLE = {}

# fp32 six-iteration solves against the fp64 oracle, relative to the largest value.  Worst measured on a B200 (1000 W) over
# all rows: discr 1.6e-4 (beta-SGP: the beta-divergence cancels to ~1e-4 of its terms), image 3.3e-6, flux 3.3e-6 (KL,
# no projection; 1.9e-8 with the flux projection), all on the 31 x 31 rows.
FP32_DISCR, FP32_IMAGE, FP32_FLUX = 1e-3, 3e-5, 3e-5
# fp32 operator: |y - ref| <= FP32_OP_C * 2^-23 * log2(ny * nx) * max|ref|; measured worst 0.49 (dense axes, 32 x 31),
# 0.17-0.31 on power-of-two, wrapped and frame transforms
FP32_OP_C = 1.0


@pytest.fixture(scope="module")
def bs():
    import beta_sgp_b200 as b
    assert b._capi.lib().bsgp_device_count() > 0, "no CUDA device: the product has no CPU path"
    return b


def _f32_psf(p):
    """p on the dyadic grid of 24 significant bits below its largest value, summing to exactly 1: representable in fp32
    and normalised to the bit, so the oracle accepts it and the fp32 plans see the same kernel."""
    step = 2.0 ** (math.ceil(math.log2(p.max())) - 24)
    q = np.round(p / step) * step
    q.flat[np.argmax(q)] += 1.0 - q.sum()          # exact: every value is a multiple of step and the sum has < 53 bits
    assert q.sum() == 1.0 and np.array_equal(q.astype(np.float32).astype(np.float64), q)
    return q


def _scene(bs, shape, kernel, seed, fwhm=3.0):
    """(gn, psf, bkg image, flux): a star field blurred by the operator the row runs (circular on the image, or the
    zero-padded one with a kernel x kernel PSF), a sloped sky, Poisson noise; all values exact in fp32."""
    from oracle import sgp_oracle as orc
    ny, nx = shape
    rng = np.random.default_rng(seed)
    ky, kx = (kernel, kernel) if kernel else shape
    psf = _f32_psf(bs.synth.moffat_psf(ky, kx, fwhm, axis_ratio=1.2, theta=0.5))
    truth = np.zeros(shape)
    n = max(2, ny * nx // 400)
    truth[rng.integers(0, ny, n), rng.integers(0, nx, n)] = 10 ** rng.uniform(2.5, 4.5, n)
    op = orc.PaddedPsf(psf, shape) if kernel else orc.CircularPsf(psf)
    blur = op.forward(truth.ravel()).reshape(shape)
    yy, xx = np.mgrid[0:ny, 0:nx]
    bkg = (300.0 + 20.0 * xx / nx - 10.0 * yy / ny).astype(np.float32).astype(np.float64)
    gn = rng.poisson(np.maximum(blur, 0) + bkg).astype(np.float64)
    return gn, psf, bkg, float((gn - bkg).sum())


BETA0 = 1.0248357
# the two runs of every row: beta-SGP with the flux projection and a 2-D background from x = gn; KL with a scalar
# background from x = 0 (the first iteration starts from the constant image)
RUNS = {
    "beta": dict(divergence="beta", init_recon=2, proj_type=1, stop_criterion=1, MAXIT=6, gamma=1e-4, beta=0.4, alpha=10.0,
                 M_alpha=3, tau=0.5, M=1, ccd_sat_level=65000, lr=1e-3, lr_exp_param=0.1, schedule_lr=True, adapt_beta=True),
    "kl": dict(divergence="kl", init_recon=0, proj_type=0, stop_criterion=1, MAXIT=6),
}


@lru_cache(maxsize=None)
def _inputs_and_oracle(shape, kernel, run):
    """Inputs of a row and the oracle's result on them; shared by the fp64 and fp32 rows of the same input."""
    import beta_sgp_b200 as bs
    from oracle import sgp_oracle as orc
    gn, psf, bkg, flux = _scene(bs, shape, kernel, seed=shape[0] * 7 + shape[1] + kernel)
    kw = dict(RUNS[run])
    div = kw.pop("divergence")
    if run == "beta":
        args = dict(bkg=bkg, flux=flux, betaParam=BETA0)
        o = orc.solve(gn, psf, bkg, divergence=div, flux=np.float64(flux), betaParam=BETA0, use_original_SGP_Afunction=not kernel,
                      verbose=False, **kw)
    else:
        args = dict(bkg=np.float64(300.0), flux=None, betaParam=1.005)
        o = orc.solve(gn, psf, np.float64(300.0), divergence=div, use_original_SGP_Afunction=not kernel, verbose=False, **kw)
    return gn, psf, args, kw, div, o


def _plan(bs, v):
    """The plan the row's solve runs on: its own Plan, or for padded rows the cached plan the front end picks."""
    if v.kernel:
        geo = bs.engine.PaddedGeometry(v.shape[0], v.shape[1], v.kernel, v.kernel)
        return bs.get_plan(geo.P, geo.P, v.dtype), True
    return bs.Plan(v.shape[0], v.shape[1], v.dtype, **v.cfg), False


def _cell(info, dtype, mk):
    """(T, MK, (threads, CTAs per SM) or FRAME) from bsgp_plan_info: a single cluster of >= 8 CTAs is frame mode;
    CTAs per SM = num_clusters * cluster_size / num_sms, rounded up (clusters of 8 or 16 may leave a few SMs idle)."""
    if info["num_clusters"] == 1 and info["cluster_size"] >= 8:
        return (dtype, mk, FRAME)
    per_sm = info["num_clusters"] * info["cluster_size"] / info["num_sms"]
    return (dtype, mk, (info["threads"], math.ceil(round(per_sm, 6))))


def _plan_cell(bs, v):
    plan, padded = _plan(bs, v)
    info = plan.info()
    mk = padded or (info["grid_ny"], info["grid_nx"]) != (info["ny"], info["nx"])
    return plan, padded, _cell(info, v.dtype, mk)


def test_variant_table_covers_every_kernel():
    reached = {v.cell for v in VARIANTS}
    assert not reached & set(UNREACHABLE), "a cell listed as unreachable is reached"
    assert reached | set(UNREACHABLE) == ALL_CELLS, sorted(map(str, ALL_CELLS - reached - set(UNREACHABLE)))


@pytest.mark.parametrize("v", VARIANTS, ids=lambda v: v.label)
def test_variant_lands_on_its_cell(bs, v):
    """A change of the automatic configuration must not move a row to another kernel unnoticed."""
    plan, padded, cell = _plan_cell(bs, v)
    info = plan.info()
    if not padded:
        plan.close()
    assert cell == v.cell, cell
    assert info["cluster_size"] == 1 or cell[2] not in ((128, 3), (256, 2)), "a cluster of several CTAs on a one-CTA launch shape"
    # the library's launch shape is the host-compiled planner's (tests/host_emul) for this device
    import emul_helper as eh
    import torch
    prop = torch.cuda.get_device_properties(info["device"])
    rc, s = eh.plan_launch((info["ny"], info["nx"]), v.dtype, 0 if padded else v.cfg.get("cluster_size", 0),
                           0 if padded else v.cfg.get("threads", 0), num_sms=prop.multi_processor_count,
                           max_smem=prop.shared_memory_per_block_optin, smem_per_sm=prop.shared_memory_per_multiprocessor)
    assert rc == 0
    for k in ("threads", "cluster_size", "smem_bytes", "resident_mask"):
        assert info[k] == s[k], (k, info[k], s[k])


def test_dense_axes_refuse_frame_mode(bs):
    """A 31 x 31 plan transforms both axes with a dense 31-point DFT, which needs one CTA per image: frame mode is refused
    (it used to run the radix FFT of the 32-point grid and fold the 61-long linear convolution on a 32-point circle)."""
    with pytest.raises(bs._capi.BsgpError, match="frame mode"):
        bs.Plan(31, 31, cluster_size=-1)


def test_set_psf_adjoint_host_refuses_wrapped_plan(bs):
    """bsgp_set_psf_adjoint_host on a wrapped plan takes the caller's image-sized buffer and returns BSGP_E_STATE before
    it copies anything (it used to copy a grid-sized block from it first)."""
    plan = bs.Plan(100, 75)
    psf = np.full((100, 75), 1.0 / 7500)
    assert bs._capi.lib().bsgp_set_psf_adjoint_host(plan._h, psf.ctypes.data, 1) == 5       # BSGP_E_STATE
    plan.close()


@pytest.mark.parametrize("run", ["beta", "kl"])
@pytest.mark.parametrize("v", VARIANTS, ids=lambda v: v.label)
def test_variant_solve_matches_oracle(bs, v, run):
    """Six iterations on every kernel variant against the oracle.
    fp64: the suite's strict bar (same iteration count, projection evaluations and line-search trials per iteration;
    discr <= 1e-10, image <= 1e-8 of its maximum, flux <= 1e-9).
    fp32: against the fp64 oracle on the same (fp32-exact) inputs; discr, image and flux held to FP32_DISCR, FP32_IMAGE,
    FP32_FLUX relative to the largest value (measured values beside them).  Trial counts are printed, not asserted (on the
    B200 they matched the oracle's on every row)."""
    gn, psf, args, kw, div, o = _inputs_and_oracle(v.shape, v.kernel, run)
    plan, padded, cell = _plan_cell(bs, v)
    assert cell == v.cell, cell
    if v.dtype == F32:
        gn, psf = gn.astype(np.float32), psf.astype(np.float32)
    bkg = args["bkg"]
    bkg = bkg[None] if np.ndim(bkg) == 2 else np.array([float(bkg)])
    flux = None if args["flux"] is None else [args["flux"]]
    where = dict(padded=True) if padded else dict(plan=plan)
    r = bs.solve_batch(gn[None], psf, bkg, divergence=div, flux=flux, betaParam=args["betaParam"], dtype=v.dtype, trace=True,
                       verbose=False, **where, **kw)
    if not padded:
        plan.close()
    it = int(r.iters[0])
    assert int(r.status[0]) == 0 and it == o.iters == kw["MAXIT"]
    e_d = np.abs(r.discr[0, :it + 1] - o.discr).max() / np.abs(o.discr).max()
    e_x = np.abs(r.x[0] - o.x).max() / np.abs(o.x).max()
    e_f = abs(float(r.x[0].sum(dtype=np.float64)) - o.x.sum()) / abs(o.x.sum())
    trials = r.trace["trials"][0, 1:it + 1]
    print(f"\n{v.label} {run} cell={v.cell} discr {e_d:.3e} image {e_x:.3e} flux {e_f:.3e} trials {list(trials)} "
          f"oracle {list(o.trace.trials)}")
    if v.dtype == F64:
        assert np.array_equal(r.trace["evals"][0, 1:it + 1], o.trace.proj_evals)
        assert int(r.proj_evals[0]) == sum(o.trace.proj_evals) + o.trace.init_proj_evals
        assert np.array_equal(trials, o.trace.trials)
        assert e_d <= 1e-10 and e_x <= 1e-8 and e_f <= 1e-9, (e_d, e_x, e_f)
    else:
        assert e_d <= FP32_DISCR and e_x <= FP32_IMAGE and e_f <= FP32_FLUX, (e_d, e_x, e_f)


@pytest.mark.parametrize("v", [v for v in VARIANTS if v.kernel], ids=lambda v: v.label)
def test_padded_output_divisors(bs, v):
    """The masked kernels divide every A and A^T by the weight of the embedded kernels (div_a, div_at: the kernel
    normalisation of convolve_fft).  The front end normalises the kernels, so the divisors it passes are 1 to the last
    bit and leave a consumer that skips its division unseen.  Kernels scaled by 4 with divisors of 4 (scaling by a power
    of two commutes with every rounding) must restore the image of the front end's padded solve."""
    gn, psf, args, kw, div, o = _inputs_and_oracle(v.shape, v.kernel, "beta")
    npdt = np.float64 if v.dtype == F64 else np.float32
    geo = bs.engine.PaddedGeometry(v.shape[0], v.shape[1], v.kernel, v.kernel)
    common = dict(divergence=div, flux=[args["flux"]], betaParam=args["betaParam"], dtype=v.dtype, verbose=False, **kw)
    ref = bs.solve_batch(gn[None].astype(npdt), psf.astype(npdt), args["bkg"][None], padded=True, **common)
    plan = bs.get_plan(geo.P, geo.P, v.dtype)
    big, div_a = geo.kernel(psf, npdt)
    bigt, div_at = geo.kernel(psf.conj().T, npdt)
    plan.set_psf(4 * big)
    plan.set_psf_adjoint(4 * bigt)
    r = bs.solve_batch(geo.embed(gn[None], npdt), None, geo.embed(args["bkg"][None], npdt), plan=plan, psf_is_set=True,
                       region=geo.region, div_a=4 * div_a, div_at=4 * div_at, adjoint_second_psf=True, **common)
    x = r.x[0][geo.rows, geo.cols]
    e_x = np.abs(x - ref.x[0]).max() / np.abs(ref.x[0]).max()
    print(f"\n{v.label} kernels x 4, divisors x 4: image {e_x:.3e} from the normalised solve")
    assert int(r.status[0]) == 0 and int(r.iters[0]) == int(ref.iters[0])
    assert e_x <= (1e-12 if v.dtype == F64 else 1e-6), e_x
    assert np.abs(r.discr[0] - ref.discr[0]).max() <= (1e-12 if v.dtype == F64 else 1e-6) * np.abs(ref.discr[0]).max()


# ------------------------------------------------------------------------------------------------
# the fp32 operator at every transform kind
# ------------------------------------------------------------------------------------------------
def _check_f32_operator(plan, x, psf):
    """apply_psf forward and adjoint with one PSF and with one PSF per image against numpy in fp64 on the same fp32
    values; returns the worst error in units of 2^-23 * log2(ny * nx) * max|ref|."""
    ny, nx = x.shape[1:]
    unit = 2.0 ** -23 * math.log2(ny * nx)
    worst = 0.0
    xd = x.astype(np.float64)
    for psfs in (psf, psf[0]):
        plan.set_psf(psfs)
        tf = np.fft.fftn(np.fft.fftshift(psfs.astype(np.float64), axes=(-2, -1)), axes=(-2, -1))
        for adj in (False, True):
            y = plan.apply_psf(x, adjoint=adj)
            ref = np.real(np.fft.ifftn((np.conj(tf) if adj else tf) * np.fft.fftn(xd, axes=(1, 2)), axes=(1, 2)))
            for i in range(x.shape[0]):
                worst = max(worst, float(np.abs(y[i] - ref[i]).max() / (unit * np.abs(ref[i]).max())))
    return worst


def _f32_operator_inputs(shape, n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n,) + shape).astype(np.float32)
    psf = rng.random((n,) + shape)
    psf /= psf.sum(axis=(1, 2), keepdims=True)
    return x, psf.astype(np.float32)


@pytest.mark.parametrize("shape,cfg", [(s, {}) for s in
                                       [(32, 32), (64, 64), (128, 128), (256, 256), (512, 512), (64, 256), (1024, 1024),
                                        (31, 31), (33, 20), (5, 7), (32, 31), (100, 75), (375, 375), (450, 450),
                                        (30, 30), (31, 29), (17, 24), (9, 12), (15, 15), (31, 64)]]
                         + [((256, 256), dict(cluster_size=g)) for g in (1, 2, 4, 8, 16)])
def test_fp32_operator_every_transform_kind(bs, shape, cfg):
    """Power-of-two radix stages, dense axes, wrapped axes, multi-CTA clusters (256^2 at G = 1 ... 16) and frame mode
    (1024^2): the fp32 operator within FP32_OP_C * 2^-23 * log2(ny * nx) of the largest value."""
    x, psf = _f32_operator_inputs(shape, 3 if shape[0] * shape[1] >= 1 << 18 else 5, shape[0] * 31 + shape[1])
    plan = bs.Plan(shape[0], shape[1], F32, **cfg)
    if "cluster_size" in cfg:
        assert plan.info()["cluster_size"] == cfg["cluster_size"]
    if shape == (1024, 1024):
        assert plan.info()["num_clusters"] == 1                     # frame mode
    worst = _check_f32_operator(plan, x, psf)
    plan.close()
    print(f"\nfp32 operator {shape} {cfg}: worst {worst:.3f} x 2^-23 log2(n) max|ref|")
    assert worst <= FP32_OP_C, worst


# ------------------------------------------------------------------------------------------------
# batches across images
# ------------------------------------------------------------------------------------------------
_BATCH_KW = dict(RUNS["beta"])
del _BATCH_KW["divergence"]


def test_frame_mode_batch_per_image_psf(bs):
    """Three images in one frame-mode launch, one PSF per image (the per-image spectrum offset of bsgp_frame_kernel), a
    different beta0 each, 2-D backgrounds: every image bit-identical to its single solve on the same plan, and at the
    fp64 bar against the oracle."""
    from oracle import sgp_oracle as orc
    plan = bs.Plan(256, 256, cluster_size=-1)
    assert plan.info()["num_clusters"] == 1 and plan.info()["cluster_size"] >= 8
    scenes = [_scene(bs, (256, 256), 0, seed=90 + i, fwhm=f) for i, f in enumerate((2.5, 3.5, 4.5))]
    gn, psf, bkg = (np.stack([s[k] for s in scenes]) for k in range(3))
    flux = np.array([s[3] for s in scenes])
    b0 = np.array([1.0248357, 0.9703266, 1.0815099])
    r = bs.solve_batch(gn, psf, bkg, divergence="beta", flux=flux, betaParam=b0, plan=plan, trace=True, verbose=False, **_BATCH_KW)
    for i in range(3):
        s = bs.solve_batch(gn[i:i + 1], psf[i], bkg[i:i + 1], divergence="beta", flux=flux[i:i + 1], betaParam=float(b0[i]), plan=plan,
                           trace=True, verbose=False, **_BATCH_KW)
        assert np.array_equal(r.x[i], s.x[0]) and np.array_equal(r.discr[i], s.discr[0]) and int(r.iters[i]) == int(s.iters[0]), i
        o = orc.solve(gn[i], psf[i], bkg[i], divergence="beta", flux=np.float64(flux[i]), betaParam=float(b0[i]), verbose=False, **_BATCH_KW)
        it = int(r.iters[i])
        assert int(r.status[i]) == 0 and it == o.iters
        assert np.array_equal(r.trace["evals"][i, 1:it + 1], o.trace.proj_evals)
        assert np.abs(r.discr[i, :it + 1] - o.discr).max() <= 1e-10 * np.abs(o.discr).max()
        assert np.abs(r.x[i] - o.x).max() <= 1e-8 * np.abs(o.x).max()
        assert abs(r.x[i].sum() - flux[i]) <= 1e-9 * flux[i]
    plan.close()


@pytest.mark.parametrize("shape,cfg", [((32, 32), {}), ((256, 256), {}), ((128, 128), dict(cluster_size=8)),
                                       ((64, 64), dict(cluster_size=-1))], ids=["small", "tile", "cluster8", "frame"])
def test_mixed_statuses_in_one_batch(bs, shape, cfg):
    """Images that end with BSGP_ST_BAD_FLUX (flux <= 0 with the flux projection) and BSGP_ST_EMPTY_BOUNDS (flux + bkg < 0:
    no positive entry in flux / (flux + bkg) * A^T gn; the reference fails there on the minimum of an empty array) between
    good ones: the bad images report their status after no iteration, the good ones are bit-identical to their single
    solves on the same plan."""
    from oracle import sgp_oracle as orc
    plan = bs.Plan(shape[0], shape[1], **cfg)
    info = plan.info()
    if cfg.get("cluster_size") == -1:
        assert info["num_clusters"] == 1
    elif "cluster_size" in cfg:
        assert info["cluster_size"] == cfg["cluster_size"]
    scenes = [_scene(bs, shape, 0, seed=40 + i) for i in range(5)]
    gn = np.stack([s[0] for s in scenes])
    psf = scenes[0][1]
    flux = np.array([s[3] for s in scenes])
    bkg = np.full(5, 300.0)
    flux[1] = -1.0                                           # BSGP_ST_BAD_FLUX
    bkg[3] = -2.0 * flux[3]                                  # BSGP_ST_EMPTY_BOUNDS
    b0 = np.array([1.0248357, 0.9703266, 1.0815099, 1.0064847, 1.0882026])
    with np.errstate(all="ignore"), pytest.raises(ValueError):
        orc.solve(gn[3], psf, np.float64(bkg[3]), divergence="beta", flux=np.float64(flux[3]), betaParam=float(b0[3]), verbose=False,
                  **_BATCH_KW)
    r = bs.solve_batch(gn, psf, bkg, divergence="beta", flux=flux, betaParam=b0, plan=plan, verbose=False, **_BATCH_KW)
    capi = bs._capi
    assert list(r.status) == [capi.ST_OK, capi.ST_BAD_FLUX, capi.ST_OK, capi.ST_EMPTY_BOUNDS, capi.ST_OK]
    assert int(r.iters[1]) == 0 and int(r.iters[3]) == 0
    for i in (0, 2, 4):
        s = bs.solve_batch(gn[i:i + 1], psf, bkg[i:i + 1], divergence="beta", flux=flux[i:i + 1], betaParam=float(b0[i]), plan=plan,
                           verbose=False, **_BATCH_KW)
        assert int(s.status[0]) == 0 and int(r.iters[i]) == int(s.iters[0]) == _BATCH_KW["MAXIT"], i
        assert np.array_equal(r.x[i], s.x[0]) and np.array_equal(r.discr[i], s.discr[0]), i
    plan.close()


# ------------------------------------------------------------------------------------------------
# device pow and the beta-divergence helpers against long double
# ------------------------------------------------------------------------------------------------
BETAS_POW = (0.5, 0.9887296104546054, 1.0001, 1.0248357, 1.5, 2.0, 2.5)


def _pow_inputs(y, rng):
    """den for p1 = den^y: the random ranges of test_pow_inline_accuracy, mantissas on both sides of the sqrt(2) split of
    pow_inline, exact powers of two and 1, |y log den| on both sides of 600 (the switch to the library pow), subnormals."""
    n = 200_000
    parts = [10.0 ** rng.uniform(lo, hi, n) for lo, hi in ((-8, 0.3), (-40, 0.3), (-300, 300))]
    hi_words = np.array([0x3ff6a09e + d for d in (-1, 0, 1)], np.int64)
    lo_words = np.array([0, 1, 0x7fffffff, 0xffffffff], np.int64)
    split = []
    for e in (-1022, -600, -40, -3, -1, 0, 1, 5, 60, 700, 1023):
        for h in hi_words:
            for lw in lo_words:
                bits = ((int(h) & 0x000fffff) | ((1023 + e) << 20)) << 32 | int(lw)
                split.append(np.array([bits], np.uint64).view(np.float64)[0])
    parts.append(np.array(split))
    parts.append(np.ldexp(1.0, np.arange(-1022, 1024, 3)))
    parts.append(np.array([1.0]))
    if y != 0.0:
        t = np.array([599.0, 599.9999, 600.0001, 601.0])
        with np.errstate(over="ignore", under="ignore"):
            edge = np.exp(np.concatenate([t, -t]) / y)
        parts.append(edge[np.isfinite(edge) & (edge >= 2.2250738585072014e-308)])
    parts.append(np.array([5e-324, 1e-320, 1e-310, 2.2250738585072014e-308 / 2, np.nextafter(2.2250738585072014e-308, 0)]))
    return np.concatenate(parts)


@pytest.mark.parametrize("beta", BETAS_POW)
def test_device_pow_against_long_double(bs, beta):
    """p1 = den^(beta - 1) of bsgp_beta_grad_terms_host is pow_inline as compiled for the GPU (rcp.approx + Newton, nvcc's
    FMA contraction), not its g++ emulation: <= 1.3 ulp against 80-bit long-double pow, the slow path included (measured
    on a B200: 1.19 ulp worst, at beta = 2.5).  u must be gn * (p1 / den) bit for bit (IEEE multiply and divide)."""
    L = bs._capi.lib()
    rng = np.random.default_rng(int(beta * 1e6))
    y = np.float64(beta) - 1.0
    den = np.ascontiguousarray(_pow_inputs(y, rng))
    gn = rng.uniform(0.5, 2.0, den.size)
    p1, u = np.empty_like(den), np.empty_like(den)
    bs._capi.check(L.bsgp_beta_grad_terms_host(den.ctypes.data, gn.ctypes.data, den.size, float(beta), p1.ctypes.data, u.ctypes.data, 0))
    with np.errstate(all="ignore"):
        ref = np.power(den.astype(np.longdouble), np.longdouble(y))
        ref64 = ref.astype(np.float64)
        assert np.array_equal(u, gn * (p1 / den), equal_nan=True)
    ok = np.isfinite(ref64) & (ref64 != 0)
    assert np.array_equal(np.isinf(p1), np.isinf(ref64))
    ulp = np.spacing(np.abs(ref64[ok])).astype(np.longdouble)
    err = np.abs(p1[ok].astype(np.longdouble) - ref[ok]) / ulp
    k = int(np.argmax(err))
    print(f"\npow beta={beta}: worst {float(err[k]):.3f} ulp at den={den[ok][k]!r} over {int(ok.sum())} values")
    assert float(err.max()) <= 1.3, (float(err.max()), den[ok][k])


def _split_fsum(t):
    """math.fsum of long-double values, exact to the 128-bit precision of (hi, lo) double pairs."""
    hi = t.astype(np.float64)
    lo = (t - hi.astype(np.longdouble)).astype(np.float64)
    return math.fsum(np.concatenate([hi, lo]).tolist())


@pytest.mark.parametrize("n", [1, 255, 256, 257, 592 * 256 + 1, 10 ** 6 + 3])
def test_beta_div_against_long_double(bs, n):
    """betaDiv (sgp.py:441-458) on a partial block, exactly one block, one grid of 592 blocks plus one element and the
    grid-stride loop, at beta in {0, 1, 1.0001, 1.5, 2}: against a long-double restatement summed exactly, relative to
    the sum of the absolute terms (near beta = 1 the value itself cancels).  Measured on a B200: 7.1e-16 worst (10^6 + 3
    elements, beta = 1.0001)."""
    rng = np.random.default_rng(n)
    model = rng.uniform(0.5, 50.0, n)
    data = rng.uniform(0.1, 60.0, n)
    y, x = model.astype(np.longdouble), data.astype(np.longdouble)
    for b in (0.0, 1.0, 1.0001, 1.5, 2.0):
        v = bs.betaDiv(model, data, b)
        bl = np.longdouble(b)
        if b == 0.0:
            terms = [x / y, -np.log(x / y), np.full(1, -np.longdouble(n))]
        elif b == 1.0:
            terms = [x * np.log(x / y), -x, y]
        else:
            k = 1 / (bl * (bl - 1))
            terms = [k * x ** bl, k * (bl - 1) * y ** bl, -k * bl * x * y ** (bl - 1)]
        t = np.concatenate(terms)
        ref, scale = _split_fsum(t), _split_fsum(np.abs(t))
        rel = abs(v - ref) / scale
        print(f"\nbetaDiv n={n} beta={b}: {rel:.2e} of sum |terms|")
        assert rel <= 1e-14, (b, rel)
