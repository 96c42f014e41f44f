"""Sharding of independent restorations over the GPUs of one box (SURVEY.md §8e).

Every stamp / subdivision / beta-init value is its own optimisation problem (the reference loops over
them one at a time: application_sgp_star_stamps.py:56-105, application_sgp_subdivisions.py:83-107), so
the batch is dealt to the ranks and nothing is exchanged until the final gather of the restored images
and their per-image scalars.  One process per GPU; torch.distributed is used for the gather only (NCCL
on the GPU box: two `all_gather_into_tensor` calls on device tensors, no host round trip; gloo in the
CPU tests).

Dealing.  Iteration counts vary by an order of magnitude (9..160) and grow as beta approaches 1, so the
images are ranked by expected cost (|beta - 1| ascending for beta-SGP, batch order otherwise) and dealt
round-robin in that ranking: every rank receives the same mix of cheap and expensive solves.

Width.  A rank that holds fewer images than the solver has cluster slots (320 subdivisions over 8 GPUs =
40 images for 71 slots) is bounded by its longest solve, not by throughput; `engine.auto_config` then
selects a wider CTA configuration (more threads per image, fewer images in flight), which roughly halves
the per-iteration latency of one image.
"""
from __future__ import annotations

import numpy as np


def expected_cost_rank(n_items, betaParam=None, divergence="beta"):
    """Permutation of 0..n-1, most expensive expected solve first (stable).  divergence may be one per image (a mixed
    batch): its beta-SGP images are ranked by |beta - 1|, its KL images follow, as engine._queue_order hands them out."""
    if isinstance(divergence, str):
        if divergence != "beta" or betaParam is None:
            return np.arange(n_items)
        is_beta = np.ones(n_items, bool)
    else:
        is_beta = np.asarray([d == "beta" for d in divergence], bool)
    b = np.broadcast_to(np.asarray(1.0 if betaParam is None else betaParam, dtype=np.float64).reshape(-1), (n_items,))
    return np.argsort(np.where(is_beta, np.abs(b - 1.0), np.inf), kind="stable")


def shard_indices(n_items, rank, world_size, cost_rank=None):
    """Indices of the batch entries owned by `rank` (ascending).  Without a ranking: rank, rank + W, rank + 2W, ...;
    with `cost_rank` (expected_cost_rank): the ranking is dealt in snake order (ranks 0..W-1, then W-1..0, ...), so no
    rank systematically receives the most expensive entry of every round."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    if cost_rank is None:
        return np.arange(rank, n_items, world_size)
    cost_rank = np.asarray(cost_rank)
    if cost_rank.shape != (n_items,):
        raise ValueError("cost_rank must be a permutation of the batch")
    pos = np.arange(n_items)
    rnd, k = pos // world_size, pos % world_size
    owner = np.where(rnd % 2 == 0, k, world_size - 1 - k)
    return np.sort(cost_rank[owner == rank])


def shard_counts(n_items, world_size, snake=False):
    if not snake:
        return [len(range(r, n_items, world_size)) for r in range(world_size)]
    pos = np.arange(n_items)
    rnd, k = pos // world_size, pos % world_size
    owner = np.where(rnd % 2 == 0, k, world_size - 1 - k)
    return [int(np.sum(owner == r)) for r in range(world_size)]


_index_cache = {}


def _gather_indices(n_items, world_size, cost_rank, dev):
    """(counts, cap, dest, keep) of the gather, with the two index tensors cached on the device: building them from host
    arrays every call is a pageable host-to-device copy, which blocks the host until the solve kernel in front of it has
    finished and so serialises the launches of the gather behind the kernel instead of queueing them under it."""
    import torch
    key = (n_items, world_size, str(dev), None if cost_rank is None else np.asarray(cost_rank).tobytes())
    hit = _index_cache.get(key)
    if hit is None:
        parts = [shard_indices(n_items, r, world_size, cost_rank) for r in range(world_size)]
        counts = [len(p_) for p_ in parts]
        cap = max(counts) if counts else 0
        dest = torch.as_tensor(np.concatenate(parts) if n_items else np.zeros(0, np.int64), device=dev, dtype=torch.long)
        keep = torch.as_tensor(np.concatenate([r * cap + np.arange(counts[r]) for r in range(world_size)]) if n_items else np.zeros(0, np.int64),
                               device=dev, dtype=torch.long)
        if len(_index_cache) > 64:
            _index_cache.clear()
        hit = _index_cache[key] = (counts, cap, dest, keep)
    return hit



def gather_to_all(local, n_items, rank, world_size, group=None, cost_rank=None):
    """All-gather per-image results.  `local` maps name -> tensor [n_local, ...] for the images of
    shard_indices(n_items, rank, world_size, cost_rank); returns name -> tensor [n_items, ...] in the original batch
    order on every rank.  The image-sized field "x" travels in its own dtype; all other fields are packed into one
    float64 matrix, so the whole gather is two collectives (shards are padded to the largest one).  Ranks with an
    empty shard contribute zero rows."""
    import torch
    import torch.distributed as dist
    names = list(local)
    ref = local[names[0]]
    dev = ref.device
    counts, cap, dest, keep = _gather_indices(n_items, world_size, cost_rank, dev)
    for name in names:
        if local[name].shape[0] != counts[rank]:
            raise ValueError(f"{name}: expected {counts[rank]} local rows, got {local[name].shape[0]}")

    def gather(t):
        """[n_local, k] -> [n_items, k] in batch order"""
        pad = torch.zeros((cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        pad[:t.shape[0]] = t
        if world_size == 1:
            allr = pad
        else:
            allr = torch.empty((world_size * cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(allr, pad, group=group)
        full = torch.empty((n_items,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        full[dest] = allr[keep]
        return full

    out = {}
    small = [n for n in names if n != "x"]
    if "x" in local:
        out["x"] = gather(local["x"])
    if small:
        widths = [int(np.prod(local[n].shape[1:])) if local[n].dim() > 1 else 1 for n in small]
        packed = torch.cat([local[n].reshape(local[n].shape[0], wd).to(torch.float64) for n, wd in zip(small, widths)], dim=1)
        full = gather(packed)
        o = 0
        for n, wd in zip(small, widths):
            out[n] = full[:, o:o + wd].reshape((n_items,) + tuple(local[n].shape[1:])).to(local[n].dtype)
            o += wd
    return out


_FIELDS = ("x", "iters", "status", "discr", "times", "beta_final", "proj_evals", "ls_trials")


def solve_batch_sharded(gn, psf, bkg, flux=None, betaParam=1.005, x0=None, obj=None, divergence="beta", group=None, device=None,
                        width="auto", timing=None, cost_rank=None, per_image=None, source=None, **kw):
    """Every rank passes the FULL batch and gets the full result back: rank r restores the images
    shard_indices(B, r, W, expected_cost_rank(...)) on its own GPU (engine.solve_batch, one persistent kernel launch) and
    the per-image results are all-gathered.  No data-path collective: the images are independent problems.

    numpy inputs -> dict of numpy arrays; CUDA tensors -> dict of CUDA tensors (inputs are sliced, solved and gathered on
    the device, asynchronously on the current stream; NCCL process group required when world_size > 1).
    psf: [ny,nx] shared or [B,ny,nx]; bkg: scalar, [B] or [B,ny,nx]; flux / betaParam: scalar or [B]; x0 / obj: [B,ny,nx].
    per_image: B keyword dicts of a mixed batch (engine.solve_batch); each rank receives the rows of its images.
    source: [B] shared observations (engine.solve_batch): gn, psf, bkg, x0 and obj then hold one entry per observation, and
    each rank receives only the observations its solves read, with the map renumbered to them; B is the number of solves.
    width: "auto" picks the CTA configuration from the local batch size (engine.auto_config), or (cluster_size, threads).
    cost_rank: optional precomputed expected_cost_rank(...) (a host array); give it when betaParam is a device tensor, so
    that the dealing does not have to copy betaParam back to the host (a synchronisation) on every call.
    timing: optional dict; with CUDA tensors it receives timing["solve"] = (start, end) CUDA events around the local solve
    (what bench.py divides the algorithmic bytes by) and timing["plan"] = the plan's info.
    Iterate snapshots (engine.solve_batch(snapshot_every=...)) are not gathered across ranks: call engine.solve_batch."""
    if "snapshot_every" in kw:
        raise ValueError("solve_batch_sharded does not support snapshot_every; call solve_batch on one GPU")
    import torch
    import torch.distributed as dist
    from . import engine
    is_dist = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if is_dist else 1
    rank = dist.get_rank(group) if is_dist else 0
    on_dev = engine._is_tensor(gn) and gn.is_cuda
    if device is None:
        device = (gn.device.index or 0) if on_dev else int(__import__("os").environ.get("LOCAL_RANK", rank))
    n_obs = int(gn.shape[0])
    if source is not None:
        source = engine._source_map(source, gn, psf, bkg, flux, betaParam, x0, obj)
    B = n_obs if source is None else int(source.size)
    ny, nx = int(gn.shape[-2]), int(gn.shape[-1])
    if per_image is not None:
        engine._check_per_image(per_image, B)
        betaParam = engine._row_betas(betaParam, per_image, B)
        flux, per_image = engine._row_flux(flux, per_image, B)
    if cost_rank is None:
        b_host = betaParam.detach().cpu().numpy() if engine._is_tensor(betaParam) else betaParam
        kinds = divergence if per_image is None else [row.get("divergence", divergence) for row in per_image]
        cost_rank = expected_cost_rank(B, b_host, kinds)
    cost_rank = np.ascontiguousarray(cost_rank)
    idx = shard_indices(B, rank, world, cost_rank)
    n_local = len(idx)
    # the observations this rank's solves read (all of them are per solve without a map), and the map renumbered to them
    obs_idx, local_source = idx, None
    if source is not None:
        obs_idx, local_source = np.unique(source[idx], return_inverse=True)
        local_source = np.ascontiguousarray(local_source.reshape(-1), dtype=np.int32)
    use_cuda = on_dev or (is_dist and dist.get_backend(group) == "nccl")
    dev = torch.device("cuda", device) if use_cuda else torch.device("cpu")
    maxit = int(kw.get("MAXIT", 500))
    if per_image is not None:
        maxit = max(int(row.get("MAXIT", maxit)) for row in per_image)     # the trace stride of the whole batch

    if on_dev:
        skey = ("sel", B, rank, world, str(gn.device), cost_rank.tobytes(), None if source is None else source.tobytes())
        sel = _index_cache.get(skey)
        if sel is None:
            sel = _index_cache[skey] = (torch.as_tensor(idx, device=gn.device, dtype=torch.long),
                                        torch.as_tensor(obs_idx, device=gn.device, dtype=torch.long))

        def take(a, per_image_ndim, obs=False):
            """this rank's entries of a per-solve array, or with obs=True of a per-observation one"""
            if a is None:
                return None
            rows, n, t = (obs_idx, n_obs, sel[1]) if obs else (idx, B, sel[0])
            if engine._is_tensor(a):
                return a.index_select(0, t) if a.dim() == per_image_ndim + 1 and a.shape[0] == n else a
            a = np.asarray(a)
            return a[rows] if a.ndim == per_image_ndim + 1 and a.shape[0] == n else a
    else:
        gn = np.asarray(gn)

        def take(a, per_image_ndim, obs=False):
            if a is None:
                return None
            rows, n = (obs_idx, n_obs) if obs else (idx, B)
            a = np.asarray(a)
            return a[rows] if a.ndim == per_image_ndim + 1 and a.shape[0] == n else a

    if n_local:
        dtype = "float32" if str(gn.dtype).endswith("float32") else "float64"
        plan = None
        if width is not None:
            cs, th = engine.auto_config(ny, nx, n_local) if width == "auto" else width
            plan = engine.get_plan(ny, nx, dtype, device, cs, th)
        bk = bkg
        if engine._is_tensor(bkg):
            bk = take(bkg, 2, True) if bkg.dim() == 3 else (take(bkg, 0, True) if bkg.dim() == 1 else bkg)
        else:
            ba = np.asarray(bkg)
            bk = ba[obs_idx] if ba.ndim >= 1 and ba.shape[0] == n_obs and ba.size > 1 else ba
        ev = None
        if timing is not None and on_dev:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        args = (take(gn, 2, True), take(psf, 2, True), bk)
        kwargs = dict(divergence=divergence, flux=take(flux, 0), betaParam=take(betaParam, 0), x0=take(x0, 2, True), obj=take(obj, 2, True),
                      device=device, plan=plan, dtype=dtype, **kw)
        if per_image is not None:
            kwargs["per_image"] = [per_image[int(i)] for i in idx]
        if local_source is not None:
            kwargs["source"] = local_source
        if ev:
            if plan is not None:
                plan.set_psf(args[1])                      # PSF spectra outside the bracket: it times the solve kernel alone
                args, kwargs = (args[0], None, args[2]), dict(kwargs, psf_is_set=True)
            ev[0].record()
        r = engine.solve_batch(*args, **kwargs)
        if ev:
            ev[1].record()
            timing["solve"] = ev
            timing["plan"] = (plan or engine.get_plan(ny, nx, dtype, device)).info()
        local = {k: (getattr(r, k) if on_dev else torch.as_tensor(np.ascontiguousarray(getattr(r, k))).to(dev)) for k in _FIELDS}
        for k in ("discr", "times"):                    # a mixed batch: this shard's largest MAXIT may be below the batch's
            t = local[k]
            if t.shape[1] < maxit + 1:
                local[k] = torch.cat([t, torch.zeros((t.shape[0], maxit + 1 - t.shape[1]), dtype=t.dtype, device=t.device)], dim=1)
    else:
        # an empty shard (B < world size): nothing to solve, zero rows for the gather (the collective must still be entered)
        xdt = gn.dtype if on_dev else (torch.float32 if str(gn.dtype).endswith("float32") else torch.float64)
        f64, i32 = dict(dtype=torch.float64, device=dev), dict(dtype=torch.int32, device=dev)
        local = dict(x=torch.zeros((0, ny, nx), dtype=xdt, device=dev), iters=torch.zeros(0, **i32), status=torch.zeros(0, **i32),
                     discr=torch.zeros((0, maxit + 1), **f64), times=torch.zeros((0, maxit + 1), **f64), beta_final=torch.zeros(0, **f64),
                     proj_evals=torch.zeros(0, **i32), ls_trials=torch.zeros(0, **i32))
    if world == 1:
        full = local                                      # shard_indices(B, 0, 1, .) is 0..B-1: nothing to gather or re-order
    else:
        full = gather_to_all(local, B, rank, world, group=group, cost_rank=cost_rank)
    if on_dev:
        return full
    return {k: v.cpu().numpy() for k, v in full.items()}
