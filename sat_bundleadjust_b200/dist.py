"""
Multi-GPU bundle adjustment: observations shard by track across the ranks of one box
(SURVEY.md section 8e).

Observations are sorted by track (bundle_adjust/ba_params.py:138-149), so rank r owns a contiguous
track range [t_r, t_{r+1}) and the contiguous observation range it induces.  Point blocks (V, g_p,
the point elimination and the back-substitution) are rank-local; the cameras are replicated.  The
exchange step is one SUM all-reduce of the rank's partial camera system per trust-region iteration
([U | g_c] after the assembly, [S | rhs] after the Schur complement) plus a handful of scalars; every
rank then factors the same reduced camera system redundantly, so all ranks take identical steps.

Plumbing only: torch.distributed (NCCL over NVLink on the GPU box, gloo in the CPU tests) moves the
bytes; the arithmetic stays in libsba_b200.so.
"""
import os

import numpy as np


def shard_ranges(pts_ind, n_pts, world_size):
    """
    Cut the track range [0, n_pts) into `world_size` contiguous pieces holding ~equal numbers of
    observations.  Returns a list of (t0, t1).  Deterministic; every rank computes the same cuts.
    When there are fewer tracks with work than ranks the trailing ranges are empty.
    """
    pts_ind = np.asarray(pts_ind)
    K = pts_ind.size
    track_ptr = np.concatenate([[0], np.cumsum(np.bincount(pts_ind, minlength=n_pts))])     # first observation of each track
    cuts = [0]
    for r in range(1, world_size):
        target = (K * r) // world_size
        t = int(np.searchsorted(track_ptr, target, side="left"))
        t = min(max(t, cuts[-1]), n_pts)
        cuts.append(t)
    cuts.append(n_pts)
    return [(cuts[r], cuts[r + 1]) for r in range(world_size)]


def local_vars(x, n_cam_vars, track_range):
    """[cameras | all points] -> [cameras | this rank's points]."""
    t0, t1 = track_range
    return np.concatenate([x[:n_cam_vars], x[n_cam_vars + 3 * t0: n_cam_vars + 3 * t1]])


def merge_vars(x_locals, n_cam_vars):
    """Per-rank solutions -> the global variable vector (cameras are identical on all ranks)."""
    return np.concatenate([x_locals[0][:n_cam_vars]] + [xl[n_cam_vars:] for xl in x_locals])


class _CudaView:
    """Zero-copy view of `count` doubles at a raw device pointer, importable by torch.as_tensor."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr, False), "version": 2}


def run_ba_optimization_distributed(p, ls_params=None, group=None, cam_prior=None):
    """
    Multi-GPU counterpart of ba_core.run_ba_optimization, to be called by every rank of an initialised
    torch.distributed NCCL process group (one process per GPU).  Every rank passes the same `p`.
    Returns (vars_init, vars_ba, err_init, err_ba, nfev, info) with the global vectors on every rank.
    `cam_prior` (a ba_priors.CameraPrior, the same on every rank) adds a Gaussian prior on the camera variables; rank 0's
    kernels add its terms once, before each exchange.

    Each rank uploads only its own shard, the per-iteration exchanges run over NVLink peer memory, and the results
    (x, err_init, err of every shard) are all-gathered on the device and brought back with one copy into pinned memory.
    """
    import time

    import torch
    import torch.distributed as dist

    from . import ba_core
    from ._lib import SbaError
    from .solver import DeviceProblem, from_device_layout, initial_vars, n_common_params

    k_common = n_common_params(p)                  # COMMON_K: the caller's vector is [K | cameras | points] (ba_params.py:167-171)
    t_start = time.perf_counter()
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    cfg = ba_core.init_optimization_config(ls_params)
    cache = getattr(p, "_sba_shard_cache", None)
    if cache is None or cache[0] != (world, p.n_pts, p.pts_ind.size):
        ranges = shard_ranges(p.pts_ind, p.n_pts, world)
        a = [tuple(int(v) for v in np.searchsorted(p.pts_ind, [t0, t1])) for t0, t1 in ranges]
        try:
            p._sba_shard_cache = ((world, p.n_pts, p.pts_ind.size), ranges, a)
        except AttributeError:
            pass
    else:
        ranges, a = cache[1], cache[2]
    if any(a1 == a0 for a0, a1 in a):
        raise ValueError("fewer tracks with observations than ranks: use a smaller process group")
    ncv = p.n_cam * p.n_params                                     # camera part of the device vector (n_params slots per camera)
    ncv_ref = ncv - (p.n_cam - 1) * k_common                       # ... and of the caller's vector
    x0 = initial_vars(p)
    stream = torch.cuda.current_stream().cuda_stream
    n_loc = [ncv + 3 * (t1 - t0) for t0, t1 in ranges]
    k_loc = [a1 - a0 for a0, a1 in a]
    longest = max(n + 2 * k for n, k in zip(n_loc, k_loc))

    def hook(ptr, count):
        t = torch.as_tensor(_CudaView(ptr, count), device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)

    def gather_obj(obj):
        out = [None] * world
        dist.all_gather_object(out, obj, group=group)
        return out

    t_prep = time.perf_counter()
    failure = None
    buf = torch.zeros(longest, dtype=torch.float64, device="cuda")
    info = None
    # The ranks must run the same engine and the same reduced-system solver (their exchange sequences differ), but each decides
    # from its own shard (tile fill, track lengths, table sizes): create, compare, and where they disagree re-create everybody
    # with the choice every shard supports (generic engine / PCG).
    create_error = None
    try:
        prob = DeviceProblem(p, stream=stream, rank=rank, world_size=world, track_range=ranges[rank])
        mine = [int(prob.engine == "pattern"), int(prob.solver == "dense")]
    except Exception as exc:                           # agreed on below: no rank may be left waiting in a collective
        create_error, prob, mine = exc, None, [-1, -1]
    choice = torch.tensor(mine, dtype=torch.int32, device="cuda")
    lo, hi = choice.clone(), choice.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    lo_l = lo.tolist()
    if min(lo_l) < 0:
        if prob is not None:
            prob.close()
        raise create_error if create_error is not None else SbaError("the problem could not be created on another rank")
    if not torch.equal(lo, hi):
        prob.close()
        prob = DeviceProblem(p, stream=stream, rank=rank, world_size=world, track_range=ranges[rank],
                             engine="pattern" if lo_l[0] else "generic", solver="dense" if lo_l[1] else "pcg")
    with prob:
        if cam_prior is not None:                      # after the re-create above: every rank, on the handle that solves
            prob.set_camera_prior(cam_prior)
        t_create = time.perf_counter()
        prob.set_allreduce(hook)                       # NCCL fall-back for exchanges that do not fit the peer buffer
        if os.environ.get("SBA_COMM", "peer") == "peer":
            prob.connect_peers(gather_obj)
        t_connect = time.perf_counter()
        xl0 = torch.from_numpy(prob._vars(local_vars(x0, ncv_ref, ranges[rank]))).cuda()
        nl, kl = n_loc[rank], k_loc[rank]
        base = buf.data_ptr()
        try:
            info = prob.solve_errors_device(xl0.data_ptr(), base, base + 8 * nl, base + 8 * (nl + kl), loss=cfg["loss"],
                                            f_scale=cfg["f_scale"], ftol=cfg["ftol"], xtol=cfg["xtol"], max_nfev=cfg["max_iter"])
        except SbaError as exc:                        # raised after the barrier below, so that no peer is left spinning
            failure = exc
        t_solve = time.perf_counter()
        dist.barrier(group=group)                      # peers keep reading each other's buffers until everybody is done
    t_close = time.perf_counter()
    # every rank learns whether any rank failed, and all raise together
    flag = torch.tensor([1.0 if failure is not None else 0.0], dtype=torch.float64, device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.SUM, group=group)
    if flag.item() > 0:
        if failure is not None and "not finite" in str(failure):
            raise ValueError("Residuals are not finite in the initial point.") from failure
        raise failure if failure is not None else SbaError("the solve failed on another rank")
    # one all-gather of [x_local | err_init | err] per rank (variable length -> padded to the longest shard), compacted on the
    # device into [x | err_init | err] and brought back with ONE copy into page-locked memory; the returned arrays are views of
    # that buffer (torch's caching host allocator recycles it once the caller drops them), so the host never re-copies them
    out = torch.empty((world, longest), dtype=torch.float64, device="cuda")
    dist.all_gather_into_tensor(out, buf, group=group)
    res = torch.cat([out[0, :ncv]] + [out[r, ncv: n_loc[r]] for r in range(world)]
                    + [out[r, n_loc[r]: n_loc[r] + k_loc[r]] for r in range(world)]
                    + [out[r, n_loc[r] + k_loc[r]: n_loc[r] + 2 * k_loc[r]] for r in range(world)])
    host = torch.empty(res.numel(), dtype=torch.float64, pin_memory=True)
    host.copy_(res, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    h = host.numpy()
    n_all, k_all = ncv + 3 * p.n_pts, sum(k_loc)
    x, err0, err1 = h[:n_all], h[n_all: n_all + k_all], h[n_all + k_all:]
    if k_common:                                                   # device layout -> [K | cameras | points]
        x = from_device_layout(x, k_common, p.n_params, p.n_cam)
    t_end = time.perf_counter()
    info["wall_s"] = {"prepare": t_prep - t_start, "create": t_create - t_prep, "connect": t_connect - t_create,
                      "solve": t_solve - t_connect, "close": t_close - t_solve, "gather": t_end - t_close}
    return x0, x, err0, err1, info["nfev"], info
