"""Shared helpers for the test-suite (test infrastructure)."""
import os

import numpy as np

from oracle import rpc_oracle
from sat_bundleadjust_b200.ba_params import BundleAdjustmentParameters

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def load_ba_golden():
    return np.load(os.path.join(GOLDEN, "ba_golden.npz"))


def load_rpc_golden():
    return np.load(os.path.join(GOLDEN, "rpc_golden.npz"))


def params_from_golden(G, name, params_cls=BundleAdjustmentParameters):
    pre = name + "/"
    ncf, npf, refw = G[pre + "opts"]
    d = {"correction_params": [str(s) for s in G[pre + "correction_params"]], "n_cam_fix": int(ncf),
         "n_pts_fix": int(npf), "ref_cam_weight": float(refw), "reduce": False, "verbose": False}
    return params_cls(G[pre + "C"], G[pre + "pts3d_init"], list(G[pre + "cameras_init"]), str(G[pre + "cam_model"]),
                      [(0, 1)], list(G[pre + "camera_centers"]), d)


def ls_from_golden(G, name):
    pre = name + "/"
    cfg = {}
    for k, v in zip(G[pre + "ls_keys"], G[pre + "ls_vals"]):
        k, v = str(k), str(v)
        cfg[k] = v if k == "loss" else (int(float(v)) if k in ("max_iter", "verbose") else float(v))
    return cfg


def rpc_from_array(a):
    r = rpc_oracle.RPCModel()
    (r.row_offset, r.col_offset, r.lat_offset, r.lon_offset, r.alt_offset,
     r.row_scale, r.col_scale, r.lat_scale, r.lon_scale, r.alt_scale) = [float(v) for v in a[:10]]
    r.row_num, r.row_den, r.col_num, r.col_den = [list(a[10 + 20 * i: 30 + 20 * i]) for i in range(4)]
    return r


def rpc_ba_params_from_golden(G, corr, params_cls=BundleAdjustmentParameters):
    cams = [rpc_from_array(a) for a in G["rpc_cams"]]
    d = {"correction_params": list(corr), "reduce": False, "verbose": False}
    return params_cls(G["rpcba/C"], G["rpcba/pts3d_init"], cams, "rpc", [(0, 1)], list(G["rpcba/camera_centers"]), d)


def dense_jacobian_from_blocks(p, Jc, Jp):
    """Assemble the dense (2K x n) Jacobian from per-observation blocks (small problems only)."""
    K, c = p.pts_ind.size, p.n_params
    n = p.n_cam * c + 3 * p.n_pts
    J = np.zeros((2 * K, n))
    for k in range(K):
        j, i = int(p.cam_ind[k]), int(p.pts_ind[k])
        J[2 * k:2 * k + 2, j * c:(j + 1) * c] = Jc[k]
        J[2 * k:2 * k + 2, p.n_cam * c + 3 * i: p.n_cam * c + 3 * i + 3] = Jp[k]
    return J


# ---- covariance bounds (test_gpu_covariance.py, test_block_oracle.py) ----------------------------------------------------
EPS = np.finfo(np.float64).eps


def scaled_cond(S, u_diag):
    """2-norm condition number of S in the basis scaled by the un-reduced diagonal U_kk (numpy, oracle side)."""
    d = np.sqrt(u_diag)
    return np.linalg.cond(S / np.outer(d, d)) if S.size else 1.0


def cond_tol(base, kappa, n):
    """
    The bound for a float64 S^-1: the fixed bound `base`, or the forward-error bound n eps kappa of a Cholesky-based inverse
    (n free camera slots, kappa = scaled_cond of S from the oracle), whichever is larger.  S = U - W V^-1 W^T is formed by
    cancellation against U, so its scaled entries carry ~eps of round-off whatever the method; satellite geometry is
    ill-conditioned by nature (a narrow-field camera's rotation and translation nearly coincide), kappa ~ 1e9 .. 1e11 here,
    which makes a fixed 1e-7 (1e-9 at the metric size) unreachable there.
    """
    return max(base, n * EPS * kappa)


def scaled_inv(A):
    """inverse in the Jacobi-scaled basis (accurate for badly scaled SPD matrices)"""
    d = np.sqrt(np.diag(A))
    return np.linalg.inv(A / np.outer(d, d)) / np.outer(d, d)


def normalised_err(A, B):
    """max_ij |A - B|_ij / sqrt(B_ii B_jj); entries where the oracle's variances are 0 must agree exactly"""
    d = np.sqrt(np.abs(np.diag(B)))
    den = np.outer(d, d)
    mask = den > 0
    err = np.zeros_like(A)
    err[mask] = np.abs(A - B)[mask] / den[mask]
    assert not np.abs(A - B)[~mask].any(), "entries where the oracle's variances are 0 must be exactly 0"
    return err.max() if err.size else 0.0


# ---- pattern-engine layout from the host harness (csrc/sba_pattern.h) -----------------------------------------------------
def _harness():
    import ctypes
    return ctypes.CDLL(os.path.join(HERE, "host_harness", "libmodel_harness.so"))


def pattern_layout(cam_ind, pts_ind, M, N, n_pts_fix=0, n_cta=148, warps=16):
    """The layout the pattern engine builds, with the units of its `warps`-wide (assembly) assignment; None if it does not apply."""
    import ctypes
    lib = _harness()
    ip = ctypes.POINTER(ctypes.c_int)
    cam = np.ascontiguousarray(cam_ind, dtype=np.int32)
    tp = np.ascontiguousarray(np.searchsorted(pts_ind, np.arange(N + 1), side="left"), dtype=np.int32)
    K = cam.size
    sizes = (ctypes.c_int * 8)()
    null = ctypes.cast(None, ip)
    args = [cam.ctypes.data_as(ip), tp.ctypes.data_as(ip), ctypes.c_longlong(K), M, N, n_pts_fix, n_cta, warps, sizes]
    lib.hh_pattern_layout(*args, *([null] * 5))
    if not sizes[0]:
        return None
    out = {"trk_new2old": np.zeros(N, np.int32), "obs_new2old": np.zeros(K, np.int32), "track_ptr": np.zeros(N + 1, np.int32),
           "units": np.zeros((sizes[1], 8), np.int32), "warp_unit0": np.zeros(n_cta * warps + 1, np.int32)}
    lib.hh_pattern_layout(*args, *[out[k].ctypes.data_as(ip) for k in ("trk_new2old", "obs_new2old", "track_ptr", "units", "warp_unit0")])
    out["n_frozen"], out["n_tiles"], out["n_runs"], out["fill"] = sizes[3], sizes[4], sizes[5], sizes[6] / 1000.0
    return out


def pattern_assignment(cam_ind, pts_ind, M, N, n_pts_fix, nc, which, warps, rows_per_task=3, n_cta=148):
    """(units (n, 8), warp_unit0) of one kernel's assignment: which 0 = jvp1 / backsub, 1 = assembly, 2 = Schur pass."""
    import ctypes
    lib = _harness()
    ip = ctypes.POINTER(ctypes.c_int)
    cam = np.ascontiguousarray(cam_ind, dtype=np.int32)
    tp = np.ascontiguousarray(np.searchsorted(pts_ind, np.arange(N + 1), side="left"), dtype=np.int32)
    cap = 4 * n_cta * warps + N
    units, wu = np.zeros((cap, 8), np.int32), np.zeros(n_cta * warps + 1, np.int32)
    w = [warps if which == k else 16 for k in range(3)]
    n = lib.hh_pattern_assignment(cam.ctypes.data_as(ip), tp.ctypes.data_as(ip), ctypes.c_longlong(cam.size), M, N, n_pts_fix, n_cta,
                                  w[0], w[1], w[2], nc, rows_per_task, which, units.ctypes.data_as(ip), cap, wu.ctypes.data_as(ip))
    assert n >= 0, n
    return units[:n], wu
