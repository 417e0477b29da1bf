"""
Device-resident bundle-adjustment problem: thin Python owner of a `sba_problem` handle.

Consumes the arrays of a `BundleAdjustmentParameters` object (ours or the reference's own,
bundle_adjust/ba_params.py:78-181) and drives libsba_b200.so through its C ABI.  All arithmetic of the
hot path runs in the sm_100a kernels of csrc/; this module only packs pointers.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import LOSS_IDS, MODEL_IDS, ProblemDesc, SolveInfo, SolveOpts, check, dptr, f64

N_CAM_PARAMS = {"affine": 8, "perspective": 11, "rpc": 9}


def rpc_table(rpc):
    """rpcm-style RPC object -> the 90-double table of include/sba_b200.h."""
    return np.concatenate([[rpc.row_offset, rpc.col_offset, rpc.lat_offset, rpc.lon_offset, rpc.alt_offset,
                            rpc.row_scale, rpc.col_scale, rpc.lat_scale, rpc.lon_scale, rpc.alt_scale],
                           np.asarray(rpc.row_num, dtype=np.float64), np.asarray(rpc.row_den, dtype=np.float64),
                           np.asarray(rpc.col_num, dtype=np.float64), np.asarray(rpc.col_den, dtype=np.float64)])


def n_common_params(p):
    """Number of calibration variables shared by all cameras (COMMON_K, bundle_adjust/ba_params.py:167-171), else 0."""
    opt = p.cam_params_to_optimize
    if "K" in opt and "COMMON_K" in opt and "T" in opt and "R" in opt:
        return 3 if p.cam_model == "affine" else 5
    return 0


def check_supported(p):
    if n_common_params(p) and p.n_cam_fix > 0:
        # the reference packs n_cam_opt cameras (ba_params.py:170) but unpacks n_cam (ba_params.py:244): with frozen
        # cameras its own vector is inconsistent, so there is no behaviour to mirror
        raise NotImplementedError("COMMON_K with n_cam_fix > 0 is inconsistent in the reference and not supported")
    if p.cam_model == "rpc" and p.n_params > 6:
        raise ValueError("cam_model 'rpc' has no calibration parameters to optimise")


def initial_vars(p):
    """
    The solver's starting vector: a copy of p.params_opt with the frozen cameras' slots overwritten by
    p.cam_params, which is what the reference's first `fun` call does to its own copy in place
    (bundle_adjust/ba_params.py:246-249 via ba_core.py:276-277).
    """
    x0 = np.array(p.params_opt, dtype=np.float64, copy=True)
    if p.n_cam_fix > 0 and not n_common_params(p):
        c = p.n_params
        x0[: p.n_cam * c].reshape(p.n_cam, c)[: p.n_cam_fix] = p.cam_params[: p.n_cam_fix, :c]
    return x0


def to_device_layout(v, n_common, n_params, n_cam):
    """[K | cam_0[:c'] ... cam_M-1[:c'] | points] (ba_params.py:167-171) -> n_params slots per camera, the shared K in camera 0's."""
    k, c, m = n_common, n_params, n_cam
    v = np.asarray(v, dtype=np.float64)
    x = np.zeros(v.size + (m - 1) * k)
    cams = x[: m * c].reshape(m, c)
    cams[:, : c - k] = v[k: k + m * (c - k)].reshape(m, c - k)
    cams[0, c - k:] = v[:k]
    x[m * c:] = v[k + m * (c - k):]
    return x


def from_device_layout(x, n_common, n_params, n_cam):
    """Inverse of to_device_layout."""
    k, c, m = n_common, n_params, n_cam
    cams = np.asarray(x)[: m * c].reshape(m, c)
    return np.concatenate([cams[0, c - k:], cams[:, : c - k].ravel(), np.asarray(x)[m * c:]])


class DeviceProblem:
    """RAII wrapper of sba_problem_create / sba_problem_destroy."""

    def __init__(self, p, stream=0, rank=0, world_size=1, rpc_float32=True, track_range=None, engine=None, solver=None,
                 cam_prior=None):
        """engine: None (automatic) | "pattern" | "generic";  solver: None (automatic) | "dense" | "pcg";
        cam_prior: None or a ba_priors.CameraPrior (see set_camera_prior)."""
        check_supported(p)
        self.lib = _lib.load()
        self.cam_model = p.cam_model
        cam_ind, pts_ind, pts2d, w = p.cam_ind, p.pts_ind, p.pts2d, p.pts2d_w
        n_pts, n_pts_fix = p.n_pts, p.n_pts_fix
        if track_range is not None:       # this rank's shard: tracks [t0, t1) and the observations they own
            t0, t1 = track_range
            a0, a1 = np.searchsorted(pts_ind, [t0, t1], side="left")
            cam_ind, pts_ind, pts2d, w = cam_ind[a0:a1], pts_ind[a0:a1] - t0, pts2d[a0:a1], w[a0:a1]
            n_pts, n_pts_fix = t1 - t0, int(np.clip(p.n_pts_fix - t0, 0, t1 - t0))
        self.n_cam, self.n_pts, self.n_obs, self.n_params = int(p.n_cam), int(n_pts), int(cam_ind.size), int(p.n_params)
        # frozen points always take their initial coordinates, whatever the caller's vector holds
        # (bundle_adjust/ba_params.py:240-243); frozen cameras are handled on the device from cam_params
        t_first = 0 if track_range is None else track_range[0]
        self._fixed_pts = np.asarray(p.pts3d[t_first: t_first + n_pts_fix], dtype=np.float64).ravel().copy()
        self._keep = [np.ascontiguousarray(cam_ind, dtype=np.int64), np.ascontiguousarray(pts_ind, dtype=np.int64),
                      f64(pts2d), f64(w), f64(p.cam_params)]
        d = ProblemDesc()
        d.cam_model = MODEL_IDS[p.cam_model]
        d.n_cam, d.n_pts, d.n_obs = self.n_cam, self.n_pts, self.n_obs
        d.n_params, d.n_cam_params = self.n_params, self._keep[4].shape[1]
        d.n_cam_fix, d.n_pts_fix = int(p.n_cam_fix), int(n_pts_fix)
        self._n_cam_fix = int(p.n_cam_fix)
        d.cam_ind = self._keep[0].ctypes.data_as(_lib.c_int64_p)
        d.pts_ind = self._keep[1].ctypes.data_as(_lib.c_int64_p)
        d.pts2d, d.pts2d_w, d.cam_params = dptr(self._keep[2]), dptr(self._keep[3]), dptr(self._keep[4])
        if p.cam_model == "rpc":
            self._keep.append(f64(np.array([rpc_table(c) for c in p.cameras])))
            d.rpc_coefs = dptr(self._keep[-1])
        d.rpc_float32 = 1 if rpc_float32 else 0
        d.rank, d.world_size = rank, world_size
        self.n_common = d.n_common = n_common_params(p)
        d.engine = {None: 0, "pattern": 1, "generic": 2}[engine]
        d.solver = {None: 0, "dense": 1, "pcg": 2}[solver]
        self.handle = ctypes.c_void_p()
        check(self.lib.sba_problem_create(ctypes.byref(self.handle), ctypes.byref(d), ctypes.c_void_p(stream)))
        self.n_vars_device = int(self.lib.sba_problem_num_vars(self.handle))
        self.engine = "pattern" if self.lib.sba_problem_engine(self.handle) == 1 else "generic"
        self.solver = "pcg" if self.lib.sba_problem_solver(self.handle) == 1 else "dense"
        # length of the caller's vector (the reference's params_opt layout); the device keeps n_params slots per camera
        self.n_vars = self.n_vars_device - (self.n_cam - 1) * self.n_common
        self._cb = None
        self.cam_prior = None
        if cam_prior is not None:
            self.set_camera_prior(cam_prior)

    def set_camera_prior(self, prior):
        """
        Gaussian prior on the camera variables (sat_bundleadjust_b200.ba_priors.CameraPrior) for the following solves,
        normal_blocks, reduced_system and covariance of this handle; None clears it.  residuals() stays the observation rows.
        """
        if prior is None:
            check(self.lib.sba_problem_set_camera_prior(self.handle, None, None))
            self.cam_prior = None
            return
        if self.n_common:
            raise NotImplementedError("camera priors are not available with COMMON_K (shared calibration)")
        if prior.mean.shape != (self.n_cam, self.n_params):
            raise ValueError("CameraPrior: mean is %s, the problem has (n_cam, n_params) = (%d, %d)"
                             % (prior.mean.shape, self.n_cam, self.n_params))
        mean, info = f64(prior.mean), f64(prior.information)
        check(self.lib.sba_problem_set_camera_prior(self.handle, dptr(mean), dptr(info)))
        self.cam_prior = prior

    def close(self):
        if getattr(self, "handle", None):
            self.lib.sba_problem_destroy(self.handle)
            self.handle = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _to_device_layout(self, v):
        return to_device_layout(v, self.n_common, self.n_params, self.n_cam)

    def _from_device_layout(self, x):
        return from_device_layout(x, self.n_common, self.n_params, self.n_cam)

    def _vars(self, x):
        """float64 device-layout vector (copy if needed) with the frozen points pinned to their initial values"""
        x = f64(x)
        assert x.size == self.n_vars
        if self.n_common:
            x = self._to_device_layout(x)
        if self._fixed_pts.size:
            off = self.n_cam * self.n_params
            if not np.array_equal(x[off: off + self._fixed_pts.size], self._fixed_pts):
                x = x.copy()
                x[off: off + self._fixed_pts.size] = self._fixed_pts
        return x

    def _no_common(self, what):
        if self.n_common:
            raise NotImplementedError("%s is not available with COMMON_K (blocks are per camera)" % what)

    # -- evaluation ------------------------------------------------------------------------------
    def residuals(self, x, loss="linear", f_scale=1.0):
        x = self._vars(x)
        r = np.empty(2 * self.n_obs)
        cost = ctypes.c_double()
        check(self.lib.sba_residuals(self.handle, dptr(x), dptr(r), LOSS_IDS[loss], f_scale, ctypes.byref(cost)))
        return r, cost.value

    def jacobian_blocks(self, x):
        """Per-observation Jacobian blocks d r / d (camera slots), d r / d point.  With COMMON_K the blocks stay per camera:
        the column of a shared variable is the sum of its slot's columns over the cameras."""
        x = self._vars(x)
        Jc = np.empty((self.n_obs, 2, self.n_params))
        Jp = np.empty((self.n_obs, 2, 3))
        check(self.lib.sba_jacobian_blocks(self.handle, dptr(x), dptr(Jc), dptr(Jp)))
        return Jc, Jp

    def normal_blocks(self, x, loss="linear", f_scale=1.0):
        self._no_common("normal_blocks")
        x = self._vars(x)
        c = self.n_params
        U = np.empty((self.n_cam, c, c))
        V = np.empty((self.n_pts, 6))
        g = np.empty(self.n_vars)
        check(self.lib.sba_normal_blocks(self.handle, dptr(x), LOSS_IDS[loss], f_scale, dptr(U), dptr(V), dptr(g)))
        return U, V, g

    def reduced_system(self, x, loss="linear", f_scale=1.0, reg=0.0):
        """(S, rhs) of the damped normal equations reduced onto the cameras, in the device layout (n_params slots per camera)."""
        x = self._vars(x)
        ns = self.n_cam * self.n_params
        S = np.empty((ns, ns), order="F")
        rhs = np.empty(ns)
        check(self.lib.sba_reduced_system(self.handle, dptr(x), LOSS_IDS[loss], ctypes.c_double(f_scale), ctypes.c_double(reg),
                                          dptr(S), dptr(rhs)))
        return S, rhs

    def covariance(self, x, loss="linear", f_scale=1.0, sigma2=None):
        """
        Posterior covariance at x (sat_bundleadjust_b200.ba_covariance has the definitions): (cov_cam (n_cam n_params)^2,
        cov_pts (n_pts, 3, 3), sigma2 (given or estimated), min_pivot_ratio).  A rank-deficient reduced camera system (gauge
        not fixed) or a free point with a singular block raises SbaError.
        """
        self._no_common("covariance")
        n_free = (self.n_cam - self._n_cam_fix) * self.n_params + 3 * (self.n_pts - self._fixed_pts.size // 3)
        dof = 2 * self.n_obs + (self.cam_prior.free_rank(self._n_cam_fix) if self.cam_prior is not None else 0) - n_free
        if not (sigma2 is not None and sigma2 > 0) and dof <= 0:
            raise ValueError("no degrees of freedom left (2 K + prior ranks - n_free = %d): sigma^2 cannot be estimated" % dof)
        x = self._vars(x)
        ns = self.n_cam * self.n_params
        cov_cam = np.empty((ns, ns), order="F")
        cov6 = np.empty((self.n_pts, 6))
        s2, ratio = ctypes.c_double(), ctypes.c_double()
        check(self.lib.sba_covariance(self.handle, dptr(x), LOSS_IDS[loss], ctypes.c_double(f_scale),
                                      ctypes.c_double(sigma2 if sigma2 is not None else 0.0), dptr(cov_cam), dptr(cov6),
                                      ctypes.byref(s2), ctypes.byref(ratio)))
        cov_pts = cov6[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(self.n_pts, 3, 3)
        return cov_cam, cov_pts, s2.value, ratio.value

    def covariance_phase_ms(self):
        """Device time of the phases of the last covariance call: reduced system, factor + pivot test, inverse, points."""
        ms = np.zeros(4)
        check(self.lib.sba_covariance_phase_ms(self.handle, dptr(ms)))
        return dict(zip(["reduced_system", "factor_pivots", "inverse", "points"], ms.tolist()))

    @staticmethod
    def make_opts(loss="linear", f_scale=1.0, ftol=1e-4, xtol=1e-10, gtol=1e-8, max_nfev=300, verbose=0,
                  max_iterations=0, timed_from=0, l2_flush_bytes=0, no_phase_timing=0):
        o = SolveOpts()
        o.loss, o.f_scale, o.ftol, o.xtol, o.gtol = LOSS_IDS[loss], f_scale, ftol, xtol, gtol
        o.max_nfev, o.verbose = int(max_nfev), int(verbose)
        o.max_iterations, o.timed_from, o.l2_flush_bytes = int(max_iterations), int(timed_from), int(l2_flush_bytes)
        o.no_phase_timing = int(no_phase_timing)
        return o

    def solve(self, x0, want_residuals=True, **kw):
        """Host buffers in, host buffers out (the end-to-end call)."""
        x0 = self._vars(x0)
        x = np.empty_like(x0)
        r = np.empty(2 * self.n_obs) if want_residuals else None
        info = SolveInfo()
        opts = self.make_opts(**kw)
        check(self.lib.sba_solve(self.handle, dptr(x0), ctypes.byref(opts), dptr(x), dptr(r) if r is not None else None,
                                 ctypes.byref(info)))
        if self.n_common:
            x = self._from_device_layout(x)
        return x, r, info.as_dict()

    def solve_with_errors(self, x0, **kw):
        """The end-to-end call of ba_core.run_ba_optimization: x, err_init, err (un-weighted pixel errors, computed on the device)."""
        x0 = self._vars(x0)
        x = np.empty_like(x0)
        err_init, err = np.empty(self.n_obs), np.empty(self.n_obs)
        info = SolveInfo()
        opts = self.make_opts(**kw)
        check(self.lib.sba_solve_errors(self.handle, dptr(x0), ctypes.byref(opts), dptr(x), dptr(err_init), dptr(err),
                                        ctypes.byref(info)))
        if self.n_common:
            x = self._from_device_layout(x)
        return x, err_init, err, info.as_dict()

    def solve_device(self, x0_ptr, x_ptr=None, r_ptr=None, **kw):
        """Device pointers (ints) in and out (device layout); nothing but the steering scalars crosses PCIe."""
        info = SolveInfo()
        opts = self.make_opts(**kw)
        check(self.lib.sba_solve_device(self.handle, ctypes.c_void_p(x0_ptr), ctypes.byref(opts),
                                        ctypes.c_void_p(x_ptr) if x_ptr else None,
                                        ctypes.c_void_p(r_ptr) if r_ptr else None, ctypes.byref(info)))
        return info.as_dict()

    def solve_errors_device(self, x0_ptr, x_ptr, err_init_ptr, err_ptr, **kw):
        """solve_with_errors with device pointers (caller's layouts)."""
        info = SolveInfo()
        opts = self.make_opts(**kw)
        vp = ctypes.c_void_p
        check(self.lib.sba_solve_errors_device(self.handle, vp(x0_ptr), ctypes.byref(opts), vp(x_ptr), vp(err_init_ptr), vp(err_ptr),
                                               ctypes.byref(info)))
        return info.as_dict()

    def assemble_device(self, x_ptr, loss="linear", f_scale=1.0):
        ms = ctypes.c_float()
        check(self.lib.sba_assemble_device(self.handle, ctypes.c_void_p(x_ptr), LOSS_IDS[loss], f_scale, ctypes.byref(ms)))
        return ms.value

    def connect_peers(self, all_gather_object):
        """
        Map the symmetric exchange buffers of all ranks (CUDA IPC over NVLink) so that the per-iteration all-reduces run
        as device-side one-shot kernels.  `all_gather_object(obj) -> list` must return every rank's object in rank order
        (e.g. a wrapper of torch.distributed.all_gather_object).
        """
        if self.lib.sba_comm_try_reuse(self.handle) == 1:      # the process already shares buffers with these peers
            return
        mine = ctypes.create_string_buffer(64)
        check(self.lib.sba_comm_export(self.handle, mine))
        handles = all_gather_object(bytes(mine.raw))
        check(self.lib.sba_comm_import(self.handle, b"".join(handles)))

    def set_allreduce(self, fn):
        """fn(device_ptr: int, count: int) must SUM-reduce `count` doubles in place across ranks."""
        def trampoline(_user, ptr, count):
            try:
                fn(int(ptr), int(count))
                return 0
            except Exception as exc:   # never let an exception cross the C boundary
                print("sba allreduce hook failed:", exc)
                return 1
        self._cb = _lib.ALLREDUCE_FN(trampoline)
        check(self.lib.sba_problem_set_allreduce(self.handle, self._cb, None))
