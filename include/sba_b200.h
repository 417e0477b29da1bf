/*
 * sba_b200 -- C ABI of the B200-native bundle-adjustment hot path (libsba_b200.so).
 *
 * The reference (centreborelli/sat-bundleadjust) has no plugin API: its hot path is ordinary Python
 * (bundle_adjust/ba_core.py) on top of scipy, plus ONE native boundary, the ctypes call into
 * lib/disp_to_h.so (bundle_adjust/s2p/triangulation.py:107-118 -> c/disp_to_h.c:40-42).
 * Each entry point below names the reference interface it replaces.  All functions return 0 on
 * success or a negative SBA_E_* code; none of them calls exit().  Unless a parameter is documented
 * as a device pointer, pointers are HOST pointers owned by the caller and host<->device copies
 * happen inside the call.  A handle is bound to the CUDA device that was current at creation and to
 * one CUDA stream; calls on the same handle must not overlap.
 */
#ifndef SBA_B200_H
#define SBA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SBA_OK 0
#define SBA_E_INVALID (-1)      /* bad argument / unsupported combination */
#define SBA_E_CUDA (-2)         /* CUDA runtime error (sba_last_error() has the text) */
#define SBA_E_NUMERIC (-3)      /* non-finite residuals at the initial point (scipy raises ValueError there) */
#define SBA_E_NOMEM (-4)

enum { SBA_MODEL_AFFINE = 0, SBA_MODEL_PERSPECTIVE = 1, SBA_MODEL_RPC = 2 };
enum { SBA_LOSS_LINEAR = 0, SBA_LOSS_HUBER = 1, SBA_LOSS_SOFT_L1 = 2, SBA_LOSS_CAUCHY = 3, SBA_LOSS_ARCTAN = 4 };

typedef struct sba_problem sba_problem;

/* Problem description = the fields of the reference's BundleAdjustmentParameters that ba_core.fun
 * reads (bundle_adjust/ba_params.py:78-181, SURVEY.md section 8b). */
typedef struct sba_problem_desc {
    int32_t cam_model;        /* SBA_MODEL_*                                   p.cam_model */
    int32_t n_cam;            /* M                                             p.n_cam */
    int32_t n_pts;            /* N (tracks held by this rank)                  p.n_pts */
    int64_t n_obs;            /* K                                             p.n_obs */
    int32_t n_params;         /* variables per camera: 3 | 5 | 6 | 8 | 11       p.n_params */
    int32_t n_cam_params;     /* columns of cam_params: 8 | 11 | 9             p.cam_params.shape[1] */
    int32_t n_cam_fix;        /* first n_cam_fix cameras are frozen            p.n_cam_fix */
    int32_t n_pts_fix;        /* first n_pts_fix points are frozen             p.n_pts_fix */
    const int64_t *cam_ind;   /* (K) camera of each observation                p.cam_ind */
    const int64_t *pts_ind;   /* (K) track of each observation, non-decreasing p.pts_ind */
    const double *pts2d;      /* (K,2) observed (col,row)                      p.pts2d */
    const double *pts2d_w;    /* (K) observation weights                       p.pts2d_w */
    const double *cam_params; /* (M, n_cam_params) initial camera parameters   p.cam_params */
    const double *rpc_coefs;  /* (M, 90) RPC tables, NULL unless cam_model == RPC:
                                 row_off col_off lat_off lon_off alt_off row_scl col_scl lat_scl lon_scl alt_scl,
                                 row_num[20] row_den[20] col_num[20] col_den[20]   p.cameras[i] (rpcm.RPCModel) */
    int32_t rpc_float32;      /* 1: round the RPC projection to float32 like ba_core.py:150 (fun parity) */
    /* multi-GPU: this rank's position among the ranks that share the cameras; the tracks are sharded */
    int32_t rank, world_size;
    /* COMMON_K (ba_params.py:167-171): the last n_common (0 | 3 | 5) of the n_params camera variables are ONE set of
       unknowns shared by all cameras.  The device vector keeps n_params slots per camera: the shared values live in
       camera 0's slots, the same slots of cameras 1..M-1 are unused and must be 0.  Requires n_cam_fix == 0. */
    int32_t n_common;
    /* Choices that sba_problem_create otherwise makes from the problem itself (0 = automatic).  The ranks of a multi-GPU solve must
       agree on both (their exchanges differ): the distributed driver creates with 0, compares, and re-creates with a common value. */
    int32_t engine;           /* 1: pattern engine (fails if it does not apply), 2: generic engine */
    int32_t solver;           /* 1: dense Cholesky of the reduced camera system, 2: matrix-free PCG */
} sba_problem_desc;

/* Solver options = the reference's ls_params (bundle_adjust/ba_core.py:222-241) + scipy's gtol default */
typedef struct sba_solve_opts {
    int32_t loss;             /* SBA_LOSS_* */
    double f_scale;
    double ftol, xtol, gtol;  /* scipy.optimize.least_squares meanings */
    int32_t max_nfev;         /* "max_iter" of the reference = max residual evaluations */
    int32_t verbose;
    /* measurement controls (not in the reference; 0 = off) */
    int32_t max_iterations;   /* stop after this many outer trust-region iterations (status 0) */
    int32_t timed_from;       /* iter_ms / phase_ms accumulate over iterations >= timed_from */
    int64_t l2_flush_bytes;   /* > 0: overwrite a scratch buffer of this size between iterations, outside
                                 the per-iteration event pairs, so that every timed iteration starts L2-cold */
    int32_t no_phase_timing;  /* 1: time whole iterations only (two events per iteration instead of ~18) */
} sba_solve_opts;

/* phases of one trust-region iteration, for sba_solve_info.phase_ms */
enum { SBA_PH_ASSEMBLE = 0,   /* fused residual + Jacobian + robust weights + U/V/g blocks (G2) */
       SBA_PH_SCALE_JVP,      /* x_scale update, |g|, J*(D^2 g) for the damping (scipy reg_term) */
       SBA_PH_POINT_PREP,     /* damped 3x3 inverse factors + Z = (Jc^T Jp) G^T */
       SBA_PH_SCHUR,          /* reduced camera system S, rhs (G3) */
       SBA_PH_CHOLESKY,       /* dense FP64 factorisation + solves (G4) */
       SBA_PH_BACKSUB,        /* point updates (G6) */
       SBA_PH_SUBSPACE,       /* second basis vector, norms, J*[t1 t2] */
       SBA_PH_STEP_EVAL,      /* x + step, residual + cost at the trial point (G1) */
       SBA_PH_COUNT };

typedef struct sba_solve_info {
    int32_t status;           /* scipy status: 0 max_nfev, 1 gtol, 2 ftol, 3 xtol, 4 ftol+xtol */
    int32_t nfev, njev;       /* residual evaluations / Jacobian (assembly) evaluations */
    int32_t iterations;       /* outer trust-region iterations */
    double cost_init, cost;   /* 0.5 * sum(rho) at x0 and at the solution */
    double optimality;        /* ||J^T f||_inf at the solution */
    double solve_ms;          /* device time of the iteration loop (CUDA events) */
    int32_t chol_retries;     /* times the reduced camera system had to be re-damped */
    int32_t gpu_launches;     /* kernels launched by this call */
    int32_t timed_iterations; /* iterations that contributed to iter_ms / phase_ms */
    double iter_ms;           /* sum of per-iteration device times (CUDA events) over the timed iterations */
    double phase_ms[8];       /* the same, split by phase (SBA_PH_*) */
    int32_t explicit_subspace_passes; /* iterations that ran the explicit J*[t1 t2] pass (= all of them: the algebraic
                                         shortcut through the normal equations cancels catastrophically) */
    int32_t pcg_solves;       /* reduced camera systems solved by block-Jacobi PCG (0 on the dense Cholesky path) ... */
    int32_t pcg_iterations;   /* ... and the CG iterations they took in total */
} sba_solve_info;

/* Optional hook for the multi-GPU exchange step: must SUM `count` doubles at device pointer `buf`
 * across all ranks, in place, enqueued on the handle's stream (e.g. torch.distributed.all_reduce). */
typedef int (*sba_allreduce_fn)(void *user, double *device_buf, int64_t count);

const char *sba_last_error(void);
int sba_version(void);

/* Replaces: the implicit set-up done on every ba_core.fun call (gathers cam_params[cam_ind], pts3d[pts_ind])
 * and ba_core.build_jacobian_sparsity (ba_core.py:186-219).  `stream` is a cudaStream_t (0 = default). */
int sba_problem_create(sba_problem **out, const sba_problem_desc *desc, void *stream);
int sba_problem_destroy(sba_problem *p);
/* Device slabs of destroyed problems are cached for the next sba_problem_create (the pipeline solves twice per run);
 * this returns them to the driver. */
int sba_release_cached_memory(void);
int sba_problem_set_allreduce(sba_problem *p, sba_allreduce_fn fn, void *user);
/* Multi-GPU exchange without the hook: a device-side one-shot all-reduce over NVLink peer memory.  Every rank calls
 * sba_comm_export (writes the 64-byte CUDA IPC handle of its symmetric buffer), the handles are gathered by any means
 * (e.g. torch.distributed.all_gather_object), and every rank calls sba_comm_import with all of them in rank order.
 * When imported, the solver uses it instead of the hook.  The problems of all ranks must be destroyed collectively. */
int sba_comm_export(sba_problem *p, void *handle_out_64_bytes);
int sba_comm_import(sba_problem *p, const void *handles_world_x_64_bytes);
/* Attach to the exchange buffers this process already shares with the same peers (kept across problems: mapping them
 * costs ~15 ms).  Returns 1 when attached, 0 when the export / gather / import sequence is needed. */
int sba_comm_try_reuse(sba_problem *p);
/* number of variables n = n_cam * n_params + 3 * n_pts */
int64_t sba_problem_num_vars(const sba_problem *p);
/* Which of the two device engines serves this problem (diagnostics / measurement): 1 = pattern-major (reduced camera
 * system of at most 132 unknowns, n_params <= 6: fused passes, nothing per-observation stored), 0 = generic (static pair
 * lists, any size up to 4096 camera unknowns).  SBA_ENGINE=generic in the environment forces 0. */
int sba_problem_engine(const sba_problem *p);
/* Solver of the reduced camera system chosen for this problem: 0 = dense Cholesky, 1 = block-Jacobi PCG. */
int sba_problem_solver(const sba_problem *p);

/* Replaces ba_core.fun(v, p) (ba_core.py:157-183): x (n) -> weighted residuals r (2K), interleaved.
 * Also returns 0.5*sum(rho(r)) for the given loss in *cost (may be NULL). */
int sba_residuals(sba_problem *p, const double *x, double *r, int32_t loss, double f_scale, double *cost);

/* Jacobian pieces at x for tests: per-observation camera block (K,2,n_params), point block (K,2,3),
 * both including observation weights but NOT the robust rescale.  Any output may be NULL. */
int sba_jacobian_blocks(sba_problem *p, const double *x, double *Jc, double *Jp);

/* Normal-equation blocks at x (robust rescale applied): U (M,c,c), V (N,6: xx xy xz yy yz zz), g (n). */
int sba_normal_blocks(sba_problem *p, const double *x, int32_t loss, double f_scale, double *U, double *V, double *g);

/* The reduced camera system of the damped normal equations at x exactly as the solver forms it (scaling D taken from
 * this one evaluation; shared calibration folded, see n_common): S = U + reg D_c^2 - W (V + reg D_p^2)^-1 W^T,
 * rhs = -(g_c - W (V + reg D_p^2)^-1 g_p).  For the parity tests of the Schur complement (there is no reference
 * counterpart: the reference never forms S).  Host buffers; S is (n_cam n_params)^2, column-major. */
int sba_reduced_system(sba_problem *p, const double *x, int32_t loss, double f_scale, double reg, double *S, double *rhs);

/* Posterior covariance at x (host pointers, caller's layouts).  sigma2 > 0: used as given; else estimated and
 * returned in *sigma2_out.  cov_cam (M*n_params)^2 column-major, cov_pts (N,6); either may be NULL.
 * SBA_E_INVALID: world_size > 1, PCG problems (no dense S), n_common > 0, dof <= 0.
 * SBA_E_NUMERIC: rank-deficient S (gauge not fixed) or a free point with a singular block.
 * J is the Jacobian of the weighted residuals at x over the free variables, rescaled for the robust loss like the solver does
 * (scipy's scale_for_robust_loss_function); H = J^T J = [[U, W], [W^T, V]], S = U - W V^-1 W^T.  cov_cam = sigma2 S^-1 (rows
 * and columns of frozen cameras 0); cov_pts[t] = sigma2 (V_t^-1 + V_t^-1 W_t^T S^-1 W_t V_t^-1) as xx xy xz yy yz zz (frozen
 * points 0).  Estimated sigma2 = 2 cost(x) / (2K - n_free) (scipy curve_fit's convention).  S is rejected as rank deficient
 * when a pivot of its Cholesky factor has L_kk^2 <= 1e-12 U_kk; *min_pivot_ratio_out (may be NULL) receives the smallest
 * L_kk^2 / U_kk over the free camera slots.  The pivot test catches round-off pivots, it does not certify full rank: in
 * ill-conditioned geometry a single free direction (e.g. the scale left by one frozen perspective camera) can pass it, so
 * fix the gauge with at least two frozen cameras or with frozen points.  The handle stays usable for solves, also after an
 * error return. */
int sba_covariance(sba_problem *p, const double *x, int32_t loss, double f_scale, double sigma2,
                   double *cov_cam, double *cov_pts, double *sigma2_out, double *min_pivot_ratio_out);
/* Device time (CUDA events) of the phases of the last sba_covariance call on this handle: reduced system (assembly, Schur
 * pass, cost), factorisation + pivot test, inverse, point pass. */
int sba_covariance_phase_ms(const sba_problem *p, double ms_out[4]);

/* Replaces scipy.optimize.least_squares(fun, x0, jac_sparsity=A, x_scale='jac', method='trf', ...)
 * as called by ba_core.run_ba_optimization (ba_core.py:284-297).
 * x0 (n) in, x (n) out, r (2K) = un-scaled residuals at the solution (res.fun), may be NULL. */
int sba_solve(sba_problem *p, const double *x0, const sba_solve_opts *opts, double *x, double *r, sba_solve_info *info);

/* sba_solve plus the two per-observation reprojection-error vectors the reference's driver returns
 * (compute_reprojection_error, ba_core.py:304-305,335-349), computed on the device: err_init (K) at x0 and err (K) at the
 * solution; either may be NULL.  Saves the 2 x 2K residual read-backs and the host-side norms of the end-to-end call. */
/* The same with device pointers (caller's layouts): nothing but the steering scalars crosses PCIe. */
int sba_solve_errors_device(sba_problem *p, const double *x0_dev, const sba_solve_opts *opts, double *x_dev,
                            double *err_init_dev, double *err_dev, sba_solve_info *info);
int sba_solve_errors(sba_problem *p, const double *x0, const sba_solve_opts *opts, double *x, double *err_init, double *err,
                     sba_solve_info *info);

/* Same solve with x0 / x / r as DEVICE pointers (inputs already resident in HBM; nothing is copied
 * to the host except the few scalars that steer the iteration). */
int sba_solve_device(sba_problem *p, const double *x0_dev, const sba_solve_opts *opts, double *x_dev, double *r_dev,
                     sba_solve_info *info);

/* One fused residual + analytic Jacobian + robust weighting + J^T J / J^T r block assembly pass at the
 * DEVICE vector x_dev, timed alone (bench: "Jacobian observations per second").  ms = device time. */
int sba_assemble_device(sba_problem *p, const double *x_dev, int32_t loss, double f_scale, float *ms);

/* Exact 2-D trust-region subproblem (host); replaces scipy/optimize/_lsq/common.py:171-219. */
int sba_tr2d(const double B[4], const double g[2], double Delta, double p_out[2]);

/* ------------------------------------------------------------------------------------------------
 * Batched RPC kernels (replace rpcm.RPCModel.projection / .localization and c/rpc.c).
 * rpc: 90 doubles, layout as sba_problem_desc.rpc_coefs.  n points, arrays are (n) each.
 * ---------------------------------------------------------------------------------------------- */
/* c/rpc.c:442-452 eval_rpci / rpcm projection: (lon,lat,alt) -> (col,row) */
int sba_rpc_projection(const double *rpc, const double *lon, const double *lat, const double *alt, int64_t n,
                       double *col, double *row);
/* cam_utils.apply_rpc_projection (cam_utils.py:217-231): ECEF (n,3) -> (n,2) incl. geo_utils.py:236-255 */
int sba_rpc_projection_ecef(const double *rpc, const double *xyz, int64_t n, double *colrow);
/* c/rpc.c:378-439 eval_rpc (iterative) / rpcm localization: (col,row,alt) -> (lon,lat); delta = first probe */
int sba_rpc_localization(const double *rpc, const double *col, const double *row, const double *alt, int64_t n,
                         double delta, double *lon, double *lat);
/* The same for n_cam cameras in ONE launch (tables (n_cam, 90)).  shared_points != 0: lon/lat/alt (col/row/alt) hold n values used for
 * every camera (one grid projected through all cameras, bundle_adjust/ba_rpcfit.py:78-95 per camera); else (n_cam, n).  Outputs (n_cam, n). */
int sba_rpc_projection_batch(const double *tables, int32_t n_cam, const double *lon, const double *lat, const double *alt, int64_t n,
                             int32_t shared_points, double *col, double *row);
int sba_rpc_localization_batch(const double *tables, int32_t n_cam, const double *col, const double *row, const double *alt, int64_t n,
                               int32_t shared_points, double delta, double *lon, double *lat);
/* Measurement only (bench.py --workload rpc): device-resident time per pass of the batched RPC kernels over n_cam cameras x n
 * points (kind 0 projection, 1 localisation, 2 triangulation between tables 2j and 2j+1), inputs uploaded once. */
int sba_rpc_throughput(int32_t kind, const double *tables_n_cam_x_90, int32_t n_cam, const double *a, const double *b,
                       const double *c, const double *d, int64_t n, double delta, int32_t reps, double *out, double *ms);

/* The reference's one native entry point, same signature and struct layout (c/disp_to_h.c:40-42,
 * c/rpc.h:14-32): two-view RPC triangulation of n_kp matches.  rpc_a / rpc_b point to `struct rpc`
 * (181 doubles).  Runs batched on the GPU; buffers are host pointers like in the reference. */
void stereo_corresp_to_lonlatalt(double *lonlatalt, float *err, float *kp_a, float *kp_b, int n_kp,
                                 void *rpc_a, void *rpc_b);
int sba_stereo_corresp_to_lonlatalt(double *lonlatalt, float *err, const float *kp_a, const float *kp_b, int64_t n_kp,
                                    const void *rpc_a, const void *rpc_b);

/* Initial 3-D points of the feature tracks, replaces the pair loop of ft_triangulate.init_pts3d
 * (bundle_adjust/feature_tracks/ft_triangulate.py:57-127): every track x every pair of `pairs` (in list order) whose two
 * cameras see the track is triangulated -- cv2.triangulatePoints' DLT for 3x4 matrices (:18-34), the two-view RPC
 * triangulation + geodetic -> ECEF for RPCs (:37-54) -- and averaged with the reference's float32 running mean, all in
 * ONE launch.  Tracks in CSR form: observations of track t are track_ptr[t] .. track_ptr[t+1]-1, cameras ascending.
 * cams: (n_cam, 12) row-major matrices, or (n_cam, 181) `struct rpc` (c/rpc.h:14-32) for SBA_MODEL_RPC.
 * pts3d_out: (n_tracks, 3) float32; tracks without a suitable pair are zero, like in the reference.  Host pointers. */
int sba_init_pts3d(int32_t cam_model, const double *cams, int32_t n_cam, const int64_t *track_ptr, const int32_t *cam_idx,
                   const double *pts2d, int64_t n_tracks, const int32_t *pairs_n_x_2, int32_t n_pairs, float *pts3d_out);
/* ft_triangulate.linear_triangulation_multiple_pts (:18-34): n matches between two 3x4 matrices -> (n,3) doubles. */
int sba_linear_triangulation(const double *P1, const double *P2, const double *pts1_n_x_2, const double *pts2_n_x_2, int64_t n,
                             double *pts3d_out);

/* Batched RPC refit, replaces ba_rpcfit.weighted_lsq (bundle_adjust/ba_rpcfit.py:88-153) for n_cam cameras at once:
 * target (n_cam, n_samples, 2) = (col,row), input_locs (n_cam, n_samples, 3) = (lon,lat,alt) -> rpc_out (n_cam, 90)
 * in the table layout above; h = ridge (1e-3), tol = RMSE change that stops the re-weighting (1e-2 px), max_iter (20).
 * n_iter_out (n_cam) / rmse_out (n_cam) may be NULL. */
int sba_rpcfit_weighted_lsq(const double *target, const double *input_locs, int32_t n_cam, int32_t n_samples, double h,
                            double tol, int32_t max_iter, double *rpc_out, int32_t *n_iter_out, double *rmse_out);

/* Outlier detection between the two bundle-adjustment passes -- device part of bundle_adjust/ba_outliers.py:14-58
 * (get_elbow_value) and :112-153 (compute_obs_to_remove).  Host buffers in and out.
 * sba_outlier_elbow: one stable radix sort of all K observations by (camera, reprojection error), then per camera the
 * elbow of the sorted curve (the sample furthest from the chord first-last, evaluated in the reference's operation
 * order so that the arg-max is bit-identical).  stats is n_cam x 5: elbow value, the order statistics at positions
 * q_lo[c] and q_hi[c] (what np.percentile interpolates between), the maximum, the arg-max position; counts (optional)
 * receives the observations per camera.
 * sba_outlier_mark: remove[k] = err[k] > thr[cam_ind[k]]. */
int sba_outlier_elbow(const double *err, const int32_t *cam_ind, int64_t K, int32_t n_cam, const int64_t *q_lo,
                      const int64_t *q_hi, double *stats, int64_t *counts);
int sba_outlier_mark(const double *err, const int32_t *cam_ind, int64_t K, int32_t n_cam, const double *thr,
                     uint8_t *remove);

/* FP64 dense Cholesky solve of an n x n SPD system on the device (host buffers in/out), exposed for
 * tests of the reduced-camera-system factorisation.  A is column-major, overwritten by L. */
int sba_cholesky_solve(double *A, double *b, int32_t n, int32_t *info);
/* The same solve repeated `reps` times on device-resident copies; *ms = mean device time (CUDA events) of one solve. */
int sba_cholesky_solve_timed(const double *A, const double *b, int32_t n, int32_t reps, double *x, double *ms);

#ifdef __cplusplus
}
#endif
#endif /* SBA_B200_H */
