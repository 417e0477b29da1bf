#!/usr/bin/env python
"""
Benchmark of the bundle-adjustment hot path (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|1m|small|cfg3|cfg3a|cfg4s]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one trust-region (Levenberg-Marquardt) iteration of the
workload the metric is quoted on ("LM iters/s and Jacobian obs/s at 1M obs"): BASELINE config 2 at twice its
track count -- synthetic 10-view perspective BA, 2e5 tracks / ~1e6 observations, soft_l1 loss,
correction_params R+T (`--workload 1m`, the default; `cfg2` is config 2 itself and is reported next to it under
"secondary" at N = 1).  At N > 1 every rank gets its own 2e5 tracks (weak scaling, the 10 cameras are shared)
and the per-iteration exchange is the SUM all-reduce of the partial camera system.

  value   = observations x iterations / second, device time (CUDA events) summed over exactly K
            iterations, inputs resident in HBM, L2 overwritten between iterations, max over ranks
  e2e     = the same unit through the public API ba_core.run_ba_optimization (host numpy buffers in,
            host numpy buffers out; problem upload, the whole solve and the read-back inside the timed region)
  roofline= algorithmic bytes / measured device time of the dominant phase of the iteration, against the
            measured HBM copy bandwidth of MEASURED_PEAKS.json
  cpu_baseline = the reference's path (oracle port: numpy residual + scipy TRF/2-point/LSMR) on this box's CPU
`--impl reference` times that CPU path alone, in the same unit, on the same workload.
`--dump-outputs DIR` writes what the last timed solve returned (camera and point variables, cost) as .npy files; the
inputs are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
Beyond 25 steps the timed iterations run as several solves of at most 25 iterations that each restart from the same
start (with W untimed iterations first), and the dump is the result of the last one: compare dumps taken with the same
--steps and --warmup.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_cam, tracks per GPU, p_vis, cam_model, correction_params, description)
    "cfg2": (10, 100000, 0.5, "perspective", ["R", "T"],
             "BASELINE config 2: synthetic 10-view perspective BA, 1e5 tracks / ~5e5 observations, soft_l1, R+T"),
    "1m": (10, 200000, 0.5, "perspective", ["R", "T"],
           "the metric's size: BASELINE config 2 at 2e5 tracks -- 10-view perspective BA, ~1e6 observations, soft_l1, R+T"),
    "5m": (10, 1000000, 0.5, "perspective", ["R", "T"],
           "10-view perspective BA, 1e6 tracks / ~5e6 observations, soft_l1, R+T (HBM-resident working set >> L2)"),
    "small": (6, 4000, 0.5, "perspective", ["R", "T"], "smoke-size: 6 views, 4e3 tracks"),
    # BASELINE configs 3 and 4 per GPU (parity / scaling cases, not the bench line): 8 x 125k tracks = 1e6 tracks, ~5e6 obs
    "cfg3": (50, 125000, 0.1, "perspective", ["R", "T"],
             "BASELINE config 3 shard: 50-view perspective BA, 1.25e5 tracks / ~6e5 observations per GPU, soft_l1, R+T"),
    "cfg3a": (50, 125000, 0.1, "affine", ["R", "T"],
              "BASELINE config 3 shard: 50-view affine BA, 1.25e5 tracks / ~6e5 observations per GPU, soft_l1, R+T"),
    "cfg3full": (50, 1000000, 0.1, "perspective", ["R", "T"],
                 "BASELINE config 3 whole: 50-view perspective BA, 1e6 tracks / ~5e6 observations per GPU, soft_l1, R+T"),
    "cfg4": (300, 625000, 0.02, "perspective", ["R", "T"],
             "BASELINE config 4: 300-view multi-date perspective BA, 6.25e5 tracks / ~3.7e6 observations per GPU (5e6 tracks / ~3e7 observations "
             "on 8 GPUs), soft_l1, R+T, matrix-free PCG on the 1800-unknown reduced camera system"),
    "rpcba": (4, 250000, 0.8, "rpc", ["R", "T"],
              "cam_model='rpc' (the pipeline default): 4 RPC cameras of the golden scene, 2.5e5 tracks / ~8e5 observations per GPU, soft_l1, R+T"),
    "cfg4s": (300, 100000, 0.02, "perspective", ["R", "T"],
              "BASELINE config 4 reduced: 300-view perspective BA, 1e5 tracks / ~6e5 observations per GPU (1800 x 1800 reduced system)"),
}
RPC_WORKLOAD = "rpc"         # BASELINE config 5: RPC refit + batched RPC projection / localisation / triangulation, 300 cameras
LS = {"loss": "soft_l1", "f_scale": 1.0}
L2_FLUSH_BYTES = 256 << 20      # > 126 MB L2
DUMP_LIMIT_BYTES = 64 * 10 ** 6  # --dump-outputs writes at most this much


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# phase -> (main kernel of the phase, as named in the ncu summaries) for the two engines of libsba_b200.so
PHASE_KERNELS = {
    "pattern": {"assemble_trial": "k_pt_assemble<", "jvp_damping": "k_pt_jvp1<", "eliminate_schur": "k_pt_schur<",
                "cholesky": "k_chol_fused<", "backsub_gram": "k_pt_backsub<"},
    "generic": {"schur": "k_schur<", "assemble": "k_assemble_points<", "point_prep": "k_point_prep<", "backsub": "k_backsub<",
                "cholesky": "k_chol_fused<", "scale_jvp": "k_jvp<1, 6, 1>", "subspace": "k_jvp<1, 6, 2>", "step_eval": "k_residual<"},
}
# C-ABI phase slots -> names used for the pattern engine (K1 doubles as trial evaluation and assembly: "step_eval" slot)
PATTERN_PHASES = {"scale_jvp": "jvp_damping", "schur": "eliminate_schur", "cholesky": "cholesky", "backsub": "backsub_gram",
                  "step_eval": "assemble_trial"}


def ncu_summary(engine, phase, workload):
    """Row of the committed ncu summary (one `ncu --set full --clock-control none` capture per kernel of this workload,
    profiles/r02_ncu_<workload>_selected_metrics.csv, written by tools/summarize_profiles.py) for the phase's main kernel."""
    kern = PHASE_KERNELS[engine].get(phase)
    name = "r02_ncu_%s_selected_metrics.csv" % workload if engine == "pattern" else "r01_ncu_full_selected_metrics.csv"
    path = os.path.join(ROOT, "profiles", name)
    if kern is None or not os.path.exists(path) or (engine == "generic" and workload != "cfg2"):
        return None, None
    import csv
    with open(path) as f:
        for row in csv.DictReader(f):
            if row["kernel"].startswith(kern):
                return row, "profiles/%s (%s, one ncu --set full capture, cold L2)" % (name, row["kernel"])
    return None, None


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (recipe of B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.proc, self.lines = None, []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_problem(workload, world):
    from sat_bundleadjust_b200 import synth
    n_cam, tracks, p_vis, model, corr, _ = WORKLOADS[workload]
    if model == "rpc":                                # the golden fixture's RPC cameras (tests/golden/rpc_golden.npz), synthetic tracks
        G = np.load(os.path.join(ROOT, "tests", "golden", "rpc_golden.npz"))
        scene = synth.make_rpc_scene(G["rpc_cams"][:n_cam], G["rpcba/camera_centers"][:n_cam], n_tracks=tracks * world, p_vis=p_vis, seed=0)
        return synth.SparseParams(scene, corr)
    if n_cam >= 100 and tracks * world > 200000:      # time-series scale: never form the dense (2M x N) correspondence matrix
        scene = synth.make_scene_sparse(n_cam=n_cam, n_tracks=tracks * world, p_vis=p_vis, cam_model=model, seed=0)
        return synth.SparseParams(scene, corr)
    scene = synth.make_scene(n_cam=n_cam, n_tracks=tracks * world, p_vis=p_vis, cam_model=model, seed=0)
    return synth.scene_to_params(scene, corr)


def algorithmic_bytes(K, N, M, c, engine):
    """SURVEY.md section 8d: int32 indices + FP64 values, J and W never materialised, camera tables once (per pass)."""
    n = M * c + 3 * N
    if engine == "pattern":
        return {
            "assemble_trial": 48 * K + 96 * N + 4 * M * c * (c + 3),    # B_asm: one fused residual + Jacobian + assembly pass (G1 + G2)
            "jvp_damping": 48 * K + 48 * N + 5 * 8 * n,                 # one J*v pass + the scale update
            "eliminate_schur": 48 * K + 120 * N + 8 * (M * c) ** 2,     # observations, x, V, g, D of the points in; S out (G3)
            "backsub_gram": 32 * K + 120 * N,                           # B_back (G6)
            "cholesky": 8 * (M * c) ** 2,
        }
    return {
        "assemble": 48 * K + 96 * N + 4 * M * c * (c + 3),          # G2: one fused residual+Jacobian+assembly pass
        "step_eval": 48 * K + 24 * N + 8 * 16 * M,                  # G1: one residual pass (no r written)
        "scale_jvp": 48 * K + 48 * N + 5 * 8 * n,                   # vector update + one J*v pass
        "subspace": 48 * K + 48 * N + 9 * 8 * n,                    # vector work + one J*[v1 v2] pass
        "point_prep": 48 * K + 24 * N + 48 * N + 48 * N + 72 * N + 24 * c * K,   # + Z write (non-algorithmic 24cK)
        "schur": 24 * c * K + 8 * (M * c) ** 2,                     # read Z once + write S
        "backsub": 24 * c * K + 72 * N + 24 * N + 4 * K,
        "cholesky": 8 * (M * c) ** 2,
    }


def dump_outputs(out_dir, arrays):
    """Writes each array of `arrays` (name -> array) as out_dir/<name>.npy in float64.  The largest output of any workload
    (1e6 tracks on one GPU: 24 MB) fits DUMP_LIMIT_BYTES whole, so nothing is sampled."""
    arrays = {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes + 1024 for a in arrays.values())       # + room for each .npy header
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def fp64_peak():
    """Measured FP64 FMA peak of this pool's B200 (tools/fp64_peak.cu, committed result profiles/r02_fp64_peak.json)."""
    path = os.path.join(ROOT, "profiles", "r02_fp64_peak.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["dfma_tflops"]), "measured (profiles/r02_fp64_peak.json, DFMA stream)"
    return 37.2, "nominal (148 SMs x 64 FMA/clk x 1.965 GHz)"


# ---------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the reference path (numpy fun + scipy TRF)
# ---------------------------------------------------------------------------------------------------
def cpu_reference_iterations(p, n_iter, n_warm=0):
    """Runs scipy TRF exactly as ba_core.py:284-297 does and returns seconds per trust-region iteration
    measured over iterations [n_warm, n_warm + n_iter) (the Jacobian + solve + evaluation of each)."""
    from scipy.optimize import least_squares
    from oracle import ba_oracle
    stamps = [time.perf_counter()]
    cpu_stamps = [time.process_time()]

    def cb(intermediate_result):
        stamps.append(time.perf_counter())
        cpu_stamps.append(time.process_time())
        if len(stamps) - 1 >= n_warm + n_iter:
            raise StopIteration      # scipy halts the iteration on StopIteration (status -2)

    x0 = p.params_opt.copy()
    A = ba_oracle.jacobian_sparsity(p)
    t0 = time.perf_counter()
    warnings.simplefilter("ignore")
    least_squares(ba_oracle.residuals, x0, jac_sparsity=A, verbose=0, x_scale="jac", method="trf", ftol=1e-15, xtol=0.0,
                  gtol=0.0, loss=LS["loss"], f_scale=LS["f_scale"], max_nfev=8 * (n_warm + n_iter) + 8, args=(p,), callback=cb)
    setup = stamps[0] - t0
    done = len(stamps) - 1
    if done <= n_warm:
        return None, done, setup, 1.0
    dt = stamps[-1] - stamps[n_warm]
    # threads actually used by the timed iterations = CPU time of the process / wall time (numpy / scipy.sparse are single-threaded on
    # this path unless a threaded BLAS picks up part of the work)
    util = (cpu_stamps[-1] - cpu_stamps[n_warm]) / dt if dt > 0 else 1.0
    return dt / (done - n_warm), done - n_warm, setup, util


def subsample_tracks(p, frac):
    """Bounded sample of the workload: keep the first `frac` of the tracks (observations are track-major)."""
    import copy
    n_keep = max(10, int(p.n_pts * frac))
    q = copy.copy(p)
    a = int(np.searchsorted(p.pts_ind, n_keep))
    q.n_pts, q.n_obs = n_keep, a
    q.pts_ind, q.cam_ind, q.pts2d, q.pts2d_w = p.pts_ind[:a], p.cam_ind[:a], p.pts2d[:a], p.pts2d_w[:a]
    q.pts3d = p.pts3d[:n_keep]
    ncv = p.n_cam * p.n_params
    q.params_opt = np.concatenate([p.params_opt[:ncv], p.params_opt[ncv: ncv + 3 * n_keep]])
    q.n_pts_fix = min(p.n_pts_fix, n_keep)
    return q


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    p = build_problem(args.workload, 1)
    K_full = p.n_obs
    # ~4.3 s per TRF iteration at 5e5 observations on one core (BASELINE.md); keep the whole run within ~4 minutes
    budget_s, per_it_full = 240.0, 4.3e-6 * 2 * K_full
    frac = min(1.0, budget_s / ((args.steps + args.warmup + 1) * per_it_full))
    q = p if frac >= 1.0 else subsample_tracks(p, frac)
    sec_it, done, setup, util = cpu_reference_iterations(q, args.steps, args.warmup)
    if sec_it is None:
        print(json.dumps({"impl": "reference", "unavailable": "scipy TRF terminated before the timed iterations"}))
        return 0
    value = q.n_obs / sec_it
    sample = ("%d TRF iterations (after %d warm-up) of scipy least_squares(trf, 2-point sparse differences, LSMR) on %s"
              % (done, args.warmup, "the full workload" if frac >= 1.0 else
                 "the first %.0f%% of the tracks (%d observations); obs x it/s is size-normalised" % (100 * frac, q.n_obs)))
    line = {
        "impl": "reference", "metric": "lm_observation_iterations_per_s", "value": value, "unit": "obs*it/s",
        "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * sec_it,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload][5], "n_obs": int(q.n_obs), "n_tracks": int(q.n_pts),
                   "n_cam": int(q.n_cam), "loss": LS["loss"]},
        "lm_iters_per_s": 1.0 / sec_it,
        "cpu_baseline": {"value": value, "unit": "obs*it/s", "cores": max(1, int(round(util))), "cpu_time_over_wall": round(util, 2), "kind": "port",
                         "sample": sample + "; cores = CPU time / wall time of the timed iterations (%d host cores present)" % (os.cpu_count() or 1)},
        "e2e": {"value": value, "unit": "obs*it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def measure_workload(workload, K, W, world, rank, local_rank, with_e2e=True, with_clocks=True, keep_outputs=False):
    """Device-timed iterations (+ phases), the fused Jacobian/assembly pass alone and the end-to-end call for one workload.
    Returns a dict of raw measurements on every rank (max over ranks already taken); with keep_outputs, also what the last
    timed solve computed ("outputs")."""
    import torch
    import torch.distributed as dist
    from sat_bundleadjust_b200 import ba_core
    from sat_bundleadjust_b200 import dist as sdist
    from sat_bundleadjust_b200.solver import DeviceProblem, initial_vars

    p = build_problem(workload, world)
    ranges = sdist.shard_ranges(p.pts_ind, p.n_pts, world)
    ncv = p.n_cam * p.n_params
    x0 = initial_vars(p)
    stream = torch.cuda.current_stream().cuda_stream
    prob = DeviceProblem(p, stream=stream, rank=rank, world_size=world, track_range=ranges[rank] if world > 1 else None)
    if world > 1:
        def hook(ptr, count):
            t = torch.as_tensor(sdist._CudaView(ptr, count), device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        prob.set_allreduce(hook)
        if os.environ.get("SBA_COMM", "peer") == "peer":
            def gather_obj(obj):
                out = [None] * world
                dist.all_gather_object(out, obj)
                return out
            prob.connect_peers(gather_obj)
    xl0 = sdist.local_vars(x0, ncv, ranges[rank]) if world > 1 else x0
    x_dev = torch.from_numpy(xl0).cuda()
    out_dev = torch.empty_like(x_dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # untimed: one short solve so that every kernel is loaded and the exchange buffers are mapped
    prob.solve_device(x_dev.data_ptr(), out_dev.data_ptr(), None, ftol=0.0, xtol=0.0, gtol=0.0, max_nfev=10 ** 6,
                      max_iterations=2, **LS)
    barrier()
    sampler = ClockSampler(local_rank) if (rank == 0 and with_clocks) else None
    # exactly K timed iterations; long runs are cut into solves of <= SEG timed iterations that each restart from
    # x0 (with W untimed iterations first), so that every timed iteration is a productive pre-convergence one
    SEG = 25

    def timed_run(no_phase_timing):
        left, acc, per_it = K, None, []
        while left > 0:
            k = min(SEG, left)
            part = prob.solve_device(x_dev.data_ptr(), out_dev.data_ptr(), None, ftol=0.0, xtol=0.0, gtol=0.0,
                                     max_nfev=10 ** 6, max_iterations=W + k, timed_from=W, l2_flush_bytes=L2_FLUSH_BYTES,
                                     no_phase_timing=no_phase_timing, **LS)
            assert part["timed_iterations"] == k, part
            per_it.append(part["iter_ms"] / k)
            last_cost = part["cost"]
            if acc is None:
                acc = part
            else:
                acc["iter_ms"] += part["iter_ms"]
                acc["timed_iterations"] += k
                acc["gpu_launches"] += part["gpu_launches"]
                for ph in acc["phase_ms"]:
                    acc["phase_ms"][ph] += part["phase_ms"][ph]
            left -= k
        acc["segment_ms_per_iteration"] = per_it
        acc["last_cost"] = last_cost
        return acc

    # the headline: whole iterations only (one CUDA-event pair per iteration); then the same K iterations again with the
    # per-phase events on (more event records per iteration, which themselves cost ~1 us each on the stream)
    info = timed_run(1)
    barrier()
    # what the headline's last solve returned to its caller: the variables in the device layout (cameras, then this rank's
    # tracks) and the cost
    x_last = out_dev.cpu().numpy() if keep_outputs else None
    info_ph = timed_run(0)
    barrier()
    keys = list(info_ph["phase_ms"].keys())
    t = torch.tensor([info["iter_ms"], info_ph["iter_ms"]] + [info_ph["phase_ms"][k] for k in keys], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t = t.cpu().numpy()
    engine = prob.engine
    phase_ms = {k: float(v) / K for k, v in zip(keys, t[2:])}
    if engine == "pattern":
        phase_ms = {PATTERN_PHASES[k]: v for k, v in phase_ms.items() if k in PATTERN_PHASES}

    # Jacobian pass alone (fused residual + analytic Jacobian + robust weights + block assembly), L2-cold
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    jac_ms = []
    for i in range(3 + 10):
        flush.fill_(i & 0xff)
        ms = prob.assemble_device(x_dev.data_ptr(), **LS)
        if i >= 3:
            jac_ms.append(ms)
    jac = torch.tensor([float(np.mean(jac_ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(jac, op=dist.ReduceOp.MAX)
    out = {"p": p, "engine": engine, "iter_ms": float(t[0]), "iter_ms_with_phase_events": float(t[1]), "phase_ms": phase_ms,
           "jac_ms": float(jac.item()), "gpu_launches": int(info["gpu_launches"]), "n_obs_local": prob.n_obs,
           "n_pts_local": prob.n_pts, "n_vars_local": prob.n_vars, "segments": info["segment_ms_per_iteration"],
           "clocks": sampler.stop() if sampler else None}
    if keep_outputs:
        out["outputs"] = {"cameras": x_last[:ncv].reshape(p.n_cam, p.n_params), "points": x_last[ncv:].reshape(-1, 3),
                          "cost": np.array([info["last_cost"]])}
    if world > 1:
        dist.barrier()      # peers may still be reading this rank's exchange buffer
    prob.close()
    del flush, x_dev, out_dev

    if with_e2e:
        # end to end through the public API (host buffers in and out; rank 0's wall clock, all ranks take part): the first call of
        # the process (first-use allocations: device slabs, pinned scalars) is reported on its own, then the mean of E2E_CALLS calls
        E2E_CALLS = 3
        ls = dict(LS, max_iter=300, verbose=0)

        def e2e_call():
            if world > 1:
                return sdist.run_ba_optimization_distributed(p, ls)[5]
            return ba_core.run_ba_optimization(p, ls, False, False, return_info=True)[5]

        walls = []
        for _ in range(1 + E2E_CALLS):
            barrier()
            t0 = time.perf_counter()
            info_e = e2e_call()
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
        wall = float(np.mean(walls[1:]))
        Kobs = int(p.n_obs)
        n_loc = out["n_vars_local"]
        # per call: int32 camera / track index + internal permutation (12 B), observation (16 B) and weight (8 B) per observation,
        # track offsets, x0 and the camera table in; x and the two per-observation error vectors out
        h2d = 36 * out["n_obs_local"] + 4 * (out["n_pts_local"] + 1) + 8 * n_loc + 8 * p.cam_params.size
        d2h = 8 * n_loc + 2 * 8 * out["n_obs_local"]
        out["e2e"] = {"value": Kobs * info_e["iterations"] / wall, "unit": "obs*it/s",
                      "h2d_bytes_per_step": int(h2d / max(1, info_e["iterations"])),
                      "d2h_bytes_per_step": int(d2h / max(1, info_e["iterations"])),
                      "wall_s": wall, "wall_s_calls": walls[1:], "calls": E2E_CALLS, "first_call_wall_s": walls[0],
                      "first_call_value": Kobs * info_e["iterations"] / walls[0],
                      "iterations": info_e["iterations"], "nfev": info_e["nfev"], "status": info_e["status"],
                      "cost": info_e["cost"], "device_ms": info_e["solve_ms"], "wall_breakdown_s": info_e.get("wall_s"),
                      "call": "ba_core.run_ba_optimization(p, {'loss': 'soft_l1', 'f_scale': 1.0, 'max_iter': 300})"}
    return out


def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W, K = args.warmup, args.steps
    m = measure_workload(args.workload, K, W, world, rank, local_rank, keep_outputs=args.dump_outputs is not None)
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, m["outputs"])
    second = None
    if world == 1 and not args.no_secondary and args.workload != "cfg2":
        second = measure_workload("cfg2", K, W, world, rank, local_rank, with_e2e=True, with_clocks=False)

    if rank == 0:
        peak, peak_src = load_peaks()
        f64_peak, f64_src = fp64_peak()
        p = m["p"]
        M, c, Kobs = p.n_cam, p.n_params, int(p.n_obs)
        K_loc, N_loc = m["n_obs_local"], m["n_pts_local"]
        engine, phase_ms, iter_ms, jac_ms = m["engine"], m["phase_ms"], m["iter_ms"], m["jac_ms"]
        ab = algorithmic_bytes(K_loc, N_loc, M, c, engine)
        asm_key = "assemble_trial" if engine == "pattern" else "assemble"
        # the dominant kernel of the iteration (the dense Cholesky is one CTA of latency, not a streaming kernel)
        dominant = max((k for k in phase_ms if k != "cholesky"), key=lambda k: phase_ms[k])
        row, row_src = ncu_summary(engine, dominant, args.workload)
        traffic = (float(row["dram rd MB"]) + float(row["dram wr MB"])) * 1e6 if row else None
        fp64_frac = float(row["fp64 pipe %"]) / 100.0 if row else None
        # FP64 work of the dominant kernel: thread-level FP64 instructions counted by ncu for one launch (FMA = 2 flop)
        flop = float(row["fp64 Gflop"]) * 1e9 if row and row.get("fp64 Gflop") else None
        roof_all = {k: {"ms": phase_ms[k], "algorithmic_bytes": ab.get(k),
                        "achieved_GBps": ab[k] / (phase_ms[k] * 1e-3) / 1e9 if phase_ms[k] > 0 and k in ab else None}
                    for k in phase_ms}
        ach = ab[dominant] / (phase_ms[dominant] * 1e-3) / 1e9
        jac_ach = ab[asm_key] / (jac_ms * 1e-3) / 1e9
        seg = np.array(m["segments"])
        line = {
            "metric": "lm_observation_iterations_per_s", "value": Kobs * K / (iter_ms * 1e-3), "unit": "obs*it/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": iter_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload][5], "n_obs": Kobs, "n_tracks": int(p.n_pts), "n_cam": int(M),
                       "n_params_per_cam": int(c), "loss": LS["loss"], "tracks_per_gpu": int(N_loc), "engine": engine,
                       "parallelism": "tracks sharded over %d GPU(s), cameras replicated" % world,
                       "exchange": ("none" if world == 1 else os.environ.get("SBA_COMM", "peer") +
                                    (" (per iteration: [U|g_c|cost], 21 scalars, [S|rhs] in block-upper form, 7 scalars; one-shot all-reduces over NVLink peer memory inside the producing kernels, no launch of their own)" if engine == "pattern"
                                     else " (per iteration: [U|g_c], [S|rhs], 5 scalar groups)")),
                       "l2": "256 MiB scratch overwritten between timed iterations (outside the event pairs)"},
            "lm_iters_per_s": K / (iter_ms * 1e-3),
            "ms_per_step_segments": {"mean": float(seg.mean()), "min": float(seg.min()), "max": float(seg.max()), "n": int(seg.size)},
            "jacobian_obs_per_s": Kobs / (jac_ms * 1e-3),
            "jacobian_pass_ms": jac_ms,
            "clocks": m["clocks"], "e2e": m["e2e"], "gpu_launches": m["gpu_launches"],
            "roofline": {"kernel": dominant + " (" + PHASE_KERNELS[engine].get(dominant, "?").rstrip("<") + ")", "bound": "hbm",
                         "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": traffic, "traffic_source": row_src, "peak_source": peak_src,
                         # the roofline that actually binds this FP64 path: FP64 pipe issue slots used (ncu), and the counted FP64
                         # work of one launch over the live kernel time against the measured DFMA peak
                         "fp64_pipe_frac": fp64_frac,
                         "fp64": ({"flop_per_launch": flop, "achieved_tflops": flop / (phase_ms[dominant] * 1e-3) / 1e12,
                                   "peak_tflops": f64_peak, "frac": flop / (phase_ms[dominant] * 1e-3) / 1e12 / f64_peak,
                                   "peak_source": f64_src} if flop else None),
                         "jacobian_assembly": {"achieved": jac_ach, "frac": jac_ach / peak, "ms": jac_ms,
                                               "algorithmic_bytes": ab[asm_key]}},
            "phases_ms_per_iteration": phase_ms, "phases": roof_all,
            "ms_per_step_with_phase_events": m["iter_ms_with_phase_events"] / K,
        }
        if second is not None:
            q = second["p"]
            line["secondary"] = [{"workload": WORKLOADS["cfg2"][5], "n_obs": int(q.n_obs), "engine": second["engine"],
                                  "value": int(q.n_obs) * K / (second["iter_ms"] * 1e-3), "unit": "obs*it/s",
                                  "ms_per_step": second["iter_ms"] / K, "phases_ms_per_iteration": second["phase_ms"],
                                  "jacobian_pass_ms": second["jac_ms"], "e2e": second["e2e"]}]
        if world == 1 and not args.no_cpu_baseline:
            # bounded sample (~20 s of CPU work): 2 TRF iterations after 1 warm-up iteration on the first half of the tracks
            q = subsample_tracks(p, 0.5) if p.n_obs > 600000 else p
            sec_it, done, _, util = cpu_reference_iterations(q, 2, 1)
            line["cpu_baseline"] = {"value": q.n_obs / sec_it, "unit": "obs*it/s", "cores": max(1, int(round(util))), "cpu_time_over_wall": round(util, 2), "kind": "port",
                                    "lm_iters_per_s_at_sample_size": 1.0 / sec_it,
                                    "sample": "%d TRF iterations (after 1 warm-up iteration) of scipy least_squares (2-point sparse "
                                              "differences + LSMR) on %s; obs x it/s is size-normalised; cores = CPU time / wall time "
                                              "of the timed iterations (%d host cores present)"
                                              % (done, "the first half of the tracks (%d observations)" % q.n_obs if q is not p
                                                 else "the full workload", os.cpu_count() or 1)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ---------------------------------------------------------------------------------------------------
# BASELINE config 5: the RPC side of the path (G7-G10): projection, localisation, triangulation, refit
# ---------------------------------------------------------------------------------------------------
def run_rpc_workload(args):
    """`--workload rpc`: 300 cameras (the two reference test RPCs with jittered offsets), a 100 x 100 x 10 lon/lat/alt grid
    per camera for projection / localisation, 1e5 matches per camera pair for triangulation, 10 x 10 x 10 samples per camera
    for the refit.  --impl reference times the CPU side only: the reference's compiled C (oracle/_ref/disp_to_h.so) when it is
    there, else the pinned C port, and the oracle's weighted_lsq, on bounded samples."""
    import ctypes
    import numpy as np
    from oracle import rpc_ctypes, rpc_oracle, rpcfit_oracle
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    G = np.load(os.path.join(ROOT, "tests", "golden", "rpc_golden.npz"))
    F = np.load(os.path.join(ROOT, "tests", "golden", "rpcfit_golden.npz"))
    n_cam, reps = 300, args.steps                           # timed passes of each batched operation (after one untimed pass)
    rng = np.random.default_rng(0)
    base = [G["rpc_a"], G["rpc_b"]]
    tables = np.stack([base[j % 2].copy() for j in range(2 * n_cam)])
    tables[:, 0] += rng.uniform(-5, 5, 2 * n_cam)         # row / col offsets jittered: 600 distinct cameras
    tables[:, 1] += rng.uniform(-5, 5, 2 * n_cam)
    ra = base[0]
    gl = np.stack(np.meshgrid(np.linspace(-0.9, 0.9, 100), np.linspace(-0.9, 0.9, 100), np.linspace(-0.9, 0.9, 10), indexing="ij"), -1).reshape(-1, 3)
    lon, lat, alt = ra[3] + gl[:, 0] * ra[8], ra[2] + gl[:, 1] * ra[7], ra[4] + gl[:, 2] * ra[9]
    n = lon.size
    # CPU side: reference C where it compiled, else the pinned port
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "disp_to_h.so"))
    clib = rpc_ctypes.load_ref() if have_ref else rpc_ctypes.load_port()
    kind = "reference" if have_ref else "port"
    from tests_util_shim import rpc_from_array
    ma, mb = rpc_from_array(base[0]), rpc_from_array(base[1])
    ns = 20000                                              # bounded CPU samples
    lla_s = np.stack([lon[:ns], lat[:ns], alt[:ns]], 1)
    t0 = time.perf_counter()
    cr = rpc_ctypes.ref_project(clib, ma, lla_s[:4000]) if have_ref else rpc_ctypes.port_project(clib, ma, lla_s)
    n_proj = cr.shape[0]
    t_proj = time.perf_counter() - t0
    col_a, row_a = ma.projection(lon, lat, alt)
    col_b, row_b = mb.projection(lon, lat, alt)
    t0 = time.perf_counter()
    _ = rpc_ctypes.triangulate(clib, ma, mb, np.stack([col_a[:ns], row_a[:ns]], 1), np.stack([col_b[:ns], row_b[:ns]], 1), 0.1, ref=have_ref)
    t_tri = time.perf_counter() - t0
    t0 = time.perf_counter()
    nfit = 6
    for k in range(nfit):
        rpcfit_oracle.weighted_lsq(F["case%d/target" % k], F["case%d/input_locs" % k])
    t_fit = (time.perf_counter() - t0) / nfit
    cpu = {"projection": n_proj / t_proj, "triangulation": ns / t_tri, "refit": 1.0 / t_fit}
    if args.impl == "reference":
        line = {"impl": "reference", "metric": "rpc_triangulated_matches_per_s", "value": cpu["triangulation"], "unit": "matches/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tri, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "BASELINE config 5: RPC triangulation / projection / refit, CPU side on bounded samples"},
                "cpu_baseline": {"value": cpu["triangulation"], "unit": "matches/s", "cores": 1, "kind": kind,
                                 "sample": "%d matches through stereo_corresp_to_lonlatalt of %s" % (ns, "oracle/_ref/disp_to_h.so (the reference's C, compiled in place)" if have_ref else "the pinned C port"),
                                 "projection_points_per_s": cpu["projection"], "refit_cameras_per_s": cpu["refit"]},
                "e2e": {"value": cpu["triangulation"], "unit": "matches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0
    import torch
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    from sat_bundleadjust_b200 import _lib, ba_rpcfit
    lib = _lib.load()
    dp = _lib.dptr
    ms = ctypes.c_double()

    def thr(kind_id, a, b, c, d, delta, out_w):
        out = np.empty(out_w * n)
        _lib.check(lib.sba_rpc_throughput(kind_id, dp(tables), n_cam, dp(a), dp(b), dp(c), dp(d) if d is not None else None, n, delta, reps,
                                          dp(out), ctypes.byref(ms)))
        return ms.value, out
    f64 = _lib.f64
    ms_proj, o = thr(0, f64(lon), f64(lat), f64(alt), None, 1.0, 2)
    last = rpc_from_array(tables[n_cam - 1])
    assert np.abs(o[:n] - last.projection(lon, lat, alt)[0]).max() < 1e-6
    ms_loc, o = thr(1, f64(col_a), f64(row_a), f64(alt), None, 1.0, 2)
    ms_tri, o = thr(2, f64(col_a), f64(row_a), f64(col_b), f64(row_b), 0.1, 3)
    if args.dump_outputs is not None:
        # the headline's last pass: lon, lat, alt of every match of the last camera pair
        dump_outputs(args.dump_outputs, {"triangulation_lonlatalt": o.reshape(n, 3)})
    # refit: 300 cameras x 1000 samples through the public batched call (host buffers in and out)
    tg = np.stack([F["case%d/target" % (k % int(F["n_cases"]))] for k in range(n_cam)])
    lc = np.stack([F["case%d/input_locs" % (k % int(F["n_cases"]))] for k in range(n_cam)])
    ba_rpcfit.weighted_lsq_batch(tg[:4], lc[:4])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ba_rpcfit.weighted_lsq_batch(tg, lc)
    t_fit_gpu = time.perf_counter() - t0
    # initial triangulation of all tracks (ft_triangulate.init_pts3d, SURVEY 8f-2): every pair x every track in ONE launch; wall clock of
    # the public call (dense correspondence matrix in, float32 points out), against the oracle's pair loop on a bounded sample
    from oracle import tri_oracle
    from sat_bundleadjust_b200 import ft_triangulate, synth
    sc = synth.make_scene(n_cam=20, n_tracks=200000, p_vis=0.3, cam_model="perspective", seed=1)
    Cm = sc.correspondence_matrix()
    pairs = [(i, j) for i in range(20) for j in range(i + 1, 20)]
    ft_triangulate.init_pts3d(Cm[:, :2000], sc.cameras, "perspective", pairs)
    t0 = time.perf_counter()
    p3 = ft_triangulate.init_pts3d(Cm, sc.cameras, "perspective", pairs)
    t_init_gpu = time.perf_counter() - t0
    t0 = time.perf_counter()
    p3_cpu = tri_oracle.init_pts3d(Cm[:, :4000], sc.cameras, pairs)
    t_init_cpu = time.perf_counter() - t0
    assert np.abs(p3[:4000].astype(np.float64) - p3_cpu.astype(np.float64)).max() <= 1.0      # float32 ulp at ECEF magnitude is 0.5 m
    # end to end through the host-pointer API (the reference-facing calls): projection of every camera's grid, host buffers
    colo, rowo = np.empty(n), np.empty(n)
    n_e2e = n_cam // 10
    colb, rowb = np.empty((n_e2e, n)), np.empty((n_e2e, n))
    tb = np.ascontiguousarray(np.stack([tables[j] for j in range(0, n_cam, 10)]))
    t0 = time.perf_counter()
    _lib.check(lib.sba_rpc_projection_batch(dp(tb), n_e2e, dp(f64(lon)), dp(f64(lat)), dp(f64(alt)), n, 1, dp(colb), dp(rowb)))
    e2e_proj = n_e2e * n / (time.perf_counter() - t0)
    f64_peak, f64_src = fp64_peak()
    peak, peak_src = load_peaks()
    pts = n_cam * n
    # flop per point counted from the formulas: 4 cubics x (19 add + 36 mul) + normalisation / de-normalisation 3 x 2 + 2 x 2 + 2 div
    flop_proj = 4 * 55 + 12
    ops = {
        "projection": {"value": pts / (ms_proj * 1e-3), "unit": "points/s", "ms": ms_proj, "cpu_baseline": cpu["projection"],
                       "hbm_frac": 40 * pts / (ms_proj * 1e-3) / 1e9 / peak, "fp64_frac": flop_proj * pts / (ms_proj * 1e-3) / 1e12 / f64_peak},
        "localization": {"value": pts / (ms_loc * 1e-3), "unit": "points/s", "ms": ms_loc},
        "triangulation": {"value": pts / (ms_tri * 1e-3), "unit": "matches/s", "ms": ms_tri, "cpu_baseline": cpu["triangulation"]},
        "refit": {"value": n_cam / t_fit_gpu, "unit": "cameras/s", "ms": 1e3 * t_fit_gpu, "cpu_baseline": cpu["refit"],
                  "note": "wall clock of ba_rpcfit.weighted_lsq_batch, host buffers in and out, 1000 samples per camera"},
        "init_pts3d": {"value": Cm.shape[1] / t_init_gpu, "unit": "tracks/s", "ms": 1e3 * t_init_gpu, "cpu_baseline": 4000 / t_init_cpu,
                       "note": "wall clock of ft_triangulate.init_pts3d (20 perspective cameras, 190 pairs, 2e5 tracks, dense C in, host conversion "
                               "included); CPU = the oracle's pair loop (numpy Jacobi DLT) on 4000 tracks"},
    }
    line = {"metric": "rpc_triangulated_matches_per_s", "value": ops["triangulation"]["value"], "unit": "matches/s", "n_gpus": 1,
            "steps": reps, "warmup": 1, "ms_per_step": ms_tri, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BASELINE config 5: 300 cameras, 100 x 100 x 10 grid per camera (projection, localisation), 1e5 matches per pair "
                                   "(triangulation), 1000 samples per camera (refit)", "n_cam": n_cam, "points_per_camera": int(n)},
            "operations": ops,
            "roofline": {"kernel": "k_rpc_projection", "bound": "hbm", "achieved": 40 * pts / (ms_proj * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": ops["projection"]["hbm_frac"], "traffic": None, "peak_source": peak_src,
                         "fp64": {"flop_per_point": flop_proj, "achieved_tflops": flop_proj * pts / (ms_proj * 1e-3) / 1e12, "peak_tflops": f64_peak,
                                  "frac": ops["projection"]["fp64_frac"], "peak_source": f64_src}},
            "cpu_baseline": {"value": cpu["triangulation"], "unit": "matches/s", "cores": 1, "kind": kind,
                             "sample": "%d matches (triangulation), %d points (projection), %d refits on one core" % (ns, n_proj, nfit)},
            "e2e": {"value": e2e_proj, "unit": "points/s", "h2d_bytes_per_step": 24 * int(n), "d2h_bytes_per_step": 16 * int(n) * (n_cam // 10),
                    "call": "sba_rpc_projection_batch (host buffers, one launch), 30 cameras x 1e5 shared points"},
            "gpu_launches": int((2 + n_cam) * (reps + 1) + 3)}
    print(json.dumps(line))
    return 0


def main():
    # stdout carries exactly one JSON line: everything else that libraries print there (e.g. NCCL's version banner)
    # is sent to stderr by swapping the file descriptors for the duration of the run
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="1m", choices=sorted(WORKLOADS) + [RPC_WORKLOAD])
    ap.add_argument("--no-secondary", action="store_true", help="skip the config-2 line reported under \"secondary\" (N = 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed solve returned as DIR/<name>.npy (float64, "
                    "at most 64 MB in all; at N > 1, rank 0's cameras and tracks).  Beyond 25 steps that solve restarts from "
                    "the initial point, so compare dumps taken with the same --steps and --warmup.  bench_outputs/ is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 0)
    if args.workload == RPC_WORKLOAD:
        rc = run_rpc_workload(args)
    else:
        rc = run_reference_arm(args) if args.impl == "reference" else run_b200_arm(args)
    sys.stdout.flush()
    return rc


if __name__ == "__main__":
    sys.exit(main())
