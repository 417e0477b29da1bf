// Pattern-major engine: the four fused passes of one trust-region iteration for problems with a small reduced camera system
// (M * n_params <= PT_MAX_NS) whose tracks share their camera sets.  Layout and vocabulary: sba_pattern.h.
//
//   k_pt_assemble   trial point x + pa t1 + pb delta, residual, robust cost, analytic Jacobian and the blocks
//                   V_i, g_i (per track, reduced inside the warp) and U_j, g_j (per camera, in registers over a work
//                   unit, then in warp-private shared-memory accumulators) -- one evaluation per observation.  Doubles as
//                   the trial-cost evaluation of the step, so an accepted step needs no further pass.   (G1 + G2 of SURVEY.md 2.2)
//   k_pt_jvp1       x_scale update of the points, |g_h|^2 and |J_h g_h|^2 -> damping (scipy trf.py:485-490)
//   k_pt_schur      damped point blocks inverted, Z_a = (Jc^T Jp) G^T staged in shared memory, all products
//                   Z_a Z_b^T of a track accumulated in registers by fixed (camera pair, row chunk) lanes; one record per
//                   (unit, pass) in global memory, merged after a CTA barrier by one thread per (block, row) in unit order
//                   into the CTA's partial of S -- no Z in HBM, no pair lists, no atomics                      (G3)
//                   (k_pt_schur_mma: the same with the products on the FP64 tensor cores, opt-in, slower)
//   k_pt_backsub    point steps from the camera step, and the Gram scalars of the 2-D subspace {g, gn}    (G6)
//   k_pt_reduce_assemble / k_pt_reduce_schur   per-CTA partials -> [U | g_c | cost] / [S | rhs]; on several GPUs the all-reduce
//                   over NVLink peer memory happens inside these kernels and inside the last CTA of k_pt_jvp1 / k_pt_backsub
// Every reduction has a fixed order (static unit -> warp assignment, ordered merges, ranks summed in rank order), so results
// are reproducible bit for bit.  Included by sba_ba.cu only.
#pragma once
#include "sba_comm.cuh"
#include "sba_kernels.cuh"
#include "sba_pattern.h"

namespace sba {

constexpr int PT_CTAS = NUM_SMS;          // one persistent CTA per SM
constexpr int PT_THREADS = 512;           // assemble (<= 128 registers)
constexpr int PT_THREADS_LIGHT = 512;     // jvp1 / backsub
constexpr int PT_THREADS_SCHUR = 384;     // schur (<= 168 registers)
constexpr int PT_MAX_NS = 132;            // camera unknowns: bounds the warp-private camera accumulators of k_pt_assemble in shared memory
constexpr int PT_RC = 3;                  // rows of a camera block per Schur task

struct PatView {
    const PUnit* units;       // assignment for this kernel's CTA shape
    const int* warp_unit0;    // (n_cta * warps + 1)
    const double2* pts2d;     // internal observation order
    const double* w;
    const double* cam_static; // (M, P) initial camera parameters
    const double* rpc_tab;
    int M, P, n_cam_fix, n_cta;
    int debug_skip;           // measurement only (SBA_PT_SKIP=1): the warps walk no units, leaving the fixed cost of a pass
    long long* cycles;        // measurement only (SBA_PT_CYCLES=1): per warp, clocks spent in its unit loop (load balance of the assignment)
};

__device__ __forceinline__ double step_value2(double x, double t, double d, double pa, double pb)
{
    return x + fma(pa, t, pb * d);
}

// inverse Cholesky factor G (lower: g00 g10 g11 g20 g21 g22) of V + reg diag(d2); false (G = 0) when not positive definite
__device__ __forceinline__ bool invert_point_block_d2(double v0, double v1, double v2, double v3, double v4, double v5,
                                                      double d0, double d1, double d2, double reg, double G[6])
{
    const double a00 = v0 + reg * d0, a10 = v1, a20 = v2;
    const double a11 = v3 + reg * d1, a21 = v4, a22 = v5 + reg * d2;
    bool ok = a00 > 0.0;
    const double i00 = fast_rsqrt(a00);
    const double c10 = a10 * i00, c20 = a20 * i00;
    const double d11 = a11 - c10 * c10;
    ok = ok && d11 > 0.0;
    const double i11 = fast_rsqrt(d11);
    const double c21 = (a21 - c20 * c10) * i11;
    const double d22 = a22 - c20 * c20 - c21 * c21;
    ok = ok && d22 > 0.0;
    const double i22 = fast_rsqrt(d22);
    if (!ok) {
#pragma unroll
        for (int k = 0; k < 6; ++k) G[k] = 0.0;
        return false;
    }
    G[0] = i00; G[2] = i11; G[5] = i22;
    G[1] = -c10 * i00 * i11;
    G[4] = -c21 * i11 * i22;
    G[3] = -(c20 * i00 + c21 * G[1]) * i22;
    return true;
}

// block-wide sum of NV values per thread in a fixed order; result valid in thread 0..NV-1 (sm: NV * 32 doubles)
template <int NV>
__device__ __forceinline__ double cta_reduce_sum(double (&v)[NV], double* sm)
{
    warp_reduce_sum<NV>(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) sm[warp * NV + k] = v[k];
    }
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x < NV)
        for (int wq = 0; wq < nw; ++wq) s += sm[wq * NV + threadIdx.x];
    __syncthreads();
    return s;
}

// grid-wide sum: every CTA stores its NV totals (held by threads 0..NV-1), the last CTA to arrive adds them in CTA
// order and writes scal[slots[k]].  Returns true in the last CTA (all threads), after the sums are visible to it.
template <int NV>
__device__ __forceinline__ bool grid_sum_last(double block_total, double* partials, unsigned* counter, double* scal,
                                              const int* slots)
{
    __shared__ bool is_last;
    if (threadIdx.x < NV) partials[(size_t)blockIdx.x * NV + threadIdx.x] = block_total;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
    if (threadIdx.x < NV) {
        double s = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(partials + (size_t)b * NV + threadIdx.x);
        scal[slots[threadIdx.x]] = s;
    }
    if (threadIdx.x == 0) *counter = 0u;
    __threadfence();
    __syncthreads();
    return true;
}

// camera records of a CTA: shared copy of camrec (M x CAMREC_STRIDE) and, for RPC, of the coefficient tables
template <int MODEL>
__device__ __forceinline__ void load_cameras_shared(const PatView& A, const double* __restrict__ camrec, double* s_cam,
                                                    double* s_rpc)
{
    for (int t = threadIdx.x; t < A.M * CAMREC_STRIDE; t += blockDim.x) s_cam[t] = camrec[t];
    if (MODEL == MODEL_RPC)
        for (int t = threadIdx.x; t < A.M * RPC_TAB_STRIDE; t += blockDim.x) s_rpc[t] = A.rpc_tab[t];
}

// k-th camera (k-th set bit) of a unit's camera set
__device__ __forceinline__ int unit_camera(const PUnit& u, int k)
{
    const int nlo = __popc(u.mask_lo);
    return k < nlo ? (int)__fns(u.mask_lo, 0, k + 1) : 32 + (int)__fns(u.mask_hi, 0, k - nlo + 1);
}

// lane geometry of a unit: lane = track slot t * L + position k
struct LaneGeo {
    int L, T, k, t, cam;
    bool on;
};
__device__ __forceinline__ LaneGeo lane_geometry(const PUnit& u, int lane)
{
    LaneGeo g;
    g.L = u.L; g.T = min(32 / u.L, PT_MAX_T);
    g.t = lane / u.L; g.k = lane - g.t * u.L;
    g.on = g.t < g.T;
    g.cam = g.on ? unit_camera(u, g.k) : 0;
    return g;
}

// sum over the track slots t of a value held by lane (t, k): afterwards lanes with t == 0 hold the total (fixed tree)
__device__ __forceinline__ double slot_reduce(double v, const LaneGeo& g)
{
    for (int off = 1; off < g.T; off <<= 1) {
        const double o = __shfl_down_sync(0xffffffffu, v, (unsigned)(off * g.L) & 31);
        if (g.on && g.t + off < g.T) v += o;
    }
    return v;
}

// the same for N values at once: the N shuffles of a step are independent and pipeline, where N separate calls would walk N
// dependent shuffle chains one after the other (27 values at the end of every unit of the assembly kernel)
template <int N>
__device__ __forceinline__ void slot_reduce_n(double (&v)[N], const LaneGeo& g)
{
    for (int off = 1; off < g.T; off <<= 1) {
        const unsigned delta = (unsigned)(off * g.L) & 31;
        const bool take = g.on && g.t + off < g.T;
        double o[N];
#pragma unroll
        for (int q = 0; q < N; ++q) o[q] = __shfl_down_sync(0xffffffffu, v[q], delta);
#pragma unroll
        for (int q = 0; q < N; ++q) if (take) v[q] += o[q];
    }
}

// The inputs of the NEXT tile of a unit are requested into L1 while the current tile is computed: a warp has only a
// dozen tiles to walk, so an exposed HBM round trip per tile would dominate the kernel.  Addresses are arithmetic (no
// index arrays), one prefetch per lane and array; lanes of a track share cache lines.
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// Jacobian rows of one observation from the geometry alone, scaled by the row scales (weight x robust rescale) that
// k_pt_assemble stored for this observation at the current point: the passes after the assembly need neither the
// observed pixel nor the loss.
template <int MODEL, int NC>
__device__ __forceinline__ void eval_scaled(const double* __restrict__ rec, const double* __restrict__ rpc_j, double X, double Y,
                                            double Z, double2 sc, bool cam_free, bool pt_free, ObsEval<MODEL, NC>& e)
{
    double u, v;
    full_side<MODEL, NC, true>(rec, rpc_j, X, Y, Z, u, v, e.Jc, e.Jp);
    const double a0 = cam_free ? sc.x : 0.0, a1 = cam_free ? sc.y : 0.0;
#pragma unroll
    for (int k = 0; k < NC; ++k) { e.Jc[k] *= a0; e.Jc[NC + k] *= a1; }
    const double b0 = pt_free ? sc.x : 0.0, b1 = pt_free ? sc.y : 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) { e.Jp[k] *= b0; e.Jp[3 + k] *= b1; }
}

// ------------------------------------------------------------------------------------------------
// K1: trial point + fused residual / Jacobian / block assembly
//   x_new = x + pa (g idsq) + pb delta  (initial != 0: x_new = x)
//   outputs: x_new, camrec_new (by CTA 0), V_new, g_new (point part), per-CTA partials of [U | g_c] and of the cost
// shared: s_cam[M*40] | s_rpc[M*90] | s_acc[nwarps][M*NV] | s_stage[nwarps][9][32] | s_red
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC>
__global__ void __launch_bounds__(PT_THREADS, 1)
k_pt_assemble(PatView A, const double* __restrict__ x, const double* __restrict__ g, const double* __restrict__ idsq,
              const double* __restrict__ idsq_c, const double* __restrict__ delta, const double* __restrict__ scal,
              int initial, int ns, int loss, double f_scale, double* __restrict__ x_new, double* __restrict__ camrec_new,
              double* __restrict__ V_new, double* __restrict__ g_new, double2* __restrict__ osc_new, double* __restrict__ partials)
{
    constexpr int NU = NC * (NC + 1) / 2, NV = NU + NC;
    extern __shared__ double smem[];
    double* s_cam = smem;
    double* s_rpc = s_cam + A.M * CAMREC_STRIDE;
    double* s_acc = s_rpc + (MODEL == MODEL_RPC ? A.M * RPC_TAB_STRIDE : 0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double* s_stage = s_acc + nw * A.M * NV;
    double* s_red = s_stage + nw * 9 * 33;
    const double pa = initial ? 0.0 : scal[SC_PA], pb = initial ? 0.0 : scal[SC_PB];
    // --- prologue: camera records of the trial point (every CTA, same arithmetic; CTA 0 publishes them) ---
    if (threadIdx.x < A.M) {
        const int j = threadIdx.x;
        double v[MAX_CAM_PARAMS];
#pragma unroll
        for (int s = 0; s < MAX_CAM_PARAMS; ++s) {
            double val = 0.0;
            if (s < A.P) {
                if (s < NC) {
                    const size_t e = (size_t)j * NC + s;
                    const double xv = initial ? x[e] : step_value2(x[e], g[e] * idsq_c[e], delta[e], pa, pb);
                    if (blockIdx.x == 0) x_new[e] = xv;
                    val = j >= A.n_cam_fix ? xv : A.cam_static[(size_t)j * A.P + s];
                } else {
                    val = A.cam_static[(size_t)j * A.P + s];
                }
            }
            v[s] = val;
        }
        build_camrec(v, MODEL, s_cam + j * CAMREC_STRIDE);
    }
    if (MODEL == MODEL_RPC)
        for (int t = threadIdx.x; t < A.M * RPC_TAB_STRIDE; t += blockDim.x) s_rpc[t] = A.rpc_tab[t];
    for (int t = threadIdx.x; t < nw * A.M * NV; t += blockDim.x) s_acc[t] = 0.0;
    __syncthreads();
    if (blockIdx.x == 0)
        for (int t = threadIdx.x; t < A.M * CAMREC_STRIDE; t += blockDim.x) camrec_new[t] = s_cam[t];

    double cost[1] = {0.0};
    double* stg = s_stage + warp * 9 * 33;           // stride 33: the (track, value) lanes below read conflict-free
    double* my_acc = s_acc + warp * A.M * NV;            // camera blocks of this warp's units: private, no ordering needed
    const int u0 = A.warp_unit0[blockIdx.x * nw + warp], u1 = A.debug_skip ? u0 : A.warp_unit0[blockIdx.x * nw + warp + 1];
    const long long cyc0 = clock64();
    for (int u = u0; u < u1; ++u) {
        const PUnit un = A.units[u];
        const LaneGeo G = lane_geometry(un, lane);
        const bool cam_free = G.cam >= A.n_cam_fix, pt_free = un.pts_free != 0;
        const double* rec = s_cam + G.cam * CAMREC_STRIDE;
        const double* rpc_j = MODEL == MODEL_RPC ? s_rpc + G.cam * RPC_TAB_STRIDE : nullptr;
        double acc[NV];
#pragma unroll
        for (int q = 0; q < NV; ++q) acc[q] = 0.0;
        for (int tb = 0; tb < un.ntrk; tb += G.T) {
            const int tt = tb + G.t;
            const bool on = G.on && tt < un.ntrk;
            const int nact = min(G.T, un.ntrk - tb);
            if (G.on && tt + G.T < un.ntrk) {          // next tile
                const size_t an = (size_t)un.obs0 + (size_t)(tt + G.T) * G.L + G.k, en = (size_t)ns + 3 * (size_t)(un.trk0 + tt + G.T);
                prefetch_l1(A.pts2d + an); prefetch_l1(A.w + an); prefetch_l1(x + en);
                if (!initial) { prefetch_l1(g + en); prefetch_l1(idsq + en); prefetch_l1(delta + en); }
            }
            double vals[9];
#pragma unroll
            for (int q = 0; q < 9; ++q) vals[q] = 0.0;
            if (on) {
                const int i = un.trk0 + tt;
                const size_t a = (size_t)un.obs0 + (size_t)tt * G.L + G.k;
                const size_t e3 = (size_t)ns + 3 * (size_t)i;
                const double2 ob = A.pts2d[a];
                const double wv = A.w[a];
                double X = x[e3], Y = x[e3 + 1], Z = x[e3 + 2];
                if (!initial) {
                    X = step_value2(X, g[e3] * idsq[e3], delta[e3], pa, pb);
                    Y = step_value2(Y, g[e3 + 1] * idsq[e3 + 1], delta[e3 + 1], pa, pb);
                    Z = step_value2(Z, g[e3 + 2] * idsq[e3 + 2], delta[e3 + 2], pa, pb);
                }
                if (G.k == 0) { x_new[e3] = X; x_new[e3 + 1] = Y; x_new[e3 + 2] = Z; }
                ObsEval<MODEL, NC> e;
                {
                    // residual, robust cost and row scales (kept for the later passes at this point), then the scaled rows
                    double u, v;
                    full_side<MODEL, NC, true>(rec, rpc_j, X, Y, Z, u, v, e.Jc, e.Jp);
                    double f0 = wv * (u - ob.x), f1 = wv * (v - ob.y), c0, c1;
                    const double s0 = wv * loss_rescale(loss, f_scale, f0, c0);
                    const double s1 = wv * loss_rescale(loss, f_scale, f1, c1);
                    osc_new[a] = make_double2(s0, s1);
                    e.f0 = f0; e.f1 = f1; e.cost = c0 + c1;
                    const double a0 = cam_free ? s0 : 0.0, a1 = cam_free ? s1 : 0.0;
#pragma unroll
                    for (int q = 0; q < NC; ++q) { e.Jc[q] *= a0; e.Jc[NC + q] *= a1; }
                    const double b0 = pt_free ? s0 : 0.0, b1 = pt_free ? s1 : 0.0;
#pragma unroll
                    for (int q = 0; q < 3; ++q) { e.Jp[q] *= b0; e.Jp[3 + q] *= b1; }
                }
                cost[0] += e.cost;
                vals[0] = e.Jp[0] * e.Jp[0] + e.Jp[3] * e.Jp[3];
                vals[1] = e.Jp[0] * e.Jp[1] + e.Jp[3] * e.Jp[4];
                vals[2] = e.Jp[0] * e.Jp[2] + e.Jp[3] * e.Jp[5];
                vals[3] = e.Jp[1] * e.Jp[1] + e.Jp[4] * e.Jp[4];
                vals[4] = e.Jp[1] * e.Jp[2] + e.Jp[4] * e.Jp[5];
                vals[5] = e.Jp[2] * e.Jp[2] + e.Jp[5] * e.Jp[5];
                vals[6] = e.Jp[0] * e.f0 + e.Jp[3] * e.f1;
                vals[7] = e.Jp[1] * e.f0 + e.Jp[4] * e.f1;
                vals[8] = e.Jp[2] * e.f0 + e.Jp[5] * e.f1;
                int q = 0;
#pragma unroll
                for (int r = 0; r < NC; ++r) {
#pragma unroll
                    for (int c = 0; c <= r; ++c) { acc[q] = fma(e.Jc[NC + r], e.Jc[NC + c], fma(e.Jc[r], e.Jc[c], acc[q])); ++q; }
                }
#pragma unroll
                for (int r = 0; r < NC; ++r) acc[NU + r] = fma(e.Jc[NC + r], e.f1, fma(e.Jc[r], e.f0, acc[NU + r]));
            }
            // per-track sums of the 9 point values: one lane per (track, value)
#pragma unroll
            for (int q = 0; q < 9; ++q) stg[q * 33 + lane] = vals[q];
            __syncwarp();
            for (int s = lane; s < 9 * nact; s += 32) {
                const int tr = s / 9, q = s - 9 * tr;
                const double* src = stg + q * 33 + tr * G.L;
                double tsum = 0.0;
                for (int m = 0; m < G.L; ++m) tsum += src[m];
                const int it = un.trk0 + tb + tr;
                if (q < 6) V_new[6 * (size_t)it + q] = tsum;
                else g_new[(size_t)ns + 3 * (size_t)it + (q - 6)] = tsum;
            }
            __syncwarp();
        }
        // flush the camera blocks of the unit: sum over the track slots, then into the warp's accumulators
        slot_reduce_n<NV>(acc, G);
        if (G.on && G.t == 0) {
            double* dst = my_acc + G.cam * NV;
#pragma unroll
            for (int q = 0; q < NV; ++q) dst[q] += acc[q];
        }
        __syncwarp();
    }
    if (A.cycles && lane == 0) A.cycles[blockIdx.x * nw + warp] = clock64() - cyc0;
    const double ctot = cta_reduce_sum<1>(cost, s_red);       // contains __syncthreads: all flushes are complete
    for (int t = threadIdx.x; t < A.M * NV; t += blockDim.x) {
        double sum = 0.0;
        for (int wq = 0; wq < nw; ++wq) sum += s_acc[wq * A.M * NV + t];     // warp order: fixed
        partials[(size_t)t * A.n_cta + blockIdx.x] = sum;
    }
    if (threadIdx.x == 0) partials[(size_t)A.M * NV * A.n_cta + blockIdx.x] = ctot;
}

// Sum of the per-CTA partials of k_pt_assemble -> camsys = [U (M, NC, NC) | g_c (M NC) | cost].  One CTA; one warp per
// value, lanes stride over the CTAs, fixed shuffle tree.  fold != 0 (single GPU): also derive the camera scaling.
//   dsq_c_new = first ? (diag U == 0 ? 1 : diag U) : max(dsq_c_cur, diag U)      (x_scale='jac', scipy common.py:598-610, squared)
__device__ __forceinline__ void cam_scale_dev(const double* __restrict__ camsys, const double* __restrict__ dsq_c_cur,
                                              int first, int M, int NC, double* __restrict__ dsq_c_new,
                                              double* __restrict__ idsq_c_new, double* __restrict__ g_new, double* scal)
{
    const int ns = M * NC;
    for (int e = threadIdx.x; e < ns; e += blockDim.x) {
        const int j = e / NC, s = e - j * NC;
        const double diag = __ldcg(camsys + (size_t)j * NC * NC + s * NC + s);
        const double d = first ? (diag == 0.0 ? 1.0 : diag) : fmax(dsq_c_cur[e], diag);
        dsq_c_new[e] = d;
        idsq_c_new[e] = 1.0 / d;
        g_new[e] = __ldcg(camsys + (size_t)M * NC * NC + e);
    }
    if (threadIdx.x == 0) scal[SC_COST_NEW] = __ldcg(camsys + (size_t)M * NC * NC + ns);
}

template <int NC>
__global__ void __launch_bounds__(256)
k_pt_reduce_assemble(const double* __restrict__ partials, int n_cta, int M, double* __restrict__ camsys, int fold,
                     const double* __restrict__ dsq_c_cur, int first, double* __restrict__ dsq_c_new,
                     double* __restrict__ idsq_c_new, double* __restrict__ g_new, double* scal, unsigned* counter, CommFused comm)
{
    constexpr int NU = NC * (NC + 1) / 2, NV = NU + NC;
    const int lane = threadIdx.x & 31;
    const int total = M * NV + 1;
    const int v = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (v < total) {
        double s = 0.0;
        for (int b = lane; b < n_cta; b += 32) s += partials[(size_t)v * n_cta + b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            if (v == M * NV) {
                camsys[(size_t)M * NC * NC + (size_t)M * NC] = s;
            } else {
                const int j = v / NV, q = v - j * NV;
                if (q < NU) {
                    int r = 0;
                    while ((r + 1) * (r + 2) / 2 <= q) ++r;
                    const int c = q - r * (r + 1) / 2;
                    camsys[(size_t)j * NC * NC + r * NC + c] = s;
                    camsys[(size_t)j * NC * NC + c * NC + r] = s;
                } else {
                    camsys[(size_t)M * NC * NC + (size_t)j * NC + (q - NU)] = s;
                }
            }
        }
    }
    if (!fold) return;
    // the last CTA to finish derives the camera scaling from the complete sums
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x == 0) *counter = 0u;
    if (comm.on) cta_allreduce(comm.c, camsys, M * NC * NC + M * NC + 1, comm.seq, scal);      // multi-GPU: [U | g_c | cost] summed over the ranks
    cam_scale_dev(camsys, dsq_c_cur, first, M, NC, dsq_c_new, idsq_c_new, g_new, scal);
}

__global__ void __launch_bounds__(256)
k_pt_cam_scale(const double* __restrict__ camsys, const double* __restrict__ dsq_c_cur, int first, int M, int NC,
               double* __restrict__ dsq_c_new, double* __restrict__ idsq_c_new, double* __restrict__ g_new, double* scal)
{
    cam_scale_dev(camsys, dsq_c_cur, first, M, NC, dsq_c_new, idsq_c_new, g_new, scal);
}

// ------------------------------------------------------------------------------------------------
// device-side control (shared by the single-thread kernel and the folded epilogue; the damping rule control_reg_dev is
// in sba_kernels.cuh, shared with the generic engine)
// ------------------------------------------------------------------------------------------------
// 2-D subspace {g_h, gn_h}: the Gram scalars of (t1, delta) are turned into those of the orthogonalised pair (t1, t2 = delta -
// alpha t1), then the exact 2-D trust-region problem is solved (scipy trf.py:496-509).  Step = pa t1 + pb delta.
__device__ __forceinline__ void control_tr2d_gram_dev(double* scal, double delta_arg)
{
    const double Delta = delta_arg < 0.0 ? scal[SC_DELTA] : delta_arg;
    const double gg = scal[SC_GG], gd = scal[SC_P_GD], dd = scal[SC_P_DD];
    const double b11 = scal[SC_A], c12 = scal[SC_P_C12], c22 = scal[SC_P_C22];
    const double t11 = scal[SC_P_T11], t1d = scal[SC_P_T1D], tdd = scal[SC_P_TDD];
    const double alpha = gg > 0.0 ? gd / gg : 0.0;
    double ww = dd - alpha * gd;                       // |gn_h - alpha g_h|^2
    if (!(ww > 1e-14 * dd)) ww = 0.0;                  // gn_h parallel to g_h to rounding: the subspace is 1-D
    const double b12 = c12 - alpha * b11, b22 = c22 - 2.0 * alpha * c12 + alpha * alpha * b11;
    const double t12 = t1d - alpha * t11, t22 = fmax(0.0, tdd - 2.0 * alpha * t1d + alpha * alpha * t11);
    const double n1 = sqrt(gg);
    const bool rank2 = ww > 0.0 && b22 > 0.0;
    const double n2 = rank2 ? sqrt(ww) : 1.0;
    const double B00 = b11 / (n1 * n1), B01 = rank2 ? b12 / (n1 * n2) : 0.0, B11 = rank2 ? b22 / (n2 * n2) : 1.0;
    const double gS0 = n1, gS1 = 0.0;                  // w is orthogonal to g_h by construction
    double pS[2];
    solve_trust_region_2d(B00, B01, B11, gS0, gS1, Delta, pS);
    const double c1 = pS[0] / n1, c2 = rank2 ? pS[1] / n2 : 0.0;
    scal[SC_C1] = c1;
    scal[SC_C2] = c2;
    scal[SC_PA] = c1 - c2 * alpha;
    scal[SC_PB] = c2;
    scal[SC_PRED] = -(0.5 * (B00 * pS[0] * pS[0] + 2.0 * B01 * pS[0] * pS[1] + B11 * pS[1] * pS[1]) + gS0 * pS[0] + gS1 * pS[1]);
    scal[SC_STEPH] = sqrt(pS[0] * pS[0] + pS[1] * pS[1]);
    scal[SC_STEPN] = sqrt(fmax(0.0, c1 * c1 * t11 + 2.0 * c1 * c2 * t12 + c2 * c2 * t22));
    scal[SC_B22] = b22;                                // diagnostics read by the host
}

__global__ void k_pt_control_tr2d(double* scal, double delta_arg)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) control_tr2d_gram_dev(scal, delta_arg);
}

// ------------------------------------------------------------------------------------------------
// K2: scaling of the points + |g_h|^2, |x D|^2, |x|^2, max|g| + |J_h g_h|^2  (-> damping)
//   dsq_p = first ? (diag V == 0 ? 1 : diag V) : max(dsq_p, diag V), idsq_p = 1 / dsq_p   (in place, one writer per track)
// shared: s_cam | s_rpc | s_t1c[ns] | s_red
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC>
__global__ void __launch_bounds__(PT_THREADS_LIGHT, 1)
k_pt_jvp1(PatView A, const double* __restrict__ x, const double* __restrict__ camrec, const double* __restrict__ V,
          const double* __restrict__ g, const double* __restrict__ dsq_c, const double* __restrict__ idsq_c,
          double* __restrict__ dsq, double* __restrict__ idsq, const double2* __restrict__ osc, int first, int ns,
          int count_cameras, int rank, double* partials, unsigned* counter, double* scal, int fold_ctl, double delta_arg, CommFused comm)
{
    extern __shared__ double smem[];
    double* s_cam = smem;
    double* s_rpc = s_cam + A.M * CAMREC_STRIDE;
    double* s_t1c = s_rpc + (MODEL == MODEL_RPC ? A.M * RPC_TAB_STRIDE : 0);
    double* s_red = s_t1c + ns;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    load_cameras_shared<MODEL>(A, camrec, s_cam, s_rpc);
    for (int e = threadIdx.x; e < ns; e += blockDim.x) s_t1c[e] = g[e] * idsq_c[e];
    __syncthreads();
    double acc[4] = {0.0, 0.0, 0.0, 0.0};       // gg, xs, xx, |J t1|^2
    double gmax = 0.0;
    if (blockIdx.x == 0 && count_cameras) {
        for (int e = threadIdx.x; e < ns; e += blockDim.x) {
            const double gv = g[e], xv = x[e];
            acc[0] += gv * gv * idsq_c[e];
            acc[1] += xv * xv * dsq_c[e];
            acc[2] += xv * xv;
            gmax = fmax(gmax, fabs(gv));
        }
    }
    const int u0 = A.warp_unit0[blockIdx.x * nw + warp], u1 = A.debug_skip ? u0 : A.warp_unit0[blockIdx.x * nw + warp + 1];
    const long long cyc0 = clock64();
    for (int u = u0; u < u1; ++u) {
        const PUnit un = A.units[u];
        const LaneGeo G = lane_geometry(un, lane);
        const bool cam_free = G.cam >= A.n_cam_fix, pt_free = un.pts_free != 0;
        const double* rec = s_cam + G.cam * CAMREC_STRIDE;
        const double* rpc_j = MODEL == MODEL_RPC ? s_rpc + G.cam * RPC_TAB_STRIDE : nullptr;
        const double* t1c = s_t1c + G.cam * NC;
        for (int tb = 0; tb < un.ntrk; tb += G.T) {
            const int tt = tb + G.t;
            if (!(G.on && tt < un.ntrk)) continue;
            if (tt + G.T < un.ntrk) {          // next tile
                const size_t in = (size_t)(un.trk0 + tt + G.T), en = (size_t)ns + 3 * in;
                prefetch_l1(osc + (size_t)un.obs0 + (size_t)(tt + G.T) * G.L + G.k);
                prefetch_l1(x + en); prefetch_l1(g + en); prefetch_l1(dsq + en); prefetch_l1(V + 6 * in);
            }
            const int i = un.trk0 + tt;
            const size_t a = (size_t)un.obs0 + (size_t)tt * G.L + G.k;
            const size_t e3 = (size_t)ns + 3 * (size_t)i;
            const double2 sc = osc[a];
            const double X = x[e3], Y = x[e3 + 1], Z = x[e3 + 2];
            const double vd[3] = {V[6 * (size_t)i], V[6 * (size_t)i + 3], V[6 * (size_t)i + 5]};
            double t1p[3], d2[3], gp[3];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                gp[q] = g[e3 + q];
                d2[q] = first ? (vd[q] == 0.0 ? 1.0 : vd[q]) : fmax(dsq[e3 + q], vd[q]);
                const double id = fast_rcp(d2[q]);
                t1p[q] = gp[q] * id;
                if (G.k == 0) { dsq[e3 + q] = d2[q]; idsq[e3 + q] = id; }
            }
            if (G.k == 0) {
                acc[0] += gp[0] * t1p[0] + gp[1] * t1p[1] + gp[2] * t1p[2];
                acc[1] += X * X * d2[0] + Y * Y * d2[1] + Z * Z * d2[2];
                acc[2] += X * X + Y * Y + Z * Z;
                gmax = fmax(gmax, fmax(fabs(gp[0]), fmax(fabs(gp[1]), fabs(gp[2]))));
            }
            ObsEval<MODEL, NC> e;
            eval_scaled<MODEL, NC>(rec, rpc_j, X, Y, Z, sc, cam_free, pt_free, e);
            double y0 = e.Jp[0] * t1p[0] + e.Jp[1] * t1p[1] + e.Jp[2] * t1p[2];
            double y1 = e.Jp[3] * t1p[0] + e.Jp[4] * t1p[1] + e.Jp[5] * t1p[2];
#pragma unroll
            for (int q = 0; q < NC; ++q) { y0 += e.Jc[q] * t1c[q]; y1 += e.Jc[NC + q] * t1c[q]; }
            acc[3] = fma(y1, y1, fma(y0, y0, acc[3]));
        }
    }
    if (A.cycles && lane == 0) A.cycles[blockIdx.x * nw + warp] = clock64() - cyc0;
    if (A.cycles && threadIdx.x == 0) { unsigned sm; asm("mov.u32 %0, %%smid;" : "=r"(sm)); A.cycles[(size_t)4 * PT_CTAS * 32 + blockIdx.x] = sm; }
    // max |g| of this rank (non-negative doubles order like their bit patterns; the slot is zeroed by the host)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_down_sync(0xffffffffu, gmax, o));
    if (lane == 0 && gmax > 0.0)
        atomicMax((unsigned long long*)(scal + SC_GMAX_SLOTS + rank), (unsigned long long)__double_as_longlong(gmax));
    const double tot = cta_reduce_sum<4>(acc, s_red);
    __shared__ int slots[4];
    if (threadIdx.x == 0) { slots[0] = SC_GG; slots[1] = SC_XS; slots[2] = SC_XX; slots[3] = SC_A; }
    __syncthreads();
    const bool last = grid_sum_last<4>(tot, partials, counter, scal, slots);
    if (last && comm.on) cta_allreduce(comm.c, scal + SC_COST, SC_GGN - SC_COST, comm.seq, scal);
    if (last && fold_ctl && threadIdx.x == 0) control_reg_dev(scal, delta_arg, -1.0);
}

// ------------------------------------------------------------------------------------------------
// K3: point elimination + Schur complement in shared memory
// shared: s_cam | s_rpc | s_Z[nwarps][32 * ZP]
// The CTA's partial of S is stored by upper block rows: block (j, j' >= j) at NC*NC * (j M - j (j-1)/2 + j' - j), row-major NC x NC.
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline int pt_block_offset(int j, int jp, int M, int NC)
{
    return NC * NC * (j * M - j * (j - 1) / 2 + (jp - j));
}

// tasks of a lane in one pass over a unit: (position pair ka <= kb, row chunk h); few tasks (short tracks): npar groups of
// lanes take every npar-th track slot of a tile in parallel
template <int NC>
struct SchurTasks {
    static constexpr int NCH = (NC + PT_RC - 1) / PT_RC;
    int ntask, npass, npar, par;
    int ka[2], kb[2], hh[2];
    bool tv[2];
    __device__ __forceinline__ void unit(int L, int lane)
    {
        ntask = L * (L + 1) / 2 * NCH;
        npass = (ntask + 63) / 64;
        npar = ntask <= 16 ? 32 / ntask : 1;
        par = npar > 1 ? lane / ntask : 0;
    }
    __device__ __forceinline__ void pass(int L, int lane, int p)
    {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int tau = p * 64 + q * 32 + lane;
            tv[q] = tau < ntask;
            if (npar > 1) { tau = lane - par * ntask; tv[q] = q == 0 && par < npar; }
            const int pr = tv[q] ? tau / NCH : 0;
            hh[q] = tv[q] ? tau - pr * NCH : 0;
            int a = 0, rem = pr;
            while (rem >= L - a) { rem -= L - a; ++a; }
            ka[q] = a; kb[q] = a + rem;
        }
    }
};

// One record per (unit, pass): the lane-private sums of a pass, [2 tasks][32 lanes][NA values] then [NC rhs values][32 lanes]
// (rows a pass does not use are neither written nor read).  Records are written when a warp leaves a unit and merged into
// the CTA's shared-memory S after all warps are done, warp by warp in unit order: fixed summation order without any
// waiting inside the main loop.
template <int NC> __host__ __device__ constexpr int pt_record_doubles() { return (2 * PT_RC * NC + NC) * 32; }

template <int MODEL, int NC>
__global__ void __launch_bounds__(PT_THREADS_SCHUR, 1)
k_pt_schur(PatView A, const double* __restrict__ x, const double* __restrict__ camrec, const double* __restrict__ V,
           const double* __restrict__ g, const double* __restrict__ dsq, const double2* __restrict__ osc,
           const double* __restrict__ scal, int ns, double* __restrict__ records, double* __restrict__ partials, double* bad_points)
{
    constexpr int ZS = NC * 3, ZP = ZS + 1;
    constexpr int NA = PT_RC * NC;                       // accumulators per task
    constexpr int REC = pt_record_doubles<NC>();
    extern __shared__ double smem[];
    const int nS = NC * NC * (A.M * (A.M + 1) / 2);
    double* s_cam = smem;
    double* s_rpc = s_cam + A.M * CAMREC_STRIDE;
    double* s_Z = s_rpc + (MODEL == MODEL_RPC ? A.M * RPC_TAB_STRIDE : 0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double reg = scal[SC_REG];
    load_cameras_shared<MODEL>(A, camrec, s_cam, s_rpc);
    __syncthreads();
    double* zs = s_Z + (size_t)warp * (32 * ZP + PT_RC * 3);          // tail padding: the last chunk may read past row NC-1
    int nbad = 0;
    const int u0 = A.warp_unit0[blockIdx.x * nw + warp], u1 = A.debug_skip ? u0 : A.warp_unit0[blockIdx.x * nw + warp + 1];
    SchurTasks<NC> tk;
    const long long cyc0 = clock64();
    for (int u = u0; u < u1; ++u) {
        const PUnit un = A.units[u];
        const LaneGeo G = lane_geometry(un, lane);
        const bool cam_free = G.cam >= A.n_cam_fix, pt_free = un.pts_free != 0;
        const double* rec = s_cam + G.cam * CAMREC_STRIDE;
        const double* rpc_j = MODEL == MODEL_RPC ? s_rpc + G.cam * RPC_TAB_STRIDE : nullptr;
        tk.unit(G.L, lane);
        for (int pass = 0; pass < tk.npass; ++pass) {
            tk.pass(G.L, lane, pass);
            double acc[2][NA], accR[NC];
#pragma unroll
            for (int q = 0; q < 2; ++q)
#pragma unroll
                for (int m = 0; m < NA; ++m) acc[q][m] = 0.0;
#pragma unroll
            for (int r = 0; r < NC; ++r) accR[r] = 0.0;
            for (int tb = 0; tb < un.ntrk; tb += G.T) {
                const int tt = tb + G.t;
                const bool on = G.on && tt < un.ntrk;
                const int nact = min(G.T, un.ntrk - tb);
                if (G.on && tt + G.T < un.ntrk) {          // next tile
                    const size_t in = (size_t)(un.trk0 + tt + G.T), en = (size_t)ns + 3 * in;
                    prefetch_l1(osc + (size_t)un.obs0 + (size_t)(tt + G.T) * G.L + G.k);
                    prefetch_l1(x + en); prefetch_l1(g + en); prefetch_l1(dsq + en); prefetch_l1(V + 6 * in);
                }
                if (on) {
                    const int i = un.trk0 + tt;
                    const size_t a = (size_t)un.obs0 + (size_t)tt * G.L + G.k;
                    const size_t e3 = (size_t)ns + 3 * (size_t)i;
                    const double2 sc = osc[a];
                    const double X = x[e3], Y = x[e3 + 1], Z = x[e3 + 2];
                    const double* v = V + 6 * (size_t)i;
                    double Gm[6], qv[3] = {0.0, 0.0, 0.0};
                    bool ok = false;
                    if (pt_free) ok = invert_point_block_d2(v[0], v[1], v[2], v[3], v[4], v[5], dsq[e3], dsq[e3 + 1], dsq[e3 + 2], reg, Gm);
                    if (!ok) {
#pragma unroll
                        for (int m = 0; m < 6; ++m) Gm[m] = 0.0;
                        if (pt_free && G.k == 0 && pass == 0) ++nbad;
                    } else {
                        const double g0 = g[e3], g1 = g[e3 + 1], g2 = g[e3 + 2];
                        qv[0] = Gm[0] * g0;
                        qv[1] = Gm[1] * g0 + Gm[2] * g1;
                        qv[2] = Gm[3] * g0 + Gm[4] * g1 + Gm[5] * g2;
                    }
                    ObsEval<MODEL, NC> e;
                    eval_scaled<MODEL, NC>(rec, rpc_j, X, Y, Z, sc, cam_free, pt_free, e);
                    double* z = zs + lane * ZP;
#pragma unroll
                    for (int r = 0; r < NC; ++r) {
                        const double w0 = e.Jc[r] * e.Jp[0] + e.Jc[NC + r] * e.Jp[3];
                        const double w1 = e.Jc[r] * e.Jp[1] + e.Jc[NC + r] * e.Jp[4];
                        const double w2 = e.Jc[r] * e.Jp[2] + e.Jc[NC + r] * e.Jp[5];
                        const double z0 = w0 * Gm[0], z1 = w0 * Gm[1] + w1 * Gm[2], z2 = w0 * Gm[3] + w1 * Gm[4] + w2 * Gm[5];
                        z[3 * r] = z0; z[3 * r + 1] = z1; z[3 * r + 2] = z2;
                        if (pass == 0) accR[r] = fma(z2, qv[2], fma(z1, qv[1], fma(z0, qv[0], accR[r])));
                    }
                }
                __syncwarp();
                for (int ts = tk.par; ts < nact; ts += tk.npar) {
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        if (!tk.tv[q]) continue;
                        const double* za = zs + (ts * G.L + tk.ka[q]) * ZP + tk.hh[q] * PT_RC * 3;
                        const double* zb = zs + (ts * G.L + tk.kb[q]) * ZP;
                        double Ar[PT_RC * 3];
#pragma unroll
                        for (int m = 0; m < PT_RC * 3; ++m) Ar[m] = za[m];
#pragma unroll
                        for (int s = 0; s < NC; ++s) {
                            const double b0 = zb[3 * s], b1 = zb[3 * s + 1], b2 = zb[3 * s + 2];
#pragma unroll
                            for (int r = 0; r < PT_RC; ++r)
                                acc[q][r * NC + s] = fma(Ar[3 * r + 2], b2, fma(Ar[3 * r + 1], b1, fma(Ar[3 * r], b0, acc[q][r * NC + s])));      // three chained DFMA
                        }
                    }
                }
                __syncwarp();
            }
            if (tk.npar > 1) {        // sum over the parallel groups (fixed tree); group 0 keeps the result
                for (int off = 1; off < tk.npar; off <<= 1) {
#pragma unroll
                    for (int m = 0; m < NA; ++m) {
                        const double o = __shfl_down_sync(0xffffffffu, acc[0][m], (unsigned)(off * tk.ntask));
                        if (tk.tv[0] && tk.par + off < tk.npar) acc[0][m] += o;
                    }
                }
            }
            // the record of this (unit, pass): task-major ([q][lane][NA], transposed through the warp's Z area so that the
            // stores are coalesced and the merge below reads the NA values of a task as one contiguous span), then the rhs rows
            double* rp = records + (size_t)(un.rec + pass) * REC;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                if (pass * 64 + q * 32 >= tk.ntask) continue;        // warp-uniform: no lane has this task
#pragma unroll
                for (int m = 0; m < NA; ++m) zs[lane * NA + m] = acc[q][m];
                __syncwarp();
                for (int e = lane; e < 32 * NA; e += 32) rp[q * 32 * NA + e] = zs[e];
                __syncwarp();
            }
            if (pass == 0) {
                slot_reduce_n<NC>(accR, G);
#pragma unroll
                for (int r = 0; r < NC; ++r) rp[(2 * NA + r) * 32 + lane] = accR[r];
            }
        }
    }
    if (A.cycles && lane == 0) A.cycles[blockIdx.x * nw + warp] = clock64() - cyc0;
    if (nbad) atomicAdd(bad_points, (double)nbad);
    __threadfence();
    __syncthreads();
    // Merge: every entry of the CTA's partial S (and rhs) is owned by one thread, which adds up the contributions of the
    // CTA's units in unit order -- parallel over the entries, fixed summation order, no read-modify-write conflicts.  Where a
    // unit's record holds the entry follows from its camera set: positions ka, kb of the two cameras -> pair -> task -> lane.
    // The unit descriptors go through shared memory (the Z areas are free now) and the record loads are issued eight units at
    // a time (units that do not contain the entry read a zero), so the L2 round trips overlap.
    {
        constexpr int NCH = SchurTasks<NC>::NCH;
        constexpr int MU = 4;
        const int cu0 = A.warp_unit0[blockIdx.x * nw], cu1 = A.warp_unit0[(blockIdx.x + 1) * nw];
        const int ncu = cu1 - cu0;
        // per unit: mask (2 ints), L, rec -> 4 ints; capacity of the Z area
        int* s_units = reinterpret_cast<int*>(s_Z);
        const int cap = (int)(((size_t)nw * (32 * ZP + PT_RC * 3) * sizeof(double)) / (4 * sizeof(int))) - 1;
        for (int c0 = 0; c0 < max(ncu, 1); c0 += cap) {        // a CTA without units still writes its (zero) partial
            const int nc_here = min(cap, ncu - c0);
            __syncthreads();
            for (int q = threadIdx.x; q < nc_here; q += blockDim.x) {
                const PUnit un = A.units[cu0 + c0 + q];
                s_units[4 * q] = (int)un.mask_lo; s_units[4 * q + 1] = (int)un.mask_hi; s_units[4 * q + 2] = un.L; s_units[4 * q + 3] = un.rec;
            }
            if (threadIdx.x == 0) { s_units[4 * nc_here] = 0; }
            __syncthreads();
            // one thread per (camera block, row) -- the NC entries of a row are contiguous in a task's record -- and one per
            // camera for the rhs; MU units at a time: NC * MU independent loads in flight
            const int nrow = (A.M * (A.M + 1) / 2) * NC;
            for (int task = threadIdx.x; task < nrow + A.M; task += blockDim.x) {
                double sum[NC];
                const bool is_S = task < nrow;
                int ja = 0, jb = 0, h = 0, mrow = 0;
                size_t t0;       // first entry of this thread in the partial vector
                if (is_S) {
                    int bq = task / NC;
                    const int r = task - bq * NC;
                    t0 = (size_t)bq * NC * NC + (size_t)r * NC;
                    while (bq >= A.M - ja) { bq -= A.M - ja; ++ja; }
                    jb = ja + bq;
                    h = r / PT_RC; mrow = (r - h * PT_RC) * NC;
                } else {
                    ja = jb = task - nrow;
                    t0 = (size_t)nS + (size_t)ja * NC;
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) sum[c] = c0 == 0 ? 0.0 : partials[(t0 + c) * A.n_cta + blockIdx.x];
                for (int q0 = 0; q0 < nc_here; q0 += MU) {
                    double val[MU][NC];
#pragma unroll
                    for (int qq = 0; qq < MU; ++qq) {
                        const int q = min(q0 + qq, nc_here - 1);
                        const unsigned long long mask = ((unsigned long long)(unsigned)s_units[4 * q + 1] << 32) | (unsigned)s_units[4 * q];
                        const int L = s_units[4 * q + 2], rec0 = s_units[4 * q + 3];
                        const bool has = q0 + qq < nc_here && ((mask >> ja) & 1ull) && ((mask >> jb) & 1ull);
                        const int ka = __popcll(mask & ((1ull << ja) - 1ull)), kb = __popcll(mask & ((1ull << jb) - 1ull));
                        const double* src;
                        int stride;
                        if (is_S) {
                            const int tau = (ka * L - ka * (ka - 1) / 2 + (kb - ka)) * NCH + h;
                            src = records + (size_t)(rec0 + (tau >> 6)) * REC + (((tau >> 5) & 1) * 32 + (tau & 31)) * NA + mrow;
                            stride = 1;
                        } else {
                            src = records + (size_t)rec0 * REC + (2 * NA) * 32 + ka;
                            stride = 32;
                        }
#pragma unroll
                        for (int c = 0; c < NC; ++c) val[qq][c] = has ? __ldcg(src + c * stride) : 0.0;
                    }
#pragma unroll
                    for (int qq = 0; qq < MU; ++qq)
#pragma unroll
                        for (int c = 0; c < NC; ++c) sum[c] += val[qq][c];
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) partials[(t0 + c) * A.n_cta + blockIdx.x] = sum[c];
            }
        }
    }
}

// D += A (8 x 4, row-major fragment: lane holds A[lane / 4][lane % 4]) x B (4 x 8, column-major fragment: lane holds
// B[lane % 4][lane / 4]); a lane owns D[lane / 4][2 (lane % 4)] and the column next to it.  FP64 tensor-core path (DMMA):
// one warp instruction does the 256 FMAs that cost 8 DFMA instructions plus their operand loads on the FP64 pipe.
__device__ __forceinline__ void mma_f64_884(double (&d)[2], double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}
template <int NC> __host__ __device__ constexpr int pt_record_doubles_mma() { return PT_MMA_TILES * 64 + NC * 32; }

// K3, tensor-core variant (SBA_PT_SCHUR=mma; NOT the default): the same elimination, with the products Z_a Z_b^T of all camera
// pairs of a track formed as the Gram matrix of the track's stacked Z rows by m8n8k4 DMMA (k = 3 padded to 4).  When a tile lies
// on the diagonal of the Gram matrix both triangles are computed; the merge reads the upper one.  Results agree with the DFMA
// kernel to rounding (tests/test_gpu_ba.py::test_schur_kernel_variants).  Measured on B200 at 1e6 observations: 236 us against
// 127 us -- the DFMA kernel already spreads the (pair, row chunk) tasks of a track over the 32 lanes, so both issue ~80 warp
// instructions per track, and with 3 warps per scheduler the DMMA chain (fragment loads -> 10 dependent-accumulator MMAs) hides
// less latency than 54 independent DFMAs per lane.  tools/dmma_lat.cu: DMMA issues at 16 cycles per SM sub-partition (37 TFLOP/s)
// from 3 warps on, so the pipe itself is not the limit.
template <int MODEL, int NC>
__global__ void __launch_bounds__(PT_THREADS_SCHUR, 1)
k_pt_schur_mma(PatView A, const double* __restrict__ x, const double* __restrict__ camrec, const double* __restrict__ V,
           const double* __restrict__ g, const double* __restrict__ dsq, const double2* __restrict__ osc,
           const double* __restrict__ scal, int ns, double* __restrict__ records, double* __restrict__ partials, double* bad_points)
{
    constexpr int ZS = NC * 3, ZP = ZS + 1;
    constexpr int NTP = PT_MMA_TILES;
    constexpr int REC = pt_record_doubles_mma<NC>();
    extern __shared__ double smem[];
    const int nS = NC * NC * (A.M * (A.M + 1) / 2);
    double* s_cam = smem;
    double* s_rpc = s_cam + A.M * CAMREC_STRIDE;
    double* s_Z = s_rpc + (MODEL == MODEL_RPC ? A.M * RPC_TAB_STRIDE : 0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double reg = scal[SC_REG];
    load_cameras_shared<MODEL>(A, camrec, s_cam, s_rpc);
    __syncthreads();
    double* zs = s_Z + (size_t)warp * (32 * ZP + PT_RC * 3);          // tail padding: the last chunk may read past row NC-1
    int nbad = 0;
    const int u0 = A.warp_unit0[blockIdx.x * nw + warp], u1 = A.debug_skip ? u0 : A.warp_unit0[blockIdx.x * nw + warp + 1];
    const int frow = lane >> 2, fk = lane & 3;           // fragment coordinates of the lane: row of the 8 x 4 operand, k index
    const long long cyc0 = clock64();
    for (int u = u0; u < u1; ++u) {
        const PUnit un = A.units[u];
        const LaneGeo G = lane_geometry(un, lane);
        const bool cam_free = G.cam >= A.n_cam_fix, pt_free = un.pts_free != 0;
        const double* rec = s_cam + G.cam * CAMREC_STRIDE;
        const double* rpc_j = MODEL == MODEL_RPC ? s_rpc + G.cam * RPC_TAB_STRIDE : nullptr;
        // Gram matrix of a track's stacked Z rows (L NC rows x 3): 8 x 8 tiles, upper triangle, tile (i, j) = number j (j + 1) / 2 + i.
        // One pass when R <= 6 (the tile -> (i, j) map is then static and every operand fragment is loaded once per track).
        const int nrows = G.L * NC, R = (nrows + 7) >> 3, ntile = R * (R + 1) / 2, npass = (ntile + NTP - 1) / NTP;
        int foff[6];                                         // offset of the lane's element of row block i inside a track's Z rows
        bool fok[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int row = 8 * i + frow, pos = row / NC;
            fok[i] = row < nrows && fk < 3;
            foff[i] = fok[i] ? pos * ZP + (row - pos * NC) * 3 + fk : 0;
        }
        for (int pass = 0; pass < npass; ++pass) {
            double C[NTP][2], accR[NC];
#pragma unroll
            for (int q = 0; q < NTP; ++q) { C[q][0] = 0.0; C[q][1] = 0.0; }
#pragma unroll
            for (int r = 0; r < NC; ++r) accR[r] = 0.0;
            for (int tb = 0; tb < un.ntrk; tb += G.T) {
                const int tt = tb + G.t;
                const bool on = G.on && tt < un.ntrk;
                const int nact = min(G.T, un.ntrk - tb);
                if (G.on && tt + G.T < un.ntrk) {          // next tile
                    const size_t in = (size_t)(un.trk0 + tt + G.T), en = (size_t)ns + 3 * in;
                    prefetch_l1(osc + (size_t)un.obs0 + (size_t)(tt + G.T) * G.L + G.k);
                    prefetch_l1(x + en); prefetch_l1(g + en); prefetch_l1(dsq + en); prefetch_l1(V + 6 * in);
                }
                if (on) {
                    const int i = un.trk0 + tt;
                    const size_t a = (size_t)un.obs0 + (size_t)tt * G.L + G.k;
                    const size_t e3 = (size_t)ns + 3 * (size_t)i;
                    const double2 sc = osc[a];
                    const double X = x[e3], Y = x[e3 + 1], Z = x[e3 + 2];
                    const double* v = V + 6 * (size_t)i;
                    double Gm[6], qv[3] = {0.0, 0.0, 0.0};
                    bool ok = false;
                    if (pt_free) ok = invert_point_block_d2(v[0], v[1], v[2], v[3], v[4], v[5], dsq[e3], dsq[e3 + 1], dsq[e3 + 2], reg, Gm);
                    if (!ok) {
#pragma unroll
                        for (int m = 0; m < 6; ++m) Gm[m] = 0.0;
                        if (pt_free && G.k == 0 && pass == 0) ++nbad;
                    } else {
                        const double g0 = g[e3], g1 = g[e3 + 1], g2 = g[e3 + 2];
                        qv[0] = Gm[0] * g0;
                        qv[1] = Gm[1] * g0 + Gm[2] * g1;
                        qv[2] = Gm[3] * g0 + Gm[4] * g1 + Gm[5] * g2;
                    }
                    ObsEval<MODEL, NC> e;
                    eval_scaled<MODEL, NC>(rec, rpc_j, X, Y, Z, sc, cam_free, pt_free, e);
                    double* z = zs + lane * ZP;
#pragma unroll
                    for (int r = 0; r < NC; ++r) {
                        const double w0 = e.Jc[r] * e.Jp[0] + e.Jc[NC + r] * e.Jp[3];
                        const double w1 = e.Jc[r] * e.Jp[1] + e.Jc[NC + r] * e.Jp[4];
                        const double w2 = e.Jc[r] * e.Jp[2] + e.Jc[NC + r] * e.Jp[5];
                        const double z0 = w0 * Gm[0], z1 = w0 * Gm[1] + w1 * Gm[2], z2 = w0 * Gm[3] + w1 * Gm[4] + w2 * Gm[5];
                        z[3 * r] = z0; z[3 * r + 1] = z1; z[3 * r + 2] = z2;
                        if (pass == 0) accR[r] = fma(z2, qv[2], fma(z1, qv[1], fma(z0, qv[0], accR[r])));
                    }
                }
                __syncwarp();
                if (npass == 1) {
                    for (int ts = 0; ts < nact; ++ts) {
                        const double* zt = zs + ts * G.L * ZP;
                        double fr[6];
#pragma unroll
                        for (int i = 0; i < 6; ++i) fr[i] = (i < R && fok[i]) ? zt[foff[i]] : 0.0;
#pragma unroll
                        for (int j = 0; j < 6; ++j) {
                            if (j < R) {                               // warp-uniform
#pragma unroll
                                for (int i = 0; i <= j; ++i) mma_f64_884(C[j * (j + 1) / 2 + i], fr[i], fr[j]);
                            }
                        }
                    }
                } else {
                    // many row blocks (long tracks): the tiles of this pass are decoded at run time, two operand loads per MMA
                    for (int ts = 0; ts < nact; ++ts) {
                        const double* zt = zs + ts * G.L * ZP;
                        int j = 0, s0 = pass * NTP;
                        while ((j + 1) * (j + 2) / 2 <= s0) ++j;
                        int i = s0 - j * (j + 1) / 2;
#pragma unroll
                        for (int q = 0; q < NTP; ++q) {
                            if (s0 + q < ntile) {                      // warp-uniform
                                const int ra = 8 * i + frow, pa = ra / NC, rb = 8 * j + frow, pb = rb / NC;
                                const double fa = (ra < nrows && fk < 3) ? zt[pa * ZP + (ra - pa * NC) * 3 + fk] : 0.0;
                                const double fb = (rb < nrows && fk < 3) ? zt[pb * ZP + (rb - pb * NC) * 3 + fk] : 0.0;
                                mma_f64_884(C[q], fa, fb);
                                if (++i > j) { i = 0; ++j; }
                            }
                        }
                    }
                }
                __syncwarp();
            }
            // the record of this (unit, pass): the accumulator tiles, row-major 8 x 8 each (a lane owns two adjacent columns), then the rhs rows
            double* rp = records + (size_t)(un.rec + pass) * REC;
#pragma unroll
            for (int q = 0; q < NTP; ++q)
                if (pass * NTP + q < ntile) { rp[q * 64 + 2 * lane] = C[q][0]; rp[q * 64 + 2 * lane + 1] = C[q][1]; }
            if (pass == 0) {
                slot_reduce_n<NC>(accR, G);
#pragma unroll
                for (int r = 0; r < NC; ++r) rp[(size_t)NTP * 64 + r * 32 + lane] = accR[r];
            }
        }
    }
    if (A.cycles && lane == 0) A.cycles[blockIdx.x * nw + warp] = clock64() - cyc0;
    if (nbad) atomicAdd(bad_points, (double)nbad);
    __threadfence();
    __syncthreads();
    // Merge: every entry of the CTA's partial S (and rhs) is owned by one thread, which adds up the contributions of the
    // CTA's units in unit order -- parallel over the entries, fixed summation order, no read-modify-write conflicts.  Where a
    // unit's record holds the entry follows from its camera set: positions ka, kb of the two cameras -> pair -> task -> lane.
    // The unit descriptors go through shared memory (the Z areas are free now) and the record loads are issued eight units at
    // a time (units that do not contain the entry read a zero), so the L2 round trips overlap.
    {
        constexpr int MU = 4;
        const int cu0 = A.warp_unit0[blockIdx.x * nw], cu1 = A.warp_unit0[(blockIdx.x + 1) * nw];
        const int ncu = cu1 - cu0;
        // per unit: mask (2 ints), L, rec -> 4 ints; capacity of the Z area
        int* s_units = reinterpret_cast<int*>(s_Z);
        const int cap = (int)(((size_t)nw * (32 * ZP + PT_RC * 3) * sizeof(double)) / (4 * sizeof(int))) - 1;
        for (int c0 = 0; c0 < max(ncu, 1); c0 += cap) {        // a CTA without units still writes its (zero) partial
            const int nc_here = min(cap, ncu - c0);
            __syncthreads();
            for (int q = threadIdx.x; q < nc_here; q += blockDim.x) {
                const PUnit un = A.units[cu0 + c0 + q];
                s_units[4 * q] = (int)un.mask_lo; s_units[4 * q + 1] = (int)un.mask_hi; s_units[4 * q + 2] = un.L; s_units[4 * q + 3] = un.rec;
            }
            if (threadIdx.x == 0) { s_units[4 * nc_here] = 0; }
            __syncthreads();
            // one thread per (camera block, row) -- the NC entries of a row are contiguous in a task's record -- and one per
            // camera for the rhs; MU units at a time: NC * MU independent loads in flight
            const int nrow = (A.M * (A.M + 1) / 2) * NC;
            for (int task = threadIdx.x; task < nrow + A.M; task += blockDim.x) {
                double sum[NC];
                const bool is_S = task < nrow;
                int ja = 0, jb = 0, r_in = 0;
                size_t t0;       // first entry of this thread in the partial vector
                if (is_S) {
                    int bq = task / NC;
                    const int r = task - bq * NC;
                    t0 = (size_t)bq * NC * NC + (size_t)r * NC;
                    while (bq >= A.M - ja) { bq -= A.M - ja; ++ja; }
                    jb = ja + bq;
                    r_in = r;
                } else {
                    ja = jb = task - nrow;
                    t0 = (size_t)nS + (size_t)ja * NC;
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) sum[c] = c0 == 0 ? 0.0 : partials[(t0 + c) * A.n_cta + blockIdx.x];
                for (int q0 = 0; q0 < nc_here; q0 += MU) {
                    double val[MU][NC];
#pragma unroll
                    for (int qq = 0; qq < MU; ++qq) {
                        const int q = min(q0 + qq, nc_here - 1);
                        const unsigned long long mask = ((unsigned long long)(unsigned)s_units[4 * q + 1] << 32) | (unsigned)s_units[4 * q];
                        const int rec0 = s_units[4 * q + 3];
                        const bool has = q0 + qq < nc_here && ((mask >> ja) & 1ull) && ((mask >> jb) & 1ull);
                        const int ka = __popcll(mask & ((1ull << ja) - 1ull)), kb = __popcll(mask & ((1ull << jb) - 1ull));
                        if (is_S) {
                            // entry (row r_in of camera ka, column c of camera kb) of the unit's Gram matrix -> tile, element
                            const int grow = ka * NC + r_in;
#pragma unroll
                            for (int c = 0; c < NC; ++c) {
                                const int gcol = kb * NC + c;
                                const int lo = min(grow, gcol), hi = max(grow, gcol);       // the Gram matrix is symmetric: upper triangle stored
                                const int ti = lo >> 3, tj = hi >> 3, tile = tj * (tj + 1) / 2 + ti, ps = tile / NTP;
                                const double* src = records + (size_t)(rec0 + ps) * REC + (tile - ps * NTP) * 64 + (lo & 7) * 8 + (hi & 7);
                                val[qq][c] = has ? __ldcg(src) : 0.0;
                            }
                        } else {
                            const double* src = records + (size_t)rec0 * REC + (size_t)NTP * 64 + ka;
#pragma unroll
                            for (int c = 0; c < NC; ++c) val[qq][c] = has ? __ldcg(src + c * 32) : 0.0;
                        }
                    }
#pragma unroll
                    for (int qq = 0; qq < MU; ++qq)
#pragma unroll
                        for (int c = 0; c < NC; ++c) sum[c] += val[qq][c];
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) partials[(t0 + c) * A.n_cta + blockIdx.x] = sum[c];
            }
        }
    }
}

// Sum of the per-CTA Schur partials -> reduced camera system S (ns x ns column-major, symmetric, both triangles) and its
// right-hand side:  S_jj' = [j == j'] (U_j + reg D_j^2) - sum,  rhs_j = -g_j + sum.  One warp per value.
// add_diag: rank 0 only (the all-reduce over ranks then counts U and the damping once).
// Multi-GPU (comm.on): the values go to the rank's exchange slot instead (block-upper layout, nS + ns doubles -- smaller than
// the symmetric S), the last CTA to finish publishes the flags, every CTA waits for the peers' flags and the warps sum
// the R contributions of their values in rank order straight out of peer memory (one remote load per lane) into S: the
// all-reduce of [S | rhs] costs no launch of its own.  The grid is <= one CTA per SM, so all CTAs are resident while they wait.
template <int NC>
__device__ __forceinline__ void reduce_schur_store(int v, double val, int M, double* __restrict__ S)
{
    const int ns = M * NC, nS = NC * NC * (M * (M + 1) / 2);
    if (v >= nS) { S[(size_t)ns * ns + (v - nS)] = val; return; }
    int b = v / (NC * NC);
    const int rs = v - b * NC * NC, r = rs / NC, c = rs - r * NC;
    int j = 0;
    while (b >= M - j) { b -= M - j; ++j; }
    const int jp = j + b;
    S[(size_t)(j * NC + r) + (size_t)(jp * NC + c) * ns] = val;
    if (j != jp) S[(size_t)(jp * NC + c) + (size_t)(j * NC + r) * ns] = val;
}

template <int NC>
__global__ void __launch_bounds__(512)
k_pt_reduce_schur(const double* __restrict__ partials, int n_cta, int M, int n_cam_fix, const double* __restrict__ camsys,
                  const double* __restrict__ dsq_c, double* scal, int add_diag, double* __restrict__ S, CommFused comm,
                  unsigned* counter)
{
    const int lane = threadIdx.x & 31;
    const int ns = M * NC, nS = NC * NC * (M * (M + 1) / 2), total = nS + ns;
    const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = gridDim.x * (blockDim.x >> 5);
    const int parity = (int)(comm.seq & 1ull);
    double* mine = comm.on ? comm.c.data[comm.c.me] + (long long)parity * comm.c.cap : nullptr;
    const double reg = scal[SC_REG];
    for (int v = gw; v < total; v += nwarps) {
        double s = 0.0;
        for (int b = lane; b < n_cta; b += 32) s += partials[(size_t)v * n_cta + b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane != 0) continue;
        double val;
        if (v >= nS) {
            val = (add_diag ? -camsys[(size_t)M * NC * NC + (v - nS)] : 0.0) + s;
        } else {
            int b = v / (NC * NC);
            const int rs = v - b * NC * NC, r = rs / NC, c = rs - r * NC;
            int j = 0;
            while (b >= M - j) { b -= M - j; ++j; }
            val = -s;
            if (b == 0 && add_diag) {
                val += camsys[(size_t)j * NC * NC + r * NC + c];
                if (r == c) val += (j < n_cam_fix) ? 1.0 : reg * dsq_c[(size_t)j * NC + r];
            }
        }
        if (comm.on) mine[v] = val;
        else reduce_schur_store<NC>(v, val, M, S);
    }
    if (!comm.on) return;
    __threadfence_system();
    __shared__ bool last;
    __shared__ int ok;
    __syncthreads();
    if (threadIdx.x == 0) { last = (atomicAdd(counter, 1u) == gridDim.x - 1); ok = 1; }
    __syncthreads();
    const CommView& c = comm.c;
    if (last) {
        __threadfence_system();
        if (threadIdx.x < c.world && threadIdx.x != c.me)
            st_release_sys(c.flag[threadIdx.x] + parity * COMM_MAX_RANKS + c.me, comm.seq);
        if (threadIdx.x == 0) *counter = 0u;
    }
    if (threadIdx.x < c.world && threadIdx.x != c.me) {
        const unsigned long long* f = c.flag[c.me] + parity * COMM_MAX_RANKS + threadIdx.x;
        const long long t0 = clock64();
        while (ld_acquire_sys(f) < comm.seq) {
            if (clock64() - t0 > c.timeout_cycles) { ok = 0; break; }  // a peer is gone: report instead of hanging
        }
    }
    __syncthreads();
    if (!ok) {
        if (threadIdx.x == 0) scal[SC_COMM_FAIL] = 1.0;
        return;
    }
    for (int v = gw; v < total; v += nwarps) {
        double part = 0.0;
        if (lane < c.world) part = ld_volatile_f64(c.data[lane] + (long long)parity * c.cap + v);
        double acc = 0.0;
        for (int r = 0; r < c.world; ++r) acc += __shfl_sync(0xffffffffu, part, r);
        if (lane == 0) reduce_schur_store<NC>(v, acc, M, S);
    }
}

// ------------------------------------------------------------------------------------------------
// K4: back-substitution dp_i = -(V_i + reg D_i^2)^-1 (g_i + W_i^T dc) and the Gram scalars of {t1, delta}
//   sums: g.delta, |D delta|^2, (J t1).(J delta), |J delta|^2, |t1|^2, t1.delta, |delta|^2
// shared: s_cam | s_rpc | s_dc[ns] | s_t1c[ns] | s_stage[nwarps][3][32] | s_red
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC>
__global__ void __launch_bounds__(PT_THREADS_LIGHT, 1)
k_pt_backsub(PatView A, const double* __restrict__ x, const double* __restrict__ camrec, const double* __restrict__ V,
             const double* __restrict__ g, const double* __restrict__ dsq, const double* __restrict__ idsq,
             const double* __restrict__ dsq_c, const double* __restrict__ idsq_c, const double2* __restrict__ osc,
             double* __restrict__ delta, int ns, int count_cameras, double* partials, unsigned* counter, double* scal, int fold_ctl,
             CommFused comm)
{
    extern __shared__ double smem[];
    double* s_cam = smem;
    double* s_rpc = s_cam + A.M * CAMREC_STRIDE;
    double* s_dc = s_rpc + (MODEL == MODEL_RPC ? A.M * RPC_TAB_STRIDE : 0);
    double* s_t1c = s_dc + ns;
    double* s_stage = s_t1c + ns;
    double* s_red = s_stage + (blockDim.x >> 5) * 3 * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double reg = scal[SC_REG];
    load_cameras_shared<MODEL>(A, camrec, s_cam, s_rpc);
    for (int e = threadIdx.x; e < ns; e += blockDim.x) { s_dc[e] = delta[e]; s_t1c[e] = g[e] * idsq_c[e]; }
    __syncthreads();
    double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // gd, dd, c12, c22, t11, t1d, tdd
    if (blockIdx.x == 0 && count_cameras) {
        for (int e = threadIdx.x; e < ns; e += blockDim.x) {
            const double d = s_dc[e], t = s_t1c[e];
            acc[0] += g[e] * d; acc[1] += dsq_c[e] * d * d; acc[4] += t * t; acc[5] += t * d; acc[6] += d * d;
        }
    }
    double* stg = s_stage + warp * 3 * 32;
    const int u0 = A.warp_unit0[blockIdx.x * nw + warp], u1 = A.debug_skip ? u0 : A.warp_unit0[blockIdx.x * nw + warp + 1];
    const long long cyc0 = clock64();
    for (int u = u0; u < u1; ++u) {
        const PUnit un = A.units[u];
        const LaneGeo G = lane_geometry(un, lane);
        const bool cam_free = G.cam >= A.n_cam_fix, pt_free = un.pts_free != 0;
        const double* rec = s_cam + G.cam * CAMREC_STRIDE;
        const double* rpc_j = MODEL == MODEL_RPC ? s_rpc + G.cam * RPC_TAB_STRIDE : nullptr;
        const double* dc = s_dc + G.cam * NC;
        const double* t1c = s_t1c + G.cam * NC;
        for (int tb = 0; tb < un.ntrk; tb += G.T) {
            const int tt = tb + G.t;
            const bool on = G.on && tt < un.ntrk;
            if (G.on && tt + G.T < un.ntrk) {          // next tile
                const size_t in = (size_t)(un.trk0 + tt + G.T), en = (size_t)ns + 3 * in;
                prefetch_l1(osc + (size_t)un.obs0 + (size_t)(tt + G.T) * G.L + G.k);
                prefetch_l1(x + en); prefetch_l1(g + en); prefetch_l1(dsq + en); prefetch_l1(idsq + en); prefetch_l1(V + 6 * in);
            }
            ObsEval<MODEL, NC> e;
            double yc0 = 0.0, yc1 = 0.0;
            size_t e3 = 0;
            if (on) {
                const int i = un.trk0 + tt;
                const size_t a = (size_t)un.obs0 + (size_t)tt * G.L + G.k;
                e3 = (size_t)ns + 3 * (size_t)i;
                eval_scaled<MODEL, NC>(rec, rpc_j, x[e3], x[e3 + 1], x[e3 + 2], osc[a], cam_free, pt_free, e);
#pragma unroll
                for (int q = 0; q < NC; ++q) { yc0 += e.Jc[q] * dc[q]; yc1 += e.Jc[NC + q] * dc[q]; }
                stg[lane] = e.Jp[0] * yc0 + e.Jp[3] * yc1;
                stg[32 + lane] = e.Jp[1] * yc0 + e.Jp[4] * yc1;
                stg[64 + lane] = e.Jp[2] * yc0 + e.Jp[5] * yc1;
            }
            __syncwarp();
            if (on) {
                const int i = un.trk0 + tt;
                double s0 = 0.0, s1 = 0.0, s2 = 0.0;
                const int l0 = G.t * G.L;
                for (int m = 0; m < G.L; ++m) { s0 += stg[l0 + m]; s1 += stg[32 + l0 + m]; s2 += stg[64 + l0 + m]; }
                const double* v = V + 6 * (size_t)i;
                const double gp0 = g[e3], gp1 = g[e3 + 1], gp2 = g[e3 + 2];
                double Gm[6];
                double d0 = 0.0, d1 = 0.0, d2 = 0.0;
                if (pt_free && invert_point_block_d2(v[0], v[1], v[2], v[3], v[4], v[5], dsq[e3], dsq[e3 + 1], dsq[e3 + 2], reg, Gm)) {
                    const double v0 = gp0 + s0, v1 = gp1 + s1, v2 = gp2 + s2;
                    const double t0 = Gm[0] * v0, t1 = Gm[1] * v0 + Gm[2] * v1, t2 = Gm[3] * v0 + Gm[4] * v1 + Gm[5] * v2;
                    d0 = -(Gm[0] * t0 + Gm[1] * t1 + Gm[3] * t2);
                    d1 = -(Gm[2] * t1 + Gm[4] * t2);
                    d2 = -(Gm[5] * t2);
                }
                const double tp0 = gp0 * idsq[e3], tp1 = gp1 * idsq[e3 + 1], tp2 = gp2 * idsq[e3 + 2];
                if (G.k == 0) {
                    delta[e3] = d0; delta[e3 + 1] = d1; delta[e3 + 2] = d2;
                    acc[0] += gp0 * d0 + gp1 * d1 + gp2 * d2;
                    acc[1] += dsq[e3] * d0 * d0 + dsq[e3 + 1] * d1 * d1 + dsq[e3 + 2] * d2 * d2;
                    acc[4] += tp0 * tp0 + tp1 * tp1 + tp2 * tp2;
                    acc[5] += tp0 * d0 + tp1 * d1 + tp2 * d2;
                    acc[6] += d0 * d0 + d1 * d1 + d2 * d2;
                }
                const double jd0 = yc0 + e.Jp[0] * d0 + e.Jp[1] * d1 + e.Jp[2] * d2;
                const double jd1 = yc1 + e.Jp[3] * d0 + e.Jp[4] * d1 + e.Jp[5] * d2;
                double jt0 = e.Jp[0] * tp0 + e.Jp[1] * tp1 + e.Jp[2] * tp2;
                double jt1 = e.Jp[3] * tp0 + e.Jp[4] * tp1 + e.Jp[5] * tp2;
#pragma unroll
                for (int q = 0; q < NC; ++q) { jt0 += e.Jc[q] * t1c[q]; jt1 += e.Jc[NC + q] * t1c[q]; }
                acc[2] = fma(jt1, jd1, fma(jt0, jd0, acc[2]));
                acc[3] = fma(jd1, jd1, fma(jd0, jd0, acc[3]));
            }
            __syncwarp();
        }
    }
    if (A.cycles && lane == 0) A.cycles[blockIdx.x * nw + warp] = clock64() - cyc0;
    const double tot = cta_reduce_sum<7>(acc, s_red);
    __shared__ int slots[7];
    if (threadIdx.x == 0) {
        slots[0] = SC_P_GD; slots[1] = SC_P_DD; slots[2] = SC_P_C12; slots[3] = SC_P_C22; slots[4] = SC_P_T11; slots[5] = SC_P_T1D;
        slots[6] = SC_P_TDD;
    }
    __syncthreads();
    const bool last = grid_sum_last<7>(tot, partials, counter, scal, slots);
    if (last && comm.on) cta_allreduce(comm.c, scal + SC_P_GD, 7, comm.seq, scal);
    if (last && fold_ctl && threadIdx.x == 0) control_tr2d_gram_dev(scal, -1.0);
}

// ------------------------------------------------------------------------------------------------
// boundary permutations: the caller's order <-> the internal (pattern-major) order
// ------------------------------------------------------------------------------------------------
// x_int = [cameras | points of internal track t = points of caller's track new2old[t]]
__global__ void k_pt_points_in(const double* __restrict__ x_ext, const int* __restrict__ new2old, long long N, int ns,
                               double* __restrict__ x_int)
{
    const long long n3 = 3 * N;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ns + n3; q += (long long)gridDim.x * blockDim.x) {
        if (q < ns) { x_int[q] = x_ext[q]; continue; }
        const long long e = q - ns, t = e / 3;
        x_int[q] = x_ext[ns + 3 * (long long)new2old[t] + (e - 3 * t)];
    }
}
__global__ void k_pt_points_out(const double* __restrict__ x_int, const int* __restrict__ new2old, long long N, int ns,
                                double* __restrict__ x_ext)
{
    const long long n3 = 3 * N;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ns + n3; q += (long long)gridDim.x * blockDim.x) {
        if (q < ns) { x_ext[q] = x_int[q]; continue; }
        const long long e = q - ns, t = e / 3;
        x_ext[ns + 3 * (long long)new2old[t] + (e - 3 * t)] = x_int[q];
    }
}
// per-observation records of `width` doubles: out_ext[new2old[a]] = in_int[a]
__global__ void k_pt_obs_out(const double* __restrict__ in_int, const int* __restrict__ new2old, long long K, int width,
                             double* __restrict__ out_ext)
{
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < K * width; q += (long long)gridDim.x * blockDim.x) {
        const long long a = q / width;
        out_ext[(long long)new2old[a] * width + (q - a * width)] = in_int[q];
    }
}
__global__ void k_pt_obs_in(const double* __restrict__ in_ext, const int* __restrict__ new2old, long long K, int width,
                            double* __restrict__ out_int)
{
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < K * width; q += (long long)gridDim.x * blockDim.x) {
        const long long a = q / width;
        out_int[q] = in_ext[(long long)new2old[a] * width + (q - a * width)];
    }
}
// internal per-observation index arrays from the track permutation (one thread per internal track)
__global__ void k_pt_build_obs(const int* __restrict__ trk_new2old, const int* __restrict__ track_ptr_old,
                               const int* __restrict__ track_ptr_new, const int* __restrict__ cam_ext, int N,
                               int* __restrict__ obs_new2old, int* __restrict__ cam_int, int* __restrict__ pts_int)
{
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < N; t += gridDim.x * blockDim.x) {
        const int o = trk_new2old[t], a0 = track_ptr_old[o], L = track_ptr_old[o + 1] - a0, b0 = track_ptr_new[t];
        for (int k = 0; k < L; ++k) { obs_new2old[b0 + k] = a0 + k; cam_int[b0 + k] = cam_ext[a0 + k]; pts_int[b0 + k] = t; }
    }
}
__global__ void k_pt_fill(double* __restrict__ dst, double v, long long n)
{
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) dst[q] = v;
}

}  // namespace sba
