// Device kernels of the bundle-adjustment hot path (sm_100a).  Included by sba_ba.cu only.
//
// Data layout in HBM (all FP64 values, int32 indices):
//   track-major (the reference's observation order, bundle_adjust/ba_params.py:138-149):
//       cam_ind[K], pts_ind[K], pts2d[K] (double2), w[K], track_ptr[N+1]
//       tile_obs[T+1]: "warp tiles" = runs of whole tracks holding <= 32 observations (one observation per
//       lane, point blocks reduced inside the warp through shared memory); a track longer than 32
//       observations forms a tile of its own and is looped over by its warp
//   camera-major copy (static, built once): cm_obs[K] (observation id), cm_pts[K], cm_pts2d[K], cm_w[K],
//       cam_ptr[M+1]; chunk table = (camera, [beg,end)) work items of <= CHUNK observations
//   obs_of[M][N]: observation id of (camera, track) or -1
//   variables x[n] = [camera blocks M*nc | points 3N]  (bundle_adjust/ba_params.py:151-173)
//   camrec[M][16]: per-camera prepared record (cos/sin of the Euler angles + parameters)
//   V[N][6], F[N][6] (inverse Cholesky factor of the damped point block), q[N][3], Z[K][nc][3]
//   camsys = [U (M, nc, nc) | g_c (M*nc)],  S = [S (ns x ns, column-major) | rhs (ns)]
// J itself is never stored: every pass recomputes the per-observation Jacobian in registers.
#pragma once
#include "sba_internal.cuh"
#include "sba_tr2d.h"

namespace sba {

constexpr int TPB = 128;          // threads per block of the reduction kernels
constexpr int CHUNK = 1024;       // observations per camera-major work item
constexpr int WPB = TPB / 32;     // warps (= tiles) per block of the tile kernels

// ------------------------------------------------------------------------------------------------
// reductions
// ------------------------------------------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void warp_reduce_sum(double (&v)[NV])
{
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        v[k] = x;
    }
}

// Sum of v[k] over the block; the result for value k is returned in thread k (k < NV <= NT).
// sm must hold NV * (NT / 32) doubles.
template <int NV, int NT>
__device__ __forceinline__ double block_reduce_sum(double (&v)[NV], double* sm)
{
    static_assert(NV <= NT, "more values than threads");
    warp_reduce_sum<NV>(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) sm[warp * NV + k] = v[k];
    }
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x < NV) {
#pragma unroll
        for (int wq = 0; wq < NT / 32; ++wq) s += sm[wq * NV + threadIdx.x];
    }
    __syncthreads();
    return s;
}

// Grid-wide deterministic sum: every block stores its NV partial sums, the last block to arrive adds
// them up in a fixed order and writes out[k].  counter must be zero on entry and is reset on exit.
template <int NV, int NT>
__device__ __forceinline__ void grid_sum_finalize(double block_total, double* partials, unsigned* counter,
                                                  double* out, const int* out_slot, double* sm)
{
    __shared__ bool is_last;
    if (threadIdx.x < NV) partials[(size_t)blockIdx.x * NV + threadIdx.x] = block_total;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(counter, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // every thread of the last block adds a fixed, strided subset of the per-block partials; the block
    // reduction that follows has a fixed shape too, so the result does not depend on which block is last
    double acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += NT) {
#pragma unroll
        for (int k = 0; k < NV; ++k) acc[k] += __ldcg(partials + (size_t)b * NV + k);
    }
    const double tot = block_reduce_sum<NV, NT>(acc, sm);
    if (threadIdx.x < NV) out[out_slot[threadIdx.x]] = tot;
    if (threadIdx.x == 0) *counter = 0u;
}

struct Slots {
    int s[8];
};

// ------------------------------------------------------------------------------------------------
// per-camera preparation
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void write_camrec(const double (&v)[MAX_CAM_PARAMS], double* __restrict__ r, int model)
{
    build_camrec(v, model, r);
}

// n_common > 0 (COMMON_K, ba_params.py:167-171, :254-255): the last n_common of the nc variables are shared by all
// cameras and live in camera 0's slots; the same slots of the other cameras are unused (zero, never stepped)
__global__ void k_prepare_cameras(const double* __restrict__ x, const double* __restrict__ cam_static,
                                  double* __restrict__ camrec, int M, int P, int nc, int n_cam_fix, int n_common, int model)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    double v[MAX_CAM_PARAMS];
#pragma unroll
    for (int s = 0; s < MAX_CAM_PARAMS; ++s) {
        double val = 0.0;
        if (s < P) {
            const int src = (s >= nc - n_common) ? 0 : j;
            val = (s < nc && j >= n_cam_fix) ? x[(size_t)src * nc + s] : cam_static[(size_t)j * P + s];
        }
        v[s] = val;
    }
    write_camrec(v, camrec + (size_t)j * CAMREC_STRIDE, model);
}

// ------------------------------------------------------------------------------------------------
// observation evaluation shared by all passes: weighted, robust-rescaled residual and Jacobian rows
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC>
struct ObsEval {
    double f0, f1, cost;
    double Jc[2 * (NC > 0 ? NC : 1)];
    double Jp[6];
};

// robust rescale of one observation's residual pair and Jacobian rows (weights folded in)
template <int MODEL, int NC, bool WITH_JP>
__device__ __forceinline__ void finish_obs(double u, double v, double ox, double oy, double w, int loss, double f_scale,
                                           bool cam_free, bool pt_free, ObsEval<MODEL, NC>& e)
{
    double f0 = w * (u - ox), f1 = w * (v - oy), c0, c1;
    const double s0 = w * loss_rescale(loss, f_scale, f0, c0);
    const double s1 = w * loss_rescale(loss, f_scale, f1, c1);
    e.f0 = f0; e.f1 = f1; e.cost = c0 + c1;
    const double a0 = cam_free ? s0 : 0.0, a1 = cam_free ? s1 : 0.0;
#pragma unroll
    for (int k = 0; k < NC; ++k) { e.Jc[k] *= a0; e.Jc[NC + k] *= a1; }
    if (WITH_JP) {
        const double b0 = pt_free ? s0 : 0.0, b1 = pt_free ? s1 : 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) { e.Jp[k] *= b0; e.Jp[3 + k] *= b1; }
    }
}

// camera block (+ point block) of one observation
template <int MODEL, int NC, bool WITH_JP>
__device__ __forceinline__ void eval_obs(const double* __restrict__ rec, const double* __restrict__ rpc_j, double X,
                                         double Y, double Z, double ox, double oy, double w, int loss, double f_scale,
                                         bool cam_free, bool pt_free, ObsEval<MODEL, NC>& e)
{
    double u, v;
    full_side<MODEL, NC, WITH_JP>(rec, rpc_j, X, Y, Z, u, v, e.Jc, e.Jp);
    finish_obs<MODEL, NC, WITH_JP>(u, v, ox, oy, w, loss, f_scale, cam_free, pt_free, e);
}

// point block only
template <int MODEL>
__device__ __forceinline__ void eval_obs_point(const double* __restrict__ rec, const double* __restrict__ rpc_j,
                                               double X, double Y, double Z, double ox, double oy, double w, int loss,
                                               double f_scale, bool pt_free, ObsEval<MODEL, 0>& e)
{
    double u, v;
    point_side<MODEL>(rec, rpc_j, X, Y, Z, u, v, e.Jp);
    finish_obs<MODEL, 0, true>(u, v, ox, oy, w, loss, f_scale, false, pt_free, e);
}

struct ObsArrays {
    const int* cam_ind;
    const int* pts_ind;
    const double2* pts2d;
    const double* w;
    const int* track_ptr;
    const int* tile_obs;     // T+1 observation offsets of the warp tiles
    int n_tiles;
};

// tile of this warp: first observation and number of observations (0 when the warp has no tile)
__device__ __forceinline__ void warp_tile(const ObsArrays& o, int& ob, int& nobs)
{
    const int tile = blockIdx.x * WPB + (threadIdx.x >> 5);
    ob = 0; nobs = 0;
    if (tile < o.n_tiles) { ob = o.tile_obs[tile]; nobs = o.tile_obs[tile + 1] - ob; }
}

template <int NV>
__device__ __forceinline__ void warp_allreduce_sum(double (&v)[NV])
{
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        v[k] = x;
    }
}

// ------------------------------------------------------------------------------------------------
// G1: residual `fun` (+ robust cost)
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(256)
k_residual(ObsArrays o, const double* __restrict__ xp, const double* __restrict__ camrec,
           const double* __restrict__ rpc_tab, long long K, int loss, double f_scale, int rpc_f32,
           double2* __restrict__ r_out, double* partials, unsigned* counter, double* scal, int slot)
{
    __shared__ double sm[1 * (256 / 32)];
    double acc[1] = {0.0};
    // two observations per trip, all their loads requested before either is used: at ~1.6 observations per resident thread
    // the kernel is a chain of dependent memory round trips (index -> point -> result), not a bandwidth problem
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long a0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; a0 < K; a0 += 2 * stride) {
        const long long a1 = a0 + stride;
        const bool two = a1 < K;
        const long long b = two ? a1 : a0;
        const int j0 = o.cam_ind[a0], i0 = o.pts_ind[a0], j1 = o.cam_ind[b], i1 = o.pts_ind[b];
        const double2 ob0 = o.pts2d[a0], ob1 = o.pts2d[b];
        const double w0 = o.w[a0], w1 = o.w[b];
        const double X0 = xp[3 * (size_t)i0], Y0 = xp[3 * (size_t)i0 + 1], Z0 = xp[3 * (size_t)i0 + 2];
        const double X1 = xp[3 * (size_t)i1], Y1 = xp[3 * (size_t)i1 + 1], Z1 = xp[3 * (size_t)i1 + 2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h == 1 && !two) break;
            const long long a = h ? a1 : a0;
            const int j = h ? j1 : j0;
            const CamRec c = load_camrec(camrec + (size_t)j * CAMREC_STRIDE);
            double u, v;
            project<MODEL>(c, MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, h ? X1 : X0, h ? Y1 : Y0,
                           h ? Z1 : Z0, u, v);
            if (MODEL == MODEL_RPC && rpc_f32) { u = (double)(float)u; v = (double)(float)v; }
            const double2 ob = h ? ob1 : ob0;
            const double w = h ? w1 : w0;
            const double f0 = w * (u - ob.x), f1 = w * (v - ob.y);
            if (r_out) r_out[a] = make_double2(f0, f1);
            acc[0] += loss_cost(loss, f0, f_scale) + loss_cost(loss, f1, f_scale);
        }
    }
    const double tot = block_reduce_sum<1, 256>(acc, sm);
    __shared__ int slots[1];
    if (threadIdx.x == 0) slots[0] = slot;
    __syncthreads();
    grid_sum_finalize<1, 256>(tot, partials, counter, scal, slots, sm);
}

// un-weighted reprojection error of every observation, err_k = |(r_2k, r_2k+1) / w_k|_2  (ba_core.py:335-349);
// individually rounded operations in numpy's order, so the values equal the host expression bit for bit
__global__ void k_reproj_error(const double2* __restrict__ r, const double* __restrict__ w, long long K,
                               double* __restrict__ err)
{
    for (long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x; a < K; a += (long long)gridDim.x * blockDim.x) {
        const double2 f = r[a];
        const double wa = w[a];
        const double q0 = __ddiv_rn(f.x, wa), q1 = __ddiv_rn(f.y, wa);
        err[a] = __dsqrt_rn(__dadd_rn(__dmul_rn(q0, q0), __dmul_rn(q1, q1)));
    }
}

// ------------------------------------------------------------------------------------------------
// G2a: point side of the assembly -- V_i = sum Jp^T Jp, g_p = sum Jp^T f.
// One observation per lane (coalesced index / observation loads, no divergence in the Jacobian); the 9 sums
// of each track are formed by the lane of its first observation from the warp's shared-memory slice.
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(TPB, MODEL == MODEL_RPC ? 3 : 6)
k_assemble_points(ObsArrays o, const double* __restrict__ xp, const double* __restrict__ camrec,
                  const double* __restrict__ rpc_tab, int n_pts_fix, int loss, double f_scale,
                  double* __restrict__ V, double* __restrict__ gp_out, double* partials, unsigned* counter,
                  double* scal)
{
    __shared__ double sv[WPB][9][32];
    __shared__ int strk[WPB][32];
    __shared__ int sseg[WPB][32];
    __shared__ double sm[1 * (TPB / 32)];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ob, nobs;
    warp_tile(o, ob, nobs);
    double acc[1] = {0.0};
    if (nobs <= 32) {
        double vals[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) vals[k] = 0.0;
        int i = -1, a = -1;
        if (lane < nobs) {
            a = ob + lane;
            i = o.pts_ind[a];
            const int j = o.cam_ind[a];
            const double2 ob2 = o.pts2d[a];
            ObsEval<MODEL, 0> e;
            eval_obs_point<MODEL>(camrec + (size_t)j * CAMREC_STRIDE,
                                  MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, xp[3 * (size_t)i],
                                  xp[3 * (size_t)i + 1], xp[3 * (size_t)i + 2], ob2.x, ob2.y, o.w[a], loss, f_scale,
                                  i >= n_pts_fix, e);
            acc[0] = e.cost;
            vals[0] = e.Jp[0] * e.Jp[0] + e.Jp[3] * e.Jp[3];
            vals[1] = e.Jp[0] * e.Jp[1] + e.Jp[3] * e.Jp[4];
            vals[2] = e.Jp[0] * e.Jp[2] + e.Jp[3] * e.Jp[5];
            vals[3] = e.Jp[1] * e.Jp[1] + e.Jp[4] * e.Jp[4];
            vals[4] = e.Jp[1] * e.Jp[2] + e.Jp[4] * e.Jp[5];
            vals[5] = e.Jp[2] * e.Jp[2] + e.Jp[5] * e.Jp[5];
            vals[6] = e.Jp[0] * e.f0 + e.Jp[3] * e.f1;
            vals[7] = e.Jp[1] * e.f0 + e.Jp[4] * e.f1;
            vals[8] = e.Jp[2] * e.f0 + e.Jp[5] * e.f1;
        }
#pragma unroll
        for (int k = 0; k < 9; ++k) sv[warp][k][lane] = vals[k];
        // tracks of the tile: the lane holding a track's first observation publishes (track, first lane, length)
        const bool head = lane < nobs && a == o.track_ptr[i];
        const unsigned heads = __ballot_sync(0xffffffffu, head);
        const int ntr = __popc(heads);
        if (head) {
            const int rank = __popc(heads & ((1u << lane) - 1u));
            strk[warp][rank] = i;
            sseg[warp][rank] = lane | ((o.track_ptr[i + 1] - a) << 8);
        }
        __syncwarp();
        // one lane per (track, value): 9 * ntr short sums instead of 9 long ones on the head lanes
        for (int s = lane; s < 9 * ntr; s += 32) {
            const int tr = s / 9, k = s - 9 * tr;
            const int seg = sseg[warp][tr], l0 = seg & 0xff, l1 = l0 + (seg >> 8);
            double t = 0.0;
            for (int m = l0; m < l1; ++m) t += sv[warp][k][m];
            const int it = strk[warp][tr];
            if (k < 6) V[6 * (size_t)it + k] = t;
            else gp_out[3 * (size_t)it + (k - 6)] = t;
        }
    } else {
        // a single long track: the warp strides over its observations
        const int i = o.pts_ind[ob];
        const double X = xp[3 * (size_t)i], Y = xp[3 * (size_t)i + 1], Z = xp[3 * (size_t)i + 2];
        double vals[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) vals[k] = 0.0;
        for (int a = ob + lane; a < ob + nobs; a += 32) {
            const int j = o.cam_ind[a];
            const double2 ob2 = o.pts2d[a];
            ObsEval<MODEL, 0> e;
            eval_obs_point<MODEL>(camrec + (size_t)j * CAMREC_STRIDE,
                                  MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, X, Y, Z, ob2.x, ob2.y,
                                  o.w[a], loss, f_scale, i >= n_pts_fix, e);
            acc[0] += e.cost;
            vals[0] += e.Jp[0] * e.Jp[0] + e.Jp[3] * e.Jp[3];
            vals[1] += e.Jp[0] * e.Jp[1] + e.Jp[3] * e.Jp[4];
            vals[2] += e.Jp[0] * e.Jp[2] + e.Jp[3] * e.Jp[5];
            vals[3] += e.Jp[1] * e.Jp[1] + e.Jp[4] * e.Jp[4];
            vals[4] += e.Jp[1] * e.Jp[2] + e.Jp[4] * e.Jp[5];
            vals[5] += e.Jp[2] * e.Jp[2] + e.Jp[5] * e.Jp[5];
            vals[6] += e.Jp[0] * e.f0 + e.Jp[3] * e.f1;
            vals[7] += e.Jp[1] * e.f0 + e.Jp[4] * e.f1;
            vals[8] += e.Jp[2] * e.f0 + e.Jp[5] * e.f1;
        }
        warp_allreduce_sum<9>(vals);
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) V[6 * (size_t)i + k] = vals[k];
#pragma unroll
            for (int k = 0; k < 3; ++k) gp_out[3 * (size_t)i + k] = vals[6 + k];
        }
    }
    const double tot = block_reduce_sum<1, TPB>(acc, sm);
    __shared__ int slots[1];
    if (threadIdx.x == 0) slots[0] = SC_COST;
    __syncthreads();
    grid_sum_finalize<1, TPB>(tot, partials, counter, scal, slots, sm);
}

// ------------------------------------------------------------------------------------------------
// G2b: camera side of the assembly -- U_j = sum Jc^T Jc, g_c = sum Jc^T f.
// Camera-major: every block works on one chunk of ONE camera, so the camera record is block-uniform,
// the accumulators stay in registers and no atomics are needed; partial sums per chunk are combined
// in a fixed order by k_reduce_cameras.
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC>
__global__ void __launch_bounds__(TPB)
k_assemble_cameras(const int* __restrict__ chunk_cam, const int* __restrict__ chunk_beg,
                   const int* __restrict__ chunk_end, const int* __restrict__ cm_pts,
                   const double2* __restrict__ cm_pts2d, const double* __restrict__ cm_w,
                   const double* __restrict__ xp, const double* __restrict__ camrec,
                   const double* __restrict__ rpc_tab, int n_cam_fix, int loss, double f_scale,
                   double* __restrict__ cam_partials)
{
    constexpr int NU = NC * (NC + 1) / 2, NV = NU + NC;
    __shared__ double sm[NV * (TPB / 32)];
    __shared__ double srec[CAMREC_STRIDE];
    const int ch = blockIdx.x, j = chunk_cam[ch];
    if (threadIdx.x < CAMREC_STRIDE) srec[threadIdx.x] = camrec[(size_t)j * CAMREC_STRIDE + threadIdx.x];
    __syncthreads();
    double acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.0;
    if (j >= n_cam_fix) {
        const double* rpc_j = MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr;
        for (int t = chunk_beg[ch] + threadIdx.x; t < chunk_end[ch]; t += TPB) {
            const int i = cm_pts[t];
            const double X = xp[3 * (size_t)i], Y = xp[3 * (size_t)i + 1], Z = xp[3 * (size_t)i + 2];
            const double2 ob = cm_pts2d[t];
            ObsEval<MODEL, NC> e;
            eval_obs<MODEL, NC, false>(srec, rpc_j, X, Y, Z, ob.x, ob.y, cm_w[t], loss, f_scale, true, false, e);
            int k = 0;
#pragma unroll
            for (int r = 0; r < NC; ++r) {
#pragma unroll
                for (int c = 0; c <= r; ++c) {
                    acc[k] += e.Jc[r] * e.Jc[c] + e.Jc[NC + r] * e.Jc[NC + c];
                    ++k;
                }
            }
#pragma unroll
            for (int r = 0; r < NC; ++r) acc[NU + r] += e.Jc[r] * e.f0 + e.Jc[NC + r] * e.f1;
        }
    }
    const double tot = block_reduce_sum<NV, TPB>(acc, sm);
    if (threadIdx.x < NV) cam_partials[(size_t)ch * NV + threadIdx.x] = tot;
}

// one block per camera: sum of its chunks -> camsys_local = [U (M,nc,nc) | g_c (M*nc)].
// One warp per value, lanes stride over the chunks, fixed-shape shuffle tree -> deterministic.
template <int NC>
__global__ void __launch_bounds__(128)
k_reduce_cameras(const double* __restrict__ cam_partials, const int* __restrict__ first_chunk, int M,
                 double* __restrict__ camsys)
{
    constexpr int NU = NC * (NC + 1) / 2, NV = NU + NC;
    const int j = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = first_chunk[j], c1 = first_chunk[j + 1];
    for (int k = warp; k < NV; k += 4) {
        double s = 0.0;
        for (int ch = c0 + lane; ch < c1; ch += 32) s += cam_partials[(size_t)ch * NV + k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane != 0) continue;
        if (k < NU) {
            int r = 0;
            while ((r + 1) * (r + 2) / 2 <= k) ++r;
            const int c = k - r * (r + 1) / 2;
            camsys[(size_t)j * NC * NC + r * NC + c] = s;
            camsys[(size_t)j * NC * NC + c * NC + r] = s;
        } else {
            camsys[(size_t)M * NC * NC + (size_t)j * NC + (k - NU)] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// x_scale='jac' update + first vector of the 2-D subspace + norms
//   sinv = max-so-far column norm of J (zero columns -> 1 on the first call)   scipy common.py:598-610
//   t1   = g / sinv^2   (= d * g_h, the scaled steepest-descent direction mapped back to x space)
// sums: |g_h|^2, |x sinv|^2, |x|^2 ; max |g|
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_scale_dots(const double* __restrict__ camsys, const double* __restrict__ V, const double* __restrict__ x,
             double* __restrict__ g, double* __restrict__ sinv, double* __restrict__ t1, long long n, int ns, int nc,
             int M, int n_common, int first, int count_cameras, int rank, double* partials, unsigned* counter, double* scal)
{
    __shared__ double sm[4 * (256 / 32)];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};   // gg, xs, xx, gmax
    double gmax = 0.0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        double diag, gv;
        if (idx < ns) {
            const int j = (int)idx / nc, s = (int)idx % nc;
            diag = camsys[(size_t)j * nc * nc + s * nc + s];
            gv = camsys[(size_t)M * nc * nc + idx];
            if (s >= nc - n_common) {        // shared column: its squared norm and gradient are the sums over the cameras
                if (j == 0) {
                    for (int jj = 1; jj < M; ++jj) {
                        diag += camsys[(size_t)jj * nc * nc + s * nc + s];
                        gv += camsys[(size_t)M * nc * nc + (size_t)jj * nc + s];
                    }
                } else {
                    diag = 0.0; gv = 0.0;
                }
            }
            g[idx] = gv;
        } else {
            const long long e = idx - ns;
            const long long i = e / 3;
            const int k = (int)(e - 3 * i);
            diag = V[6 * i + (k == 0 ? 0 : (k == 1 ? 3 : 5))];
            gv = g[idx];
        }
        const double nrm = sqrt(diag);
        double si;
        if (first) si = (nrm == 0.0) ? 1.0 : nrm;
        else si = fmax(sinv[idx], nrm);
        sinv[idx] = si;
        const double xv = x[idx];
        t1[idx] = gv / (si * si);
        gmax = fmax(gmax, fabs(gv));
        if (idx >= ns || count_cameras) {
            const double gh = gv / si, xsv = xv * si;
            acc[0] += gh * gh;
            acc[1] += xsv * xsv;
            acc[2] += xv * xv;
        }
    }
    // block max
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_down_sync(0xffffffffu, gmax, o));
    __shared__ double smax[256 / 32];
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = gmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = 0.0;
        for (int k = 0; k < 256 / 32; ++k) m = fmax(m, smax[k]);
        // non-negative doubles order like their bit patterns
        atomicMax((unsigned long long*)(scal + SC_GMAX_SLOTS + rank), (unsigned long long)__double_as_longlong(m));
    }
    acc[3] = 0.0;
    const double tot = block_reduce_sum<4, 256>(acc, sm);
    __shared__ int slots[4];
    if (threadIdx.x == 0) { slots[0] = SC_GG; slots[1] = SC_XS; slots[2] = SC_XX; slots[3] = SC_SCRATCH; }
    __syncthreads();
    grid_sum_finalize<4, 256>(tot, partials, counter, scal, slots, sm);
}

// ------------------------------------------------------------------------------------------------
// J * [v1 v2] over all observations; sums |Jv1|^2 (, Jv1.Jv2, |Jv2|^2)
// ------------------------------------------------------------------------------------------------
template <int MODEL, int NC, int NVEC>
__global__ void __launch_bounds__(TPB, (MODEL == MODEL_RPC || NC > 6) ? 3 : 6)
k_jvp(ObsArrays o, const double* __restrict__ xp, const double* __restrict__ camrec,
      const double* __restrict__ rpc_tab, long long K, int ns, int n_cam_fix, int n_pts_fix, int loss, double f_scale,
      const double* __restrict__ v1, const double* __restrict__ v2, const double* __restrict__ v1c,
      const double* __restrict__ v2c, double* partials, unsigned* counter, double* scal, Slots out)
{
    __shared__ double sm[3 * (TPB / 32)];
    double acc[3] = {0.0, 0.0, 0.0};
    for (long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x; a < K; a += (long long)gridDim.x * blockDim.x) {
        const int j = o.cam_ind[a], i = o.pts_ind[a];
        const double X = xp[3 * (size_t)i], Y = xp[3 * (size_t)i + 1], Z = xp[3 * (size_t)i + 2];
        const double2 ob = o.pts2d[a];
        ObsEval<MODEL, NC> e;
        eval_obs<MODEL, NC, true>(camrec + (size_t)j * CAMREC_STRIDE,
                                  MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, X, Y, Z, ob.x, ob.y,
                                  o.w[a], loss, f_scale, j >= n_cam_fix, i >= n_pts_fix, e);
        double y0 = 0.0, y1 = 0.0, z0 = 0.0, z1 = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            const double a1 = v1c[(size_t)j * NC + k];        // camera part (expanded copy when variables are shared)
            y0 += e.Jc[k] * a1; y1 += e.Jc[NC + k] * a1;
            if (NVEC == 2) { const double a2 = v2c[(size_t)j * NC + k]; z0 += e.Jc[k] * a2; z1 += e.Jc[NC + k] * a2; }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double a1 = v1[ns + 3 * (size_t)i + k];
            y0 += e.Jp[k] * a1; y1 += e.Jp[3 + k] * a1;
            if (NVEC == 2) { const double a2 = v2[ns + 3 * (size_t)i + k]; z0 += e.Jp[k] * a2; z1 += e.Jp[3 + k] * a2; }
        }
        acc[0] += y0 * y0 + y1 * y1;
        if (NVEC == 2) { acc[1] += y0 * z0 + y1 * z1; acc[2] += z0 * z0 + z1 * z1; }
    }
    const double tot = block_reduce_sum<3, TPB>(acc, sm);
    __shared__ int slots[3];
    if (threadIdx.x < 3) slots[threadIdx.x] = out.s[threadIdx.x];
    __syncthreads();
    grid_sum_finalize<3, TPB>(tot, partials, counter, scal, slots, sm);
}

// ------------------------------------------------------------------------------------------------
// G3a: point elimination prep -- damped 3x3 block -> inverse Cholesky factor G (lower, 6 values),
//      q = G g_p, and per observation Z = (Jc^T Jp) G^T  (nc x 3).
// Warp tiles: the lane of a track's first observation inverts its block and publishes G through shared
// memory; every lane then builds its observation's Z, which leaves the warp as one contiguous, coalesced
// span (observations of a tile are adjacent in Z) staged through shared memory.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool invert_point_block(const double* __restrict__ v, double s0, double s1, double s2,
                                                   double reg, double G[6])
{
    const double a00 = v[0] + reg * s0 * s0, a10 = v[1], a20 = v[2];
    const double a11 = v[3] + reg * s1 * s1, a21 = v[4], a22 = v[5] + reg * s2 * s2;
    bool ok = a00 > 0.0;
    const double c00 = sqrt(a00), c10 = a10 / c00, c20 = a20 / c00;
    const double d11 = a11 - c10 * c10;
    ok = ok && d11 > 0.0;
    const double c11 = sqrt(d11), c21 = (a21 - c20 * c10) / c11;
    const double d22 = a22 - c20 * c20 - c21 * c21;
    ok = ok && d22 > 0.0;
    const double c22 = sqrt(d22);
    if (!ok) {
#pragma unroll
        for (int k = 0; k < 6; ++k) G[k] = 0.0;
        return false;
    }
    G[0] = 1.0 / c00; G[2] = 1.0 / c11; G[5] = 1.0 / c22;     // g00 g10 g11 g20 g21 g22
    G[1] = -c10 * G[0] * G[2];
    G[4] = -c21 * G[2] * G[5];
    G[3] = -(c20 * G[0] + c21 * G[1]) * G[5];
    return true;
}

// G, q of track i (frozen or degenerate points get G = 0, i.e. no step and no coupling)
__device__ __forceinline__ void point_factor(int i, int ns, int n_pts_fix, double reg, const double* __restrict__ V,
                                             const double* __restrict__ g, const double* __restrict__ sinv,
                                             double* __restrict__ F, double* __restrict__ q, double* scal, double G[6])
{
    double qq[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < 6; ++k) G[k] = 0.0;
    if (i >= n_pts_fix) {
        const size_t e = ns + 3 * (size_t)i;
        if (invert_point_block(V + 6 * (size_t)i, sinv[e], sinv[e + 1], sinv[e + 2], reg, G)) {
            const double g0 = g[e], g1 = g[e + 1], g2 = g[e + 2];
            qq[0] = G[0] * g0;
            qq[1] = G[1] * g0 + G[2] * g1;
            qq[2] = G[3] * g0 + G[4] * g1 + G[5] * g2;
        } else {
            atomicAdd(scal + SC_BAD_POINTS, 1.0);
        }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) F[6 * (size_t)i + k] = G[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) q[3 * (size_t)i + k] = qq[k];
}

template <int MODEL, int NC>
__device__ __forceinline__ void obs_Z(const ObsEval<MODEL, NC>& e, const double G[6], double* __restrict__ z)
{
#pragma unroll
    for (int r = 0; r < NC; ++r) {
        const double w0 = e.Jc[r] * e.Jp[0] + e.Jc[NC + r] * e.Jp[3];
        const double w1 = e.Jc[r] * e.Jp[1] + e.Jc[NC + r] * e.Jp[4];
        const double w2 = e.Jc[r] * e.Jp[2] + e.Jc[NC + r] * e.Jp[5];
        z[3 * r + 0] = w0 * G[0];
        z[3 * r + 1] = w0 * G[1] + w1 * G[2];
        z[3 * r + 2] = w0 * G[3] + w1 * G[4] + w2 * G[5];
    }
}

template <int MODEL, int NC>
__global__ void __launch_bounds__(TPB, (MODEL == MODEL_RPC || NC > 6) ? 3 : 6)
k_point_prep(ObsArrays o, const double* __restrict__ xp, const double* __restrict__ camrec,
             const double* __restrict__ rpc_tab, int ns, int n_cam_fix, int n_pts_fix, int loss,
             double f_scale, const double* __restrict__ V, const double* __restrict__ g,
             const double* __restrict__ sinv, double* __restrict__ F, double* __restrict__ q, double* __restrict__ Zout,
             double* scal)
{
    constexpr int ZS = NC * 3, ZP = ZS + 1;      // padded lane stride (odd): conflict-free 64-bit accesses
    const double reg = scal[SC_REG];
    __shared__ double sG[WPB][6][32];
    __shared__ double sZ[WPB][32 * ZP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ob, nobs;
    warp_tile(o, ob, nobs);
    if (nobs == 0) return;
    if (nobs <= 32) {
        int i = -1, a = -1, beg = 0;
        if (lane < nobs) {
            a = ob + lane;
            i = o.pts_ind[a];
            beg = o.track_ptr[i];
            if (a == beg) {
                double G[6];
                point_factor(i, ns, n_pts_fix, reg, V, g, sinv, F, q, scal, G);
#pragma unroll
                for (int k = 0; k < 6; ++k) sG[warp][k][lane] = G[k];
            }
        }
        __syncwarp();
        if (lane < nobs) {
            double G[6];
            const int hl = beg - ob;
#pragma unroll
            for (int k = 0; k < 6; ++k) G[k] = sG[warp][k][hl];
            const int j = o.cam_ind[a];
            const double2 ob2 = o.pts2d[a];
            ObsEval<MODEL, NC> e;
            eval_obs<MODEL, NC, true>(camrec + (size_t)j * CAMREC_STRIDE,
                                      MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr,
                                      xp[3 * (size_t)i], xp[3 * (size_t)i + 1], xp[3 * (size_t)i + 2], ob2.x, ob2.y, o.w[a],
                                      loss, f_scale, j >= n_cam_fix, i >= n_pts_fix, e);
            obs_Z<MODEL, NC>(e, G, &sZ[warp][lane * ZP]);
        }
        __syncwarp();
        double* dst = Zout + (size_t)ob * ZS;
        for (int t = lane; t < nobs * ZS; t += 32) dst[t] = sZ[warp][(t / ZS) * ZP + (t % ZS)];
    } else {
        const int i = o.pts_ind[ob];
        double G[6];
        if (lane == 0) point_factor(i, ns, n_pts_fix, reg, V, g, sinv, F, q, scal, G);
#pragma unroll
        for (int k = 0; k < 6; ++k) G[k] = __shfl_sync(0xffffffffu, G[k], 0);
        const double X = xp[3 * (size_t)i], Y = xp[3 * (size_t)i + 1], Z = xp[3 * (size_t)i + 2];
        for (int a = ob + lane; a < ob + nobs; a += 32) {
            const int j = o.cam_ind[a];
            const double2 ob2 = o.pts2d[a];
            ObsEval<MODEL, NC> e;
            eval_obs<MODEL, NC, true>(camrec + (size_t)j * CAMREC_STRIDE,
                                      MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, X, Y, Z, ob2.x,
                                      ob2.y, o.w[a], loss, f_scale, j >= n_cam_fix, i >= n_pts_fix, e);
            obs_Z<MODEL, NC>(e, G, Zout + (size_t)a * ZS);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// G3b: Schur complement blocks from explicit pair lists.
// The structure of S is static over a solve, so the list of (observation a of camera j, observation b of camera j')
// pairs that share a track is built once per problem (k_pair_count / k_pair_fill, ordered by block, then by camera
// j's camera-major order: deterministic).  Work item = a slice of <= SLICE pairs of ONE block (j, j'): every lane
// has a valid pair (no failed look-ups, no divergence), acc += Z_a Z_b^T stays in registers (rows
// ROW0..ROW0+NR-1), diagonal blocks also accumulate Z_a q_i.  No atomics: one partial per slice, summed in a fixed
// order by k_schur_finalize.
// ------------------------------------------------------------------------------------------------
constexpr int SLICE = 1024;

// one warp per (chunk of camera j, partner j') item: number of tracks of the chunk that j' also sees
__global__ void k_pair_count(const int* __restrict__ chunk_cam, const int* __restrict__ chunk_beg,
                             const int* __restrict__ chunk_end, const int* __restrict__ cm_pts,
                             const int* __restrict__ obs_of, int N, const int* __restrict__ item_base,
                             const int* __restrict__ item_chunk, int n_items, int* __restrict__ counts)
{
    const int item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n_items) return;
    const int ch = item_chunk[item], j = chunk_cam[ch], jp = j + (item - item_base[ch]);
    int cnt = 0;
    if (jp == j) cnt = chunk_end[ch] - chunk_beg[ch];
    else {
        const int* row = obs_of + (size_t)jp * N;
        for (int t = chunk_beg[ch] + lane; t < chunk_end[ch]; t += 32) cnt += row[cm_pts[t]] >= 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if (lane == 0) counts[item] = cnt;
}

// same traversal, writes the pairs of the item at pairs[item_off[item] ...] in camera-major order
__global__ void k_pair_fill(const int* __restrict__ chunk_cam, const int* __restrict__ chunk_beg,
                            const int* __restrict__ chunk_end, const int* __restrict__ cm_obs,
                            const int* __restrict__ cm_pts, const int* __restrict__ obs_of, int N,
                            const int* __restrict__ item_base, const int* __restrict__ item_chunk, int n_items,
                            const int* __restrict__ item_off, int2* __restrict__ pairs)
{
    const int item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n_items) return;
    const int ch = item_chunk[item], j = chunk_cam[ch], jp = j + (item - item_base[ch]);
    const int* row = obs_of + (size_t)jp * N;
    int out = item_off[item];
    const int beg = chunk_beg[ch], end = chunk_end[ch];
    for (int t0 = beg; t0 < end; t0 += 32) {
        const int t = t0 + lane;
        int a = -1, b = -1;
        if (t < end) {
            a = cm_obs[t];
            b = (jp == j) ? a : row[cm_pts[t]];
        }
        const unsigned m = __ballot_sync(0xffffffffu, b >= 0);
        if (b >= 0) pairs[out + __popc(m & ((1u << lane) - 1u))] = make_int2(a, b);
        out += __popc(m);
    }
}

template <int NC, int ROW0, int NR>
__global__ void __launch_bounds__(TPB, 3)
k_schur(const int* __restrict__ slice_block, const int* __restrict__ slice_p0, const int* __restrict__ slice_p1,
        const int* __restrict__ sb_j, const int* __restrict__ sb_jp, const int2* __restrict__ pairs,
        const int* __restrict__ pts_ind, const double* __restrict__ Zin, const double* __restrict__ q,
        double* __restrict__ schur_partials)
{
    constexpr int NV = NR * NC + NR, NVALL = NC * NC + NC;
    constexpr int EPT = SLICE / TPB;                       // pairs per thread
    // 16-byte vector loads of the Z records when every offset involved is even
    constexpr bool VEC = ((NC * 3) % 2 == 0) && ((NR * 3) % 2 == 0) && ((ROW0 * 3) % 2 == 0);
    __shared__ double sm[NV * (TPB / 32)];
    const int sl = blockIdx.x, blk = slice_block[sl];
    const bool diag = sb_j[blk] == sb_jp[blk];
    const int p0 = slice_p0[sl], p1 = slice_p1[sl];
    double acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.0;
    int2 pr[EPT];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int p = p0 + threadIdx.x + e * TPB;
        pr[e] = p < p1 ? pairs[p] : make_int2(-1, -1);
    }
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
        const int a = pr[e].x, b = pr[e].y;
        if (a < 0) continue;
        double A[NR * 3], B[NC * 3];
        const double* za = Zin + (size_t)a * NC * 3 + ROW0 * 3;
        const double* zb = Zin + (size_t)b * NC * 3;
        if (VEC) {
            const double2* za2 = reinterpret_cast<const double2*>(za);
            const double2* zb2 = reinterpret_cast<const double2*>(zb);
#pragma unroll
            for (int k = 0; k < NR * 3 / 2; ++k) { const double2 v = za2[k]; A[2 * k] = v.x; A[2 * k + 1] = v.y; }
#pragma unroll
            for (int k = 0; k < NC * 3 / 2; ++k) { const double2 v = zb2[k]; B[2 * k] = v.x; B[2 * k + 1] = v.y; }
        } else {
#pragma unroll
            for (int k = 0; k < NR * 3; ++k) A[k] = za[k];
#pragma unroll
            for (int k = 0; k < NC * 3; ++k) B[k] = zb[k];
        }
#pragma unroll
        for (int s = 0; s < NC; ++s) {
#pragma unroll
            for (int r = 0; r < NR; ++r)
                acc[r * NC + s] += A[3 * r] * B[3 * s] + A[3 * r + 1] * B[3 * s + 1] + A[3 * r + 2] * B[3 * s + 2];
        }
        if (diag) {
            const int i = pts_ind[a];
            const double q0 = q[3 * (size_t)i], q1 = q[3 * (size_t)i + 1], q2 = q[3 * (size_t)i + 2];
#pragma unroll
            for (int r = 0; r < NR; ++r) acc[NR * NC + r] += A[3 * r] * q0 + A[3 * r + 1] * q1 + A[3 * r + 2] * q2;
        }
    }
    const double tot = block_reduce_sum<NV, TPB>(acc, sm);
    if (threadIdx.x < NV) {
        const int k = threadIdx.x;
        const int pos = (k < NR * NC) ? (ROW0 * NC + k) : (NC * NC + ROW0 + (k - NR * NC));
        schur_partials[(size_t)sl * NVALL + pos] = tot;
    }
}

// one block per (j, j') block: S_jj' = [j==j'] (U_j + reg diag(sinv_c^2)) - sum over the block's slices ;
// rhs_j = -g_j + sum.  One warp per value: lanes stride over the slices, fixed-shape shuffle tree -> deterministic.
template <int NC>
__global__ void __launch_bounds__(256)
k_schur_finalize(const double* __restrict__ schur_partials, const int* __restrict__ sb_first,
                 const int* __restrict__ sb_j, const int* __restrict__ sb_jp, int M, int n_cam_fix,
                 const double* __restrict__ camsys_local, const double* __restrict__ sinv,
                 const double* __restrict__ scal, int add_diag, int n_common, double* __restrict__ S)
{
    constexpr int NVALL = NC * NC + NC, NW = 8, G = 4;      // 8 warps, 4 values per warp in flight
    const double reg = scal[SC_REG];
    const int blk = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j = sb_j[blk], jp = sb_jp[blk];
    const int ns = M * NC;
    const int s0 = sb_first[blk], s1 = sb_first[blk + 1];
    for (int k0 = warp; k0 < NVALL; k0 += NW * G) {
        double sum[G];
#pragma unroll
        for (int u = 0; u < G; ++u) sum[u] = 0.0;
        for (int sl = s0 + lane; sl < s1; sl += 32)
#pragma unroll
            for (int u = 0; u < G; ++u) {
                const int k = k0 + NW * u;
                if (k < NVALL) sum[u] += schur_partials[(size_t)sl * NVALL + k];
            }
#pragma unroll
        for (int u = 0; u < G; ++u)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum[u] += __shfl_xor_sync(0xffffffffu, sum[u], o);
        if (lane != 0) continue;
#pragma unroll
        for (int u = 0; u < G; ++u) {
            const int k = k0 + NW * u;
            if (k >= NVALL) continue;
            const double s = sum[u];
            if (k < NC * NC) {
                const int r = k / NC, c = k % NC;
                double val = -s;
                if (j == jp) {
                    val += camsys_local[(size_t)j * NC * NC + r * NC + c];
                    if (r == c && add_diag && !(j > 0 && r >= NC - n_common)) {      // unused shared slots: see k_fold_common
                        const double si = sinv[(size_t)j * NC + r];
                        val += (j < n_cam_fix) ? 1.0 : reg * si * si;
                    }
                }
                S[(size_t)(j * NC + r) + (size_t)(jp * NC + c) * ns] = val;
                if (j != jp) S[(size_t)(jp * NC + c) + (size_t)(j * NC + r) * ns] = val;
            } else if (j == jp) {
                const int r = k - NC * NC;
                S[(size_t)ns * ns + (size_t)j * NC + r] = -camsys_local[(size_t)M * NC * NC + (size_t)j * NC + r] + s;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// COMMON_K (ba_params.py:167-171): the last n_common variables of every camera are ONE set of unknowns.  The blocks
// are assembled per camera as usual; the reduced system is then folded, S' = P^T S P with P the 0/1 map from
// [shared | per-camera] unknowns to per-camera slots: rows and columns of the shared slots of cameras 1..M-1 are
// added onto camera 0's and replaced by identity rows with a zero right-hand side (their step is 0).
// One CTA; S is ns x ns column-major followed by the right-hand side.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_fold_common(double* __restrict__ S, int ns, int nc, int M, int n_common)
{
    double* rhs = S + (size_t)ns * ns;
    const int s0 = nc - n_common;
    // rows (and the right-hand side)
    for (int t = threadIdx.x; t < n_common * (ns + 1); t += blockDim.x) {
        const int s = s0 + t / (ns + 1), col = t % (ns + 1);
        double* base = col < ns ? S + (size_t)col * ns : rhs;
        double acc = base[s];
        for (int j = 1; j < M; ++j) { acc += base[j * nc + s]; base[j * nc + s] = 0.0; }
        base[s] = acc;
    }
    __syncthreads();
    // columns
    for (int t = threadIdx.x; t < n_common * ns; t += blockDim.x) {
        const int s = s0 + t / ns, row = t % ns;
        double acc = S[(size_t)s * ns + row];
        for (int j = 1; j < M; ++j) { acc += S[(size_t)(j * nc + s) * ns + row]; S[(size_t)(j * nc + s) * ns + row] = 0.0; }
        S[(size_t)s * ns + row] = acc;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < n_common * (M - 1); t += blockDim.x) {
        const int e = (1 + t / n_common) * nc + s0 + t % n_common;
        S[(size_t)e * ns + e] = 1.0;
    }
}

// camera part of a variable vector with the shared slots of camera 0 copied to every camera (what J acts on)
__global__ void k_expand_common(const double* __restrict__ src, double* __restrict__ dst, int ns, int nc, int n_common)
{
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < ns; e += gridDim.x * blockDim.x) {
        const int s = e % nc;
        dst[e] = s >= nc - n_common ? src[s] : src[e];
    }
}

// ------------------------------------------------------------------------------------------------
// G6: back-substitution  dp_i = -G^T (q_i + sum_a Z_a^T dc_cam(a)), warp tiles like k_point_prep
// ------------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(TPB)
k_backsub(ObsArrays o, int ns, const double* __restrict__ F, const double* __restrict__ q,
          const double* __restrict__ Zin, const double* __restrict__ dcam, double* __restrict__ delta)
{
    constexpr int ZS = NC * 3, ZP = ZS + 1;
    __shared__ double sv[WPB][3][32];
    __shared__ double sZ[WPB][32 * ZP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ob, nobs;
    warp_tile(o, ob, nobs);
    if (nobs == 0) return;
    if (nobs <= 32) {
        const double* src = Zin + (size_t)ob * ZS;
        for (int t = lane; t < nobs * ZS; t += 32) sZ[warp][(t / ZS) * ZP + (t % ZS)] = src[t];
        __syncwarp();
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        int i = -1, a = -1;
        if (lane < nobs) {
            a = ob + lane;
            i = o.pts_ind[a];
            const int j = o.cam_ind[a];
            const double* z = &sZ[warp][lane * ZP];
#pragma unroll
            for (int r = 0; r < NC; ++r) {
                const double dc = dcam[(size_t)j * NC + r];
                s0 += z[3 * r] * dc; s1 += z[3 * r + 1] * dc; s2 += z[3 * r + 2] * dc;
            }
        }
        sv[warp][0][lane] = s0; sv[warp][1][lane] = s1; sv[warp][2][lane] = s2;
        __syncwarp();
        if (lane < nobs) {
            const int beg = o.track_ptr[i];
            if (a == beg) {
                const int L = o.track_ptr[i + 1] - beg;
                double t0 = q[3 * (size_t)i], t1 = q[3 * (size_t)i + 1], t2 = q[3 * (size_t)i + 2];
                for (int m = 0; m < L; ++m) { t0 += sv[warp][0][lane + m]; t1 += sv[warp][1][lane + m]; t2 += sv[warp][2][lane + m]; }
                const double* G = F + 6 * (size_t)i;
                delta[ns + 3 * (size_t)i + 0] = -(G[0] * t0 + G[1] * t1 + G[3] * t2);
                delta[ns + 3 * (size_t)i + 1] = -(G[2] * t1 + G[4] * t2);
                delta[ns + 3 * (size_t)i + 2] = -(G[5] * t2);
            }
        }
    } else {
        const int i = o.pts_ind[ob];
        double s[3] = {0.0, 0.0, 0.0};
        for (int a = ob + lane; a < ob + nobs; a += 32) {
            const int j = o.cam_ind[a];
            const double* z = Zin + (size_t)a * ZS;
#pragma unroll
            for (int r = 0; r < NC; ++r) {
                const double dc = dcam[(size_t)j * NC + r];
                s[0] += z[3 * r] * dc; s[1] += z[3 * r + 1] * dc; s[2] += z[3 * r + 2] * dc;
            }
        }
        warp_allreduce_sum<3>(s);
        if (lane == 0) {
            const double t0 = s[0] + q[3 * (size_t)i], t1 = s[1] + q[3 * (size_t)i + 1], t2 = s[2] + q[3 * (size_t)i + 2];
            const double* G = F + 6 * (size_t)i;
            delta[ns + 3 * (size_t)i + 0] = -(G[0] * t0 + G[1] * t1 + G[3] * t2);
            delta[ns + 3 * (size_t)i + 1] = -(G[2] * t1 + G[4] * t2);
            delta[ns + 3 * (size_t)i + 2] = -(G[5] * t2);
        }
    }
}

// g_h.gn_h = sum g d  and  |gn_h|^2 = sum (sinv d)^2      (d = Gauss-Newton step delta)
__global__ void __launch_bounds__(256)
k_dot_g_delta(const double* __restrict__ g, const double* __restrict__ sinv, const double* __restrict__ delta,
              long long n, int ns, int count_cameras, double* partials, unsigned* counter, double* scal)
{
    __shared__ double sm[2 * (256 / 32)];
    double acc[2] = {0.0, 0.0};
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        if (idx >= ns || count_cameras) {
            const double d = delta[idx], sd = sinv[idx] * d;
            acc[0] += g[idx] * d;
            acc[1] += sd * sd;
        }
    }
    const double tot = block_reduce_sum<2, 256>(acc, sm);
    __shared__ int slots[2];
    if (threadIdx.x == 0) { slots[0] = SC_GGN; slots[1] = SC_DD; }
    __syncthreads();
    grid_sum_finalize<2, 256>(tot, partials, counter, scal, slots, sm);
}

// second basis vector, orthogonalised explicitly (the Gauss-Newton step is nearly parallel to the gradient
// whenever the damping is large, so forming |w|^2 from the Gram matrix would cancel catastrophically):
//   t2 = delta - alpha t1 ,  alpha = (g_h.gn_h)/|g_h|^2 read from the scalar block (no host round trip)
// sums: |w|^2 = |sinv t2|^2, w.g_h = t2.g, |t1|^2, t1.t2, |t2|^2
__global__ void __launch_bounds__(256)
k_build_t2(const double* __restrict__ g, const double* __restrict__ sinv, const double* __restrict__ delta,
           const double* __restrict__ t1, double* __restrict__ t2, long long n, int ns, int count_cameras,
           double* partials, unsigned* counter, double* scal)
{
    __shared__ double sm[5 * (256 / 32)];
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const double gg = scal[SC_GG];
    const double alpha = gg > 0.0 ? scal[SC_GGN] / gg : 0.0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const double a = t1[idx], b = delta[idx] - alpha * a;
        t2[idx] = b;
        if (idx >= ns || count_cameras) {
            const double wv = sinv[idx] * b;
            acc[0] += wv * wv;
            acc[1] += b * g[idx];
            acc[2] += a * a;
            acc[3] += a * b;
            acc[4] += b * b;
        }
    }
    const double tot = block_reduce_sum<5, 256>(acc, sm);
    __shared__ int slots[5];
    if (threadIdx.x == 0) { slots[0] = SC_WW; slots[1] = SC_WG; slots[2] = SC_T11; slots[3] = SC_T12; slots[4] = SC_T22; }
    __syncthreads();
    grid_sum_finalize<5, 256>(tot, partials, counter, scal, slots, sm);
}

__device__ __forceinline__ double step_value(double x, double a, double d, double ca, double cb)
{
    return x + fma(ca, a, cb * d);
}

__global__ void __launch_bounds__(256)
k_step(const double* __restrict__ x, const double* __restrict__ t1, const double* __restrict__ delta,
       const double* __restrict__ scal, double* __restrict__ x_new, long long n, const double* __restrict__ cam_static,
       double* __restrict__ camrec_new, int M, int P, int nc, int n_cam_fix, int n_common, int model)
{
    const double ca = scal[SC_C1], cb = scal[SC_C2];
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long idx = gid; idx < n; idx += (long long)gridDim.x * blockDim.x)
        x_new[idx] = step_value(x[idx], t1[idx], delta[idx], ca, cb);
    // the first M threads also prepare the camera records of the trial point (same expression as above,
    // so the records match x_new bit for bit)
    if (gid < M) {
        const int j = (int)gid;
        double v[MAX_CAM_PARAMS];
#pragma unroll
        for (int s = 0; s < MAX_CAM_PARAMS; ++s) {
            double val = 0.0;
            if (s < P) {
                if (s < nc && j >= n_cam_fix) {
                    const size_t e = (size_t)((s >= nc - n_common) ? 0 : j) * nc + s;
                    val = step_value(x[e], t1[e], delta[e], ca, cb);
                } else {
                    val = cam_static[(size_t)j * P + s];
                }
            }
            v[s] = val;
        }
        write_camrec(v, camrec_new + (size_t)j * CAMREC_STRIDE, model);
    }
}

// ------------------------------------------------------------------------------------------------
// device-side control: the damping rule and the 2-D trust-region solve run as single-thread kernels on the
// already reduced scalars, so that the host reads the scalar block once per trial step instead of three times
// ------------------------------------------------------------------------------------------------
// damping from the Cauchy step (scipy trf.py:485-490): reg = -min_{0<=t<=Delta/|g_h|} (a t^2 + b t) / Delta^2
// delta_arg < 0: first iteration, Delta = |x0 * scale_inv| (or 1);  reg_override >= 0: use that value (re-damping).
// Also run in the epilogue of the pattern engine's K2 (k_pt_jvp1).
__device__ __forceinline__ void control_reg_dev(double* scal, double delta_arg, double reg_override)
{
    double Delta = delta_arg;
    if (Delta < 0.0) {
        Delta = sqrt(scal[SC_XS]);
        if (Delta == 0.0) Delta = 1.0;
    }
    scal[SC_DELTA] = Delta;
    if (reg_override >= 0.0) { scal[SC_REG] = reg_override; return; }
    const double gg = scal[SC_GG];
    const double qa = 0.5 * scal[SC_A], qb = -gg;
    const double to_tr = Delta / sqrt(gg);
    double ag = 0.0;
    ag = fmin(ag, to_tr * (qa * to_tr + qb));
    if (qa != 0.0) {
        const double ext = -0.5 * qb / qa;
        if (ext > 0.0 && ext < to_tr) ag = fmin(ag, ext * (qa * ext + qb));
    }
    scal[SC_REG] = -ag / (Delta * Delta);
}

__global__ void k_control_reg(double* scal, double delta_arg, double reg_override)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) control_reg_dev(scal, delta_arg, reg_override);
}

// exact 2-D trust-region step in span{g_h, gn_h} (scipy trf.py:496-509) for the radius `delta_arg`
// (< 0: the radius stored by k_control_reg)
__global__ void k_control_tr2d(double* scal, double delta_arg)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const double Delta = delta_arg < 0.0 ? scal[SC_DELTA] : delta_arg;
    const double gg = scal[SC_GG], ww = scal[SC_WW], wg = scal[SC_WG];
    const double t11 = scal[SC_T11], t12 = scal[SC_T12], t22 = scal[SC_T22];
    const double b11 = scal[SC_B11], b12 = scal[SC_B12], b22 = scal[SC_B22];
    // orthonormal basis s1 = g_h/|g_h|, s2 = w/|w| ; x-space images t1/|g_h|, t2/|w|
    const double n1 = sqrt(gg);
    const bool rank2 = ww > 0.0;
    const double n2 = rank2 ? sqrt(ww) : 1.0;
    const double B00 = b11 / (n1 * n1), B01 = rank2 ? b12 / (n1 * n2) : 0.0, B11 = rank2 ? b22 / (n2 * n2) : 1.0;
    const double gS0 = n1, gS1 = rank2 ? wg / n2 : 0.0;
    double pS[2];
    solve_trust_region_2d(B00, B01, B11, gS0, gS1, Delta, pS);
    const double c1 = pS[0] / n1, c2 = rank2 ? pS[1] / n2 : 0.0;
    scal[SC_C1] = c1;
    scal[SC_C2] = c2;
    scal[SC_PRED] = -(0.5 * (B00 * pS[0] * pS[0] + 2.0 * B01 * pS[0] * pS[1] + B11 * pS[1] * pS[1]) + gS0 * pS[0] + gS1 * pS[1]);
    scal[SC_STEPH] = sqrt(pS[0] * pS[0] + pS[1] * pS[1]);
    scal[SC_STEPN] = sqrt(fmax(0.0, c1 * c1 * t11 + 2.0 * c1 * c2 * t12 + c2 * c2 * t22));
}

// per-observation Jacobian blocks for tests (weights applied, no robust rescale)
template <int MODEL, int NC>
__global__ void k_jac_blocks(ObsArrays o, const double* __restrict__ xp, const double* __restrict__ camrec,
                             const double* __restrict__ rpc_tab, long long K, int n_cam_fix, int n_pts_fix,
                             double* __restrict__ Jc, double* __restrict__ Jp)
{
    for (long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x; a < K; a += (long long)gridDim.x * blockDim.x) {
        const int j = o.cam_ind[a], i = o.pts_ind[a];
        const double2 ob = o.pts2d[a];
        ObsEval<MODEL, NC> e;
        eval_obs<MODEL, NC, true>(camrec + (size_t)j * CAMREC_STRIDE,
                                  MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr, xp[3 * (size_t)i],
                                  xp[3 * (size_t)i + 1], xp[3 * (size_t)i + 2], ob.x, ob.y, o.w[a], LOSS_LINEAR, 1.0,
                                  j >= n_cam_fix, i >= n_pts_fix, e);
        if (Jc)
            for (int k = 0; k < 2 * NC; ++k) Jc[(size_t)a * 2 * NC + k] = e.Jc[k];
        if (Jp)
            for (int k = 0; k < 6; ++k) Jp[(size_t)a * 6 + k] = e.Jp[k];
    }
}

// scatter for obs_of[M][N]
// camera-major copies (static) of the per-observation data, from the camera-major permutation cm_obs
__global__ void k_gather_camera_major(const int* __restrict__ cm_obs, const int* __restrict__ pts_ind,
                                      const double2* __restrict__ pts2d, const double* __restrict__ w, long long K,
                                      int* __restrict__ cm_pts, double2* __restrict__ cm_pts2d, double* __restrict__ cm_w)
{
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < K; t += (long long)gridDim.x * blockDim.x) {
        const int a = cm_obs[t];
        cm_pts[t] = pts_ind[a]; cm_pts2d[t] = pts2d[a]; cm_w[t] = w[a];
    }
}

__global__ void k_fill_obs_of(const int* __restrict__ cam_ind, const int* __restrict__ pts_ind, long long K, int N,
                              int* __restrict__ obs_of)
{
    for (long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x; a < K; a += (long long)gridDim.x * blockDim.x)
        obs_of[(size_t)cam_ind[a] * N + pts_ind[a]] = (int)a;
}

}  // namespace sba
