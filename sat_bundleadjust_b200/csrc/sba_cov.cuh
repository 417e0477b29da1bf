// Posterior covariance at a point x (sba_covariance).  Included by sba_ba.cu after sba_kernels.cuh.
//
// With H = J^T J = [[U, W], [W^T, V]] over the free variables and S = U - W V^-1 W^T (the undamped reduced camera system,
// formed by the solver's own Schur path and factored S = L L^T by its Cholesky kernels):
//   cameras   Sigma_cc = s2 S^-1                                          k_cov_inverse + k_cov_finish
//   track t   Sigma_t  = s2 (V_t^-1 + sum_{a,b} Y_a S^-1[a,b] Y_b^T),  Y_a = V_t^-1 W_a^T     k_cov_points
// where W_a = Jc_a^T Jp_a (nc x 3) is the coupling block of observation a of the track.  J is never stored: k_cov_points
// recomputes every observation's (robust-rescaled) Jacobian rows in registers, like every other pass.
#pragma once
#include <math_constants.h>

#include "sba_kernels.cuh"

namespace sba {

// Gauge / rank test on the factor L of S: pivot k of a free camera slot is rejected when L_kk^2 <= thr * U_kk (U = the
// un-reduced camera block at the same x; S is formed by cancellation against U, so a pivot of that relative size is round-off).
// out[0] = smallest ratio L_kk^2 / U_kk over the free slots, out[1] = first rejected slot (-1: none), out[2] = its ratio.
// A failed factorisation (fail = k + 1, non-positive pivot k) rejects slot k with ratio 0.  One CTA.
__global__ void __launch_bounds__(256)
k_cov_pivots(const double* __restrict__ L, const double* __restrict__ camsys, int ns, int nc, int n_cam_fix,
             const double* __restrict__ fail, double thr, double* __restrict__ out)
{
    __shared__ double s_min[256];
    __shared__ int s_bad[256];
    const int tid = threadIdx.x;
    const int failed = (int)*fail;
    double mn = CUDART_INF;
    int bad = ns;
    if (failed) {
        mn = 0.0;
        bad = failed - 1;
    } else {
        for (int k = n_cam_fix * nc + tid; k < ns; k += 256) {
            const int j = k / nc, r = k - j * nc;
            const double u = camsys[(size_t)j * nc * nc + r * nc + r];
            const double l = L[(size_t)k * ns + k];
            const double ratio = u > 0.0 ? l * l / u : 0.0;
            mn = fmin(mn, ratio);
            if (!(ratio > thr) && k < bad) bad = k;
        }
    }
    s_min[tid] = mn; s_bad[tid] = bad;
    __syncthreads();
    for (int h = 128; h > 0; h >>= 1) {
        if (tid < h) { s_min[tid] = fmin(s_min[tid], s_min[tid + h]); s_bad[tid] = min(s_bad[tid], s_bad[tid + h]); }
        __syncthreads();
    }
    if (tid == 0) {
        const int b = s_bad[0];
        out[0] = s_min[0];
        out[1] = b < ns ? (double)b : -1.0;
        if (b < ns) {
            const int j = b / nc, r = b - j * nc;
            const double u = camsys[(size_t)j * nc * nc + r * nc + r], l = L[(size_t)b * ns + b];
            out[2] = (failed || !(u > 0.0)) ? 0.0 : l * l / u;
        } else {
            out[2] = 0.0;
        }
    }
}

// S^-1 = L^-T L^-1 from the lower triangle of the factor (column-major, ns x ns; the upper triangle is not read: the blocked
// factorisation leaves S there).  One CTA per 32 columns c0.. of the identity, every size up to the dense limit (ns <= 4096):
// forward substitution L Z = E, then backward L^T X = Z, both left-looking over 32-row blocks.  A block step is a 32 x 32
// tile product over the finished blocks (tiles of L and of the CTA's own columns staged in shared memory, L read from L2)
// followed by a 32 x 32 triangular solve of the diagonal block by one warp (lane = column).  The CTA's columns live in X
// (global, the output) between steps; rows of Z above c0 are zero and are never touched by the forward pass.
constexpr int CI_LD = 33;
__global__ void __launch_bounds__(256)
k_cov_inverse(const double* __restrict__ L, int ns, double* __restrict__ X)
{
    __shared__ double Lt[32 * CI_LD], Xt[32 * CI_LD], Zs[32 * CI_LD];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c0 = blockIdx.x * 32, nblk = (ns + 31) / 32, K0 = blockIdx.x;
    const int c = lane;                            // this thread's column of the tile product; rows warp + 8 u
    const bool col_ok = c0 + c < ns;
    // acc[u] = sum over the row tiles of A[j][r] * Xcols[r][c], j = warp + 8 u
    auto tile_step = [&](bool forward, int K, int R, double (&acc)[4]) {
        const int k0 = 32 * K, r0 = 32 * R;
        for (int e = tid; e < 1024; e += 256) {
            const int hi = e >> 5, lo = e & 31;
            // forward: A[j][r] = L[k0 + j, r0 + r] (rows of block K, columns of block R < K), consecutive j coalesced
            // backward: A[j][r] = L[r0 + r, k0 + j] (transposed: rows of block R > K), consecutive r coalesced
            if (forward) Lt[lo * CI_LD + hi] = (k0 + lo < ns && r0 + hi < ns) ? L[(size_t)(r0 + hi) * ns + k0 + lo] : 0.0;
            else Lt[hi * CI_LD + lo] = (k0 + hi < ns && r0 + lo < ns) ? L[(size_t)(k0 + hi) * ns + r0 + lo] : 0.0;
            Xt[lo * CI_LD + hi] = (r0 + lo < ns && c0 + hi < ns) ? X[(size_t)(c0 + hi) * ns + r0 + lo] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < 32; ++r) {
            const double xv = Xt[r * CI_LD + c];
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[u] = fma(Lt[(warp + 8 * u) * CI_LD + r], xv, acc[u]);
        }
        __syncthreads();
    };
    auto load_diag = [&](int k0) {                 // Lt[j][s] = L[k0 + j, k0 + s], lower triangle of the diagonal block
        for (int e = tid; e < 1024; e += 256) {
            const int s = e >> 5, j = e & 31;
            Lt[j * CI_LD + s] = (s <= j && k0 + j < ns) ? L[(size_t)(k0 + s) * ns + k0 + j] : (s == j ? 1.0 : 0.0);
        }
    };
    // ---- forward: Z_K = L_KK^-1 (E_K - sum_{R < K} L_KR Z_R), blocks K >= K0 (Z is zero above c0) ----
    for (int K = K0; K < nblk; ++K) {
        const int k0 = 32 * K;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int R = K0; R < K; ++R) tile_step(true, K, R, acc);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = warp + 8 * u;
            Zs[j * CI_LD + c] = (k0 + j == c0 + c ? 1.0 : 0.0) - acc[u];
        }
        load_diag(k0);
        __syncthreads();
        if (warp == 0) {
            for (int j = 0; j < 32; ++j) {
                double v = Zs[j * CI_LD + c];
                for (int s = 0; s < j; ++s) v = fma(-Lt[j * CI_LD + s], Zs[s * CI_LD + c], v);
                Zs[j * CI_LD + c] = v / Lt[j * CI_LD + j];
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = warp + 8 * u;
            if (k0 + j < ns && col_ok) X[(size_t)(c0 + c) * ns + k0 + j] = Zs[j * CI_LD + c];
        }
        __syncthreads();
    }
    // ---- backward: X_K = L_KK^-T (Z_K - sum_{R > K} L_RK^T X_R), from the last block up ----
    for (int K = nblk - 1; K >= 0; --K) {
        const int k0 = 32 * K;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int R = K + 1; R < nblk; ++R) tile_step(false, K, R, acc);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = warp + 8 * u;
            const double z = (K >= K0 && k0 + j < ns && col_ok) ? X[(size_t)(c0 + c) * ns + k0 + j] : 0.0;
            Zs[j * CI_LD + c] = z - acc[u];
        }
        load_diag(k0);
        __syncthreads();
        if (warp == 0) {
            for (int j = 31; j >= 0; --j) {
                double v = Zs[j * CI_LD + c];
                for (int s = j + 1; s < 32; ++s) v = fma(-Lt[s * CI_LD + j], Zs[s * CI_LD + c], v);
                Zs[j * CI_LD + c] = v / Lt[j * CI_LD + j];
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = warp + 8 * u;
            if (k0 + j < ns && col_ok) X[(size_t)(c0 + c) * ns + k0 + j] = Zs[j * CI_LD + c];
        }
        __syncthreads();
    }
}

// in place: X <- s2 (X + X^T) / 2 (exactly symmetric), rows and columns of the frozen slots [0, n_fix) set to 0
__global__ void __launch_bounds__(256)
k_cov_finish(double* __restrict__ X, int ns, int n_fix, double s2)
{
    const long long total = (long long)ns * ns;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(e / ns), i = (int)(e - (long long)j * ns);
        if (i < j) continue;                       // the thread of (i, j), i >= j, owns both mirror entries
        double v = i == j ? X[e] : 0.5 * (X[e] + X[(size_t)i * ns + j]);
        v = (i < n_fix || j < n_fix) ? 0.0 : s2 * v;
        X[e] = v;
        X[(size_t)i * ns + j] = v;
    }
}

// coupling block W = Jc^T Jp (NC x 3, row-major) of observation a, and its contribution Jp^T Jp to V (xx xy xz yy yz zz);
// returns the camera (-1 and zeros when a is past the track)
template <int MODEL, int NC>
__device__ __forceinline__ int cov_obs(const ObsArrays& o, int a, bool valid, int i, const double* __restrict__ xp,
                                       const double* __restrict__ camrec, const double* __restrict__ rpc_tab, int n_cam_fix,
                                       bool pt_free, int loss, double f_scale, double (&W)[NC * 3], double (&Vp)[6])
{
#pragma unroll
    for (int k = 0; k < NC * 3; ++k) W[k] = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) Vp[k] = 0.0;
    if (!valid) return -1;
    const int j = o.cam_ind[a];
    const double2 ob = o.pts2d[a];
    ObsEval<MODEL, NC> e;
    eval_obs<MODEL, NC, true>(camrec + (size_t)j * CAMREC_STRIDE, MODEL == MODEL_RPC ? rpc_tab + (size_t)j * RPC_TAB_STRIDE : nullptr,
                              xp[3 * (size_t)i], xp[3 * (size_t)i + 1], xp[3 * (size_t)i + 2], ob.x, ob.y, o.w[a], loss, f_scale,
                              j >= n_cam_fix, pt_free, e);
#pragma unroll
    for (int r = 0; r < NC; ++r)
#pragma unroll
        for (int m = 0; m < 3; ++m) W[3 * r + m] = e.Jc[r] * e.Jp[m] + e.Jc[NC + r] * e.Jp[3 + m];
    Vp[0] = e.Jp[0] * e.Jp[0] + e.Jp[3] * e.Jp[3];
    Vp[1] = e.Jp[0] * e.Jp[1] + e.Jp[3] * e.Jp[4];
    Vp[2] = e.Jp[0] * e.Jp[2] + e.Jp[3] * e.Jp[5];
    Vp[3] = e.Jp[1] * e.Jp[1] + e.Jp[4] * e.Jp[4];
    Vp[4] = e.Jp[1] * e.Jp[2] + e.Jp[4] * e.Jp[5];
    Vp[5] = e.Jp[2] * e.Jp[2] + e.Jp[5] * e.Jp[5];
    return j;
}

// Y = Vinv W^T (3 x NC, stored [m][r] as Y[3 r + m]), Vinv symmetric (xx xy xz yy yz zz)
template <int NC>
__device__ __forceinline__ void cov_Y(const double (&Vi)[6], const double (&W)[NC * 3], double (&Y)[NC * 3])
{
#pragma unroll
    for (int r = 0; r < NC; ++r) {
        const double w0 = W[3 * r], w1 = W[3 * r + 1], w2 = W[3 * r + 2];
        Y[3 * r + 0] = Vi[0] * w0 + Vi[1] * w1 + Vi[2] * w2;
        Y[3 * r + 1] = Vi[1] * w0 + Vi[3] * w1 + Vi[4] * w2;
        Y[3 * r + 2] = Vi[2] * w0 + Vi[4] * w1 + Vi[5] * w2;
    }
}

// Marginal covariance of the tracks, over the warp tiles of the internal track order (runs of whole tracks of <= 32
// observations; a longer track is a tile of its own).  Output: s2 V_t^-1 + sum_{a,b} Y_a C[a,b] Y_b^T with C = s2 S^-1, upper
// triangle (xx xy xz yy yz zz), in the caller's track order (trk_new2old: internal -> caller, NULL when they agree).  Frozen
// points are 0; a free point whose block V_t is not positive definite is 0 and counted in *bad.  C is read from shared memory
// when it fits (c_in_smem), else from L2.
//
// k_cov_points: the tiles of <= 32 observations, one warp per tile (grid-stride), lane = observation, several tracks per warp.
// Every lane evaluates its observation's Jacobian rows once (robust rescale in registers); the per-lane V contributions, the
// Y_a = V_t^-1 W_a^T and the per-lane results go through the warp's shared-memory slots, and every lane sums the slots of its
// own track's lane segment (fixed order, no shuffles across tracks).  Per lane the pair loop is T_a = sum_b C[a,b] Y_b^T
// over its track, then Y_a T_a.
constexpr int COV_THREADS = 128, COV_WARPS = COV_THREADS / 32;

template <int NC>
__host__ __device__ constexpr int cov_warp_doubles() { return (12 + 3 * NC) * 32; }      // V slots, Y slots, result slots

template <int MODEL, int NC>
__global__ void __launch_bounds__(COV_THREADS)
k_cov_points(ObsArrays o, const int* __restrict__ tile_obs, int n_tiles, const double* __restrict__ xp,
             const double* __restrict__ camrec, const double* __restrict__ rpc_tab, int n_cam_fix, int n_pts_fix, int loss,
             double f_scale, const double* __restrict__ C, int ns, int c_in_smem, double s2, const int* __restrict__ trk_new2old,
             double* __restrict__ out, double* __restrict__ bad)
{
    extern __shared__ double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* sw = sm + (size_t)warp * cov_warp_doubles<NC>();
    double *sV = sw, *sY = sw + 6 * 32, *sA = sw + (6 + 3 * NC) * 32;
    int* sJ = (int*)(sm + (size_t)COV_WARPS * cov_warp_doubles<NC>()) + warp * 32;
    double* sC = sm + (size_t)COV_WARPS * cov_warp_doubles<NC>() + COV_WARPS * 32 / 2;
    if (c_in_smem) {
        for (int e = threadIdx.x; e < ns * ns; e += blockDim.x) sC[e] = C[e];
        __syncthreads();
    }
    const double* Cv = c_in_smem ? sC : C;
    for (int tile = blockIdx.x * COV_WARPS + warp; tile < n_tiles; tile += gridDim.x * COV_WARPS) {
        const int ob = tile_obs[tile], nobs = tile_obs[tile + 1] - ob;
        if (nobs > 32) continue;                              // long track: k_cov_long_tracks
        const bool valid = lane < nobs;
        const int a = ob + (valid ? lane : 0);
        const int t = o.pts_ind[a], beg = o.track_ptr[t], len = o.track_ptr[t + 1] - beg, hl = beg - ob;
        const bool pt_free = t >= n_pts_fix;
        double W[NC * 3], Vp[6];
        const int ja = cov_obs<MODEL, NC>(o, a, valid, t, xp, camrec, rpc_tab, n_cam_fix, pt_free, loss, f_scale, W, Vp);
#pragma unroll
        for (int k = 0; k < 6; ++k) sV[k * 32 + lane] = Vp[k];
        __syncwarp();
        double V[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (valid)
            for (int b = hl; b < hl + len; ++b)
#pragma unroll
                for (int k = 0; k < 6; ++k) V[k] += sV[k * 32 + b];
        double G[6], Vi[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        const bool ok = valid && pt_free && invert_point_block(V, 0.0, 0.0, 0.0, 0.0, G);
        if (ok) {                                            // V^-1 = G^T G, G lower (g00 g10 g11 g20 g21 g22)
            Vi[0] = G[0] * G[0] + G[1] * G[1] + G[3] * G[3];
            Vi[1] = G[1] * G[2] + G[3] * G[4];
            Vi[2] = G[3] * G[5];
            Vi[3] = G[2] * G[2] + G[4] * G[4];
            Vi[4] = G[4] * G[5];
            Vi[5] = G[5] * G[5];
        }
        double Ya[NC * 3];
        cov_Y<NC>(Vi, W, Ya);                                 // 0 unless ok
#pragma unroll
        for (int k = 0; k < NC * 3; ++k) sY[k * 32 + lane] = Ya[k];
        sJ[lane] = ja < 0 ? 0 : ja;
        __syncwarp();
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (ok) {
            double T[NC * 3];
#pragma unroll
            for (int k = 0; k < NC * 3; ++k) T[k] = 0.0;
            for (int b = hl; b < hl + len; ++b) {
                const double* Ccol = Cv + (size_t)sJ[b] * NC * ns + (size_t)ja * NC;   // C[ja NC + r, jb NC + s]
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    const double y0 = sY[(3 * s) * 32 + b], y1 = sY[(3 * s + 1) * 32 + b], y2 = sY[(3 * s + 2) * 32 + b];
#pragma unroll
                    for (int r = 0; r < NC; ++r) {
                        const double cv = Ccol[(size_t)s * ns + r];
                        T[3 * r] = fma(cv, y0, T[3 * r]);
                        T[3 * r + 1] = fma(cv, y1, T[3 * r + 1]);
                        T[3 * r + 2] = fma(cv, y2, T[3 * r + 2]);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < NC; ++r) {
                acc[0] += Ya[3 * r] * T[3 * r];
                acc[1] += Ya[3 * r] * T[3 * r + 1];
                acc[2] += Ya[3 * r] * T[3 * r + 2];
                acc[3] += Ya[3 * r + 1] * T[3 * r + 1];
                acc[4] += Ya[3 * r + 1] * T[3 * r + 2];
                acc[5] += Ya[3 * r + 2] * T[3 * r + 2];
            }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) sA[k * 32 + lane] = acc[k];
        __syncwarp();
        if (valid && lane == hl) {                            // the track's first lane writes it
            double res[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                double v = s2 * Vi[k];
                for (int b = hl; b < hl + len; ++b) v += sA[k * 32 + b];
                res[k] = v;
            }
            if (pt_free && !ok) atomicAdd(bad, 1.0);
            const int dst = trk_new2old ? trk_new2old[t] : t;
#pragma unroll
            for (int k = 0; k < 6; ++k) out[6 * (size_t)dst + k] = res[k];
        }
        __syncwarp();                                         // the slots are reused by the next tile
    }
}

// k_cov_long_tracks: the tiles of one track of more than 32 observations, one warp per track.  Pass 1 forms V_t (warp sum)
// and inverts it; pass 2 runs over (chunk, chunk) pairs of 32 observations, the partner chunk's Y recomputed in registers and
// shuffled from its lane (O(L^2) work, nothing stored per observation).
template <int MODEL, int NC>
__global__ void __launch_bounds__(128)
k_cov_long_tracks(ObsArrays o, const int* __restrict__ tile_obs, int n_tiles, const double* __restrict__ xp,
                  const double* __restrict__ camrec, const double* __restrict__ rpc_tab, int n_cam_fix, int n_pts_fix, int loss,
                  double f_scale, const double* __restrict__ C, int ns, double s2, const int* __restrict__ trk_new2old,
                  double* __restrict__ out, double* __restrict__ bad)
{
    const double* Cv = C;
    const int lane = threadIdx.x & 31;
    const int warps = gridDim.x * (blockDim.x >> 5);
    for (int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); tile < n_tiles; tile += warps) {
        const int ob = tile_obs[tile];
        if (tile_obs[tile + 1] - ob <= 32) continue;
        const int t = o.pts_ind[ob];
        const int dst = trk_new2old ? trk_new2old[t] : t;
        double res[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (t >= n_pts_fix) {
            const int beg = o.track_ptr[t], len = o.track_ptr[t + 1] - beg, nch = (len + 31) / 32;
            double W[NC * 3], Vp[6], V[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            int ja = -1;
            for (int ch = 0; ch < nch; ++ch) {
                const int q = 32 * ch + lane;
                ja = cov_obs<MODEL, NC>(o, beg + q, q < len, t, xp, camrec, rpc_tab, n_cam_fix, true, loss, f_scale, W, Vp);
#pragma unroll
                for (int k = 0; k < 6; ++k) V[k] += Vp[k];
            }
            warp_allreduce_sum<6>(V);
            double G[6];
            if (invert_point_block(V, 0.0, 0.0, 0.0, 0.0, G)) {
                // V^-1 = G^T G, G lower (g00 g10 g11 g20 g21 g22)
                double Vi[6];
                Vi[0] = G[0] * G[0] + G[1] * G[1] + G[3] * G[3];
                Vi[1] = G[1] * G[2] + G[3] * G[4];
                Vi[2] = G[3] * G[5];
                Vi[3] = G[2] * G[2] + G[4] * G[4];
                Vi[4] = G[4] * G[5];
                Vi[5] = G[5] * G[5];
                double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                for (int c1 = 0; c1 < nch; ++c1) {
                    const int qa = 32 * c1 + lane;
                    if (nch > 1)
                        ja = cov_obs<MODEL, NC>(o, beg + qa, qa < len, t, xp, camrec, rpc_tab, n_cam_fix, true, loss, f_scale, W, Vp);
                    double Ya[NC * 3], T[NC * 3];
                    cov_Y<NC>(Vi, W, Ya);
#pragma unroll
                    for (int k = 0; k < NC * 3; ++k) T[k] = 0.0;
                    const int jrow = ja < 0 ? 0 : ja;
                    for (int c2 = 0; c2 < nch; ++c2) {
                        double Yb[NC * 3];
                        int jb = ja;
                        if (c2 == c1) {
#pragma unroll
                            for (int k = 0; k < NC * 3; ++k) Yb[k] = Ya[k];
                        } else {
                            const int qb = 32 * c2 + lane;
                            double Wb[NC * 3];
                            jb = cov_obs<MODEL, NC>(o, beg + qb, qb < len, t, xp, camrec, rpc_tab, n_cam_fix, true, loss, f_scale, Wb, Vp);
                            cov_Y<NC>(Vi, Wb, Yb);
                        }
                        const int nb = min(32, len - 32 * c2);
                        for (int bb = 0; bb < nb; ++bb) {
                            const int jbb = __shfl_sync(0xffffffffu, jb, bb);
                            const double* Ccol = Cv + (size_t)jbb * NC * ns + (size_t)jrow * NC;   // C[jrow NC + r, jbb NC + s]
#pragma unroll
                            for (int s = 0; s < NC; ++s) {
                                const double y0 = __shfl_sync(0xffffffffu, Yb[3 * s], bb);
                                const double y1 = __shfl_sync(0xffffffffu, Yb[3 * s + 1], bb);
                                const double y2 = __shfl_sync(0xffffffffu, Yb[3 * s + 2], bb);
#pragma unroll
                                for (int r = 0; r < NC; ++r) {
                                    const double cv = Ccol[(size_t)s * ns + r];
                                    T[3 * r] = fma(cv, y0, T[3 * r]);
                                    T[3 * r + 1] = fma(cv, y1, T[3 * r + 1]);
                                    T[3 * r + 2] = fma(cv, y2, T[3 * r + 2]);
                                }
                            }
                        }
                    }
                    if (ja >= 0) {
#pragma unroll
                        for (int r = 0; r < NC; ++r) {
                            acc[0] += Ya[3 * r] * T[3 * r];
                            acc[1] += Ya[3 * r] * T[3 * r + 1];
                            acc[2] += Ya[3 * r] * T[3 * r + 2];
                            acc[3] += Ya[3 * r + 1] * T[3 * r + 1];
                            acc[4] += Ya[3 * r + 1] * T[3 * r + 2];
                            acc[5] += Ya[3 * r + 2] * T[3 * r + 2];
                        }
                    }
                }
                warp_allreduce_sum<6>(acc);
#pragma unroll
                for (int k = 0; k < 6; ++k) res[k] = fma(s2, Vi[k], acc[k]);
            } else if (lane == 0) {
                atomicAdd(bad, 1.0);
            }
        }
        if (lane < 6) {
            double v = res[0];
#pragma unroll
            for (int k = 1; k < 6; ++k) v = lane == k ? res[k] : v;
            out[6 * (size_t)dst + lane] = v;
        }
    }
}

}  // namespace sba
