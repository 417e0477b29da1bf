// Gaussian priors on the camera variables (sba_problem_set_camera_prior): per camera j a mean mu_j and a symmetric positive
// semi-definite information matrix L_j (n_params x n_params), which add
//     0.5 sum_j (x_j - mu_j)^T L_j (x_j - mu_j)
// to the cost.  This is scipy's least_squares on the augmented residual [r ; C_j (x_j - mu_j)] with L_j = C_j^T C_j and the
// robust loss on the observation rows only, so every camera-side quantity of the iteration gets one prior term:
//     U_j += L_j,  g_c,j += L_j (x_j - mu_j),  cost += 0.5 d^T L d,  |J v|^2 += v_c^T L v_c (and the cross terms).
// The term is added once, by rank 0, before the multi-GPU exchange of the quantity it belongs to, so the ranks stay
// bit-identical.  A zero L adds exact zeros.  Frozen cameras' blocks are stored as zeros.
//
// The device functions below are the per-camera quadratic forms both engines share (the pattern engine calls them inside
// k_pt_reduce_assemble, k_pt_jvp1 and k_pt_backsub); the kernels are the generic engine's, launched only when a prior is set.
// Included by sba_ba.cu only.
#pragma once
#include "sba_kernels.cuh"

namespace sba {

// info == nullptr: no prior (or a rank other than 0, which adds nothing)
struct CamPrior {
    const double* mean;       // (M * nc): the params_opt camera layout
    const double* info;       // (M, nc, nc), symmetric; frozen cameras' blocks 0
};

// (L_j (x_j - mu_j))_r
__device__ __forceinline__ double prior_grad_row(CamPrior pr, int j, int r, int nc, const double* __restrict__ x)
{
    const double* L = pr.info + ((size_t)j * nc + r) * nc;
    const double* m = pr.mean + (size_t)j * nc;
    const double* xj = x + (size_t)j * nc;
    double s = 0.0;
    for (int c = 0; c < nc; ++c) s = fma(L[c], xj[c] - m[c], s);
    return s;
}

// a_j^T L_j b_j (a, b: camera vectors of ns entries)
__device__ __forceinline__ double prior_form(CamPrior pr, int j, int nc, const double* a, const double* b)
{
    const double* L = pr.info + (size_t)j * nc * nc;
    const double* aj = a + (size_t)j * nc;
    const double* bj = b + (size_t)j * nc;
    double s = 0.0;
    for (int r = 0; r < nc; ++r) {
        double t = 0.0;
        for (int c = 0; c < nc; ++c) t = fma(L[r * nc + c], bj[c], t);
        s = fma(aj[r], t, s);
    }
    return s;
}

// (sum_e a_e (L b)_e, sum_e b_e (L b)_e) over this thread's camera slots e = threadIdx.x, + blockDim.x, ... < ns: its share of
// a^T L b and b^T L b.  Out of line, so that the register allocation of the tile loops of the calling kernels stays as it is.
__device__ __noinline__ double2 prior_forms_rows(CamPrior pr, int ns, int nc, const double* a, const double* b)
{
    double sa = 0.0, sb = 0.0;
    for (int e = threadIdx.x; e < ns; e += blockDim.x) {
        const double* L = pr.info + (size_t)e * nc;
        const double* bj = b + (size_t)(e / nc) * nc;
        double t = 0.0;
        for (int c = 0; c < nc; ++c) t = fma(L[c], bj[c], t);
        sa = fma(a[e], t, sa);
        sb = fma(b[e], t, sb);
    }
    return make_double2(sa, sb);
}

// 0.5 (x_j - mu_j)^T L_j (x_j - mu_j)
__device__ __forceinline__ double prior_cost_cam(CamPrior pr, int j, int nc, const double* __restrict__ x)
{
    const double* L = pr.info + (size_t)j * nc * nc;
    const double* m = pr.mean + (size_t)j * nc;
    const double* xj = x + (size_t)j * nc;
    double s = 0.0;
    for (int r = 0; r < nc; ++r) {
        double t = 0.0;
        for (int c = 0; c < nc; ++c) t = fma(L[r * nc + c], xj[c] - m[c], t);
        s = fma(xj[r] - m[r], t, s);
    }
    return 0.5 * s;
}

// sum over the cameras of prior_cost_cam, by the 32 lanes of one warp in a fixed order (result in every lane)
__device__ __forceinline__ double prior_cost_warp(CamPrior pr, int M, int nc, const double* __restrict__ x)
{
    double s = 0.0;
    for (int j = threadIdx.x & 31; j < M; j += 32) s += prior_cost_cam(pr, j, nc, x);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

// ---- generic engine ------------------------------------------------------------------------------------------------------
// camsys = [U (M, nc, nc) | g_c (M nc)] of this rank, after k_reduce_cameras: U_j += L_j, g_c,j += L_j (x_j - mu_j).
// One thread per camera slot (j, r): row r of U_j and g_c,j[r].
__global__ void __launch_bounds__(256)
k_prior_cameras(CamPrior pr, const double* __restrict__ x, int M, int nc, double* __restrict__ camsys)
{
    const int ns = M * nc;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < ns; e += gridDim.x * blockDim.x) {
        const int j = e / nc, r = e - j * nc;
        double* U = camsys + (size_t)j * nc * nc + (size_t)r * nc;
        const double* L = pr.info + (size_t)e * nc;
        for (int c = 0; c < nc; ++c) U[c] += L[c];
        camsys[(size_t)M * nc * nc + e] += prior_grad_row(pr, j, r, nc, x);
    }
}

// Scalar prior terms, one CTA of 256 threads, fixed summation order; a slot < 0 is skipped:
//   scal[s_cost] += 0.5 sum_j (x_j - mu_j)^T L_j (x_j - mu_j)           (x camera part; x may be null when s_cost < 0)
//   scal[s11] += v1^T L v1,  scal[s12] += v1^T L v2,  scal[s22] += v2^T L v2    (camera parts of v1, v2)
__global__ void __launch_bounds__(256)
k_prior_scalars(CamPrior pr, int M, int nc, const double* __restrict__ x, int s_cost, const double* __restrict__ v1,
                const double* __restrict__ v2, int s11, int s12, int s22, double* scal)
{
    __shared__ double sm[4 * (256 / 32)];
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
        if (s_cost >= 0) a0 += prior_cost_cam(pr, j, nc, x);
        if (s11 >= 0) a1 += prior_form(pr, j, nc, v1, v1);
        if (s12 >= 0) a2 += prior_form(pr, j, nc, v1, v2);
        if (s22 >= 0) a3 += prior_form(pr, j, nc, v2, v2);
    }
    double acc[4] = {a0, a1, a2, a3};
    const double tot = block_reduce_sum<4, 256>(acc, sm);
    const int slot = threadIdx.x == 0 ? s_cost : threadIdx.x == 1 ? s11 : threadIdx.x == 2 ? s12 : threadIdx.x == 3 ? s22 : -1;
    if (threadIdx.x < 4 && slot >= 0) scal[slot] += tot;
}

}  // namespace sba
