// TEST INFRASTRUCTURE: host build (g++) of the header-only model math in csrc/sba_models.cuh so that
// the analytic Jacobians can be checked on a machine without a GPU.  Not part of the product library.
#include "../../sat_bundleadjust_b200/csrc/sba_models.cuh"
#include "../../sat_bundleadjust_b200/csrc/sba_tr2d.h"
#include "../../sat_bundleadjust_b200/csrc/sba_index.h"
#include "../../sat_bundleadjust_b200/csrc/sba_pattern.h"

using namespace sba;

template <int MODEL, int NC>
static void run(const double* camrec, const double* rpc, const double* X, double* uv, double* Jc, double* Jp)
{
    CamRec c = load_camrec(camrec);
    project_jac<MODEL, NC>(c, rpc, X[0], X[1], X[2], uv[0], uv[1], Jc, Jp);
}

extern "C" {

// camrec: prepared record (cos/sin + params); returns 0 on success
int hh_project(int model, const double* camrec, const double* rpc, const double* X, double* uv)
{
    CamRec c = load_camrec(camrec);
    if (model == MODEL_PERSPECTIVE) project<MODEL_PERSPECTIVE>(c, rpc, X[0], X[1], X[2], uv[0], uv[1]);
    else if (model == MODEL_AFFINE) project<MODEL_AFFINE>(c, rpc, X[0], X[1], X[2], uv[0], uv[1]);
    else project<MODEL_RPC>(c, rpc, X[0], X[1], X[2], uv[0], uv[1]);
    return 0;
}

int hh_project_jac(int model, int nc, const double* camrec, const double* rpc, const double* X,
                   double* uv, double* Jc, double* Jp)
{
#define CASE(M, N) if (model == M && nc == N) { run<M, N>(camrec, rpc, X, uv, Jc, Jp); return 0; }
    CASE(MODEL_PERSPECTIVE, 3) CASE(MODEL_PERSPECTIVE, 6) CASE(MODEL_PERSPECTIVE, 11)
    CASE(MODEL_AFFINE, 3) CASE(MODEL_AFFINE, 5) CASE(MODEL_AFFINE, 8)
    CASE(MODEL_RPC, 3) CASE(MODEL_RPC, 6)
#undef CASE
    return 1;
}

// v: full camera parameter vector; builds the prepared record the kernels use
void hh_build_camrec(const double* v, int model, double* rec) { build_camrec(v, model, rec); }

int hh_point_side(int model, const double* rec, const double* rpc, const double* X, double* uv, double* Jp)
{
    if (model == MODEL_PERSPECTIVE) point_side<MODEL_PERSPECTIVE>(rec, rpc, X[0], X[1], X[2], uv[0], uv[1], Jp);
    else if (model == MODEL_AFFINE) point_side<MODEL_AFFINE>(rec, rpc, X[0], X[1], X[2], uv[0], uv[1], Jp);
    else point_side<MODEL_RPC>(rec, rpc, X[0], X[1], X[2], uv[0], uv[1], Jp);
    return 0;
}

int hh_full_side(int model, int nc, const double* rec, const double* rpc, const double* X, double* uv, double* Jc,
                 double* Jp)
{
#define CASE(M, N) if (model == M && nc == N) { full_side<M, N, true>(rec, rpc, X[0], X[1], X[2], uv[0], uv[1], Jc, Jp); return 0; }
    CASE(MODEL_PERSPECTIVE, 3) CASE(MODEL_PERSPECTIVE, 6) CASE(MODEL_PERSPECTIVE, 11)
    CASE(MODEL_AFFINE, 3) CASE(MODEL_AFFINE, 5) CASE(MODEL_AFFINE, 8)
    CASE(MODEL_RPC, 3) CASE(MODEL_RPC, 6)
#undef CASE
    return 1;
}

double hh_loss_rescale(int loss, double f_scale, double f, double* f_out, double* cost)
{
    double s = loss_rescale(loss, f_scale, f, *cost);
    *f_out = f;
    return s;
}

int hh_tr2d(const double* B, const double* g, double Delta, double* p)
{
    return solve_trust_region_2d(B[0], B[1], B[3], g[0], g[1], Delta, p) ? 1 : 0;
}

// one evaluated trial point (csrc/sba_tr2d.h tr_outcome): returns the termination code, -1 for none
int hh_tr_outcome(double cost, double cost_new, double predicted, double step_h_norm, double step_norm, double x_norm,
                  double Delta, double ftol, double xtol, double* Delta_out, int* accept)
{
    const TrOutcome r = tr_outcome(cost, cost_new, predicted, step_h_norm, step_norm, x_norm, Delta, ftol, xtol);
    *Delta_out = r.Delta;
    *accept = r.accept ? 1 : 0;
    return r.status;
}

// host index construction of a problem (csrc/sba_index.h): sizes first (pass NULL outputs), then the arrays
int hh_host_index(const long long* cam_ind, const long long* pts_ind, long long K, int M, int N, int chunk, int max_threads,
                  int* sizes /* [n_chunks, n_tiles+1] */, int* cam, int* pts, int* track_ptr, int* cam_cnt, int* cm_obs,
                  int* ch_cam, int* ch_beg, int* ch_end, int* first_chunk, int* tile_obs)
{
    HostIndex h;
    const int rc = build_host_index((const int64_t*)cam_ind, (const int64_t*)pts_ind, K, M, N, chunk, max_threads, h);
    if (rc) return rc;
    sizes[0] = (int)h.ch_cam.size(); sizes[1] = (int)h.tile_obs.size();
    if (!cam) return 0;
    std::copy(h.cam.begin(), h.cam.end(), cam); std::copy(h.pts.begin(), h.pts.end(), pts);
    std::copy(h.track_ptr.begin(), h.track_ptr.end(), track_ptr); std::copy(h.cam_cnt.begin(), h.cam_cnt.end(), cam_cnt);
    std::copy(h.cm_obs.begin(), h.cm_obs.end(), cm_obs);
    std::copy(h.ch_cam.begin(), h.ch_cam.end(), ch_cam); std::copy(h.ch_beg.begin(), h.ch_beg.end(), ch_beg);
    std::copy(h.ch_end.begin(), h.ch_end.end(), ch_end); std::copy(h.first_chunk.begin(), h.first_chunk.end(), first_chunk);
    std::copy(h.tile_obs.begin(), h.tile_obs.end(), tile_obs);
    return 0;
}


// pattern-major layout (csrc/sba_pattern.h): sizes first (NULL outputs), then the arrays.
// sizes = [ok, n_units, 0, n_frozen_tracks, n_tiles, n_runs]; units (of the `warps`-wide assignment) as 8 ints each
int hh_pattern_layout(const int* cam, const int* track_ptr, long long K, int M, int N, int n_pts_fix, int n_cta, int warps,
                      int* sizes, int* trk_new2old, int* obs_new2old, int* track_ptr_new, int* units, int* warp_unit0)
{
    PatternLayout L;
    build_pattern_layout(cam, track_ptr, K, M, N, n_pts_fix, n_cta, warps + 8, warps, std::max(1, warps - 4), 6, 3, L);
    sizes[0] = L.ok ? 1 : 0; sizes[1] = (int)L.wide.units.size(); sizes[2] = 0; sizes[3] = L.n_frozen_tracks;
    sizes[4] = (int)L.n_tiles; sizes[5] = L.n_runs; sizes[6] = (int)(1000.0 * L.fill);
    if (!L.ok || !trk_new2old) return 0;
    std::copy(L.trk_new2old.begin(), L.trk_new2old.end(), trk_new2old);
    for (int t = 0; t < N; ++t)          // the observation permutation the device derives (k_pt_build_obs)
        for (int k = 0, a0 = track_ptr[L.trk_new2old[t]], b0 = L.track_ptr[t]; k < L.track_ptr[t + 1] - b0; ++k) obs_new2old[b0 + k] = a0 + k;
    std::copy(L.track_ptr.begin(), L.track_ptr.end(), track_ptr_new);
    static_assert(sizeof(PUnit) == 8 * sizeof(int), "PUnit layout");
    std::copy((const int*)L.wide.units.data(), (const int*)L.wide.units.data() + 8 * L.wide.units.size(), units);
    std::copy(L.wide.warp_unit0.begin(), L.wide.warp_unit0.end(), warp_unit0);
    return 0;
}


// units of one kernel shape (which: 0 light, 1 wide, 2 narrow) for explicit warp counts; returns the number of units
int hh_pattern_assignment(const int* cam, const int* track_ptr, long long K, int M, int N, int n_pts_fix, int n_cta, int w_light, int w_wide,
                          int w_narrow, int nc, int rows_per_task, int which, int* units, int max_units, int* warp_unit0)
{
    PatternLayout L;
    build_pattern_layout(cam, track_ptr, K, M, N, n_pts_fix, n_cta, w_light, w_wide, w_narrow, nc, rows_per_task, L);
    if (!L.ok) return -1;
    const PatternAssignment& A = which == 0 ? L.light : (which == 1 ? L.wide : L.narrow);
    if ((int)A.units.size() > max_units) return -2;
    std::copy((const int*)A.units.data(), (const int*)A.units.data() + 8 * A.units.size(), units);
    std::copy(A.warp_unit0.begin(), A.warp_unit0.end(), warp_unit0);
    return (int)A.units.size();
}

int hh_tile_cost(int L, int nc, int rows_per_task, int kind) { return pattern_tile_cost(L, nc, rows_per_task, kind); }
int hh_unit_cost(int kind, int rows_per_task) { return pattern_unit_cost(kind, rows_per_task); }

}
