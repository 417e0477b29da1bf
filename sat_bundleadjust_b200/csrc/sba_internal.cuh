// Internal declarations shared by the translation units of libsba_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/sba_b200.h"
#include "sba_models.cuh"

namespace sba {

void set_error(const std::string& msg);

#define SBA_CUDA(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            ::sba::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + ":" + \
                             std::to_string(__LINE__) + ")");                                       \
            return SBA_E_CUDA;                                                                      \
        }                                                                                           \
    } while (0)

#define SBA_TRY(expr)                \
    do {                             \
        int _r = (expr);             \
        if (_r != SBA_OK) return _r; \
    } while (0)

constexpr int NUM_SMS = 148;   // B200

// ---- scalar block (device, mirrored to pinned host memory) --------------------------------------
// Grouped so that every multi-GPU exchange is one contiguous SUM all-reduce.
enum Scal {
    // group A (SUM over ranks): after assembly + scale update + first J*v
    SC_COST = 0,          // 0.5 sum rho at x (assembly pass)
    SC_GG,                // |g_h|^2
    SC_XS,                // |x * scale_inv|^2
    SC_XX,                // |x|^2
    SC_A,                 // |J_h g_h|^2
    SC_GMAX_SLOTS,        // max |g|, one slot per rank (16 slots), combined on the host
    // group B
    SC_GGN = SC_GMAX_SLOTS + 16,   // g_h . gn_h
    SC_DD,                // |gn_h|^2
    // group C: second basis vector t2 = delta - alpha t1
    SC_WW, SC_WG, SC_T11, SC_T12, SC_T22,
    // group C' (only the explicit J*[t1 t2] pass)
    SC_B11, SC_B12, SC_B22,
    // group D
    SC_COST_NEW,
    // local diagnostics (never reduced)
    SC_BAD_POINTS,        // points whose damped 3x3 block was not positive definite
    SC_CHOL_FAIL,         // reduced camera system factorisation failed (pivot index + 1)
    SC_SCRATCH,
    // device-side control (single-thread kernels; identical on every rank because their inputs are all-reduced)
    SC_DELTA,             // trust-region radius in use
    SC_REG,               // damping of the Gauss-Newton system
    SC_C1, SC_C2,         // step = c1 t1 + c2 t2
    SC_PRED,              // predicted reduction of the 2-D model
    SC_STEPH,             // |step_h| (scaled space)
    SC_STEPN,             // |step|   (x space)
    SC_COMM_FAIL,         // a peer did not arrive within the time-out of the peer-memory all-reduce
    // pattern engine, group P (SUM over ranks): Gram scalars of the pair {t1 = D^-2 g, delta = Gauss-Newton step}
    SC_P_GD,              // g . delta            (= g_h . gn_h)
    SC_P_DD,              // |D delta|^2          (= |gn_h|^2)
    SC_P_C12,             // (J t1) . (J delta)
    SC_P_C22,             // |J delta|^2
    SC_P_T11,             // |t1|^2
    SC_P_T1D,             // t1 . delta
    SC_P_TDD,             // |delta|^2
    // pattern engine, device-side control: step = pa t1 + pb delta
    SC_PA, SC_PB,
    SC_COUNT
};
constexpr int H_SCAL_COUNT = SC_COUNT + 8;      // pinned host mirror: the scalar block + the CG state of the PCG path

struct ChunkTable {          // camera-major work items
    int n = 0;
    int* cam = nullptr;      // device
    int* beg = nullptr;
    int* end = nullptr;
    std::vector<int> h_cam, h_first_of_cam;   // host: chunk -> camera ; camera -> first chunk (size M+1)
};

}  // namespace sba

struct sba_problem {
    // description
    int model = 0, M = 0, N = 0, nc = 0, P = 0, n_cam_fix = 0, n_pts_fix = 0, rpc_f32 = 0;
    int64_t K = 0;
    int64_t n = 0;           // number of variables
    int rank = 0, world = 1;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;          // side stream: the camera-major half of the assembly overlaps the track-major half
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    sba_allreduce_fn allreduce = nullptr;
    void* allreduce_user = nullptr;

    // static device data, track-major (the reference's observation order)
    int *cam_ind = nullptr, *pts_ind = nullptr, *track_ptr = nullptr;
    double *pts2d = nullptr, *w = nullptr, *cam_static = nullptr, *rpc_tab = nullptr;
    // static device data, camera-major copy
    int *cm_obs = nullptr, *cm_pts = nullptr, *cam_ptr = nullptr, *obs_of = nullptr;
    double *cm_pts2d = nullptr, *cm_w = nullptr;
    sba::ChunkTable chunks;
    int n_schur_items = 0;   // (chunk, partner camera) partial slots
    int *item_base = nullptr;                                  // device: first slot of every chunk (n_chunks + 1)
    int *item_chunk = nullptr;                                 // device: slot -> chunk
    int *sb_j = nullptr, *sb_jp = nullptr, *sb_first = nullptr; // device: (j,j') blocks and their first slice
    int *pairs = nullptr;                                      // device: int2 (a, b) observation pairs, block-major
    int *slice_block = nullptr, *slice_p0 = nullptr, *slice_p1 = nullptr;   // device: <= SLICE pairs of one block each
    long long n_pairs = 0;
    int *tile_obs = nullptr;                                   // device: warp-tile observation offsets (n_tiles + 1)
    int n_tiles = 0;
    int n_schur_blocks = 0;

    // iteration state (device)
    double *x = nullptr, *x_new = nullptr, *g = nullptr, *sinv = nullptr, *delta = nullptr, *t1 = nullptr, *t2 = nullptr;
    double *camrec = nullptr, *camrec_new = nullptr;
    double *V = nullptr, *F = nullptr, *q = nullptr, *Z = nullptr;
    double *camsys_local = nullptr, *camsys = nullptr;     // [U (M*nc*nc) | g_c (M*nc)]
    double *S = nullptr;                                   // [S (ns*ns) | rhs (ns)], ns = M*nc
    bool comm_split = false;                               // two-launch all-reduce (push, pull) instead of the fused kernel
    int n_common = 0;                                      // COMMON_K: trailing per-camera variables shared by all cameras
    double *cvec = nullptr;                                // 3 * ns: camera parts of delta, t1, t2 with the shared slots expanded
    double *chol_work = nullptr;                           // 34*(ns+32) scratch of the blocked factorisation
    double *cam_partials = nullptr, *schur_partials = nullptr, *red_partials = nullptr;
    unsigned* counters = nullptr;
    double* scal = nullptr;          // device scalar block
    double* h_scal = nullptr;        // pinned host mirror
    double* r_out = nullptr;         // (2K) residual output buffer
    double* err_out = nullptr;       // (K) per-observation reprojection errors (sba_solve_errors)
    double *io_x = nullptr;          // (n) staging for host-pointer entry points
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int launches = 0;
    // measurement: event ring for per-phase timing, scratch for L2 flushes
    std::vector<cudaEvent_t> ev_pool;
    int ev_used = 0;
    // peer-memory all-reduce (multi-GPU): own symmetric buffer + mapped peer buffers
    void* comm_buf = nullptr;
    void* comm_peer[16] = {nullptr};
    long long comm_cap = 0;                  // doubles per parity
    unsigned long long comm_seq = 0;
    bool comm_ready = false;
    std::vector<void*> arena_chunks;         // device slabs owned by this problem
    std::vector<size_t> arena_chunk_bytes;
    char* arena_ptr = nullptr;
    size_t arena_left = 0;
    void* flush_buf = nullptr;
    size_t flush_bytes = 0;

    // ---- G5: matrix-free PCG on the reduced camera system (csrc/sba_pcg.cuh), generic engine only ----
    bool use_pcg = false;
    double pcg_tol = 1e-8;
    int pcg_max_it = 500;
    long long pcg_iterations = 0, pcg_solves = 0;       // totals of the last solve (diagnostics)
    double *pcg_vec = nullptr, *pcg_diag = nullptr, *pcg_L = nullptr, *pcg_w = nullptr, *pcg_s = nullptr;

    // ---- pattern engine (csrc/sba_pattern.h): internal track order = tracks grouped by visibility pattern ----
    int engine = 0;                                      // 0: generic (pair lists), 1: pattern-major
    int n_pts_fix_int = 0;                               // frozen tracks in the internal order: tracks [0, n_pts_fix_int)
    std::vector<int> h_trk_new2old, h_obs_new2old;       // host copies (test-only entry points un-permute on the host)
    int *trk_new2old = nullptr, *obs_new2old = nullptr;  // device
    void* pt_units[3] = {nullptr, nullptr, nullptr};                // device PUnit[]: assignments for the three CTA shapes
    int* pt_warp_unit0[3] = {nullptr, nullptr, nullptr};
    int pt_n_cta = 0;
    double *V2 = nullptr, *g2 = nullptr, *camsys2 = nullptr;        // second buffer set (trial point)
    long long* pt_cycles = nullptr;                                 // SBA_PT_CYCLES=1: per-warp clocks of the last launch of each kernel shape (3 x 148 x 32)
    bool pt_obs_uploaded = false;                                   // observations / weights already uploaded to r_out / err_out by the helper thread of problem creation
    bool pt_schur_mma = false;                                      // K3 variant (SBA_PT_SCHUR=mma): FP64 tensor-core Gram tiles instead of the DFMA task kernel -- measured slower, kept as a switch
    double *dsq = nullptr, *idsq = nullptr;                         // (n) squared column scales of the points and their reciprocals
    double *dsqc = nullptr, *dsqc2 = nullptr, *idsqc = nullptr, *idsqc2 = nullptr;   // (ns) the same for the cameras, double-buffered
    double *pt_partials = nullptr;                                  // per-CTA partial sums, [value][cta]
    double *osc = nullptr, *osc2 = nullptr;                         // (2K) per-observation robust row scales at the current / trial point
    double *pt_records = nullptr;                                   // Schur records, one per (unit, pass)
    double *r_int = nullptr, *e_int = nullptr;                      // (2K), (K) residuals / errors in internal order

    // ---- Gaussian prior on the camera variables (sba_problem_set_camera_prior, sba_prior.cuh), allocated on first use ----
    bool has_prior = false;
    double *prior_mean = nullptr, *prior_info = nullptr;           // (M nc), (M, nc, nc) symmetrised; frozen cameras' blocks 0
    long long prior_rank_sum = 0;                                   // sum over the free cameras of rank(L_j): degrees of freedom it adds

    // ---- posterior covariance (sba_covariance), allocated by its first call ----
    double *cov_cam = nullptr, *cov_pts = nullptr;                  // (ns x ns) s2 S^-1, (N, 6) point blocks in the caller's order
    double *cov_diag = nullptr;                                     // pivot test: min ratio, rejected slot, its ratio; bad points
    int* cov_tile_obs = nullptr;                                    // pattern engine: warp tiles of the point pass (internal order)
    int cov_n_tiles = 0;
    cudaEvent_t cov_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    double cov_ms[4] = {0.0, 0.0, 0.0, 0.0};                        // device time of the phases of the last call
};
