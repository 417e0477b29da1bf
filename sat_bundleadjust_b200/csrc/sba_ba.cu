// Host side of the bundle-adjustment hot path: problem set-up, kernel launches and the
// trust-region (Levenberg-Marquardt type) iteration.
//
// The iteration reproduces scipy's `trf_no_bounds` (scipy/optimize/_lsq/trf.py:415-587), which is what
// the reference runs through scipy.optimize.least_squares (bundle_adjust/ba_core.py:284-297), with two
// changes: the Jacobian is analytic instead of 2-point finite differences, and the regularised
// Gauss-Newton step  (J_h^T J_h + reg I) p = -g_h  is solved exactly through the Schur complement onto the
// cameras + dense Cholesky instead of LSMR.  Everything else keeps scipy's definitions:
//   * variables scaled by D = diag(max-so-far column norm of J)  (x_scale='jac', common.py:598-610)
//   * damping  reg = -min_t q(-t g_h) / Delta^2  from the Cauchy step            (trf.py:485-490)
//   * step from the exact 2-D trust-region problem in span{g_h, gn_h}           (trf.py:496-509)
//   * Delta <- 0.25 |step| if ratio < 0.25 ; Delta <- 2 Delta if ratio > 0.75 and the step hit the
//     boundary (common.py:222-245); initial Delta = |x0 * scale_inv|             (trf.py:443)
//   * termination: dF < ftol F with ratio > 0.25 | |dx| < xtol (xtol + |x|) | |g|_inf < gtol |
//     nfev == max_nfev                                                           (common.py:705-717)
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "sba_comm.cuh"
#include "sba_cov.cuh"
#include "sba_index.h"
#include "sba_kernels.cuh"
#include "sba_pattern.cuh"
#include "sba_pcg.cuh"
#include "sba_tr2d.h"

namespace sba {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }
int launch_cholesky_solve(double* A_dev, double* b_dev, double* x_dev, int n, double* fail_dev, double* work_dev,
                          cudaStream_t stream, bool write_factor);

static inline int grid_for(long long work, int threads, int max_blocks)
{
    long long b = (work + threads - 1) / threads;
    if (b < 1) b = 1;
    if (b > max_blocks) b = max_blocks;
    return (int)b;
}

// Device memory of a problem comes from a few large slabs (cudaMalloc / cudaFree of ~50 separate buffers was
// measured at up to 0.8 s per problem on a busy box); 256-byte aligned bump allocation, freed all at once.
// Slabs of destroyed problems are kept in a process-wide pool (up to SLAB_POOL_MAX bytes) and handed to the next
// problem: the pipeline solves twice per run (before / after outlier removal) and cudaFree + cudaMalloc of the same
// ~0.5 GB cost 5-25 ms per solve.  sba_release_cached_memory() empties the pool.
struct Slab { void* ptr; size_t bytes; int device; };
static std::mutex g_pool_mutex;
static std::vector<Slab> g_slab_pool;
static std::vector<double*> g_pinned_pool;          // pinned scalar blocks (SC_COUNT doubles)
static size_t g_pool_bytes = 0;

// Symmetric exchange buffer of the multi-GPU solve: one per process, kept (with its CUDA IPC mappings of the peers' buffers)
// across problems -- opening the handles costs ~15 ms per call, more than a third of a solve at the bench size.
struct CommGlobal {
    void* buf = nullptr;
    void* peer[16] = {nullptr};
    long long cap = 0;                 // doubles per parity
    unsigned long long seq = 0;        // exchange counter, the same on every rank
    int world = 0, rank = -1, device = -1;
    bool ready = false;
};
static CommGlobal g_comm;
static void comm_release()
{
    if (!g_comm.buf) return;
    for (int r = 0; r < g_comm.world; ++r)
        if (g_comm.ready && r != g_comm.rank && g_comm.peer[r]) cudaIpcCloseMemHandle(g_comm.peer[r]);
    cudaFree(g_comm.buf);
    g_comm = CommGlobal();
}
static long long comm_needed(const sba_problem* p)
{
    const long long ns = (long long)p->M * p->nc;
    const long long dense = p->use_pcg ? 0 : ns * ns + ns;
    return std::max<long long>({dense, ns * p->nc + ns + 1, (long long)p->M * (p->nc * (p->nc + 1) / 2 + p->nc), (long long)SC_COUNT, 1LL << 16});
}
constexpr size_t SLAB_POOL_MAX = (size_t)16 << 30;

static void* pool_take(size_t want, int device, size_t* got)
{
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    int best = -1;
    for (int i = 0; i < (int)g_slab_pool.size(); ++i) {
        const Slab& c = g_slab_pool[i];
        if (c.device != device || c.bytes < want || c.bytes > 2 * want + ((size_t)64 << 20)) continue;
        if (best < 0 || c.bytes < g_slab_pool[best].bytes) best = i;
    }
    if (best < 0) return nullptr;
    const Slab c = g_slab_pool[best];
    g_slab_pool.erase(g_slab_pool.begin() + best);
    g_pool_bytes -= c.bytes;
    *got = c.bytes;
    return c.ptr;
}

static void pool_give(void* ptr, size_t bytes, int device)
{
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        if (g_pool_bytes + bytes <= SLAB_POOL_MAX) {
            g_slab_pool.push_back({ptr, bytes, device});
            g_pool_bytes += bytes;
            return;
        }
    }
    cudaFree(ptr);
}

static int arena_alloc(sba_problem* p, void** ptr, size_t bytes)
{
    constexpr size_t ALIGN = 256, CHUNK_BYTES = 64u << 20;
    bytes = (bytes + ALIGN - 1) / ALIGN * ALIGN;
    if (bytes == 0) bytes = ALIGN;
    if (bytes > p->arena_left) {
        size_t want = bytes > CHUNK_BYTES ? bytes : CHUNK_BYTES;
        void* chunk = pool_take(want, p->device, &want);
        if (!chunk) SBA_CUDA(cudaMalloc(&chunk, want));
        p->arena_chunks.push_back(chunk);
        p->arena_chunk_bytes.push_back(want);
        if (bytes >= CHUNK_BYTES) { *ptr = chunk; return SBA_OK; }     // dedicated slab, keep the open chunk
        p->arena_ptr = (char*)chunk;
        p->arena_left = want;
    }
    *ptr = p->arena_ptr;
    p->arena_ptr += bytes;
    p->arena_left -= bytes;
    return SBA_OK;
}

template <typename T>
static int dev_alloc(sba_problem* p, T** ptr, size_t count)
{
    *ptr = nullptr;
    return arena_alloc(p, (void**)ptr, count * sizeof(T));
}

template <typename T>
static int dev_upload(sba_problem* p, T** ptr, const std::vector<T>& h, cudaStream_t s)
{
    SBA_TRY(dev_alloc(p, ptr, h.size()));
    if (!h.empty()) SBA_CUDA(cudaMemcpyAsync(*ptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
    return SBA_OK;
}

static bool valid_nc(int model, int nc)
{
    if (model == MODEL_PERSPECTIVE) return nc == 3 || nc == 6 || nc == 11;
    if (model == MODEL_AFFINE) return nc == 3 || nc == 5 || nc == 8;
    if (model == MODEL_RPC) return nc == 3 || nc == 6;
    return false;
}

#define SBA_DISPATCH(p, MACRO)                                                          \
    switch ((p)->model * 16 + (p)->nc) {                                                \
    case MODEL_PERSPECTIVE * 16 + 3: MACRO(MODEL_PERSPECTIVE, 3); break;                \
    case MODEL_PERSPECTIVE * 16 + 6: MACRO(MODEL_PERSPECTIVE, 6); break;                \
    case MODEL_PERSPECTIVE * 16 + 11: MACRO(MODEL_PERSPECTIVE, 11); break;              \
    case MODEL_AFFINE * 16 + 3: MACRO(MODEL_AFFINE, 3); break;                          \
    case MODEL_AFFINE * 16 + 5: MACRO(MODEL_AFFINE, 5); break;                          \
    case MODEL_AFFINE * 16 + 8: MACRO(MODEL_AFFINE, 8); break;                          \
    case MODEL_RPC * 16 + 3: MACRO(MODEL_RPC, 3); break;                                \
    case MODEL_RPC * 16 + 6: MACRO(MODEL_RPC, 6); break;                                \
    default: set_error("unsupported (cam_model, n_params) combination"); return SBA_E_INVALID; \
    }

#define SBA_DISPATCH_MODEL(p, MACRO)                            \
    switch ((p)->model) {                                       \
    case MODEL_PERSPECTIVE: MACRO(MODEL_PERSPECTIVE); break;    \
    case MODEL_AFFINE: MACRO(MODEL_AFFINE); break;              \
    default: MACRO(MODEL_RPC); break;                           \
    }

static ObsArrays obs_arrays(const sba_problem* p)
{
    ObsArrays o;
    o.cam_ind = p->cam_ind; o.pts_ind = p->pts_ind; o.pts2d = (const double2*)p->pts2d; o.w = p->w;
    o.track_ptr = p->track_ptr;
    o.tile_obs = p->tile_obs; o.n_tiles = p->n_tiles;
    return o;
}

static int check_launch(sba_problem* p)
{
    p->launches++;
    SBA_CUDA(cudaGetLastError());
    return SBA_OK;
}

// ---- per-phase / per-iteration device timing (CUDA events on the solver's stream) --------------------
struct PhaseTimer {
    sba_problem* p;
    bool on = false;
    struct Rec { int phase, e0, e1; };
    std::vector<Rec> recs;
    int open_e0 = -1, open_phase = -1;
    int get_event()
    {
        if (p->ev_used == (int)p->ev_pool.size()) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return -1;
            p->ev_pool.push_back(e);
        }
        return p->ev_used++;
    }
    void begin(int phase)
    {
        if (!on) return;
        open_e0 = get_event();
        open_phase = phase;
        if (open_e0 >= 0) cudaEventRecord(p->ev_pool[open_e0], p->stream);
    }
    void end()
    {
        if (!on || open_e0 < 0) return;
        const int e1 = get_event();
        if (e1 >= 0) {
            cudaEventRecord(p->ev_pool[e1], p->stream);
            recs.push_back({open_phase, open_e0, e1});
        }
        open_e0 = -1;
    }
    // phase == -1 marks a whole iteration
    void resolve(sba_solve_info* info)
    {
        for (const Rec& r : recs) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, p->ev_pool[r.e0], p->ev_pool[r.e1]) != cudaSuccess) continue;
            if (r.phase < 0) { info->iter_ms += ms; info->timed_iterations++; }
            else info->phase_ms[r.phase] += ms;
        }
    }
};

// ------------------------------------------------------------------------------------------------
// launches
// ------------------------------------------------------------------------------------------------
static int run_prepare(sba_problem* p, const double* x, double* camrec)
{
    k_prepare_cameras<<<grid_for(p->M, 128, 1 << 20), 128, 0, p->stream>>>(x, p->cam_static, camrec, p->M, p->P, p->nc,
                                                                             p->n_cam_fix, p->n_common, p->model);
    return check_launch(p);
}

static int run_residual(sba_problem* p, const double* x, const double* camrec, int loss, double f_scale, double* r_out,
                        int slot, int rpc_f32)
{
    const int grid = grid_for(p->K, 256, NUM_SMS * 8);
#define L(MODEL)                                                                                                  \
    k_residual<MODEL><<<grid, 256, 0, p->stream>>>(obs_arrays(p), x + (size_t)p->M * p->nc, camrec, p->rpc_tab, p->K, \
                                                   loss, f_scale, rpc_f32, (double2*)r_out, p->red_partials,       \
                                                   p->counters + 0, p->scal, slot)
    SBA_DISPATCH_MODEL(p, L);
#undef L
    return check_launch(p);
}

static int allreduce_any(sba_problem* p, double* buf, long long count);
static CommView comm_view(const sba_problem* p);
static CommFused comm_fused(sba_problem* p, long long count);

// fused residual + analytic Jacobian + robust weighting + block assembly at x (camrec must be prepared).
// The track-major half (V, g_p) runs on the solver's stream, the camera-major half (U, g_c) on a side stream.
static int run_assemble(sba_problem* p, const double* x, const double* camrec, int loss, double f_scale)
{
    const double* xp = x + (size_t)p->M * p->nc;
    SBA_CUDA(cudaEventRecord(p->ev_fork, p->stream));
    SBA_CUDA(cudaStreamWaitEvent(p->stream2, p->ev_fork, 0));
    {
#define L(MODEL, NC)                                                                                                   \
    k_assemble_cameras<MODEL, NC><<<p->chunks.n, TPB, 0, p->stream2>>>(                                               \
        p->chunks.cam, p->chunks.beg, p->chunks.end, p->cm_pts, (const double2*)p->cm_pts2d, p->cm_w, xp, camrec,      \
        p->rpc_tab, p->n_cam_fix, loss, f_scale, p->cam_partials);                                                     \
    SBA_TRY(check_launch(p));                                                                                          \
    k_reduce_cameras<NC><<<p->M, 128, 0, p->stream2>>>(p->cam_partials, p->cam_ptr /* first chunk table */, p->M,      \
                                                       p->camsys_local)
        SBA_DISPATCH(p, L);
#undef L
        SBA_TRY(check_launch(p));
    }
    SBA_CUDA(cudaEventRecord(p->ev_join, p->stream2));
    {
        const int grid = (p->n_tiles + WPB - 1) / WPB;
#define L(MODEL)                                                                                                      \
    k_assemble_points<MODEL><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), xp, camrec, p->rpc_tab, p->n_pts_fix, loss,      \
                                                          f_scale, p->V, p->g + (size_t)p->M * p->nc, p->red_partials,   \
                                                          p->counters + 1, p->scal)
        SBA_DISPATCH_MODEL(p, L);
#undef L
        SBA_TRY(check_launch(p));
    }
    SBA_CUDA(cudaStreamWaitEvent(p->stream, p->ev_join, 0));
    if (p->world > 1) {
        const size_t cnt = (size_t)p->M * p->nc * p->nc + (size_t)p->M * p->nc;
        SBA_CUDA(cudaMemcpyAsync(p->camsys, p->camsys_local, cnt * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
        SBA_TRY(allreduce_any(p, p->camsys, (long long)cnt));
    }
    return SBA_OK;
}

static CommView comm_view(const sba_problem* p)
{
    CommView c;
    for (int r = 0; r < COMM_MAX_RANKS; ++r) { c.data[r] = nullptr; c.flag[r] = nullptr; }
    for (int r = 0; r < p->world; ++r) {
        c.data[r] = (double*)p->comm_peer[r];
        c.flag[r] = (unsigned long long*)((double*)p->comm_peer[r] + 2 * p->comm_cap);
    }
    c.cap = p->comm_cap; c.me = p->rank; c.world = p->world;
    // 60 s by default (SBA_COMM_TIMEOUT_S): ranks make a host round trip per trial step, so ordinary skew (a busy host, first-touch
    // IPC mapping, verbose output) must not be mistaken for a lost peer
    static const double timeout_s = getenv("SBA_COMM_TIMEOUT_S") ? atof(getenv("SBA_COMM_TIMEOUT_S")) : 60.0;
    c.timeout_cycles = (long long)(timeout_s * 1.9e9);
    return c;
}

// Exchange descriptor for a kernel that does its all-reduce of `count` doubles in its own epilogue (cta_allreduce): takes the
// next exchange number when the peer buffers are mapped, the message fits and SBA_COMM_FUSED is not 0; else on == 0 and
// the caller falls back to allreduce_any() after the kernel.
static CommFused comm_fused(sba_problem* p, long long count)
{
    static const bool enabled = !(getenv("SBA_COMM_FUSED") && atoi(getenv("SBA_COMM_FUSED")) == 0);
    CommFused f;
    f.on = 0; f.seq = 0;
    if (p->world > 1 && p->comm_ready && !p->comm_split && enabled && count <= p->comm_cap) {
        f.c = comm_view(p);
        f.seq = ++g_comm.seq;
        f.on = 1;
    } else {
        for (int r = 0; r < COMM_MAX_RANKS; ++r) { f.c.data[r] = nullptr; f.c.flag[r] = nullptr; }
        f.c.cap = 0; f.c.timeout_cycles = 0; f.c.me = 0; f.c.world = 1;
    }
    return f;
}

// SUM all-reduce of `count` doubles at device pointer `buf`, in place, on the solver's stream: peer memory when the
// symmetric buffers are mapped (sba_comm_import), else the caller's hook (NCCL through torch.distributed)
static int allreduce_any(sba_problem* p, double* buf, long long count)
{
    if (p->world <= 1) return SBA_OK;
    if (p->comm_ready && count <= p->comm_cap) {
        const CommView c = comm_view(p);
        const unsigned long long seq = ++g_comm.seq;
        const int grid = grid_for(count, 256, 16);
        if (p->comm_split) {        // SBA_COMM_SPLIT=1: the two-launch form (push, then pull)
            k_comm_push<<<grid, 256, 0, p->stream>>>(c, buf, count, seq, p->counters + 8);
            SBA_TRY(check_launch(p));
            k_comm_pull<<<grid, 256, 0, p->stream>>>(c, buf, count, seq, p->scal);
            return check_launch(p);
        }
        k_comm_allreduce<<<grid, 256, 0, p->stream>>>(c, buf, count, seq, p->counters + 8, p->scal);
        return check_launch(p);
    }
    if (!p->allreduce || p->allreduce(p->allreduce_user, buf, count) != 0) {
        set_error("allreduce callback failed");
        return SBA_E_INVALID;
    }
    return SBA_OK;
}

static int allreduce_scal(sba_problem* p, int first, int count) { return allreduce_any(p, p->scal + first, count); }

static int fetch_scal(sba_problem* p)
{
    SBA_CUDA(cudaMemcpyAsync(p->h_scal, p->scal, SC_COUNT * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

static int run_scale_dots(sba_problem* p, int first)
{
    SBA_CUDA(cudaMemsetAsync(p->scal + SC_GMAX_SLOTS, 0, 16 * sizeof(double), p->stream));
    const int grid = grid_for(p->n, 256, NUM_SMS * 8);
    k_scale_dots<<<grid, 256, 0, p->stream>>>(p->camsys, p->V, p->x, p->g, p->sinv, p->t1, p->n, p->M * p->nc, p->nc, p->M,
                                              p->n_common, first, p->rank == 0, p->rank, p->red_partials, p->counters + 2, p->scal);
    return check_launch(p);
}

static int run_jvp(sba_problem* p, int loss, double f_scale, int nvec, Slots out)
{
    const int grid = grid_for(p->K, TPB, NUM_SMS * 16);
    const int ns = p->M * p->nc;
    const double *v1c = p->t1, *v2c = p->t2;
    if (p->n_common) {       // J acts on per-camera slots: expand the shared ones
        k_expand_common<<<grid_for(ns, 256, 64), 256, 0, p->stream>>>(p->t1, p->cvec + ns, ns, p->nc, p->n_common);
        if (nvec == 2) k_expand_common<<<grid_for(ns, 256, 64), 256, 0, p->stream>>>(p->t2, p->cvec + 2 * ns, ns, p->nc, p->n_common);
        SBA_TRY(check_launch(p));
        v1c = p->cvec + ns; v2c = p->cvec + 2 * ns;
    }
#define L(MODEL, NC)                                                                                                  \
    if (nvec == 1)                                                                                                    \
        k_jvp<MODEL, NC, 1><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), p->x + (size_t)p->M * p->nc, p->camrec,        \
                                                         p->rpc_tab, p->K, p->M * p->nc, p->n_cam_fix, p->n_pts_fix,   \
                                                         loss, f_scale, p->t1, p->t2, v1c, v2c, p->red_partials,       \
                                                         p->counters + 3, p->scal, out);                               \
    else                                                                                                              \
        k_jvp<MODEL, NC, 2><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), p->x + (size_t)p->M * p->nc, p->camrec,        \
                                                         p->rpc_tab, p->K, p->M * p->nc, p->n_cam_fix, p->n_pts_fix,   \
                                                         loss, f_scale, p->t1, p->t2, v1c, v2c, p->red_partials,       \
                                                         p->counters + 3, p->scal, out)
    SBA_DISPATCH(p, L);
#undef L
    return check_launch(p);
}

// G5: the camera step from block-Jacobi PCG on the reduced camera system, matrix-free (sba_pcg.cuh).  Needs Z, F, q of
// k_point_prep.  Tolerance: |r|_{M^-1} <= pcg_tol |r0|_{M^-1}; the trust-region step only uses the result as the second
// direction of its 2-D subspace (scipy solves the same system with LSMR to 1e-6), so an inexact solve costs convergence
// speed, never correctness.
static int run_pcg(sba_problem* p)
{
    const int ns = p->M * p->nc, nc = p->nc;
    const int nv = nc * (nc + 1) / 2 + nc;
    double* cg = p->pcg_vec + 5 * (size_t)ns;
    const int grid_t = (p->n_tiles + WPB - 1) / WPB;
#define PCG_NC(MACRO)                                              \
    switch (nc) {                                                  \
    case 3: MACRO(3); break;                                       \
    case 5: MACRO(5); break;                                       \
    case 6: MACRO(6); break;                                       \
    case 8: MACRO(8); break;                                       \
    default: MACRO(11); break;                                     \
    }
#define L(NC) k_pcg_diag<NC><<<p->chunks.n, TPB, 0, p->stream>>>(p->chunks.beg, p->chunks.end, p->cm_obs, p->cm_pts, p->Z, p->q, p->cam_partials)
    PCG_NC(L);
#undef L
    SBA_TRY(check_launch(p));
    k_pcg_sum<<<p->M, 128, 0, p->stream>>>(p->cam_partials, p->cam_ptr, nv, cg, 0, p->pcg_diag);
    SBA_TRY(check_launch(p));
    SBA_TRY(allreduce_any(p, p->pcg_diag, (long long)p->M * nv));
#define L(NC) k_pcg_init<NC><<<1, 1024, 0, p->stream>>>(p->pcg_diag, p->camsys, p->sinv, p->scal, p->M, p->n_cam_fix, p->pcg_L, p->pcg_vec, p->scal + SC_CHOL_FAIL)
    PCG_NC(L);
#undef L
    SBA_TRY(check_launch(p));
    const int max_it = p->pcg_max_it;
    int it = 0;
    while (it < max_it) {
        const int batch = std::min(8, max_it - it);
        for (int b = 0; b < batch; ++b) {
#define L(NC)                                                                                                                  \
    k_pcg_tracks<NC><<<grid_t, TPB, 0, p->stream>>>(obs_arrays(p), p->Z, p->pcg_vec + 3 * (size_t)ns, cg, p->pcg_s);             \
    k_pcg_cameras<NC><<<p->chunks.n, TPB, 0, p->stream>>>(p->chunks.beg, p->chunks.end, p->cm_obs, p->cm_pts, p->Z, p->pcg_s, cg, \
                                                          p->cam_partials)
            PCG_NC(L);
#undef L
            SBA_TRY(check_launch(p)); p->launches++;
            k_pcg_sum<<<p->M, 128, 0, p->stream>>>(p->cam_partials, p->cam_ptr, nc, cg, 1, p->pcg_w);
            SBA_TRY(check_launch(p));
            SBA_TRY(allreduce_any(p, p->pcg_w, (long long)ns));
#define L(NC) k_pcg_update<NC><<<1, 1024, 0, p->stream>>>(p->pcg_w, p->camsys, p->sinv, p->scal, p->pcg_L, p->M, p->n_cam_fix, p->pcg_tol, max_it, p->pcg_vec)
            PCG_NC(L);
#undef L
            SBA_TRY(check_launch(p));
        }
        it += batch;
        // the host only looks at the flag between batches (converged launches inside a batch return at once)
        SBA_CUDA(cudaMemcpyAsync(p->h_scal + SC_COUNT, cg, PCG_SCAL * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        SBA_CUDA(cudaStreamSynchronize(p->stream));
        if (p->h_scal[SC_COUNT + 2] != 0.0) break;
    }
    p->pcg_iterations += (long long)p->h_scal[SC_COUNT + 3];
    p->pcg_solves += 1;
    SBA_CUDA(cudaMemcpyAsync(p->delta, p->pcg_vec, (size_t)ns * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
#undef PCG_NC
    return SBA_OK;
}

// Schur complement + Cholesky solve + back-substitution for a given damping `reg`
static int run_gauss_newton_step(sba_problem* p, int loss, double f_scale, PhaseTimer& tm, bool stop_after_schur = false)
{
    const int ns = p->M * p->nc;
    const double* xp = p->x + (size_t)ns;
    SBA_CUDA(cudaMemsetAsync(p->scal + SC_BAD_POINTS, 0, 2 * sizeof(double), p->stream));
    tm.begin(SBA_PH_POINT_PREP);
    {
        const int grid = (p->n_tiles + WPB - 1) / WPB;
#define L(MODEL, NC)                                                                                                    \
    k_point_prep<MODEL, NC><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), xp, p->camrec, p->rpc_tab, ns, p->n_cam_fix,       \
                                                         p->n_pts_fix, loss, f_scale, p->V, p->g, p->sinv, p->F,    \
                                                         p->q, p->Z, p->scal)
        SBA_DISPATCH(p, L);
#undef L
        SBA_TRY(check_launch(p));
    }
    tm.end();
    if (p->use_pcg) {
        if (stop_after_schur) { set_error("the reduced camera system is not formed on the PCG path"); return SBA_E_INVALID; }
        tm.begin(SBA_PH_SCHUR);
        SBA_TRY(run_pcg(p));
        tm.end();
    } else {
    tm.begin(SBA_PH_SCHUR);
    {
#define SCHUR_ARGS                                                                                                     \
    p->slice_block, p->slice_p0, p->slice_p1, p->sb_j, p->sb_jp, (const int2*)p->pairs, p->pts_ind, p->Z, p->q,          \
        p->schur_partials
        switch (p->nc) {
        case 3: k_schur<3, 0, 3><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS); break;
        case 5: k_schur<5, 0, 5><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS); break;
        case 6: k_schur<6, 0, 6><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS); break;
        case 8: k_schur<8, 0, 8><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS); break;
        case 11:
            k_schur<11, 0, 6><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS);
            SBA_TRY(check_launch(p));
            k_schur<11, 6, 5><<<p->n_schur_items, TPB, 0, p->stream>>>(SCHUR_ARGS);
            break;
        default: set_error("bad nc"); return SBA_E_INVALID;
        }
        SBA_TRY(check_launch(p));
#undef SCHUR_ARGS
#define FIN_ARGS                                                                                                       \
    p->schur_partials, p->sb_first, p->sb_j, p->sb_jp, p->M, p->n_cam_fix, p->camsys_local, p->sinv, p->scal,           \
        p->rank == 0, p->n_common, p->S
        switch (p->nc) {
        case 3: k_schur_finalize<3><<<p->n_schur_blocks, 256, 0, p->stream>>>(FIN_ARGS); break;
        case 5: k_schur_finalize<5><<<p->n_schur_blocks, 256, 0, p->stream>>>(FIN_ARGS); break;
        case 6: k_schur_finalize<6><<<p->n_schur_blocks, 256, 0, p->stream>>>(FIN_ARGS); break;
        case 8: k_schur_finalize<8><<<p->n_schur_blocks, 256, 0, p->stream>>>(FIN_ARGS); break;
        default: k_schur_finalize<11><<<p->n_schur_blocks, 256, 0, p->stream>>>(FIN_ARGS); break;
        }
        SBA_TRY(check_launch(p));
#undef FIN_ARGS
    }
    SBA_TRY(allreduce_any(p, p->S, (long long)ns * ns + ns));
    if (p->n_common) {
        k_fold_common<<<1, 256, 0, p->stream>>>(p->S, ns, p->nc, p->M, p->n_common);
        SBA_TRY(check_launch(p));
    }
    tm.end();
    if (stop_after_schur) return SBA_OK;
    tm.begin(SBA_PH_CHOLESKY);
    SBA_TRY(launch_cholesky_solve(p->S, p->S + (size_t)ns * ns, p->delta, ns, p->scal + SC_CHOL_FAIL, p->chol_work,
                                  p->stream, false));
    p->launches++;
    tm.end();
    }
    tm.begin(SBA_PH_BACKSUB);
    {
        const int grid = (p->n_tiles + WPB - 1) / WPB;
        const double* dcam = p->delta;
        if (p->n_common) {
            k_expand_common<<<grid_for(ns, 256, 64), 256, 0, p->stream>>>(p->delta, p->cvec, ns, p->nc, p->n_common);
            SBA_TRY(check_launch(p));
            dcam = p->cvec;
        }
        switch (p->nc) {
        case 3: k_backsub<3><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), ns, p->F, p->q, p->Z, dcam, p->delta); break;
        case 5: k_backsub<5><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), ns, p->F, p->q, p->Z, dcam, p->delta); break;
        case 6: k_backsub<6><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), ns, p->F, p->q, p->Z, dcam, p->delta); break;
        case 8: k_backsub<8><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), ns, p->F, p->q, p->Z, dcam, p->delta); break;
        default: k_backsub<11><<<grid, TPB, 0, p->stream>>>(obs_arrays(p), ns, p->F, p->q, p->Z, dcam, p->delta); break;
        }
        SBA_TRY(check_launch(p));
    }
    tm.end();
    return SBA_OK;
}


#include "sba_pattern_host.inl"

// ------------------------------------------------------------------------------------------------
// the iteration: one driver for both engines, which differ only in the launch sequences below
// ------------------------------------------------------------------------------------------------
// state of a fresh solve from the start vector in p->x
static int trf_reset(sba_problem* p)
{
    if (p->engine == 1) return pt_reset_state(p);
    SBA_CUDA(cudaMemsetAsync(p->scal, 0, SC_COUNT * sizeof(double), p->stream));
    return SBA_OK;
}

// the cost at x0 into scal[SC_COST_NEW], by the same kernels as every later trial point
static int trf_cost_x0(sba_problem* p, const sba_solve_opts* o)
{
    if (p->engine == 1) return pt_run_assemble(p, 1, 1, o->loss, o->f_scale);
    SBA_TRY(run_prepare(p, p->x, p->camrec));
    SBA_TRY(run_residual(p, p->x, p->camrec, o->loss, o->f_scale, nullptr, SC_COST_NEW, 0));
    return allreduce_scal(p, SC_COST_NEW, 1);
}

// the blocks at x0 (the pattern engine's cost evaluation has computed them already)
static int trf_blocks_x0(sba_problem* p, const sba_solve_opts* o)
{
    if (p->engine == 1) { pt_accept(p); return SBA_OK; }
    return run_assemble(p, p->x, p->camrec, o->loss, o->f_scale);
}

// everything from the blocks at x to the scalars of the 2-D subproblem, with no host round trip.
// reg_override >= 0: re-damp the system of this iteration with that value
static int trf_step(sba_problem* p, const sba_solve_opts* o, PhaseTimer& tm, bool first, double Delta, double reg_override)
{
    const int loss = o->loss;
    const double fs = o->f_scale;
    const int ns = p->M * p->nc;
    if (p->engine == 1) {
        if (reg_override < 0.0) {
            tm.begin(SBA_PH_SCALE_JVP);
            SBA_TRY(pt_run_jvp1(p, first ? 1 : 0, loss, fs, Delta));       // and the damping
            tm.end();
        } else {
            k_control_reg<<<1, 32, 0, p->stream>>>(p->scal, Delta, reg_override);
            SBA_TRY(check_launch(p));
        }
        tm.begin(SBA_PH_SCHUR);
        SBA_TRY(pt_run_schur(p, loss, fs));
        tm.end();
        tm.begin(SBA_PH_CHOLESKY);
        SBA_TRY(launch_cholesky_solve(p->S, p->S + (size_t)ns * ns, p->delta, ns, p->scal + SC_CHOL_FAIL, p->chol_work, p->stream, false));
        p->launches++;
        tm.end();
        tm.begin(SBA_PH_BACKSUB);
        SBA_TRY(pt_run_backsub(p, loss, fs));
        tm.end();
        return SBA_OK;
    }
    const int elem_grid = grid_for(p->n, 256, NUM_SMS * 8);
    if (reg_override < 0.0) {
        tm.begin(SBA_PH_SCALE_JVP);
        SBA_TRY(run_scale_dots(p, first ? 1 : 0));
        Slots sa; sa.s[0] = SC_A; sa.s[1] = SC_SCRATCH; sa.s[2] = SC_SCRATCH;
        SBA_TRY(run_jvp(p, loss, fs, 1, sa));
        SBA_TRY(allreduce_scal(p, SC_COST, SC_GGN - SC_COST));
        tm.end();
    }
    k_control_reg<<<1, 32, 0, p->stream>>>(p->scal, Delta, reg_override);
    SBA_TRY(check_launch(p));
    SBA_TRY(run_gauss_newton_step(p, loss, fs, tm));
    tm.begin(SBA_PH_SUBSPACE);
    k_dot_g_delta<<<elem_grid, 256, 0, p->stream>>>(p->g, p->sinv, p->delta, p->n, ns, p->rank == 0, p->red_partials,
                                                    p->counters + 4, p->scal);
    SBA_TRY(check_launch(p));
    SBA_TRY(allreduce_scal(p, SC_GGN, 2));
    k_build_t2<<<elem_grid, 256, 0, p->stream>>>(p->g, p->sinv, p->delta, p->t1, p->t2, p->n, ns, p->rank == 0,
                                                 p->red_partials, p->counters + 5, p->scal);
    SBA_TRY(check_launch(p));
    Slots sb; sb.s[0] = SC_B11; sb.s[1] = SC_B12; sb.s[2] = SC_B22;
    SBA_TRY(run_jvp(p, loss, fs, 2, sb));
    SBA_TRY(allreduce_scal(p, SC_WW, 8));      // [ww wg t11 t12 t22 | b11 b12 b22] in one exchange
    tm.end();
    return SBA_OK;
}

// trial point x_new = x + c1 t1 + c2 t2 for radius `radius` (< 0: the one on the device) and its cost into scal[SC_COST_NEW]
static int trf_trial(sba_problem* p, const sba_solve_opts* o, double radius)
{
    if (p->engine == 1) {
        if (radius >= 0.0) {        // else K4 has solved the 2-D subproblem already
            k_pt_control_tr2d<<<1, 32, 0, p->stream>>>(p->scal, radius);
            SBA_TRY(check_launch(p));
        }
        return pt_run_assemble(p, 0, 0, o->loss, o->f_scale);     // K1: the cost, and the blocks should x_new be accepted
    }
    k_control_tr2d<<<1, 32, 0, p->stream>>>(p->scal, radius);
    SBA_TRY(check_launch(p));
    k_step<<<grid_for(p->n, 256, NUM_SMS * 8), 256, 0, p->stream>>>(p->x, p->t1, p->t2, p->scal, p->x_new, p->n, p->cam_static,
                                                                    p->camrec_new, p->M, p->P, p->nc, p->n_cam_fix, p->n_common,
                                                                    p->model);
    SBA_TRY(check_launch(p));
    SBA_TRY(run_residual(p, p->x_new, p->camrec_new, o->loss, o->f_scale, nullptr, SC_COST_NEW, 0));
    return allreduce_scal(p, SC_COST_NEW, 1);
}

// the trial point becomes the current point; its blocks are needed unless the solve terminates
static int trf_accept(sba_problem* p, const sba_solve_opts* o, PhaseTimer& tm, bool terminating, int& njev)
{
    if (p->engine == 1) {
        pt_accept(p);               // the trial evaluation already holds the blocks of the new point
        ++njev;
        return SBA_OK;
    }
    std::swap(p->x, p->x_new);
    std::swap(p->camrec, p->camrec_new);
    if (terminating) return SBA_OK;
    tm.begin(SBA_PH_ASSEMBLE);
    SBA_TRY(run_assemble(p, p->x, p->camrec, o->loss, o->f_scale));
    tm.end();
    ++njev;
    return SBA_OK;
}

static int solve_trf(sba_problem* p, const sba_solve_opts* o, sba_solve_info* info)
{
    std::memset(info, 0, sizeof(*info));
    if (o->max_nfev < 1) { set_error("max_nfev must be >= 1"); return SBA_E_INVALID; }
    p->launches = 0;
    p->pcg_iterations = 0; p->pcg_solves = 0;
    SBA_TRY(trf_reset(p));
    SBA_CUDA(cudaEventRecord(p->ev0, p->stream));
    SBA_TRY(trf_cost_x0(p, o));
    SBA_TRY(fetch_scal(p));
    double cost = p->h_scal[SC_COST_NEW];
    if (!std::isfinite(cost)) { set_error("Residuals are not finite in the initial point."); return SBA_E_NUMERIC; }
    info->cost_init = cost;
    SBA_TRY(trf_blocks_x0(p, o));
    int nfev = 1, njev = 1, iteration = 0, status = -1, chol_retries = 0;
    double Delta = -1.0, g_norm = 0.0;   // Delta < 0: not initialised yet (the device sets |x0 * scale_inv|)
    bool first = true;
    PhaseTimer tm, it_tm;
    tm.p = it_tm.p = p;
    p->ev_used = 0;
    if (o->l2_flush_bytes > 0 && (size_t)o->l2_flush_bytes > p->flush_bytes) {
        if (p->flush_buf) cudaFree(p->flush_buf);
        p->flush_buf = nullptr; p->flush_bytes = 0;
        SBA_CUDA(cudaMalloc(&p->flush_buf, (size_t)o->l2_flush_bytes));
        p->flush_bytes = (size_t)o->l2_flush_bytes;
    }
    // scalars of the 2-D subproblem that are not finite when the damped system had no usable solution
    const int chk0 = p->engine == 1 ? SC_P_GD : SC_GGN, chk1 = p->engine == 1 ? SC_P_C22 : SC_B22;

    auto enqueue_trial = [&](double radius) -> int {
        tm.begin(SBA_PH_STEP_EVAL);
        SBA_TRY(trf_trial(p, o, radius));
        tm.end();
        return SBA_OK;
    };
    // everything from the blocks at x to the first trial point
    auto enqueue_iteration = [&](double reg_override) -> int {
        SBA_TRY(trf_step(p, o, tm, first, Delta, reg_override));
        return enqueue_trial(-1.0);
    };

    while (true) {
        if (o->max_iterations > 0 && iteration >= o->max_iterations) break;
        if (nfev >= o->max_nfev) break;
        it_tm.on = iteration >= o->timed_from && (o->timed_from > 0 || o->l2_flush_bytes > 0 || o->max_iterations > 0);
        tm.on = it_tm.on && !o->no_phase_timing;     // the ~16 extra event records per iteration cost ~1 us each on the stream
        if (o->l2_flush_bytes > 0)
            SBA_CUDA(cudaMemsetAsync(p->flush_buf, iteration & 0xff, (size_t)o->l2_flush_bytes, p->stream));
        it_tm.begin(-1);
        // One host read per trial point.  scipy tests |g|_inf < gtol before it computes a step; here the first trial
        // point of the iteration is already in flight when the test is made, and is simply discarded if it fires.
        SBA_TRY(enqueue_iteration(-1.0));
        SBA_TRY(fetch_scal(p));
        const double* h = p->h_scal;
        if (h[SC_COMM_FAIL] != 0.0) { set_error("peer-memory all-reduce timed out (a rank is missing)"); return SBA_E_CUDA; }
        for (int attempt = 0; h[SC_CHOL_FAIL] != 0.0 || !std::isfinite(h[chk0]) || !std::isfinite(h[chk1]); ++attempt) {
            if (attempt >= 30) { set_error("reduced camera system could not be factorised"); return SBA_E_NUMERIC; }
            // re-damp: J_h has unit column norms, so reg is relative to 1
            ++chol_retries;
            SBA_TRY(enqueue_iteration(std::max(h[SC_REG] * 10.0, 1e-12)));
            SBA_TRY(fetch_scal(p));
            h = p->h_scal;
        }
        first = false;
        Delta = h[SC_DELTA];
        const double x_norm = std::sqrt(h[SC_XX]);
        g_norm = 0.0;
        for (int r = 0; r < 16; ++r) g_norm = std::max(g_norm, h[SC_GMAX_SLOTS + r]);
        if (o->verbose >= 2)
            printf("[sba] it %3d nfev %3d cost %.10e |g|inf %.3e Delta %.3e reg %.3e\n", iteration, nfev, cost, g_norm, Delta,
                   h[SC_REG]);
        if (g_norm < o->gtol) { status = 1; break; }

        double cost_new;
        TrOutcome tr;
        while (true) {
            ++nfev;
            cost_new = h[SC_COST_NEW];
            tr = tr_outcome(cost, cost_new, h[SC_PRED], h[SC_STEPH], h[SC_STEPN], x_norm, Delta, o->ftol, o->xtol);
            Delta = tr.Delta;
            if (tr.accept || tr.status >= 0 || nfev >= o->max_nfev) break;
            // rejected: same model, smaller radius, new trial point (no new factorisation, like scipy)
            SBA_TRY(enqueue_trial(Delta));
            SBA_TRY(fetch_scal(p));
            h = p->h_scal;
        }
        if (tr.accept) {
            cost = cost_new;
            SBA_TRY(trf_accept(p, o, tm, tr.status >= 0, njev));
        }
        it_tm.end();
        ++iteration;
        if (tr.status >= 0) { status = tr.status; break; }
    }
    if (status < 0) status = 0;
    SBA_CUDA(cudaEventRecord(p->ev1, p->stream));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    float ms = 0.f;
    SBA_CUDA(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
    info->status = status; info->nfev = nfev; info->njev = njev; info->iterations = iteration;
    info->cost = cost; info->optimality = g_norm; info->solve_ms = ms; info->chol_retries = chol_retries;
    info->gpu_launches = p->launches;
    info->explicit_subspace_passes = iteration;
    info->pcg_solves = (int)p->pcg_solves; info->pcg_iterations = (int)p->pcg_iterations;
    tm.resolve(info);
    it_tm.resolve(info);
    return SBA_OK;
}

// residuals at the internal vector x (camrec prepared) into a device buffer in the CALLER's observation order
static int residuals_ext(sba_problem* p, const double* x, const double* camrec, int loss, double f_scale, double* r_ext_dev,
                         int slot, int rpc_f32)
{
    if (p->engine == 0) return run_residual(p, x, camrec, loss, f_scale, r_ext_dev, slot, rpc_f32);
    SBA_TRY(run_residual(p, x, camrec, loss, f_scale, r_ext_dev ? p->r_int : nullptr, slot, rpc_f32));
    if (r_ext_dev) SBA_TRY(pt_obs_out(p, p->r_int, 2, r_ext_dev));
    return SBA_OK;
}

// un-weighted reprojection errors of the residuals just computed by residuals_ext, caller's order
static int reproj_errors_ext(sba_problem* p, const double* r_ext_dev, double* err_ext_dev)
{
    const int grid = grid_for(p->K, 256, NUM_SMS * 8);
    if (p->engine == 0) {
        k_reproj_error<<<grid, 256, 0, p->stream>>>((const double2*)r_ext_dev, p->w, p->K, err_ext_dev);
        return check_launch(p);
    }
    k_reproj_error<<<grid, 256, 0, p->stream>>>((const double2*)p->r_int, p->w, p->K, p->e_int);
    SBA_TRY(check_launch(p));
    return pt_obs_out(p, p->e_int, 1, err_ext_dev);
}

// caller's variable vector (device) -> internal vector; and back
static int vars_in(sba_problem* p, const double* x_ext_dev, double* dst)
{
    if (p->engine == 0) {
        SBA_CUDA(cudaMemcpyAsync(dst, x_ext_dev, (size_t)p->n * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
        return SBA_OK;
    }
    return pt_x_in(p, x_ext_dev, dst);
}
static int vars_out(sba_problem* p, const double* src, double* x_ext_dev)
{
    if (p->engine == 0) {
        SBA_CUDA(cudaMemcpyAsync(x_ext_dev, src, (size_t)p->n * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
        return SBA_OK;
    }
    return pt_x_out(p, src, x_ext_dev);
}

}  // namespace sba

using namespace sba;

// ------------------------------------------------------------------------------------------------
// C ABI: problem life cycle
// ------------------------------------------------------------------------------------------------
extern "C" const char* sba_last_error(void) { return g_error.c_str(); }
extern "C" int sba_version(void) { return 100; }

extern "C" int sba_release_cached_memory(void)
{
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    int dev = 0;
    cudaGetDevice(&dev);
    for (const Slab& c : g_slab_pool) { cudaSetDevice(c.device); cudaFree(c.ptr); }
    for (double* h : g_pinned_pool) cudaFreeHost(h);
    g_slab_pool.clear(); g_pinned_pool.clear(); g_pool_bytes = 0;
    comm_release();
    cudaSetDevice(dev);
    return SBA_OK;
}

extern "C" int sba_problem_destroy(sba_problem* p)
{
    if (!p) return SBA_OK;
    cudaSetDevice(p->device);
    if (p->stream2) cudaStreamSynchronize(p->stream2);
    cudaStreamSynchronize(p->stream);               // nothing of this problem may still be running on the slabs
    if (p->engine == 1) pt_print_cycles(p);
    for (size_t i = 0; i < p->arena_chunks.size(); ++i) pool_give(p->arena_chunks[i], p->arena_chunk_bytes[i], p->device);
    // the exchange buffer and its peer mappings belong to the process (g_comm), not to the problem
    if (p->h_scal) { std::lock_guard<std::mutex> lock(g_pool_mutex); g_pinned_pool.push_back(p->h_scal); }
    if (p->ev0) cudaEventDestroy(p->ev0);
    if (p->ev1) cudaEventDestroy(p->ev1);
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    if (p->ev_join) cudaEventDestroy(p->ev_join);
    if (p->stream2) cudaStreamDestroy(p->stream2);
    for (cudaEvent_t e : p->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : p->cov_ev) if (e) cudaEventDestroy(e);
    if (p->flush_buf) cudaFree(p->flush_buf);
    delete p;
    return SBA_OK;
}

static int problem_create_impl(sba_problem* p, const sba_problem_desc* d)
{
    const int M = p->M, N = p->N, nc = p->nc;
    const int64_t K = p->K;
    cudaStream_t s = p->stream;
    const bool timing = getenv("SBA_TIMING") != nullptr;
    auto t_prev = std::chrono::steady_clock::now();
    auto stamp = [&](const char* what) {
        if (!timing) return;
        cudaStreamSynchronize(s);
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[sba create] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
        t_prev = now;
    };
    // --- indices: int64 -> int32, track offsets, camera-major order, chunks, warp tiles (host, O(K), a few threads) ---
    HostIndex hidx;
    const bool try_pattern = d->engine != 2 && !(p->use_pcg && d->engine == 0) && pattern_engine_applicable(p, d->engine == 1);
    if (d->engine == 1 && !try_pattern) { set_error("the pattern engine does not apply to this problem (size, n_params or shared calibration)"); return SBA_E_INVALID; }
    // The two big uploads of the pattern engine (observations 16 B and weights 8 B per observation, from pageable host memory: the
    // driver stages them synchronously, ~2.4 ms per million observations) do not depend on the layout: a helper thread issues them
    // on the problem's stream while this thread builds the host index and the pattern layout.
    std::thread uploader;
    struct Joiner { std::thread& t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{uploader};
    cudaError_t up_err = cudaSuccess;
    if (try_pattern) {
        SBA_TRY(dev_alloc(p, &p->r_out, 2 * (size_t)K));
        SBA_TRY(dev_alloc(p, &p->err_out, (size_t)K));
        p->pt_obs_uploaded = true;
        uploader = std::thread([&up_err, p, d, K, s]() {
            up_err = cudaSetDevice(p->device);
            if (up_err == cudaSuccess) up_err = cudaMemcpyAsync(p->r_out, d->pts2d, 2 * (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s);
            if (up_err == cudaSuccess) up_err = cudaMemcpyAsync(p->err_out, d->pts2d_w, (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s);
        });
    }
    int irc = build_host_index(d->cam_ind, d->pts_ind, K, M, N, CHUNK, 8, hidx, try_pattern);
    if (irc == 1) { set_error("cam_ind / pts_ind out of range"); return SBA_E_INVALID; }
    if (irc == 2) { set_error("pts_ind must be non-decreasing (observations sorted by track)"); return SBA_E_INVALID; }
    std::vector<int>&cam = hidx.cam, &pts = hidx.pts, &track_ptr = hidx.track_ptr, &cm_obs = hidx.cm_obs;
    std::vector<int>&ch_cam = hidx.ch_cam, &ch_beg = hidx.ch_beg, &ch_end = hidx.ch_end, &first_chunk = hidx.first_chunk;
    std::vector<int>& tile_obs = hidx.tile_obs;
    stamp("host index pass");
    if (try_pattern) {
        PatternLayout lay;
        if (const char* e = getenv("SBA_PT_SCHUR")) p->pt_schur_mma = std::strcmp(e, "mma") == 0;
        build_pattern_layout(cam.data(), track_ptr.data(), K, M, N, p->n_pts_fix, PT_CTAS, PT_THREADS_LIGHT / 32, PT_THREADS / 32, PT_THREADS_SCHUR / 32, nc, p->pt_schur_mma ? 0 : PT_RC,
                             lay);
        stamp("pattern layout");
        // A tile holds tracks with ONE camera set: when the visibility patterns are too diverse (many cameras, random visibility)
        // the tiles stay mostly empty and the generic engine, which packs arbitrary tracks into a warp, is the faster one
        // (it costs ~1.9x the pattern engine at full tiles).  Small problems keep the pattern engine; SBA_ENGINE=pattern forces it.
        const char* eng = getenv("SBA_ENGINE");
        if (lay.ok && K >= 65536 && lay.fill < 0.5 && d->engine != 1 && !(eng && std::strcmp(eng, "pattern") == 0)) {
            lay.ok = false;
            lay.why = "visibility patterns too diverse (tile fill " + std::to_string(lay.fill) + ")";
        }
        if (uploader.joinable()) uploader.join();
        if (up_err != cudaSuccess) { set_error(std::string("upload of the observations: ") + cudaGetErrorString(up_err)); return SBA_E_CUDA; }
        if (lay.ok) {
            const int rc = pattern_create(p, d, hidx, lay);
            stamp("pattern uploads + state");
            return rc;
        }
        p->pt_obs_uploaded = false;                    // the generic engine uploads into its own layout
        if (timing) fprintf(stderr, "[sba create] pattern engine not applicable: %s\n", lay.why.c_str());
        if (d->engine == 1) { set_error(("the pattern engine does not apply: " + lay.why).c_str()); return SBA_E_INVALID; }
        irc = build_host_index(d->cam_ind, d->pts_ind, K, M, N, CHUNK, 8, hidx);       // the generic engine needs the camera-major tables too
        if (irc) { set_error("cam_ind / pts_ind invalid"); return SBA_E_INVALID; }
    }
    p->chunks.n = (int)ch_cam.size();
    p->chunks.h_cam = ch_cam;
    p->chunks.h_first_of_cam = first_chunk;
    // Schur: (j <= j') blocks; the partial of (chunk ch, partner j') lives at item_base[ch] + (j' - cam(ch))
    std::vector<int> item_base(ch_cam.size() + 1, 0), sb_j, sb_jp;
    for (size_t c = 0; c < ch_cam.size(); ++c) item_base[c + 1] = item_base[c] + (M - ch_cam[c]);
    std::vector<int> item_chunk(item_base.back());
    for (size_t c = 0; c < ch_cam.size(); ++c)
        for (int t = item_base[c]; t < item_base[c + 1]; ++t) item_chunk[t] = (int)c;
    for (int j = 0; j < M; ++j)
        for (int jp = j; jp < M; ++jp) { sb_j.push_back(j); sb_jp.push_back(jp); }
    p->n_schur_items = item_base.back();
    p->n_schur_blocks = (int)sb_j.size();
    p->n_tiles = (int)tile_obs.size() - 1;
    stamp("host tables");
    SBA_TRY(dev_upload(p, &p->cam_ind, cam, s));
    SBA_TRY(dev_upload(p, &p->pts_ind, pts, s));
    SBA_TRY(dev_upload(p, &p->track_ptr, track_ptr, s));
    SBA_TRY(dev_upload(p, &p->cm_obs, cm_obs, s));
    SBA_TRY(dev_upload(p, &p->cam_ptr, first_chunk, s));   // camera -> first chunk (used by k_reduce_cameras)
    SBA_TRY(dev_upload(p, &p->chunks.cam, ch_cam, s));
    SBA_TRY(dev_upload(p, &p->chunks.beg, ch_beg, s));
    SBA_TRY(dev_upload(p, &p->chunks.end, ch_end, s));
    SBA_TRY(dev_upload(p, &p->item_base, item_base, s));
    SBA_TRY(dev_upload(p, &p->item_chunk, item_chunk, s));
    SBA_TRY(dev_upload(p, &p->tile_obs, tile_obs, s));
    SBA_TRY(dev_upload(p, &p->sb_j, sb_j, s));
    SBA_TRY(dev_upload(p, &p->sb_jp, sb_jp, s));

    SBA_TRY(dev_alloc(p, &p->pts2d, 2 * (size_t)K));
    SBA_CUDA(cudaMemcpyAsync(p->pts2d, d->pts2d, 2 * (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s));
    SBA_TRY(dev_alloc(p, &p->w, (size_t)K));
    SBA_CUDA(cudaMemcpyAsync(p->w, d->pts2d_w, (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s));
    SBA_TRY(dev_alloc(p, &p->cam_static, (size_t)M * p->P));
    SBA_CUDA(cudaMemcpyAsync(p->cam_static, d->cam_params, (size_t)M * p->P * sizeof(double), cudaMemcpyHostToDevice, s));
    if (p->model == MODEL_RPC) {
        SBA_TRY(dev_alloc(p, &p->rpc_tab, (size_t)M * RPC_TAB_STRIDE));
        SBA_CUDA(cudaMemcpyAsync(p->rpc_tab, d->rpc_coefs, (size_t)M * RPC_TAB_STRIDE * sizeof(double),
                                 cudaMemcpyHostToDevice, s));
    }
    // camera-major copies of the observation data: gathered on the device from the track-major arrays
    SBA_TRY(dev_alloc(p, &p->cm_pts, (size_t)K)); SBA_TRY(dev_alloc(p, &p->cm_pts2d, 2 * (size_t)K)); SBA_TRY(dev_alloc(p, &p->cm_w, (size_t)K));
    k_gather_camera_major<<<grid_for(K, 256, NUM_SMS * 8), 256, 0, s>>>(p->cm_obs, p->pts_ind, (const double2*)p->pts2d, p->w, K,
                                                                       p->cm_pts, (double2*)p->cm_pts2d, p->cm_w);
    SBA_CUDA(cudaGetLastError());
    if (!p->use_pcg) {
        SBA_TRY(dev_alloc(p, &p->obs_of, (size_t)M * N));
        SBA_CUDA(cudaMemsetAsync(p->obs_of, 0xFF, (size_t)M * N * sizeof(int), s));
        k_fill_obs_of<<<grid_for(K, 256, NUM_SMS * 8), 256, 0, s>>>(p->cam_ind, p->pts_ind, K, N, p->obs_of);
        SBA_CUDA(cudaGetLastError());
    }
    stamp("uploads + obs_of");
    // --- static pair lists of the Schur complement: count, scan on the host, fill (dense path only) ---
    if (p->use_pcg) {
        p->n_schur_items = 0; p->n_schur_blocks = 0; p->n_pairs = 0;
    } else {
        const int n_items = item_base.back();
        int *d_counts = nullptr, *d_off = nullptr;
        SBA_TRY(dev_alloc(p, &d_counts, (size_t)n_items));
        SBA_TRY(dev_alloc(p, &d_off, (size_t)n_items));
        k_pair_count<<<(n_items + 3) / 4, 128, 0, s>>>(p->chunks.cam, p->chunks.beg, p->chunks.end, p->cm_pts, p->obs_of, N,
                                                      p->item_base, p->item_chunk, n_items, d_counts);
        SBA_CUDA(cudaGetLastError());
        std::vector<int> counts(n_items), off(n_items);
        SBA_CUDA(cudaMemcpyAsync(counts.data(), d_counts, (size_t)n_items * sizeof(int), cudaMemcpyDeviceToHost, s));
        SBA_CUDA(cudaStreamSynchronize(s));
        // pair list order: block (j, j'), then the chunks of camera j
        std::vector<int> slice_block, slice_p0, slice_p1, sb_first;
        long long total = 0;
        for (size_t blk = 0; blk < sb_j.size(); ++blk) {
            const int j = sb_j[blk], jp = sb_jp[blk];
            const long long blk_begin = total;
            for (int c = first_chunk[j]; c < first_chunk[j + 1]; ++c) {
                const int item = item_base[c] + (jp - j);
                off[item] = (int)total;
                total += counts[item];
            }
            sb_first.push_back((int)slice_block.size());
            for (long long q0 = blk_begin; q0 < total; q0 += SLICE) {
                slice_block.push_back((int)blk); slice_p0.push_back((int)q0); slice_p1.push_back((int)std::min(q0 + SLICE, total));
            }
        }
        sb_first.push_back((int)slice_block.size());
        if (total > 2000000000LL) { set_error("pair list too large: use the matrix-free path"); return SBA_E_INVALID; }
        p->n_pairs = total;
        p->n_schur_items = (int)slice_block.size();
        SBA_CUDA(cudaMemcpyAsync(d_off, off.data(), (size_t)n_items * sizeof(int), cudaMemcpyHostToDevice, s));
        SBA_TRY(dev_alloc(p, &p->pairs, (size_t)std::max<long long>(total, 1) * 2));
        k_pair_fill<<<(n_items + 3) / 4, 128, 0, s>>>(p->chunks.cam, p->chunks.beg, p->chunks.end, p->cm_obs, p->cm_pts,
                                                     p->obs_of, N, p->item_base, p->item_chunk, n_items, d_off,
                                                     (int2*)p->pairs);
        SBA_CUDA(cudaGetLastError());
        SBA_TRY(dev_upload(p, &p->slice_block, slice_block, s));
        SBA_TRY(dev_upload(p, &p->slice_p0, slice_p0, s));
        SBA_TRY(dev_upload(p, &p->slice_p1, slice_p1, s));
        SBA_TRY(dev_upload(p, &p->sb_first, sb_first, s));
        SBA_CUDA(cudaStreamSynchronize(s));   // `off` and the slice vectors go out of scope
    }

    stamp("pair lists");
    // --- iteration state ---
    const size_t n = (size_t)p->n, ns = (size_t)M * nc;
    SBA_TRY(dev_alloc(p, &p->x, n)); SBA_TRY(dev_alloc(p, &p->x_new, n)); SBA_TRY(dev_alloc(p, &p->g, n));
    SBA_TRY(dev_alloc(p, &p->sinv, n)); SBA_TRY(dev_alloc(p, &p->delta, n)); SBA_TRY(dev_alloc(p, &p->t1, n));
    SBA_TRY(dev_alloc(p, &p->t2, n)); SBA_TRY(dev_alloc(p, &p->io_x, n));
    SBA_TRY(dev_alloc(p, &p->camrec, (size_t)M * CAMREC_STRIDE)); SBA_TRY(dev_alloc(p, &p->camrec_new, (size_t)M * CAMREC_STRIDE));
    SBA_TRY(dev_alloc(p, &p->V, 6 * (size_t)N)); SBA_TRY(dev_alloc(p, &p->F, 6 * (size_t)N)); SBA_TRY(dev_alloc(p, &p->q, 3 * (size_t)N));
    SBA_TRY(dev_alloc(p, &p->Z, (size_t)K * nc * 3));
    // tracks without observations are never touched by the tile kernels: their blocks must read as zero
    for (double* buf : {p->g, p->sinv, p->delta, p->t1, p->t2, p->x_new}) SBA_CUDA(cudaMemsetAsync(buf, 0, n * sizeof(double), s));
    SBA_CUDA(cudaMemsetAsync(p->V, 0, 6 * (size_t)N * sizeof(double), s));
    SBA_CUDA(cudaMemsetAsync(p->F, 0, 6 * (size_t)N * sizeof(double), s));
    SBA_CUDA(cudaMemsetAsync(p->q, 0, 3 * (size_t)N * sizeof(double), s));
    SBA_TRY(dev_alloc(p, &p->camsys_local, ns * nc + ns));
    if (p->world > 1) SBA_TRY(dev_alloc(p, &p->camsys, ns * nc + ns));
    else p->camsys = p->camsys_local;
    if (p->use_pcg) {
        const size_t nvc = (size_t)nc * (nc + 1) / 2 + nc;
        SBA_TRY(dev_alloc(p, &p->pcg_vec, 5 * ns + PCG_SCAL)); SBA_TRY(dev_alloc(p, &p->pcg_diag, (size_t)M * nvc));
        SBA_TRY(dev_alloc(p, &p->pcg_L, ns * nc)); SBA_TRY(dev_alloc(p, &p->pcg_w, ns)); SBA_TRY(dev_alloc(p, &p->pcg_s, 3 * (size_t)N));
        SBA_CUDA(cudaMemsetAsync(p->pcg_vec, 0, (5 * ns + PCG_SCAL) * sizeof(double), s));
        SBA_CUDA(cudaMemsetAsync(p->pcg_s, 0, 3 * (size_t)N * sizeof(double), s));
    } else {
        SBA_TRY(dev_alloc(p, &p->S, ns * ns + ns));
        SBA_TRY(dev_alloc(p, &p->chol_work, (size_t)34 * (ns + 32)));
    }
    SBA_TRY(dev_alloc(p, &p->cvec, (size_t)3 * ns));
    const size_t nv_cam = (size_t)nc * (nc + 1) / 2 + nc;
    SBA_TRY(dev_alloc(p, &p->cam_partials, (size_t)p->chunks.n * nv_cam));
    SBA_TRY(dev_alloc(p, &p->schur_partials, (size_t)std::max(p->n_schur_items, 1) * (nc * nc + nc)));
    SBA_CUDA(cudaMemsetAsync(p->schur_partials, 0, (size_t)std::max(p->n_schur_items, 1) * (nc * nc + nc) * sizeof(double), s));
    SBA_TRY(dev_alloc(p, &p->red_partials, (size_t)std::max(NUM_SMS * 16, (p->n_tiles + WPB - 1) / WPB + 1) * 8));
    SBA_TRY(dev_alloc(p, &p->counters, 16));
    SBA_CUDA(cudaMemsetAsync(p->counters, 0, 16 * sizeof(unsigned), s));
    SBA_TRY(dev_alloc(p, &p->scal, SC_COUNT));
    SBA_CUDA(cudaMemsetAsync(p->scal, 0, SC_COUNT * sizeof(double), s));
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        if (!g_pinned_pool.empty()) { p->h_scal = g_pinned_pool.back(); g_pinned_pool.pop_back(); }
    }
    if (!p->h_scal) SBA_CUDA(cudaMallocHost((void**)&p->h_scal, H_SCAL_COUNT * sizeof(double)));
    SBA_TRY(dev_alloc(p, &p->r_out, 2 * (size_t)K));
    SBA_TRY(dev_alloc(p, &p->err_out, (size_t)K));
    SBA_CUDA(cudaEventCreate(&p->ev0));
    SBA_CUDA(cudaEventCreate(&p->ev1));
    SBA_CUDA(cudaStreamCreateWithFlags(&p->stream2, cudaStreamNonBlocking));
    SBA_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
    SBA_CUDA(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
    SBA_CUDA(cudaStreamSynchronize(s));   // host staging vectors go out of scope
    stamp("state buffers");
    return SBA_OK;
}

extern "C" int sba_problem_create(sba_problem** out, const sba_problem_desc* d, void* stream)
{
    if (!out || !d) { set_error("null argument"); return SBA_E_INVALID; }
    *out = nullptr;
    if (d->n_cam < 1 || d->n_pts < 1 || d->n_obs < 1 || d->n_obs > 2000000000LL) { set_error("empty or oversized problem"); return SBA_E_INVALID; }
    if (!valid_nc(d->cam_model, d->n_params)) { set_error("unsupported (cam_model, n_params) combination"); return SBA_E_INVALID; }
    const int P = d->cam_model == MODEL_AFFINE ? 8 : (d->cam_model == MODEL_PERSPECTIVE ? 11 : 9);
    if (d->n_cam_params != P) { set_error("cam_params has the wrong number of columns for this camera model"); return SBA_E_INVALID; }
    if (d->cam_model == MODEL_RPC && !d->rpc_coefs) { set_error("rpc_coefs required for cam_model rpc"); return SBA_E_INVALID; }
    if (!d->cam_ind || !d->pts_ind || !d->pts2d || !d->pts2d_w || !d->cam_params) { set_error("null array"); return SBA_E_INVALID; }
    if (d->n_cam_fix < 0 || d->n_cam_fix > d->n_cam || d->n_pts_fix < 0 || d->n_pts_fix > d->n_pts) { set_error("bad n_cam_fix / n_pts_fix"); return SBA_E_INVALID; }
    if (d->n_common < 0 || d->n_common > 5 || d->n_common >= d->n_params || (d->n_common > 0 && d->n_cam_fix > 0)) {
        // the reference's COMMON_K packing is only self-consistent without frozen cameras (ba_params.py:170 vs :244)
        set_error("bad n_common (shared calibration needs n_cam_fix == 0)");
        return SBA_E_INVALID;
    }
    if (d->world_size < 1 || d->world_size > 16 || d->rank < 0 || d->rank >= d->world_size) { set_error("bad rank / world_size"); return SBA_E_INVALID; }
    // Solver of the reduced camera system: dense Cholesky up to PCG_ABOVE unknowns, matrix-free block-Jacobi PCG beyond
    // (SBA_SOLVER=pcg | dense overrides).  The dense path also needs a (camera, track) look-up table of n_cam * n_pts ints.
    constexpr int64_t PCG_ABOVE = 1200, PCG_MAX_NS = 65536;
    const int64_t ns_all = (int64_t)d->n_cam * d->n_params;
    bool use_pcg = ns_all > PCG_ABOVE || (double)d->n_cam * d->n_pts > 1.5e9;
    if (const char* e = getenv("SBA_SOLVER")) {
        if (std::strcmp(e, "pcg") == 0) use_pcg = true;
        if (std::strcmp(e, "dense") == 0) use_pcg = false;
    }
    if (d->solver == 1) use_pcg = false;
    if (d->solver == 2) use_pcg = true;
    if (d->engine < 0 || d->engine > 2 || d->solver < 0 || d->solver > 2) { set_error("bad engine / solver choice"); return SBA_E_INVALID; }
    if (use_pcg && d->n_common > 0) use_pcg = false;      // the shared-calibration border is only folded on the dense path
    if (!use_pcg && (double)d->n_cam * d->n_pts > 1.5e9) { set_error("unsupported size: n_cam * n_pts > 1.5e9 needs the PCG path (no shared calibration, SBA_SOLVER unset)"); return SBA_E_INVALID; }
    if (!use_pcg && ns_all > 4096) { set_error("unsupported size: more than 4096 camera unknowns need the PCG path (no shared calibration, SBA_SOLVER unset)"); return SBA_E_INVALID; }
    if (ns_all > PCG_MAX_NS) { set_error("unsupported size: more than 65536 camera unknowns"); return SBA_E_INVALID; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: sat_bundleadjust_b200 has no CPU fallback");
        return SBA_E_CUDA;
    }
    sba_problem* p = new sba_problem();
    p->model = d->cam_model; p->M = d->n_cam; p->N = d->n_pts; p->K = d->n_obs; p->nc = d->n_params; p->P = P;
    p->n_cam_fix = d->n_cam_fix; p->n_pts_fix = d->n_pts_fix; p->rpc_f32 = d->rpc_float32;
    p->rank = d->rank; p->world = d->world_size;
    p->n_common = d->n_common;
    p->use_pcg = use_pcg;
    if (const char* e = getenv("SBA_PCG_TOL")) p->pcg_tol = atof(e);
    p->n = (int64_t)p->M * p->nc + 3 * (int64_t)p->N;
    p->stream = (cudaStream_t)stream;
    cudaGetDevice(&p->device);
    if (const char* e = getenv("SBA_COMM_SPLIT")) p->comm_split = atoi(e) != 0;
    const int rc = problem_create_impl(p, d);
    if (rc != SBA_OK) { sba_problem_destroy(p); return rc; }
    *out = p;
    return SBA_OK;
}

extern "C" int sba_problem_set_allreduce(sba_problem* p, sba_allreduce_fn fn, void* user)
{
    if (!p) return SBA_E_INVALID;
    p->allreduce = fn; p->allreduce_user = user;
    return SBA_OK;
}

extern "C" int64_t sba_problem_num_vars(const sba_problem* p) { return p ? p->n : -1; }
extern "C" int sba_problem_engine(const sba_problem* p) { return p ? p->engine : -1; }
extern "C" int sba_problem_solver(const sba_problem* p) { return p ? (p->use_pcg ? 1 : 0) : -1; }

// Multi-GPU exchange over peer memory: every rank exports the IPC handle of its symmetric buffer ...
extern "C" int sba_comm_export(sba_problem* p, void* handle_out)
{
    if (!p || !handle_out) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    comm_release();                            // a fresh exchange group: drop whatever an earlier group left
    g_comm.cap = comm_needed(p);
    const size_t bytes = (size_t)(2 * g_comm.cap) * sizeof(double) + 2 * COMM_MAX_RANKS * sizeof(unsigned long long);
    SBA_CUDA(cudaMalloc(&g_comm.buf, bytes));
    SBA_CUDA(cudaMemset(g_comm.buf, 0, bytes));
    g_comm.world = p->world; g_comm.rank = p->rank; g_comm.device = p->device;
    p->comm_buf = g_comm.buf; p->comm_cap = g_comm.cap;
    cudaIpcMemHandle_t h;
    SBA_CUDA(cudaIpcGetMemHandle(&h, g_comm.buf));
    std::memcpy(handle_out, &h, sizeof(h));
    return SBA_OK;
}

// ... and maps the buffers of all ranks (handles: world x 64 bytes, in rank order; its own entry is skipped)
extern "C" int sba_comm_import(sba_problem* p, const void* handles)
{
    if (!p || !handles || !g_comm.buf || p->comm_buf != g_comm.buf) { set_error("sba_comm_export must be called first"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    for (int r = 0; r < p->world; ++r) {
        if (r == p->rank) { g_comm.peer[r] = g_comm.buf; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, (const char*)handles + (size_t)r * sizeof(h), sizeof(h));
        SBA_CUDA(cudaIpcOpenMemHandle(&g_comm.peer[r], h, cudaIpcMemLazyEnablePeerAccess));
    }
    g_comm.ready = true;
    g_comm.seq = 0;
    for (int r = 0; r < p->world; ++r) p->comm_peer[r] = g_comm.peer[r];
    p->comm_ready = true;
    return SBA_OK;
}

// Attach a new problem to the exchange buffers this process already shares with the same peers (same world, rank, device;
// large enough).  Returns 1 when attached, 0 when sba_comm_export / sba_comm_import are needed.  All ranks of a group run the
// same sequence of problems, so they agree on the answer.
extern "C" int sba_comm_try_reuse(sba_problem* p)
{
    if (!p || !g_comm.ready || g_comm.world != p->world || g_comm.rank != p->rank || g_comm.device != p->device) return 0;
    if (g_comm.cap < comm_needed(p)) return 0;
    p->comm_buf = g_comm.buf; p->comm_cap = g_comm.cap;
    for (int r = 0; r < p->world; ++r) p->comm_peer[r] = g_comm.peer[r];
    p->comm_ready = true;
    return 1;
}

// ------------------------------------------------------------------------------------------------
// C ABI: evaluation entry points
// ------------------------------------------------------------------------------------------------
extern "C" int sba_residuals(sba_problem* p, const double* x, double* r, int32_t loss, double f_scale, double* cost)
{
    if (!p || !x) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_CUDA(cudaMemcpyAsync(p->io_x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    double* xi = p->io_x;
    if (p->engine == 1) { SBA_TRY(vars_in(p, p->io_x, p->x_new)); xi = p->x_new; }
    SBA_TRY(run_prepare(p, xi, p->camrec_new));
    SBA_TRY(residuals_ext(p, xi, p->camrec_new, loss, f_scale, p->r_out, SC_COST_NEW, p->rpc_f32));
    if (r) SBA_CUDA(cudaMemcpyAsync(r, p->r_out, 2 * (size_t)p->K * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_TRY(fetch_scal(p));
    if (cost) *cost = p->h_scal[SC_COST_NEW];
    return SBA_OK;
}

extern "C" int sba_jacobian_blocks(sba_problem* p, const double* x, double* Jc, double* Jp)
{
    if (!p || !x) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_CUDA(cudaMemcpyAsync(p->io_x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    double* xi = p->io_x;
    if (p->engine == 1) { SBA_TRY(vars_in(p, p->io_x, p->x_new)); xi = p->x_new; }
    SBA_TRY(run_prepare(p, xi, p->camrec_new));
    double *dJc = nullptr, *dJp = nullptr;
    if (Jc) SBA_CUDA(cudaMalloc((void**)&dJc, (size_t)p->K * 2 * p->nc * sizeof(double)));
    if (Jp) SBA_CUDA(cudaMalloc((void**)&dJp, (size_t)p->K * 6 * sizeof(double)));
    const int grid = grid_for(p->K, 128, NUM_SMS * 16);
#define L(MODEL, NC)                                                                                               \
    k_jac_blocks<MODEL, NC><<<grid, 128, 0, p->stream>>>(obs_arrays(p), xi + (size_t)p->M * p->nc, p->camrec_new,   \
                                                         p->rpc_tab, p->K, p->n_cam_fix,                             \
                                                         p->engine == 1 ? p->n_pts_fix_int : p->n_pts_fix, dJc, dJp)
    SBA_DISPATCH(p, L);
#undef L
    SBA_TRY(check_launch(p));
    if (Jc) SBA_CUDA(cudaMemcpyAsync(Jc, dJc, (size_t)p->K * 2 * p->nc * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (Jp) SBA_CUDA(cudaMemcpyAsync(Jp, dJp, (size_t)p->K * 6 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    if (dJc) cudaFree(dJc);
    if (dJp) cudaFree(dJp);
    if (p->engine == 1) {          // test-only entry point: un-permute on the host
        if (p->h_obs_new2old.empty()) {
            p->h_obs_new2old.resize((size_t)p->K);
            SBA_CUDA(cudaMemcpy(p->h_obs_new2old.data(), p->obs_new2old, (size_t)p->K * sizeof(int), cudaMemcpyDeviceToHost));
        }
        auto unperm = [&](double* buf, size_t width) {
            std::vector<double> tmp(buf, buf + (size_t)p->K * width);
            for (int64_t a = 0; a < p->K; ++a)
                std::memcpy(buf + (size_t)p->h_obs_new2old[a] * width, tmp.data() + (size_t)a * width, width * sizeof(double));
        };
        if (Jc) unperm(Jc, 2 * (size_t)p->nc);
        if (Jp) unperm(Jp, 6);
    }
    return SBA_OK;
}

// frozen points of the internal order: the generic kernels test `track index >= n_pts_fix`, which only holds for the caller's
// order; the pattern engine carries the flag per run instead (PUnit::pts_free)
extern "C" int sba_normal_blocks(sba_problem* p, const double* x, int32_t loss, double f_scale, double* U, double* V,
                                 double* g)
{
    if (!p || !x) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    const size_t ns = (size_t)p->M * p->nc;
    if (p->engine == 1) {
        SBA_CUDA(cudaMemcpyAsync(p->io_x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        SBA_TRY(vars_in(p, p->io_x, p->x));
        SBA_TRY(pt_reset_state(p));
        SBA_TRY(pt_run_assemble(p, 1, 1, loss, f_scale));
        pt_accept(p);
        std::vector<double> Vi(V ? 6 * (size_t)p->N : 0), gi(g ? (size_t)p->n : 0);
        if (U) SBA_CUDA(cudaMemcpyAsync(U, p->camsys, ns * p->nc * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (V) SBA_CUDA(cudaMemcpyAsync(Vi.data(), p->V, Vi.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (g) SBA_CUDA(cudaMemcpyAsync(gi.data(), p->g, gi.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        SBA_CUDA(cudaStreamSynchronize(p->stream));
        for (int t = 0; t < p->N; ++t) {
            const size_t o = (size_t)p->h_trk_new2old[t];
            if (V) std::memcpy(V + 6 * o, Vi.data() + 6 * (size_t)t, 6 * sizeof(double));
            if (g) std::memcpy(g + ns + 3 * o, gi.data() + ns + 3 * (size_t)t, 3 * sizeof(double));
        }
        if (g) std::memcpy(g, gi.data(), ns * sizeof(double));
        return SBA_OK;
    }
    SBA_CUDA(cudaMemcpyAsync(p->x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    SBA_TRY(run_prepare(p, p->x, p->camrec));
    SBA_TRY(run_assemble(p, p->x, p->camrec, loss, f_scale));
    if (U) SBA_CUDA(cudaMemcpyAsync(U, p->camsys, ns * p->nc * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (V) SBA_CUDA(cudaMemcpyAsync(V, p->V, 6 * (size_t)p->N * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (g) {
        SBA_CUDA(cudaMemcpyAsync(g, p->camsys + ns * p->nc, ns * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        SBA_CUDA(cudaMemcpyAsync(g + ns, p->g + ns, 3 * (size_t)p->N * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

// The reduced camera system of the damped normal equations at x, as the solver forms it (scaling D from this one
// evaluation): S = U + reg D_c^2 - W (V + reg D_p^2)^-1 W^T and rhs = -(g_c - W (V + reg D_p^2)^-1 g_p), COMMON_K folded.
// Exposed for the parity tests of the Schur complement; host buffers, S is (M n_params)^2 column-major.
// Device part: x (host) is uploaded (then `uploaded`, if given, is recorded); afterwards p->x / p->camrec hold x, p->camsys its
// U blocks, p->S the system, and the cost at x is in scal[SC_COST_NEW] (pattern engine) or scal[SC_COST] (generic engine).
static int form_reduced_system(sba_problem* p, const double* x, int32_t loss, double f_scale, double reg,
                               cudaEvent_t uploaded = nullptr)
{
    if (p->engine == 1) {
        SBA_CUDA(cudaMemcpyAsync(p->io_x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        if (uploaded) SBA_CUDA(cudaEventRecord(uploaded, p->stream));
        SBA_TRY(vars_in(p, p->io_x, p->x));
        SBA_TRY(pt_reset_state(p));
        SBA_TRY(pt_run_assemble(p, 1, 1, loss, f_scale));
        pt_accept(p);
        SBA_TRY(pt_run_jvp1(p, 1, loss, f_scale, -1.0));
        k_control_reg<<<1, 32, 0, p->stream>>>(p->scal, -1.0, reg);
        SBA_TRY(check_launch(p));
        SBA_TRY(pt_run_schur(p, loss, f_scale));
    } else {
        SBA_CUDA(cudaMemsetAsync(p->scal, 0, SC_COUNT * sizeof(double), p->stream));
        SBA_CUDA(cudaMemcpyAsync(p->x, x, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        if (uploaded) SBA_CUDA(cudaEventRecord(uploaded, p->stream));
        SBA_TRY(run_prepare(p, p->x, p->camrec));
        SBA_TRY(run_assemble(p, p->x, p->camrec, loss, f_scale));
        SBA_TRY(run_scale_dots(p, 1));
        k_control_reg<<<1, 32, 0, p->stream>>>(p->scal, -1.0, reg);
        SBA_TRY(check_launch(p));
        PhaseTimer tm;
        tm.p = p;
        SBA_TRY(run_gauss_newton_step(p, loss, f_scale, tm, true));
    }
    return SBA_OK;
}

extern "C" int sba_reduced_system(sba_problem* p, const double* x, int32_t loss, double f_scale, double reg, double* S,
                                  double* rhs)
{
    if (!p || !x || !S || !rhs || !(reg >= 0.0)) { set_error("bad argument"); return SBA_E_INVALID; }
    if (p->world > 1) { set_error("sba_reduced_system: single-rank problems only"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    const size_t ns = (size_t)p->M * p->nc;
    SBA_TRY(form_reduced_system(p, x, loss, f_scale, reg));
    SBA_CUDA(cudaMemcpyAsync(S, p->S, ns * ns * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_CUDA(cudaMemcpyAsync(rhs, p->S + ns * ns, ns * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

// Posterior covariance at x (sba_cov.cuh has the definitions): the undamped reduced camera system through the solver's own
// Schur path, its Cholesky factor with the pivot test, S^-1, then one pass over the tracks.
constexpr double COV_PIVOT_THRESHOLD = 1e-12;
constexpr size_t COV_SMEM_MAX = 100 * 1024;     // s2 S^-1 goes to shared memory up to this size (ns <= 113)

// Warp tiles of the point pass in the internal track order (runs of whole tracks of <= 32 observations, a longer track a tile
// of its own): the generic engine has them; the pattern engine's are built once, on the first call, from its track offsets.
static int cov_tiles(sba_problem* p, const int** tiles, int* n_tiles)
{
    if (p->engine == 0) { *tiles = p->tile_obs; *n_tiles = p->n_tiles; return SBA_OK; }
    if (!p->cov_tile_obs) {
        std::vector<int> tp((size_t)p->N + 1), to(1, 0);
        SBA_CUDA(cudaMemcpyAsync(tp.data(), p->track_ptr, tp.size() * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        SBA_CUDA(cudaStreamSynchronize(p->stream));
        int cur = 0;
        for (int i = 0; i < p->N; ++i) {
            const int L = tp[i + 1] - tp[i];
            if (L == 0) continue;
            if (cur > 0 && cur + L > 32) { to.push_back(tp[i]); cur = 0; }
            cur += L;
            if (cur >= 32) { to.push_back(tp[i + 1]); cur = 0; }
        }
        if (cur > 0) to.push_back(tp[p->N]);
        SBA_TRY(dev_upload(p, &p->cov_tile_obs, to, p->stream));
        SBA_CUDA(cudaStreamSynchronize(p->stream));
        p->cov_n_tiles = (int)to.size() - 1;
    }
    *tiles = p->cov_tile_obs; *n_tiles = p->cov_n_tiles;
    return SBA_OK;
}

extern "C" int sba_covariance(sba_problem* p, const double* x, int32_t loss, double f_scale, double sigma2, double* cov_cam,
                              double* cov_pts, double* sigma2_out, double* min_pivot_ratio_out)
{
    if (!p || !x) { set_error("null argument"); return SBA_E_INVALID; }
    if (p->world > 1) { set_error("sba_covariance: single-rank problems only"); return SBA_E_INVALID; }
    if (p->use_pcg) { set_error("sba_covariance: the PCG path forms no dense reduced camera system"); return SBA_E_INVALID; }
    if (p->n_common) { set_error("sba_covariance: not available with shared calibration (n_common > 0)"); return SBA_E_INVALID; }
    const int M = p->M, nc = p->nc, ns = M * nc;
    const long long n_free = (long long)(M - p->n_cam_fix) * nc + 3LL * (p->N - p->n_pts_fix);
    const long long dof = 2 * (long long)p->K - n_free;
    if (!(sigma2 > 0.0) && dof <= 0) {
        set_error("sba_covariance: " + std::to_string(dof) + " degrees of freedom (2 K - free variables): sigma^2 cannot be estimated");
        return SBA_E_INVALID;
    }
    SBA_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = p->stream;
    if (!p->cov_cam) {
        SBA_TRY(dev_alloc(p, &p->cov_cam, (size_t)ns * ns));
        SBA_TRY(dev_alloc(p, &p->cov_pts, 6 * (size_t)p->N));
        SBA_TRY(dev_alloc(p, &p->cov_diag, 4));
        for (cudaEvent_t& e : p->cov_ev) SBA_CUDA(cudaEventCreate(&e));
    }
    const int* tiles = nullptr;
    int n_tiles = 0;
    SBA_TRY(cov_tiles(p, &tiles, &n_tiles));
    // phase 0 starts when x is on the device (the upload from pageable host memory is not device work)
    SBA_TRY(form_reduced_system(p, x, loss, f_scale, 0.0, p->cov_ev[0]));
    // the pattern engine's evaluation swapped its buffer sets (pt_accept): swap them back on every exit, so that the handle is
    // left with the same buffer roles as before the call
    struct Unswap { sba_problem* p; ~Unswap() { if (p->engine == 1) pt_accept(p); } } unswap{p};
    // sigma2 estimated: the cost at x by the residual kernel of sba_residuals, in float64 like the Jacobian rows (rpc_float32 is
    // for fun parity only).  sigma2 given: the assembly's own cost serves the finiteness check.
    int cost_slot = p->engine == 1 ? SC_COST_NEW : SC_COST;
    if (!(sigma2 > 0.0)) {
        cost_slot = SC_SCRATCH;
        SBA_TRY(run_residual(p, p->x, p->camrec, loss, f_scale, nullptr, SC_SCRATCH, 0));
    }
    SBA_CUDA(cudaEventRecord(p->cov_ev[1], s));
    // factor (frozen slots: identity rows of S) and pivot test
    SBA_TRY(launch_cholesky_solve(p->S, p->S + (size_t)ns * ns, p->delta, ns, p->scal + SC_CHOL_FAIL, p->chol_work, s, true));
    p->launches++;
    SBA_CUDA(cudaMemsetAsync(p->cov_diag, 0, 4 * sizeof(double), s));
    k_cov_pivots<<<1, 256, 0, s>>>(p->S, p->camsys, ns, nc, p->n_cam_fix, p->scal + SC_CHOL_FAIL, COV_PIVOT_THRESHOLD, p->cov_diag);
    SBA_TRY(check_launch(p));
    SBA_CUDA(cudaEventRecord(p->cov_ev[2], s));
    double* h = p->h_scal + SC_COUNT;            // the slots after the scalar block (used by the PCG path only)
    SBA_CUDA(cudaMemcpyAsync(h, p->cov_diag, 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
    SBA_CUDA(cudaMemcpyAsync(p->h_scal + cost_slot, p->scal + cost_slot, sizeof(double), cudaMemcpyDeviceToHost, s));
    SBA_CUDA(cudaStreamSynchronize(s));
    const double min_ratio = h[0], cost = p->h_scal[cost_slot];
    if (min_pivot_ratio_out) *min_pivot_ratio_out = min_ratio;
    if (h[1] >= 0.0) {
        const int k = (int)h[1];
        char msg[256];
        snprintf(msg, sizeof(msg),
                 "sba_covariance: the reduced camera system is rank deficient (gauge not fixed?): camera %d, slot %d: pivot ratio "
                 "L_kk^2 / U_kk = %.3e <= %.0e", k / nc, k % nc, h[2], COV_PIVOT_THRESHOLD);
        set_error(msg);
        return SBA_E_NUMERIC;
    }
    if (!std::isfinite(cost)) { set_error("sba_covariance: residuals are not finite at x"); return SBA_E_NUMERIC; }
    const double s2 = sigma2 > 0.0 ? sigma2 : 2.0 * cost / (double)dof;
    // s2 S^-1, exactly symmetric, frozen rows / columns 0
    k_cov_inverse<<<(ns + 31) / 32, 256, 0, s>>>(p->S, ns, p->cov_cam);
    SBA_TRY(check_launch(p));
    k_cov_finish<<<grid_for((long long)ns * ns, 256, NUM_SMS * 4), 256, 0, s>>>(p->cov_cam, ns, p->n_cam_fix * nc, s2);
    SBA_TRY(check_launch(p));
    SBA_CUDA(cudaEventRecord(p->cov_ev[3], s));
    {
        const size_t c_bytes = (size_t)ns * ns * sizeof(double);
        const int in_smem = c_bytes <= COV_SMEM_MAX;
        const int npf = p->engine == 1 ? p->n_pts_fix_int : p->n_pts_fix;
        const int* perm = p->engine == 1 ? p->trk_new2old : nullptr;
        const int grid_long = std::max(1, std::min((n_tiles + 3) / 4, NUM_SMS * 4));
#define L(MODEL, NC)                                                                                                          \
    {                                                                                                                         \
        const size_t smem = ((size_t)COV_WARPS * cov_warp_doubles<NC>() + COV_WARPS * 32 / 2) * sizeof(double) +           \
                            (in_smem ? c_bytes : 0);                                                                          \
        SBA_CUDA(cudaFuncSetAttribute(k_cov_points<MODEL, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
        const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (size_t)(200 * 1024) / smem));                      \
        const int grid = std::max(1, std::min((n_tiles + COV_WARPS - 1) / COV_WARPS, NUM_SMS * per_sm));                   \
        k_cov_points<MODEL, NC><<<grid, COV_THREADS, smem, s>>>(obs_arrays(p), tiles, n_tiles, p->x + (size_t)ns, p->camrec,  \
                                                               p->rpc_tab, p->n_cam_fix, npf, loss, f_scale, p->cov_cam, ns,   \
                                                               in_smem, s2, perm, p->cov_pts, p->cov_diag + 3);               \
        SBA_TRY(check_launch(p));                                                                                             \
        k_cov_long_tracks<MODEL, NC><<<grid_long, 128, 0, s>>>(obs_arrays(p), tiles, n_tiles, p->x + (size_t)ns, p->camrec,   \
                                                              p->rpc_tab, p->n_cam_fix, npf, loss, f_scale, p->cov_cam, ns, s2, \
                                                              perm, p->cov_pts, p->cov_diag + 3);                             \
    }
        SBA_DISPATCH(p, L);
#undef L
        SBA_TRY(check_launch(p));
    }
    SBA_CUDA(cudaEventRecord(p->cov_ev[4], s));
    if (cov_cam) SBA_CUDA(cudaMemcpyAsync(cov_cam, p->cov_cam, (size_t)ns * ns * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (cov_pts) SBA_CUDA(cudaMemcpyAsync(cov_pts, p->cov_pts, 6 * (size_t)p->N * sizeof(double), cudaMemcpyDeviceToHost, s));
    SBA_CUDA(cudaMemcpyAsync(h + 3, p->cov_diag + 3, sizeof(double), cudaMemcpyDeviceToHost, s));
    SBA_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < 4; ++k) {
        float ms = 0.f;
        SBA_CUDA(cudaEventElapsedTime(&ms, p->cov_ev[k], p->cov_ev[k + 1]));
        p->cov_ms[k] = ms;
    }
    if (h[3] != 0.0) {
        set_error("sba_covariance: " + std::to_string((long long)h[3]) + " free point(s) with a singular 3x3 block V_t");
        return SBA_E_NUMERIC;
    }
    if (sigma2_out) *sigma2_out = s2;
    return SBA_OK;
}

extern "C" int sba_covariance_phase_ms(const sba_problem* p, double* ms4)
{
    if (!p || !ms4) { set_error("null argument"); return SBA_E_INVALID; }
    for (int k = 0; k < 4; ++k) ms4[k] = p->cov_ms[k];
    return SBA_OK;
}

extern "C" int sba_solve_device(sba_problem* p, const double* x0_dev, const sba_solve_opts* opts, double* x_dev,
                                double* r_dev, sba_solve_info* info)
{
    if (!p || !x0_dev || !opts || !info) { set_error("null argument"); return SBA_E_INVALID; }
    if (p->world > 1 && !p->allreduce && !p->comm_ready) { set_error("world_size > 1 needs sba_comm_import or sba_problem_set_allreduce"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_TRY(vars_in(p, x0_dev, p->x));
    SBA_TRY(solve_trf(p, opts, info));
    if (x_dev) SBA_TRY(vars_out(p, p->x, x_dev));
    if (r_dev) {
        SBA_TRY(residuals_ext(p, p->x, p->camrec, SBA_LOSS_LINEAR, 1.0, r_dev, SC_SCRATCH, p->rpc_f32));
        info->gpu_launches = p->launches;
    }
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

extern "C" int sba_solve(sba_problem* p, const double* x0, const sba_solve_opts* opts, double* x, double* r,
                         sba_solve_info* info)
{
    if (!p || !x0 || !opts || !info) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_CUDA(cudaMemcpyAsync(p->io_x, x0, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    SBA_TRY(sba_solve_device(p, p->io_x, opts, x ? p->io_x : nullptr, r ? p->r_out : nullptr, info));
    if (x) SBA_CUDA(cudaMemcpyAsync(x, p->io_x, (size_t)p->n * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (r) SBA_CUDA(cudaMemcpyAsync(r, p->r_out, 2 * (size_t)p->K * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

extern "C" int sba_assemble_device(sba_problem* p, const double* x_dev, int32_t loss, double f_scale, float* ms)
{
    if (!p || !x_dev) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_TRY(vars_in(p, x_dev, p->x));
    if (p->engine == 1) {
        SBA_TRY(pt_reset_state(p));
        SBA_CUDA(cudaEventRecord(p->ev0, p->stream));
        SBA_TRY(pt_run_assemble(p, 1, 1, loss, f_scale));
        SBA_CUDA(cudaEventRecord(p->ev1, p->stream));
    } else {
        SBA_TRY(run_prepare(p, p->x, p->camrec));
        SBA_CUDA(cudaEventRecord(p->ev0, p->stream));
        SBA_TRY(run_assemble(p, p->x, p->camrec, loss, f_scale));
        SBA_CUDA(cudaEventRecord(p->ev1, p->stream));
    }
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    float t = 0.f;
    SBA_CUDA(cudaEventElapsedTime(&t, p->ev0, p->ev1));
    if (ms) *ms = t;
    return SBA_OK;
}

extern "C" int sba_tr2d(const double B[4], const double g[2], double Delta, double p_out[2])
{
    return sba::solve_trust_region_2d(B[0], B[1], B[3], g[0], g[1], Delta, p_out) ? 1 : 0;
}

// sba_solve plus the two per-observation error vectors the reference's driver returns (ba_core.py:304-305), computed
// on the device: err_init at x0, err at the solution (K doubles each, either may be NULL).
// sba_solve_device plus the two per-observation error vectors (device pointers, caller's order; any may be NULL)
extern "C" int sba_solve_errors_device(sba_problem* p, const double* x0_dev, const sba_solve_opts* opts, double* x_dev,
                                       double* err_init_dev, double* err_dev, sba_solve_info* info)
{
    if (!p || !x0_dev || !opts || !info) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    if (err_init_dev) {
        SBA_TRY(vars_in(p, x0_dev, p->x_new));
        SBA_TRY(run_prepare(p, p->x_new, p->camrec_new));
        SBA_TRY(residuals_ext(p, p->x_new, p->camrec_new, SBA_LOSS_LINEAR, 1.0, p->r_out, SC_SCRATCH, p->rpc_f32));
        SBA_TRY(reproj_errors_ext(p, p->r_out, err_init_dev));
    }
    SBA_TRY(sba_solve_device(p, x0_dev, opts, x_dev, err_dev ? p->r_out : nullptr, info));
    if (err_dev) SBA_TRY(reproj_errors_ext(p, p->r_out, err_dev));
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}

extern "C" int sba_solve_errors(sba_problem* p, const double* x0, const sba_solve_opts* opts, double* x, double* err_init,
                                double* err, sba_solve_info* info)
{
    if (!p || !x0 || !opts || !info) { set_error("null argument"); return SBA_E_INVALID; }
    SBA_CUDA(cudaSetDevice(p->device));
    SBA_CUDA(cudaMemcpyAsync(p->io_x, x0, (size_t)p->n * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    if (err_init) {
        SBA_TRY(vars_in(p, p->io_x, p->x_new));
        SBA_TRY(run_prepare(p, p->x_new, p->camrec_new));
        SBA_TRY(residuals_ext(p, p->x_new, p->camrec_new, SBA_LOSS_LINEAR, 1.0, p->r_out, SC_SCRATCH, p->rpc_f32));
        SBA_TRY(reproj_errors_ext(p, p->r_out, p->err_out));
        SBA_CUDA(cudaMemcpyAsync(err_init, p->err_out, (size_t)p->K * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    SBA_TRY(sba_solve_device(p, p->io_x, opts, x ? p->io_x : nullptr, err ? p->r_out : nullptr, info));
    if (x) SBA_CUDA(cudaMemcpyAsync(x, p->io_x, (size_t)p->n * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (err) {
        SBA_TRY(reproj_errors_ext(p, p->r_out, p->err_out));
        SBA_CUDA(cudaMemcpyAsync(err, p->err_out, (size_t)p->K * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    SBA_CUDA(cudaStreamSynchronize(p->stream));
    return SBA_OK;
}
