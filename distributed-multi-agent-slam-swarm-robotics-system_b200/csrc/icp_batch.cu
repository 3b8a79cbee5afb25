// Batched point-to-point ICP (mapmerge_icp_register_batch in include/occgrid_b200.h, DESIGN §6f):
// A source clouds registered against ONE target cloud.  The target's cell list is built once with
// the launches of mapmerge_icp_register (icp_build_index); then k_icp_loop_batch runs the iteration
// loops of all agents in one cooperative launch.  Every agent's points are dealt in the virtual
// blocks of k_icp_loop and its partials are folded by the same icp_fold_eval / icp_fold_solve, so
// each agent's result equals a separate mapmerge_icp_register call bit for bit, whatever the grid.
#include <cmath>

#include "icp_core.cuh"

namespace occ {

// ---- the batched loop: A source clouds against one target --------------------------------------
// Work is dealt in (agent, virtual block) items: agent a owns the virtual blocks vb_off[a] ..
// vb_off[a + 1] - 1, point i of the agent sits in its block i / kIT, lane i % kIT, exactly as in
// k_icp_loop, so every partial is the same sum.  An item is always served by CTA vb % gridDim.x,
// which therefore owns its points' working copy and correspondences across phases.  Folds are
// dealt per agent (agent a on CTA a % gridDim.x) and reuse icp_fold_eval / icp_fold_solve on a view
// of the agent's own partials; the agent's state lives in global memory.  One iteration is four
// phases separated by grid barriers: covariance | solve | move + associate | evaluate.  A converged
// agent's items and folds are skipped; the loop ends when no agent is running or at max_iteration.
struct IcpBatch {
    const double* sx; const double* sy;            // caller's clouds, agent a at [off[a], off[a + 1])
    const long long* off;                          // [n_agents + 1]
    int n_agents, max_iteration;
    long long cap;                                 // points the working copy holds
    double* px; double* py; unsigned int* corr;    // working copy of the sources, indexed like sx
    IcpIndex ix;
    double r, r2, rel_f, rel_r;
    double* partial; double* partial2;             // [n_vb][6], [n_vb][2] as in IcpLoop
    unsigned int* vb_off;                          // [n_agents + 1] first virtual block of every agent
    int* vb_agent;                                 // [n_vb] agent of every virtual block
    IcpState* state;                               // [n_agents]
    double* result;                                // [n_agents][20]
    unsigned int* bar;                             // [0, 4) grid_barrier, [4] abort flag, [5] table valid,
                                                   // [6] agents still running; zeroed before each launch
};

// Agent a's registration as k_icp_loop would see it: what icp_fold_eval and icp_fold_solve read.
__device__ __forceinline__ IcpLoop icp_agent_view(const IcpBatch& p, int a) {
    IcpLoop q;
    const long long b = __ldcg(p.off + a);
    const unsigned int vb0 = __ldcg(p.vb_off + a);
    q.px = p.px + b; q.py = p.py + b; q.n = __ldcg(p.off + a + 1) - b;
    q.ix = p.ix; q.r = p.r; q.r2 = p.r2; q.rel_f = p.rel_f; q.rel_r = p.rel_r;
    q.corr = p.corr + b;
    q.partial = p.partial + (size_t)vb0 * 6; q.partial2 = p.partial2 + (size_t)vb0 * 2;
    q.n_vb = (int)(__ldcg(p.vb_off + a + 1) - vb0);
    q.max_iteration = p.max_iteration; q.state = p.state + a; q.bar = p.bar;
    return q;
}

// apply = false: first association, which also copies the sources into the working copy.
__device__ __forceinline__ void icp_batch_assoc(const IcpBatch& p, unsigned int n_vb, bool apply) {
    __shared__ double s_U[16];
    for (unsigned int vb = blockIdx.x; vb < n_vb; vb += gridDim.x) {
        const int a = __ldcg(p.vb_agent + vb);
        const IcpState* L = p.state + a;
        if (__ldcg(&L->done)) continue;                          // uniform over the CTA
        const long long b = __ldcg(p.off + a), n = __ldcg(p.off + a + 1) - b;
        const long long i = (long long)(vb - __ldcg(p.vb_off + a)) * kIT + threadIdx.x;
        if (apply) {
            if (threadIdx.x < 16) s_U[threadIdx.x] = __ldcg(L->U + threadIdx.x);
            __syncthreads();
        }
        double v[6] = {0, 0, 0, 0, 0, 0};
        if (i < n) {
            double x, y;
            if (apply) {                                         // PointCloud::Transform, as icp_assoc_phase
                x = p.px[b + i]; y = p.py[b + i];
                const double* U = s_U;
                const double w = OCC_DADD(OCC_DADD(OCC_DMUL(U[12], x), OCC_DMUL(U[13], y)), U[15]);
                const double nx = OCC_DDIV(OCC_DADD(OCC_DADD(OCC_DMUL(U[0], x), OCC_DMUL(U[1], y)), U[3]), w);
                const double ny = OCC_DDIV(OCC_DADD(OCC_DADD(OCC_DMUL(U[4], x), OCC_DMUL(U[5], y)), U[7]), w);
                x = nx; y = ny;
            } else {
                x = p.sx[b + i]; y = p.sy[b + i];
            }
            p.px[b + i] = x; p.py[b + i] = y;
            double d2;
            const unsigned int q = icp_nearest(p.ix, x, y, p.r, p.r2, &d2);
            p.corr[b + i] = q;
            if (q != 0xffffffffu) { v[0] = 1.0; v[1] = d2; v[2] = x; v[3] = y; v[4] = p.ix.x[q]; v[5] = p.ix.y[q]; }
        }
        block_sum<6>(v, p.partial + (size_t)vb * 6);            // its syncs also retire s_U before the next item
    }
}

__device__ __forceinline__ void icp_batch_cov(const IcpBatch& p, unsigned int n_vb) {
    __shared__ double s_mean[4];
    for (unsigned int vb = blockIdx.x; vb < n_vb; vb += gridDim.x) {
        const int a = __ldcg(p.vb_agent + vb);
        const IcpState* L = p.state + a;
        if (__ldcg(&L->done)) continue;
        const long long b = __ldcg(p.off + a), n = __ldcg(p.off + a + 1) - b;
        const long long i = (long long)(vb - __ldcg(p.vb_off + a)) * kIT + threadIdx.x;
        if (threadIdx.x < 4) s_mean[threadIdx.x] = __ldcg(L->mean + threadIdx.x);
        __syncthreads();
        double v[2] = {0, 0};
        if (i < n) {                                             // as icp_cov_phase
            const unsigned int q = p.corr[b + i];
            if (q != 0xffffffffu) {
                const double sx = p.px[b + i] - s_mean[0], sy = p.py[b + i] - s_mean[1];
                const double tx = p.ix.x[q] - s_mean[2], ty = p.ix.y[q] - s_mean[3];
                v[0] = sx * tx + sy * ty;
                v[1] = sx * ty - sy * tx;
            }
        }
        block_sum<2>(v, p.partial2 + (size_t)vb * 2);
    }
}

// kind 0: first evaluation, 1: solve, 2: evaluation after a move.
__device__ __forceinline__ void icp_batch_fold(const IcpBatch& p, int kind) {
    for (int a = blockIdx.x; a < p.n_agents; a += gridDim.x) {
        IcpState* L = p.state + a;
        if (__ldcg(&L->done)) continue;
        const IcpLoop q = icp_agent_view(p, a);
        if (kind == 1) icp_fold_solve(q, L);
        else icp_fold_eval(q, L, kind == 0);
        if (kind == 2 && threadIdx.x == 0 && L->done) atomicSub(p.bar + 6, 1u);   // a counter, not a sum
    }
}

__global__ void __launch_bounds__(kIT, 3)
k_icp_loop_batch(const IcpBatch p) {
    unsigned int target = 0;
    int* abort_flag = reinterpret_cast<int*>(p.bar + 4);
    volatile unsigned int* vbar = p.bar;
    const int A = p.n_agents;
    if (blockIdx.x == 0) {                                     // check the offset table, lay out the virtual blocks
        int bad = 0;
        for (int a = threadIdx.x; a < A; a += kIT) {
            const long long b = p.off[a], e = p.off[a + 1];
            if (e < b || (a == 0 && b != 0)) bad = 1;
            p.vb_off[a] = (unsigned int)((e - b + kIT - 1) / kIT);
        }
        if (threadIdx.x == 0 && p.off[A] > p.cap) bad = 1;
        bad = __syncthreads_or(bad);
        if (!bad) {
            const unsigned long long n_vb = cta_scan_in_place<4>(p.vb_off, A, 0ull);
            if (threadIdx.x == 0) p.vb_off[A] = (unsigned int)n_vb;
        }
        if (threadIdx.x == 0) vbar[5] = bad ? 0u : 1u;
    }
    bool alive = grid_barrier(p.bar, target, abort_flag);
    if (!alive || vbar[5] == 0u) {                             // every row: identity, zeros, iterations -1 / -2
        for (int a = blockIdx.x; a < A; a += gridDim.x)
            if (threadIdx.x == 0)
                for (int k = 0; k < 20; ++k) p.result[(size_t)a * 20 + k] = k < 16 ? ((k % 5 == 0) ? 1.0 : 0.0) : (k == 18 ? (alive ? -2.0 : -1.0) : 0.0);
        return;
    }
    const unsigned int n_vb = __ldcg(p.vb_off + A);
    for (unsigned int vb = blockIdx.x * kIT + threadIdx.x; vb < n_vb; vb += gridDim.x * kIT) {
        int lo = 0, hi = A;                                    // vb_off[lo] <= vb < vb_off[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldcg(p.vb_off + mid) <= vb) lo = mid; else hi = mid;
        }
        p.vb_agent[vb] = lo;
    }
    for (int a = blockIdx.x; a < A; a += gridDim.x)
        if (threadIdx.x == 0) {
            IcpState* L = p.state + a;
            for (int i = 0; i < 16; ++i) { L->T[i] = (i % 5 == 0) ? 1.0 : 0.0; L->U[i] = L->T[i]; }
            L->fitness = L->rmse = L->iterations = L->n_corr = 0.0;
            L->mean[0] = L->mean[1] = L->mean[2] = L->mean[3] = 0.0;
            const bool empty = p.off[a + 1] == p.off[a];          // never launched: identity, zeros
            L->done = empty ? 1 : 0;
            if (!empty) atomicAdd(p.bar + 6, 1u);
        }
    alive = grid_barrier(p.bar, target, abort_flag);
    if (alive) icp_batch_assoc(p, n_vb, false);
    if (alive) alive = grid_barrier(p.bar, target, abort_flag);
    if (alive) icp_batch_fold(p, 0);
    if (alive) alive = grid_barrier(p.bar, target, abort_flag);
    for (int it = 0; alive && it < p.max_iteration && vbar[6] != 0u; ++it) {   // vbar[6] only changes in phase 4
        icp_batch_cov(p, n_vb);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
        icp_batch_fold(p, 1);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
        icp_batch_assoc(p, n_vb, true);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
        icp_batch_fold(p, 2);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
    }
    for (int a = blockIdx.x; a < A; a += gridDim.x)           // the agent's own CTA wrote its state
        if (threadIdx.x == 0) {
            const IcpState* L = p.state + a;
            double* row = p.result + (size_t)a * 20;
            for (int k = 0; k < 16; ++k) row[k] = L->T[k];
            row[16] = L->fitness; row[17] = L->rmse;
            row[18] = (!alive && !L->done) ? -1.0 : L->iterations;   // a barrier timed out: the host reports it
            row[19] = L->n_corr;
        }
}

constexpr int kIcpBatchMaxAgents = 65535;
static_assert(sizeof(IcpState) == 328, "the header states 328 bytes of state per agent");
constexpr int64_t kIcpBatchMaxPoints = 1ll << 39;          // keeps the virtual block numbers below 2^32

struct IcpBatchLayout {
    size_t cnt, start, cursor, sx, sy, sidx, block_sums, state, vb_off, bar;    // fixed part
    size_t px, py, corr, partial, partial2, vb_agent, total;                   // grows with the points
};

static IcpBatchLayout icp_batch_layout(int64_t target_points, int64_t points, int n_agents, int64_t cells) {
    IcpBatchLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    L.cnt = take((size_t)(cells + 1) * 4); L.start = take((size_t)(cells + 1) * 4); L.cursor = take((size_t)(cells + 1) * 4);
    L.sx = take((size_t)target_points * 8); L.sy = take((size_t)target_points * 8); L.sidx = take((size_t)target_points * 4);
    L.block_sums = take((size_t)((cells + kScanBlockIcp - 1) / kScanBlockIcp + 1) * 4);
    L.state = take((size_t)n_agents * sizeof(IcpState));
    L.vb_off = take((size_t)(n_agents + 1) * 4);
    L.bar = take(256);
    const size_t vbs = (size_t)((points + kIT - 1) / kIT) + (size_t)n_agents;   // >= sum over agents of ceil(n_a / kIT)
    L.px = take((size_t)points * 8); L.py = take((size_t)points * 8); L.corr = take((size_t)points * 4);
    L.partial = take(vbs * 6 * 8); L.partial2 = take(vbs * 2 * 8); L.vb_agent = take(vbs * 4);
    L.total = o;
    return L;
}

static int icp_batch_grid_cap = 0;                         // mapmerge_icp_batch_set_max_ctas

// Argument checks shared by the batched workspace query and call; sets the error message.
static bool icp_batch_args_ok(const char* who, int64_t n_target, int64_t points, int n_agents, int32_t cells_w, int32_t cells_h) {
    if (n_agents < 1 || n_agents > kIcpBatchMaxAgents) {
        set_last_error("%s: n_agents %d outside 1..%d", who, n_agents, kIcpBatchMaxAgents);
        return false;
    }
    if (n_target < 1 || n_target >= 0xffffffffll) {
        set_last_error("%s: n_target %lld outside 1..2^32 - 2", who, (long long)n_target);
        return false;
    }
    if (points < 0 || points > kIcpBatchMaxPoints) {
        set_last_error("%s: total_source_points %lld outside 0..2^39", who, (long long)points);
        return false;
    }
    if (cells_w < 1 || cells_h < 1) {
        set_last_error("%s: cells %d x %d below 1", who, (int)cells_w, (int)cells_h);
        return false;
    }
    // everything but the cell tables ((cells + 1) * 12 bytes and the scan's block sums) stays below 2^46 bytes
    const uint64_t cells = (uint64_t)cells_w * (uint64_t)cells_h;
    if (cells + 1 > (SIZE_MAX - (1ull << 46)) / 13) {
        set_last_error("%s: a cell list of %d x %d cells overflows size_t", who, (int)cells_w, (int)cells_h);
        return false;
    }
    return true;
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t mapmerge_icp_register_batch_workspace_bytes(int64_t n_target, int64_t total_source_points, int n_agents,
                                                   int32_t cells_w, int32_t cells_h) {
    if (!icp_batch_args_ok("mapmerge_icp_register_batch_workspace_bytes", n_target, total_source_points, n_agents, cells_w, cells_h))
        return 0;
    return icp_batch_layout(n_target, total_source_points, n_agents, (int64_t)cells_w * cells_h).total;
}

int mapmerge_icp_batch_set_max_ctas(int ctas) {
    if (ctas < 0) { set_last_error("mapmerge_icp_batch_set_max_ctas: ctas %d below 0", ctas); return OCCGRID_E_ARG; }
    icp_batch_grid_cap = ctas;
    return OCCGRID_OK;
}

int mapmerge_icp_register_batch(const double* d_sx, const double* d_sy, const int64_t* d_offsets, int n_agents,
                                const double* d_tx, const double* d_ty, int64_t n_target, double min_x, double min_y,
                                double cell, int32_t cells_w, int32_t cells_h, double max_correspondence_distance,
                                int32_t max_iteration, double relative_fitness, double relative_rmse, double* d_results,
                                void* d_ws, size_t ws_bytes, void* stream) {
    static const char* who = "mapmerge_icp_register_batch";
    if (!d_sx || !d_sy || !d_offsets || !d_tx || !d_ty || !d_results || !d_ws) {
        set_last_error("%s: NULL pointer", who);
        return OCCGRID_E_ARG;
    }
    if (!icp_batch_args_ok(who, n_target, 0, n_agents, cells_w, cells_h)) return OCCGRID_E_ARG;
    if (!(std::isfinite(cell) && cell > 0.0)) {
        set_last_error("%s: cell %g must be finite and > 0", who, cell);
        return OCCGRID_E_ARG;
    }
    if (!(std::isfinite(max_correspondence_distance) && max_correspondence_distance > 0.0)) {
        set_last_error("%s: threshold %g must be finite and > 0", who, max_correspondence_distance);
        return OCCGRID_E_ARG;
    }
    if (max_iteration < 0) {
        set_last_error("%s: max_iteration %d below 0", who, (int)max_iteration);
        return OCCGRID_E_ARG;
    }
    const int64_t cells = (int64_t)cells_w * cells_h;
    if (ws_bytes < icp_batch_layout(n_target, 0, n_agents, cells).total) {
        set_last_error("%s: workspace too small", who);
        return OCCGRID_E_WORKSPACE;
    }
    // the point capacity: the most points whose layout fits ws_bytes
    int64_t lo = 0, hi = kIcpBatchMaxPoints;
    while (lo < hi) {
        const int64_t mid = lo + (hi - lo + 1) / 2;
        if (icp_batch_layout(n_target, mid, n_agents, cells).total <= ws_bytes) lo = mid; else hi = mid - 1;
    }
    const IcpBatchLayout L = icp_batch_layout(n_target, lo, n_agents, cells);
    char* ws = reinterpret_cast<char*>(d_ws);
    auto at = [&](size_t off) { return reinterpret_cast<void*>(ws + off); };
    unsigned int* cnt = static_cast<unsigned int*>(at(L.cnt));
    unsigned int* bar = static_cast<unsigned int*>(at(L.bar));
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0;
    OCC_CUDA_TRY(cudaGetDevice(&dev));
    static int resident_by_device[64] = {};
    int resident = (dev >= 0 && dev < 64) ? resident_by_device[dev] : 0;
    if (resident == 0) {
        int sms = 0, per_sm = 0;
        OCC_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        OCC_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_icp_loop_batch, kIT, 0));
        if (sms <= 0 || per_sm <= 0) { set_last_error("%s: the loop kernel does not fit the device", who); return OCCGRID_E_CUDA; }
        resident = sms * per_sm;
        if (dev >= 0 && dev < 64) resident_by_device[dev] = resident;
    }
    const int grid = (icp_batch_grid_cap > 0 && icp_batch_grid_cap < resident) ? icp_batch_grid_cap : resident;
    ProfileScope ps(K_ICP_BATCH, st, 6);
    OCC_CUDA_TRY(cudaMemsetAsync(cnt, 0, (size_t)(cells + 1) * 4, st));
    icp_build_index(d_tx, d_ty, n_target, min_x, min_y, cell, cells_w, cells_h, cnt, static_cast<unsigned int*>(at(L.start)),
                    static_cast<unsigned int*>(at(L.cursor)), static_cast<unsigned int*>(at(L.block_sums)),
                    static_cast<double*>(at(L.sx)), static_cast<double*>(at(L.sy)), static_cast<unsigned int*>(at(L.sidx)), st);
    OCC_CUDA_TRY(cudaGetLastError());
    IcpBatch p;
    p.sx = d_sx; p.sy = d_sy; p.off = reinterpret_cast<const long long*>(d_offsets);
    p.n_agents = n_agents; p.max_iteration = max_iteration; p.cap = lo;
    p.px = static_cast<double*>(at(L.px)); p.py = static_cast<double*>(at(L.py)); p.corr = static_cast<unsigned int*>(at(L.corr));
    p.ix.min_x = min_x; p.ix.min_y = min_y; p.ix.cell = cell; p.ix.w = cells_w; p.ix.h = cells_h;
    p.ix.start = static_cast<const unsigned int*>(at(L.start)); p.ix.x = static_cast<const double*>(at(L.sx));
    p.ix.y = static_cast<const double*>(at(L.sy)); p.ix.idx = static_cast<const unsigned int*>(at(L.sidx));
    p.r = max_correspondence_distance; p.r2 = max_correspondence_distance * max_correspondence_distance;
    p.rel_f = relative_fitness; p.rel_r = relative_rmse;
    p.partial = static_cast<double*>(at(L.partial)); p.partial2 = static_cast<double*>(at(L.partial2));
    p.vb_off = static_cast<unsigned int*>(at(L.vb_off)); p.vb_agent = static_cast<int*>(at(L.vb_agent));
    p.state = static_cast<IcpState*>(at(L.state)); p.result = d_results; p.bar = bar;
    OCC_CUDA_TRY(cudaMemsetAsync(bar, 0, 256, st));
    void* args[] = {&p};
    OCC_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_icp_loop_batch, dim3((unsigned)grid), dim3(kIT), args, 0, st));
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
