// Point-to-point ICP of a local cloud against the global cloud (SURVEY §8 rows a13 / f3).
//
// Reference call site: server_nodes/map_merger.py:45-56
//     reg_p2p = o3d.pipelines.registration.registration_icp(local_pcd, self.global_pcd, 1.0, I,
//                   TransformationEstimationPointToPoint(), ICPConvergenceCriteria(max_iteration=30))
//     if reg_p2p.fitness < 0.6: reject
// Open3D is a third-party dependency that is absent and un-pinned here (parity unpinned); this
// follows its published algorithm (Registration.cpp / TransformationEstimation.cpp, Eigen
// Umeyama.h), restated on the CPU in oracle/icp_oracle.py:
//   * correspondences: the nearest target point of every source point, kept when its squared
//     distance is < max_dist^2; fitness = #corr / #source; inlier_rmse = sqrt(sum d^2 / #corr);
//   * update = rigid Umeyama fit of the corresponding pairs, T = update * T, source transformed
//     by update; repeated max_iteration times or until |d fitness| and |d rmse| < 1e-6.
// All clouds on this path are planar (z == 0), where the Umeyama rotation is the closed form
// theta = atan2(sum cross, sum dot) of the demeaned pairs.
//
// Device design: the target is binned into a uniform cell list (cell = max_dist / 4: counting
// sort, points of a cell contiguous); a source point searches rings of cells outwards and stops
// as soon as the best distance is within the scanned square (exact nearest neighbour, ties by
// lowest target index).  Sums are reduced in a fixed order (per-CTA partials, then one CTA), so a
// registration is reproducible bit for bit.  The whole iteration loop is ONE persistent cooperative
// kernel (k_icp_loop): two grid barriers per iteration, no host round trips, early exit on
// convergence.  The device pieces the batched call (icp_batch.cu) shares live in icp_core.cuh.
#include "icp_core.cuh"
#include "sincos_dd.cuh"

namespace occ {

__device__ __forceinline__ int icp_cell_of(double v, double lo, double cell, int n) {
    const double f = floor(OCC_DDIV(OCC_DADD(v, -lo), cell));
    return f < 0.0 ? 0 : (f > (double)(n - 1) ? n - 1 : (int)f);
}

__global__ void __launch_bounds__(kIT)
k_icp_count(const double* __restrict__ tx, const double* __restrict__ ty, long long n, double min_x, double min_y, double cell,
            int w, int h, unsigned int* __restrict__ cnt) {
    for (long long i = (long long)blockIdx.x * kIT + threadIdx.x; i < n; i += (long long)gridDim.x * kIT)
        atomicAdd(&cnt[(size_t)icp_cell_of(ty[i], min_y, cell, h) * w + icp_cell_of(tx[i], min_x, cell, w)], 1u);
}

// start[c] = exclusive sum of cnt; cursor[c] = start[c] (consumed by the fill pass).
// Exclusive scan of the per-cell counts in three launches (block sums -> scan of the block sums ->
// rescan with the carry): every block of 16 384 cells runs on its own CTA, so the index of a
// 640 k-cell map is built in tens of microseconds instead of one CTA looping for a millisecond.
__global__ void __launch_bounds__(1024)
k_icp_scan_sums(const unsigned int* __restrict__ cnt, long long cells, unsigned int* __restrict__ block_sums) {
    __shared__ unsigned int s_warp[33];
    const long long i0 = (long long)blockIdx.x * kScanBlockIcp + (long long)threadIdx.x * kScanItemsIcp;
    unsigned int sum = 0;
#pragma unroll
    for (int j = 0; j < kScanItemsIcp; ++j) sum += (i0 + j < cells) ? cnt[i0 + j] : 0u;
    unsigned int total;
    block_exclusive_scan(sum, s_warp, &total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024)
k_icp_scan_top(unsigned int* __restrict__ block_sums, int n_blocks, unsigned int* __restrict__ start, long long cells) {
    const unsigned long long total = cta_scan_in_place<1>(block_sums, n_blocks, 0ull);
    if (threadIdx.x == 0) start[cells] = (unsigned int)total;
}

__global__ void __launch_bounds__(1024)
k_icp_scan_apply(const unsigned int* __restrict__ cnt, long long cells, const unsigned int* __restrict__ block_sums,
                 unsigned int* __restrict__ start, unsigned int* __restrict__ cursor) {
    __shared__ unsigned int s_warp[33];
    const long long i0 = (long long)blockIdx.x * kScanBlockIcp + (long long)threadIdx.x * kScanItemsIcp;
    unsigned int v[kScanItemsIcp], sum = 0;
#pragma unroll
    for (int j = 0; j < kScanItemsIcp; ++j) { v[j] = (i0 + j < cells) ? cnt[i0 + j] : 0u; sum += v[j]; }
    unsigned int total;
    unsigned int run = block_sums[blockIdx.x] + block_exclusive_scan(sum, s_warp, &total);
#pragma unroll
    for (int j = 0; j < kScanItemsIcp; ++j) {
        if (i0 + j < cells) { start[i0 + j] = run; cursor[i0 + j] = run; }
        run += v[j];
    }
}

__global__ void __launch_bounds__(kIT)
k_icp_fill(const double* __restrict__ tx, const double* __restrict__ ty, long long n, double min_x, double min_y, double cell,
           int w, int h, unsigned int* __restrict__ cursor, double* __restrict__ sx, double* __restrict__ sy,
           unsigned int* __restrict__ sidx) {
    for (long long i = (long long)blockIdx.x * kIT + threadIdx.x; i < n; i += (long long)gridDim.x * kIT) {
        const double x = tx[i], y = ty[i];
        const unsigned int p = atomicAdd(&cursor[(size_t)icp_cell_of(y, min_y, cell, h) * w + icp_cell_of(x, min_x, cell, w)], 1u);
        sx[p] = x; sy[p] = y; sidx[p] = (unsigned int)i;
    }
}

// (optionally) moves this CTA's source points by the update, then finds their correspondences.
__device__ __forceinline__ void icp_assoc_phase(const IcpLoop& p, const IcpState* L, bool apply) {
    for (int vb = blockIdx.x; vb < p.n_vb; vb += gridDim.x) {
        const long long i = (long long)vb * kIT + threadIdx.x;
        double v[6] = {0, 0, 0, 0, 0, 0};
        if (i < p.n) {
            double x = p.px[i], y = p.py[i];
            if (apply) {                                         // PointCloud::Transform
                const double* U = L->U;
                const double w = OCC_DADD(OCC_DADD(OCC_DMUL(U[12], x), OCC_DMUL(U[13], y)), U[15]);
                const double nx = OCC_DDIV(OCC_DADD(OCC_DADD(OCC_DMUL(U[0], x), OCC_DMUL(U[1], y)), U[3]), w);
                const double ny = OCC_DDIV(OCC_DADD(OCC_DADD(OCC_DMUL(U[4], x), OCC_DMUL(U[5], y)), U[7]), w);
                x = nx; y = ny;
                p.px[i] = x; p.py[i] = y;
            }
            double d2;
            const unsigned int q = icp_nearest(p.ix, x, y, p.r, p.r2, &d2);
            p.corr[i] = q;
            if (q != 0xffffffffu) { v[0] = 1.0; v[1] = d2; v[2] = x; v[3] = y; v[4] = p.ix.x[q]; v[5] = p.ix.y[q]; }
        }
        block_sum<6>(v, p.partial + (size_t)vb * 6);
    }
}

__device__ __forceinline__ void icp_cov_phase(const IcpLoop& p, const IcpState* L) {
    for (int vb = blockIdx.x; vb < p.n_vb; vb += gridDim.x) {
        const long long i = (long long)vb * kIT + threadIdx.x;
        double v[2] = {0, 0};
        if (i < p.n) {
            const unsigned int q = p.corr[i];
            if (q != 0xffffffffu) {
                const double sx = p.px[i] - L->mean[0], sy = p.py[i] - L->mean[1];
                const double tx = p.ix.x[q] - L->mean[2], ty = p.ix.y[q] - L->mean[3];
                v[0] = sx * tx + sy * ty;
                v[1] = sx * ty - sy * tx;
            }
        }
        block_sum<2>(v, p.partial2 + (size_t)vb * 2);
    }
}

// Three CTAs per SM: without the bound ptxas may cut the kernel to 64 registers and spill in the
// neighbour search.
__global__ void __launch_bounds__(kIT, 3)
k_icp_loop(const IcpLoop p) {
    __shared__ IcpState L;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 16; ++i) { L.T[i] = (i % 5 == 0) ? 1.0 : 0.0; L.U[i] = L.T[i]; }
        L.fitness = L.rmse = L.iterations = L.n_corr = 0.0;
        L.mean[0] = L.mean[1] = L.mean[2] = L.mean[3] = 0.0;
        L.done = 0;
    }
    __syncthreads();
    unsigned int target = 0;
    int* abort_flag = reinterpret_cast<int*>(p.bar + 4);
    bool alive = true;
    icp_assoc_phase(p, &L, false);
    alive = grid_barrier(p.bar, target, abort_flag);
    if (alive) icp_fold_eval(p, &L, 1);
    for (int it = 0; alive && it < p.max_iteration && !L.done; ++it) {
        icp_cov_phase(p, &L);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
        icp_fold_solve(p, &L);
        icp_assoc_phase(p, &L, true);
        if (!(alive = grid_barrier(p.bar, target, abort_flag))) break;
        icp_fold_eval(p, &L, 0);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (!alive) L.iterations = -1.0;                       // a barrier timed out: the host reports it
        *p.state = L;
    }
}

struct IcpLayout {
    size_t cnt, start, cursor, sx, sy, sidx, px, py, corr, partial, partial2, state, block_sums, bar, total;
};

static IcpLayout icp_layout(int64_t target_points, int64_t source_points, int64_t cells) {
    IcpLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t blocks = (size_t)((source_points + kIT - 1) / kIT) + 1;
    L.cnt = take((size_t)(cells + 1) * 4); L.start = take((size_t)(cells + 1) * 4); L.cursor = take((size_t)(cells + 1) * 4);
    L.sx = take((size_t)target_points * 8); L.sy = take((size_t)target_points * 8); L.sidx = take((size_t)target_points * 4);
    L.px = take((size_t)source_points * 8); L.py = take((size_t)source_points * 8); L.corr = take((size_t)source_points * 4);
    L.partial = take(blocks * 6 * 8); L.partial2 = take(blocks * 2 * 8); L.state = take(sizeof(IcpState));
    L.block_sums = take((size_t)((cells + kScanBlockIcp - 1) / kScanBlockIcp + 1) * 4);
    L.bar = take(256);
    L.total = o;
    return L;
}

void icp_build_index(const double* d_tx, const double* d_ty, int64_t n_target, double min_x, double min_y, double cell,
                            int32_t cells_w, int32_t cells_h, unsigned int* cnt, unsigned int* start, unsigned int* cursor,
                            unsigned int* block_sums, double* sx, double* sy, unsigned int* sidx, cudaStream_t st) {
    const int64_t cells = (int64_t)cells_w * cells_h;
    long long gt = (n_target + kIT - 1) / kIT;
    if (gt > device_sm_count() * 16) gt = device_sm_count() * 16;
    k_icp_count<<<(int)gt, kIT, 0, st>>>(d_tx, d_ty, n_target, min_x, min_y, cell, cells_w, cells_h, cnt);
    const int scan_blocks = (int)((cells + kScanBlockIcp - 1) / kScanBlockIcp);
    k_icp_scan_sums<<<scan_blocks, 1024, 0, st>>>(cnt, cells, block_sums);
    k_icp_scan_top<<<1, 1024, 0, st>>>(block_sums, scan_blocks, start, cells);
    k_icp_scan_apply<<<scan_blocks, 1024, 0, st>>>(cnt, cells, block_sums, start, cursor);
    k_icp_fill<<<(int)gt, kIT, 0, st>>>(d_tx, d_ty, n_target, min_x, min_y, cell, cells_w, cells_h, cursor, sx, sy, sidx);
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t mapmerge_icp_workspace_bytes(int64_t target_points, int64_t source_points, int32_t cells_w, int32_t cells_h) {
    if (target_points <= 0 || source_points <= 0 || cells_w <= 0 || cells_h <= 0) return 0;
    return icp_layout(target_points, source_points, (int64_t)cells_w * cells_h).total;
}

int mapmerge_icp_register(const double* d_sx, const double* d_sy, int64_t n_source, const double* d_tx, const double* d_ty,
                          int64_t n_target, double min_x, double min_y, double cell, int32_t cells_w, int32_t cells_h,
                          double max_correspondence_distance, int32_t max_iteration, double relative_fitness, double relative_rmse,
                          double* d_result, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_sx || !d_sy || !d_tx || !d_ty || n_source <= 0 || n_target <= 0 || n_target >= 0xffffffffll || !(cell > 0.0) ||
        cells_w <= 0 || cells_h <= 0 || !(max_correspondence_distance > 0.0) || max_iteration < 0 || !d_result || !d_ws) {
        set_last_error("mapmerge_icp_register: bad arguments");
        return OCCGRID_E_ARG;
    }
    const int64_t cells = (int64_t)cells_w * cells_h;
    const IcpLayout L = icp_layout(n_target, n_source, cells);
    if (ws_bytes < L.total) { set_last_error("mapmerge_icp_register: workspace too small"); return OCCGRID_E_WORKSPACE; }
    char* ws = reinterpret_cast<char*>(d_ws);
    unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + L.cnt);
    unsigned int* start = reinterpret_cast<unsigned int*>(ws + L.start);
    unsigned int* cursor = reinterpret_cast<unsigned int*>(ws + L.cursor);
    double* sx = reinterpret_cast<double*>(ws + L.sx);
    double* sy = reinterpret_cast<double*>(ws + L.sy);
    unsigned int* sidx = reinterpret_cast<unsigned int*>(ws + L.sidx);
    double* px = reinterpret_cast<double*>(ws + L.px);
    double* py = reinterpret_cast<double*>(ws + L.py);
    unsigned int* corr = reinterpret_cast<unsigned int*>(ws + L.corr);
    double* partial = reinterpret_cast<double*>(ws + L.partial);
    double* partial2 = reinterpret_cast<double*>(ws + L.partial2);
    IcpState* state = reinterpret_cast<IcpState*>(ws + L.state);
    unsigned int* block_sums = reinterpret_cast<unsigned int*>(ws + L.block_sums);
    unsigned int* bar = reinterpret_cast<unsigned int*>(ws + L.bar);
    cudaStream_t st = (cudaStream_t)stream;
    const int gs = (int)((n_source + kIT - 1) / kIT);
    ProfileScope ps(K_ICP, st, 6);
    OCC_CUDA_TRY(cudaMemsetAsync(cnt, 0, (size_t)(cells + 1) * 4, st));
    OCC_CUDA_TRY(cudaMemcpyAsync(px, d_sx, (size_t)n_source * 8, cudaMemcpyDeviceToDevice, st));
    OCC_CUDA_TRY(cudaMemcpyAsync(py, d_sy, (size_t)n_source * 8, cudaMemcpyDeviceToDevice, st));
    icp_build_index(d_tx, d_ty, n_target, min_x, min_y, cell, cells_w, cells_h, cnt, start, cursor, block_sums, sx, sy, sidx, st);
    IcpIndex ix;
    ix.min_x = min_x; ix.min_y = min_y; ix.cell = cell; ix.w = cells_w; ix.h = cells_h;
    ix.start = start; ix.x = sx; ix.y = sy; ix.idx = sidx;
    const double r = max_correspondence_distance, r2 = r * r;
    OCC_CUDA_TRY(cudaGetLastError());
    // the iteration loop: one cooperative launch (the grid must be co-resident for its barriers)
    static int resident_by_device[64] = {};
    int dev = 0;
    OCC_CUDA_TRY(cudaGetDevice(&dev));
    int resident = (dev >= 0 && dev < 64) ? resident_by_device[dev] : 0;
    if (resident == 0) {
        int sms = 0, per_sm = 0;
        OCC_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        OCC_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_icp_loop, kIT, 0));
        if (sms <= 0 || per_sm <= 0) { set_last_error("mapmerge_icp_register: the loop kernel does not fit the device"); return OCCGRID_E_CUDA; }
        resident = sms * per_sm;
        if (dev >= 0 && dev < 64) resident_by_device[dev] = resident;
    }
    IcpLoop lp;
    lp.px = px; lp.py = py; lp.n = n_source; lp.ix = ix; lp.r = r; lp.r2 = r2;
    lp.rel_f = relative_fitness; lp.rel_r = relative_rmse;
    lp.corr = corr; lp.partial = partial; lp.partial2 = partial2; lp.n_vb = gs; lp.max_iteration = max_iteration;
    lp.state = state; lp.bar = bar;
    OCC_CUDA_TRY(cudaMemsetAsync(bar, 0, 256, st));
    void* args[] = {&lp};
    OCC_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_icp_loop, dim3((unsigned)(gs < resident ? gs : resident)), dim3(kIT), args, 0, st));
    OCC_CUDA_TRY(cudaGetLastError());
    OCC_CUDA_TRY(cudaMemcpyAsync(d_result, state, 20 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    return OCCGRID_OK;
}

}  // extern "C"
