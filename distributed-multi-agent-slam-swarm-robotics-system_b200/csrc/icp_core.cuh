// Device pieces of the ICP registration shared by the single call (icp.cu) and the batched call
// (icp_batch.cu): the target's cell list, the registration state, the fixed-order block sum, the
// exact nearest-neighbour search and the folds of the iteration loop.  See icp.cu for the algorithm.
#pragma once
#include "common.cuh"

namespace occ {

constexpr int kIT = 256;

struct IcpIndex {                 // cell list over the target cloud
    double min_x, min_y, cell;
    int w, h;
    const unsigned int* start;    // [w*h + 1]
    const double* x;              // target points sorted by cell
    const double* y;
    const unsigned int* idx;      // their indices in the caller's cloud
};

struct IcpState {                 // device-resident; the first 20 doubles are the public result
    double T[16];
    double fitness, rmse, iterations, n_corr;
    double U[16];
    double mean[4];               // source x, y; target x, y over the current correspondences
    int done;
};

// Exclusive scan of the cell counts: blocks of kScanBlockIcp cells (see icp.cu).
constexpr int kScanItemsIcp = 16;
constexpr int kScanBlockIcp = 1024 * kScanItemsIcp;


// Fixed-order block sum of N doubles per thread into out[N] (thread 0 writes).
template <int N>
__device__ __forceinline__ void block_sum(double (&v)[N], double* out) {
    __shared__ double s_part[N][kIT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[j] = OCC_DADD(v[j], __shfl_down_sync(0xffffffffu, v[j], o));
        if (lane == 0) s_part[j][warp] = v[j];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
            double a = s_part[j][0];
            for (int w = 1; w < kIT / 32; ++w) a = OCC_DADD(a, s_part[j][w]);
            out[j] = a;
        }
    }
    __syncthreads();
}

// Exact nearest neighbour of (px, py) in the cell list, squared distance < r2, ties -> lowest
// target index.  Returns the sorted position or 0xffffffff.
__device__ __forceinline__ unsigned int icp_nearest(const IcpIndex& ix, double px, double py, double r, double r2, double* d2_out) {
    const double qx = floor(OCC_DDIV(OCC_DADD(px, -ix.min_x), ix.cell)), qy = floor(OCC_DDIV(OCC_DADD(py, -ix.min_y), ix.cell));
    // distance from the query to the edge of its own (unclamped) cell, shaved for rounding
    const double fx = px - (ix.min_x + qx * ix.cell), fy = py - (ix.min_y + qy * ix.cell);
    double inner = fmin(fmin(fx, ix.cell - fx), fmin(fy, ix.cell - fy));
    inner = fmax(inner - 1e-9 * ix.cell, 0.0);
    const long long cqx = (long long)fmax(fmin(qx, 4.0e9), -4.0e9), cqy = (long long)fmax(fmin(qy, 4.0e9), -4.0e9);
    const int rmax = (int)ceil(r / ix.cell) + 1;
    double best = INFINITY;
    unsigned int best_pos = 0xffffffffu, best_idx = 0xffffffffu;
    for (int R = 0; R <= rmax; ++R) {
        const long long y_lo = cqy - R, y_hi = cqy + R, x_lo = cqx - R, x_hi = cqx + R;
        for (long long cy = y_lo; cy <= y_hi; ++cy) {
            if (cy < 0 || cy >= ix.h) continue;
            const bool edge_row = (cy == y_lo || cy == y_hi);
            const long long step = edge_row ? 1 : (2 * (long long)R > 0 ? 2 * (long long)R : 1);
            for (long long cx = x_lo; cx <= x_hi; cx += step) {              // full row on the ring's top/bottom, two cells otherwise
                if (cx < 0 || cx >= ix.w) continue;
                const size_t c = (size_t)cy * ix.w + (size_t)cx;
                const unsigned int b = ix.start[c], e = ix.start[c + 1];
                for (unsigned int p = b; p < e; ++p) {
                    const double dx = OCC_DADD(ix.x[p], -px), dy = OCC_DADD(ix.y[p], -py);
                    const double d2 = OCC_DADD(OCC_DMUL(dx, dx), OCC_DMUL(dy, dy));
                    const unsigned int id = ix.idx[p];
                    if (d2 < best || (d2 == best && id < best_idx)) { best = d2; best_pos = p; best_idx = id; }
                }
            }
        }
        const double margin = (double)R * ix.cell * (1.0 - 1e-12) + inner;      // everything unscanned is at least this far
        if (margin >= r) break;
        if (best_pos != 0xffffffffu && best <= margin * margin) break;
    }
    *d2_out = best;
    return (best_pos != 0xffffffffu && best < r2) ? best_pos : 0xffffffffu;
}

// ---- the iteration loop: ONE persistent cooperative kernel --------------------------------------
// Every CTA carries an identical copy of the registration state in shared memory: the per-block
// partial sums go through global memory, and after a grid barrier EVERY CTA folds them in the same
// fixed order and takes the same decisions (score, convergence, Umeyama update), so nothing has
// to be broadcast and an iteration costs two grid barriers instead of five launches.  Work is
// dealt in "virtual blocks" of kIT source points, so the partials — and with them every bit of the
// result — do not depend on how many CTAs the device holds.
struct IcpLoop {
    double* px; double* py; long long n;          // working copy of the source cloud
    IcpIndex ix;
    double r, r2, rel_f, rel_r;
    unsigned int* corr;
    double* partial;                               // [n_vb][6] = {count, sum d2, sum sx, sum sy, sum tx, sum ty}
    double* partial2;                              // [n_vb][2] = {sum dot, sum cross} of the demeaned pairs
    int n_vb, max_iteration;
    IcpState* state;
    unsigned int* bar;                             // [0, 4) grid_barrier words, [4] abort flag; zeroed before each launch
};

// Folds the association partials in a fixed order, scores the registration and decides whether
// the loop has converged (Registration.cpp: |d fitness| < rel_f && |d rmse| < rel_r).
__device__ __forceinline__ void icp_fold_eval(const IcpLoop& p, IcpState* L, int first) {
    double v[6] = {0, 0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < p.n_vb; b += kIT)
#pragma unroll
        for (int j = 0; j < 6; ++j) v[j] = OCC_DADD(v[j], __ldcg(p.partial + (size_t)b * 6 + j));
    __shared__ double s_tot[6];
    block_sum<6>(v, s_tot);
    if (threadIdx.x == 0) {
        const double cnt = s_tot[0];
        const double fit = p.n > 0 ? cnt / (double)p.n : 0.0;
        const double rmse = cnt > 0.0 ? sqrt(s_tot[1] / cnt) : 0.0;
        if (!first) {
            L->iterations += 1.0;
            if (fabs(L->fitness - fit) < p.rel_f && fabs(L->rmse - rmse) < p.rel_r) L->done = 1;
        }
        L->fitness = fit; L->rmse = rmse; L->n_corr = cnt;
        if (cnt > 0.0) { L->mean[0] = s_tot[2] / cnt; L->mean[1] = s_tot[3] / cnt; L->mean[2] = s_tot[4] / cnt; L->mean[3] = s_tot[5] / cnt; }
    }
    __syncthreads();
}

// Folds the covariance partials and composes the update: theta = atan2(sum cross, sum dot).
__device__ __forceinline__ void icp_fold_solve(const IcpLoop& p, IcpState* L) {
    double v[2] = {0, 0};
    for (int b = threadIdx.x; b < p.n_vb; b += kIT) {
        v[0] = OCC_DADD(v[0], __ldcg(p.partial2 + (size_t)b * 2));
        v[1] = OCC_DADD(v[1], __ldcg(p.partial2 + (size_t)b * 2 + 1));
    }
    __shared__ double s_tot[2];
    block_sum<2>(v, s_tot);
    if (threadIdx.x == 0) {
        double U[16];
        for (int i = 0; i < 16; ++i) U[i] = (i % 5 == 0) ? 1.0 : 0.0;
        if (L->n_corr > 0.0) {                                   // no correspondences -> identity (TransformationEstimation.cpp)
            const double th = atan2(s_tot[1], s_tot[0]);
            const double c = cos(th), sn = sin(th);
            U[0] = c; U[1] = -sn; U[4] = sn; U[5] = c;
            U[3] = L->mean[2] - (c * L->mean[0] - sn * L->mean[1]);
            U[7] = L->mean[3] - (sn * L->mean[0] + c * L->mean[1]);
        }
        double Tn[16];
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
                double a = 0.0;
                for (int k = 0; k < 4; ++k) a += U[4 * i + k] * L->T[4 * k + j];
                Tn[4 * i + j] = a;
            }
        for (int i = 0; i < 16; ++i) { L->T[i] = Tn[i]; L->U[i] = U[i]; }
    }
    __syncthreads();
}

// Builds the cell list of the target cloud on `st` (icp.cu): cnt must be zero; fills start
// [cells + 1], cursor and the sorted x / y / idx arrays.  The launches of mapmerge_icp_register.
void icp_build_index(const double* d_tx, const double* d_ty, int64_t n_target, double min_x, double min_y, double cell,
                     int32_t cells_w, int32_t cells_h, unsigned int* cnt, unsigned int* start, unsigned int* cursor,
                     unsigned int* block_sums, double* sx, double* sy, unsigned int* sidx, cudaStream_t st);

}  // namespace occ
