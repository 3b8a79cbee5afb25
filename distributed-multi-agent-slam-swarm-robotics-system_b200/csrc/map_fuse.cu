// Fused occupancy map (mapmerge_warp_fuse in include/occgrid_b200.h): every agent map of a stack is
// resampled into one target grid under its agent->global rigid transform, and the covering agents'
// cells are combined with an int8 max, so that free space survives the merge.  EXTENSION: the
// reference merge (map_merger.py, mapmerge.cu) only keeps occupied cells.
//
// The contract (DESIGN §6d).  Per agent, in host fp64 with every operation rounded on its own:
//   bx = (gox + 0.5*g) - tx            by = (goy + 0.5*g) - ty
//   c0 = (R00*g)/r   c1 = (R10*g)/r   c2 = ((R00*bx + R10*by) - ox_a)/r
//   c3 = (R01*g)/r   c4 = (R11*g)/r   c5 = ((R01*bx + R11*by) - oy_a)/r
// Per target cell (column j, row i):
//   u = (c0*j) + ((c1*i) + c2)         v = (c3*j) + ((c4*i) + c5)
//   agent a covers the cell iff 0 <= u < W and 0 <= v < H  (NaN never covers)
//   out[i][j] = max(-1, max over covering agents of map_a[(int)v][(int)u])
// The device evaluates u and v with __dmul_rn / __dadd_rn: nvcc would otherwise contract them to FMA.
#include <cmath>
#include <vector>

#include "common.cuh"

namespace occ {

constexpr int kFuseTile = 64;              // target cells per tile side; one CTA per tile
constexpr int kFuseThreads = 256;          // 16 cells per thread
constexpr int kFusePitch = kFuseTile + 16; // shared row pitch: 16-byte rows, no bank conflict between a warp's 4 rows
constexpr int kFuseMaxAgents = 65535;      // as mapmerge_extract_batch_*
constexpr double kRigidTol = 1e-9;         // |R^T R - I| per entry

// Per-agent record in the workspace: the six coefficients and a conservative footprint in target
// cells ([j0, j1] x [i0, i1], clamped to the target; empty when j0 > j1).
struct FuseAgent {
    double c[6];
    int32_t j0, j1, i0, i1;
};
static_assert(sizeof(FuseAgent) == 64, "FuseAgent is 64 bytes");

// Thread t of the CTA owns the 16 cells (row 8w + 4h + l/8, column 8c + l%8) of its tile, h = 0..1,
// c = 0..7, w = t / 32, l = t % 32: at every (h, c) a warp covers a 4 x 8 patch, so its gathers touch
// a few rows of the agent map under any rotation.  The running maxima stay in registers; the tile is
// staged in shared memory and stored with 16-byte stores where the target rows allow it.
__global__ void __launch_bounds__(kFuseThreads)
k_warp_fuse(const int8_t* __restrict__ maps, int n_agents, int32_t width, int32_t height, const FuseAgent* __restrict__ ag,
            int8_t* __restrict__ out, int32_t out_w, int32_t out_h, long long tiles_x, long long n_tiles, int vec_ok) {
    __shared__ unsigned int s_warp[33];
    __shared__ int s_agent[kFuseThreads];
    __shared__ double s_c[6][kFuseThreads];
    __shared__ __align__(16) int8_t s_out[kFuseTile * kFusePitch];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r_loc = 8 * warp + (lane >> 3), c_loc = lane & 7;
    const size_t map_cells = (size_t)width * (size_t)height;

    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long ty = tile / tiles_x;
        const int i0 = (int)(ty * kFuseTile), j0 = (int)((tile - ty * tiles_x) * kFuseTile);
        double row[2], col[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) row[h] = (double)(i0 + r_loc + 4 * h);
#pragma unroll
        for (int c = 0; c < 8; ++c) col[c] = (double)(j0 + 8 * c + c_loc);
        int m[2][8];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int c = 0; c < 8; ++c) m[h][c] = -1;

        for (int base = 0; base < n_agents; base += kFuseThreads) {
            const int a = base + (int)threadIdx.x;
            bool hit = false;
            if (a < n_agents) {
                const FuseAgent& f = ag[a];
                hit = f.j0 <= j0 + kFuseTile - 1 && f.j1 >= j0 && f.i0 <= i0 + kFuseTile - 1 && f.i1 >= i0;
            }
            unsigned int n_hits;
            const unsigned int pos = block_exclusive_scan<unsigned int>(hit ? 1u : 0u, s_warp, &n_hits);
            if (hit) {
                s_agent[pos] = a;
#pragma unroll
                for (int k = 0; k < 6; ++k) s_c[k][pos] = ag[a].c[k];
            }
            __syncthreads();
            for (unsigned int k = 0; k < n_hits; ++k) {
                const double c0 = s_c[0][k], c1 = s_c[1][k], c2 = s_c[2][k];
                const double c3 = s_c[3][k], c4 = s_c[4][k], c5 = s_c[5][k];
                const int8_t* __restrict__ map = maps + (size_t)s_agent[k] * map_cells;
                double ur[2], vr[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    ur[h] = __dadd_rn(__dmul_rn(c1, row[h]), c2);
                    vr[h] = __dadd_rn(__dmul_rn(c4, row[h]), c5);
                }
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double uc = __dmul_rn(c0, col[c]), vc = __dmul_rn(c3, col[c]);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const double u = __dadd_rn(uc, ur[h]), v = __dadd_rn(vc, vr[h]);
                        // For u >= 0 (false for NaN), floor(u) < W <=> u < W, and floor(u) == (int)u; the
                        // conversion saturates, so u = +inf gives INT_MAX >= W
                        const int iu = __double2int_rd(u), iv = __double2int_rd(v);
                        if (u >= 0.0 && v >= 0.0 && (unsigned int)iu < (unsigned int)width && (unsigned int)iv < (unsigned int)height) {
                            const int8_t cell = __ldg(map + (size_t)iv * (size_t)width + (size_t)iu);
                            m[h][c] = max(m[h][c], (int)cell);
                        }
                    }
                }
            }
            __syncthreads();        // s_agent / s_c are rewritten by the next chunk
        }

#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int c = 0; c < 8; ++c) s_out[(r_loc + 4 * h) * kFusePitch + 8 * c + c_loc] = (int8_t)m[h][c];
        __syncthreads();
        {
            const int r = (int)threadIdx.x >> 2, seg = ((int)threadIdx.x & 3) * 16;
            const long long gi = (long long)i0 + r, gj = (long long)j0 + seg;
            if (gi < out_h) {
                int8_t* dst = out + (size_t)gi * (size_t)out_w + (size_t)gj;
                const int8_t* src = s_out + r * kFusePitch + seg;
                if (vec_ok && gj + 16 <= out_w) {
                    *reinterpret_cast<int4*>(dst) = *reinterpret_cast<const int4*>(src);
                } else {
                    for (int k = 0; k < 16 && gj + k < out_w; ++k) dst[k] = src[k];
                }
            }
        }
        __syncthreads();            // s_out is rewritten by the next tile
    }
}

// Agent footprint in target cells from the inverse of (j, i) -> (u, v): j = j(u, v), i = i(u, v) at
// the four corners of [0, W] x [0, H], widened by 2 cells plus a relative 1e-6 for the rounding of
// u and v and the 1e-9 rigidity tolerance.  Non-finite coefficients cover nothing (u or v is then
// never finite).
static void footprint(FuseAgent& f, const double* T, double res, double out_res, int32_t width, int32_t height,
                      int32_t out_w, int32_t out_h) {
    f.j0 = f.i0 = 1;
    f.j1 = f.i1 = 0;
    for (int k = 0; k < 6; ++k)
        if (!std::isfinite(f.c[k])) return;
    const double s = res / out_res;
    double jmin = INFINITY, jmax = -INFINITY, imin = INFINITY, imax = -INFINITY;
    for (int k = 0; k < 4; ++k) {
        const double du = ((k & 1) ? (double)width : 0.0) - f.c[2], dv = ((k & 2) ? (double)height : 0.0) - f.c[5];
        // (u, v) - (c2, c5) = (g/r) R^T (j, i)  =>  (j, i) = (r/g) R (du, dv)
        const double j = s * (T[0] * du + T[1] * dv), i = s * (T[4] * du + T[5] * dv);
        jmin = fmin(jmin, j); jmax = fmax(jmax, j);
        imin = fmin(imin, i); imax = fmax(imax, i);
    }
    if (!(std::isfinite(jmin) && std::isfinite(jmax) && std::isfinite(imin) && std::isfinite(imax))) return;
    const double mj = 2.0 + 1e-6 * fmax(fabs(jmin), fabs(jmax)), mi = 2.0 + 1e-6 * fmax(fabs(imin), fabs(imax));
    const double a0 = fmax(floor(jmin - mj), 0.0), a1 = fmin(ceil(jmax + mj), (double)out_w - 1.0);
    const double b0 = fmax(floor(imin - mi), 0.0), b1 = fmin(ceil(imax + mi), (double)out_h - 1.0);
    if (a0 > a1 || b0 > b1) return;
    f.j0 = (int32_t)a0; f.j1 = (int32_t)a1;
    f.i0 = (int32_t)b0; f.i1 = (int32_t)b1;
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t mapmerge_warp_fuse_workspace_bytes(int n_agents, int32_t out_w, int32_t out_h) {
    if (n_agents < 1 || n_agents > kFuseMaxAgents) {
        set_last_error("mapmerge_warp_fuse_workspace_bytes: n_agents %d outside 1..%d", n_agents, kFuseMaxAgents);
        return 0;
    }
    if (out_w < 1 || out_h < 1) {
        set_last_error("mapmerge_warp_fuse_workspace_bytes: target size %d x %d", (int)out_w, (int)out_h);
        return 0;
    }
    return align_up((size_t)n_agents * sizeof(FuseAgent), 256);
}

int mapmerge_warp_fuse(const int8_t* d_maps, int n_agents, int32_t width, int32_t height, double res,
                       const double* origins_host, const double* T_host, double out_ox, double out_oy, double out_res,
                       int32_t out_w, int32_t out_h, int8_t* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_maps || !origins_host || !T_host || !d_out || !d_ws) {
        set_last_error("mapmerge_warp_fuse: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (n_agents < 1 || n_agents > kFuseMaxAgents) {
        set_last_error("mapmerge_warp_fuse: n_agents %d outside 1..%d", n_agents, kFuseMaxAgents);
        return OCCGRID_E_ARG;
    }
    if (width < 1 || height < 1 || out_w < 1 || out_h < 1) {
        set_last_error("mapmerge_warp_fuse: size < 1 (maps %d x %d, target %d x %d)", (int)width, (int)height, (int)out_w, (int)out_h);
        return OCCGRID_E_ARG;
    }
    if (!(std::isfinite(res) && res > 0.0) || !(std::isfinite(out_res) && out_res > 0.0)) {
        set_last_error("mapmerge_warp_fuse: resolution must be finite and > 0 (maps %g, target %g)", res, out_res);
        return OCCGRID_E_ARG;
    }
    const size_t map_cells = (size_t)width * (size_t)height;
    if (map_cells > SIZE_MAX / (size_t)n_agents) {
        set_last_error("mapmerge_warp_fuse: stack of %d maps of %d x %d overflows size_t", n_agents, (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    for (int a = 0; a < n_agents; ++a) {
        const double* T = T_host + 16 * (size_t)a;
        for (int k = 0; k < 16; ++k)
            if (!std::isfinite(T[k])) {
                set_last_error("mapmerge_warp_fuse: transform %d has a non-finite entry", a);
                return OCCGRID_E_ARG;
            }
        const double R[2][2] = {{T[0], T[1]}, {T[4], T[5]}};
        for (int p = 0; p < 2; ++p)
            for (int q = 0; q < 2; ++q) {
                const double rtr = R[0][p] * R[0][q] + R[1][p] * R[1][q];
                if (!(fabs(rtr - (p == q ? 1.0 : 0.0)) <= kRigidTol)) {
                    set_last_error("mapmerge_warp_fuse: transform %d is not rigid (|R^T R - I| > 1e-9)", a);
                    return OCCGRID_E_ARG;
                }
            }
    }
    if (ws_bytes < mapmerge_warp_fuse_workspace_bytes(n_agents, out_w, out_h)) {
        set_last_error("mapmerge_warp_fuse: workspace too small");
        return OCCGRID_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<FuseAgent> hx((size_t)n_agents);
    const double g = out_res, r = res;
    for (int a = 0; a < n_agents; ++a) {
        const double* T = T_host + 16 * (size_t)a;
        const double R00 = T[0], R01 = T[1], R10 = T[4], R11 = T[5], tx = T[3], ty = T[7];
        const double bx = (out_ox + 0.5 * g) - tx, by = (out_oy + 0.5 * g) - ty;
        FuseAgent& f = hx[a];
        f.c[0] = (R00 * g) / r;
        f.c[1] = (R10 * g) / r;
        f.c[2] = ((R00 * bx + R10 * by) - origins_host[2 * (size_t)a]) / r;
        f.c[3] = (R01 * g) / r;
        f.c[4] = (R11 * g) / r;
        f.c[5] = ((R01 * bx + R11 * by) - origins_host[2 * (size_t)a + 1]) / r;
        footprint(f, T, res, out_res, width, height, out_w, out_h);
    }
    // A copy from pageable memory has been staged by the driver when cudaMemcpyAsync returns, so hx
    // may go out of scope without a stream synchronisation.
    OCC_CUDA_TRY(cudaMemcpyAsync(d_ws, hx.data(), sizeof(FuseAgent) * (size_t)n_agents, cudaMemcpyHostToDevice, st));
    const long long tiles_x = ((long long)out_w + kFuseTile - 1) / kFuseTile;
    const long long tiles_y = ((long long)out_h + kFuseTile - 1) / kFuseTile;
    const long long n_tiles = tiles_x * tiles_y;
    const unsigned int ctas = (unsigned int)(n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL);
    const int vec_ok = (out_w % 16 == 0) && ((reinterpret_cast<uintptr_t>(d_out) & 15) == 0);
    ProfileScope ps(K_MERGE_WARP_FUSE, st, 1);
    k_warp_fuse<<<ctas, kFuseThreads, 0, st>>>(d_maps, n_agents, width, height, reinterpret_cast<const FuseAgent*>(d_ws), d_out,
                                               out_w, out_h, tiles_x, n_tiles, vec_ok);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
