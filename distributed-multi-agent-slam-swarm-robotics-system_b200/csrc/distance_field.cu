// Obstacle clearance (occgrid_distance_field / occgrid_inflate in include/occgrid_b200.h): the exact
// squared Euclidean distance transform of a grid's obstacles, and the navigation grid that blocks the
// FREE cells within a robot radius of an obstacle.  EXTENSION (DESIGN §6g): the reference treats a
// robot as a point.
//
// EDT, separable and exact (Meijster et al. 2000), integer arithmetic only, no atomics:
//   phase 1, per column: g(x, y) = |y - y'| to the nearest obstacle y' of column x, -1 when the column
//     has none.  Columns are cut into bands of 32 rows; k_edt_mask packs each (band, column) into a
//     32-bit obstacle mask, k_edt_link carries the nearest obstacle row above and below every band
//     down each column (one thread per column, one step per band), and k_edt_col finds each cell's
//     nearest obstacle from its band's mask and links with clz / ffs, one coalesced write per cell.
//   phase 2, per row: d2(x) = min over columns x' with g(x') >= 0 of (x - x')^2 + g(x')^2, the lower
//     envelope of those parabolas.  One thread per row builds the envelope as a stack of sites and
//     then walks it left to right.  A site is popped when the new parabola meets it no later than it
//     meets the one below it; the comparison of the two crossing points N1 / D1 <= N2 / D2 is made by
//     cross-multiplying in 64 bits (|N| < 2^31, D < 2^16), so nothing is divided.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace occ {

constexpr int kEdtBand = 32;                  // rows per phase-1 band (one bit each of a uint32 mask)
constexpr int kEdtMaxSide = 32768;
constexpr int kEdtMaxRobots = 65535;

__device__ __forceinline__ bool edt_obstacle(int8_t v) { return v > 50; }

// mask[b][x] bit r: cell (x, 32 b + r) is an obstacle.
__global__ void __launch_bounds__(256)
k_edt_mask(const int8_t* __restrict__ grid, int width, int height, int n_bands, unsigned int* __restrict__ mask) {
    const long long n = (long long)n_bands * width;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / width), x = (int)(i - (long long)b * width);
        const int y0 = b * kEdtBand, rows = min(kEdtBand, height - y0);
        const int8_t* p = grid + (size_t)y0 * width + x;
        unsigned int m = 0;
        for (int r = 0; r < rows; ++r) m |= (edt_obstacle(__ldg(p + (size_t)r * width)) ? 1u : 0u) << r;
        mask[i] = m;
    }
}

// link[b][x] = (last obstacle row above band b, first obstacle row below it), -1 for none.
__global__ void __launch_bounds__(128)
k_edt_link(const unsigned int* __restrict__ mask, int width, int n_bands, int2* __restrict__ link) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= width) return;
    int carry = -1;
    for (int b = 0; b < n_bands; ++b) {
        link[(size_t)b * width + x].x = carry;
        const unsigned int m = mask[(size_t)b * width + x];
        if (m) carry = b * kEdtBand + 31 - __clz((int)m);
    }
    carry = -1;
    for (int b = n_bands - 1; b >= 0; --b) {
        link[(size_t)b * width + x].y = carry;
        const unsigned int m = mask[(size_t)b * width + x];
        if (m) carry = b * kEdtBand + __ffs((int)m) - 1;
    }
}

// g[y][x]: vertical distance to the nearest obstacle of column x, -1 when the column has none.
__global__ void __launch_bounds__(256)
k_edt_col(const unsigned int* __restrict__ mask, const int2* __restrict__ link, int width, int height, int n_bands,
          int* __restrict__ g) {
    const long long n = (long long)n_bands * width;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / width), x = (int)(i - (long long)b * width);
        const int y0 = b * kEdtBand, rows = min(kEdtBand, height - y0);
        const unsigned int m = mask[i];
        const int2 ln = link[i];
        for (int r = 0; r < rows; ++r) {
            const unsigned int at_or_above = m & (0xffffffffu >> (31 - r));
            const unsigned int at_or_below = m & (0xffffffffu << r);
            const int ya = at_or_above ? y0 + 31 - __clz((int)at_or_above) : ln.x;
            const int yb = at_or_below ? y0 + __ffs((int)at_or_below) - 1 : ln.y;
            const int y = y0 + r;
            int d = -1;
            if (ya >= 0) d = y - ya;
            if (yb >= 0 && (d < 0 || yb - y < d)) d = yb - y;
            g[(size_t)y * width + x] = d;
        }
    }
}

// One thread per row: the lower envelope of (x - x')^2 + g(x')^2 over the row's columns with g >= 0,
// kept as a stack of (x', g(x')^2) in the thread's row of `stack`, then evaluated at every x.  The
// row is read from `g` before it is written to `d2`, so the two may be the same buffer.
__global__ void __launch_bounds__(128)
k_edt_row(const int* g, int width, int height, int2* __restrict__ stack, int* d2) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= height) return;
    const int* gr = g + (size_t)y * width;
    int2* st = stack + (size_t)y * width;
    int n = 0;
    for (int u = 0; u < width; ++u) {
        const int gu = gr[u];
        if (gu < 0) continue;
        const int g2u = gu * gu;
        while (n >= 2) {
            const int2 b = st[n - 1], a = st[n - 2];
            // b is hidden when u's crossing with b, N_bu / 2(u - b), is not right of b's crossing with
            // a, N_ab / 2(b - a)
            const long long n_ab = (long long)b.x * b.x - (long long)a.x * a.x + (long long)b.y - a.y;
            const long long n_bu = (long long)u * u - (long long)b.x * b.x + (long long)g2u - b.y;
            if (n_bu * (long long)(b.x - a.x) <= n_ab * (long long)(u - b.x)) --n;
            else break;
        }
        st[n++] = make_int2(u, g2u);
    }
    int* out = d2 + (size_t)y * width;
    if (n == 0) {                                 // no obstacle anywhere in the grid
        for (int x = 0; x < width; ++x) out[x] = -1;
        return;
    }
    int k = 0;
    int2 cur = st[0];
    int2 nxt = n > 1 ? st[1] : make_int2(0, 0);
    for (int x = 0; x < width; ++x) {
        long long fc = (long long)(x - cur.x) * (x - cur.x) + cur.y;
        while (k + 1 < n) {
            const long long fn = (long long)(x - nxt.x) * (x - nxt.x) + nxt.y;
            if (fn > fc) break;
            ++k; cur = nxt; fc = fn;
            if (k + 1 < n) nxt = st[k + 1];
        }
        out[x] = (int)fc;
    }
}

// nav = 100 where the cell is FREE and 0 <= d2 <= max_d2, else the grid's value.
__global__ void __launch_bounds__(256)
k_inflate(const int8_t* __restrict__ grid, const int* __restrict__ d2, long long n, long long max_d2, int8_t* __restrict__ nav) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        const int8_t v = grid[c];
        const int d = d2[c];
        nav[c] = (v == OCCGRID_CELL_FREE && d >= 0 && (long long)d <= max_d2) ? (int8_t)OCCGRID_CELL_OCCUPIED : v;
    }
}

// Robot blockIdx.y puts its footprint back: every cell within max_d2 of its cell gets the grid's value.
// Footprints may overlap; every writer of a cell writes the same value.
__global__ void __launch_bounds__(256)
k_inflate_footprint(const int8_t* __restrict__ grid, int width, int height, double ox, double oy, double res,
                    const double* __restrict__ robot_xy, long long max_d2, int reach, int8_t* __restrict__ nav) {
    const int a = blockIdx.y;
    const double qx = (robot_xy[2 * a] - ox) / res, qy = (robot_xy[2 * a + 1] - oy) / res;
    // int() truncates toward zero, so the cell is inside iff -1 < q < size (false for NaN and inf)
    if (!(qx > -1.0 && qx < (double)width && qy > -1.0 && qy < (double)height)) return;
    const int rx = (int)qx, ry = (int)qy;
    const int x0 = max(rx - reach, 0), x1 = min(rx + reach, width - 1);
    const int y0 = max(ry - reach, 0), y1 = min(ry + reach, height - 1);
    const long long bw = x1 - x0 + 1, n = bw * (y1 - y0 + 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = y0 + (int)(i / bw), x = x0 + (int)(i % bw);
        const long long dx = x - rx, dy = y - ry;
        if (dx * dx + dy * dy <= max_d2) {
            const size_t c = (size_t)y * width + x;
            nav[c] = grid[c];
        }
    }
}

// Workspace layout; every offset is 256-aligned.
struct EdtLayout {
    size_t mask, link, d2, stack, total;
    int n_bands;
};

static EdtLayout edt_layout(int32_t width, int32_t height) {
    EdtLayout L;
    L.n_bands = (height + kEdtBand - 1) / kEdtBand;
    const size_t w = (size_t)width, cells = (size_t)width * (size_t)height;
    L.mask = 0;
    L.link = align_up(L.mask + 4 * w * L.n_bands, 256);
    L.d2 = align_up(L.link + 8 * w * L.n_bands, 256);
    L.stack = align_up(L.d2 + 4 * cells, 256);
    L.total = align_up(L.stack + 8 * cells, 256);
    return L;
}

static int edt_check(const char* who, int32_t width, int32_t height) {
    if (width < 1 || height < 1 || width > kEdtMaxSide || height > kEdtMaxSide) {
        set_last_error("%s: width x height %d x %d: each must be in 1..%d", who, (int)width, (int)height, kEdtMaxSide);
        return OCCGRID_E_ARG;
    }
    return OCCGRID_OK;
}

// The four EDT launches: grid -> d2, through the workspace's mask, link and stack.
static void edt_run(const int8_t* d_grid, int32_t width, int32_t height, int32_t* d_d2, char* ws, const EdtLayout& L,
                    cudaStream_t st) {
    unsigned int* mask = reinterpret_cast<unsigned int*>(ws + L.mask);
    int2* link = reinterpret_cast<int2*>(ws + L.link);
    const long long items = (long long)L.n_bands * width;
    const unsigned int gb = (unsigned int)std::min((items + 255) / 256, (long long)device_sm_count() * 16);
    k_edt_mask<<<gb, 256, 0, st>>>(d_grid, width, height, L.n_bands, mask);
    k_edt_link<<<(width + 127) / 128, 128, 0, st>>>(mask, width, L.n_bands, link);
    k_edt_col<<<gb, 256, 0, st>>>(mask, link, width, height, L.n_bands, d_d2);
    k_edt_row<<<(height + 127) / 128, 128, 0, st>>>(d_d2, width, height, reinterpret_cast<int2*>(ws + L.stack), d_d2);
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t occgrid_distance_field_workspace_bytes(int32_t width, int32_t height) {
    if (edt_check("occgrid_distance_field_workspace_bytes", width, height) != OCCGRID_OK) return 0;
    return edt_layout(width, height).total;
}

int occgrid_distance_field(const int8_t* d_grid, int32_t width, int32_t height, int32_t* d_d2, void* d_ws, size_t ws_bytes,
                           void* stream) {
    if (!d_grid || !d_d2 || !d_ws) {
        set_last_error("occgrid_distance_field: NULL pointer");
        return OCCGRID_E_ARG;
    }
    const int rc = edt_check("occgrid_distance_field", width, height);
    if (rc != OCCGRID_OK) return rc;
    const EdtLayout L = edt_layout(width, height);
    if (ws_bytes < L.total) { set_last_error("occgrid_distance_field: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_DISTANCE_FIELD, st, 4);
    edt_run(d_grid, width, height, d_d2, reinterpret_cast<char*>(d_ws), L, st);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int occgrid_inflate(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy, double res, int64_t max_d2,
                    const double* d_robot_xy, int32_t n_robots, int8_t* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grid || !d_out || !d_ws || (n_robots > 0 && !d_robot_xy)) {
        set_last_error("occgrid_inflate: NULL pointer");
        return OCCGRID_E_ARG;
    }
    const int rc = edt_check("occgrid_inflate", width, height);
    if (rc != OCCGRID_OK) return rc;
    if (max_d2 < 0) {
        set_last_error("occgrid_inflate: max_d2 %lld must be >= 0", (long long)max_d2);
        return OCCGRID_E_ARG;
    }
    if (n_robots < 0 || n_robots > kEdtMaxRobots) {
        set_last_error("occgrid_inflate: n_robots %d outside 0..%d", (int)n_robots, kEdtMaxRobots);
        return OCCGRID_E_ARG;
    }
    if (!(std::isfinite(res) && res > 0.0)) {
        set_last_error("occgrid_inflate: resolution must be finite and > 0 (got %g)", res);
        return OCCGRID_E_ARG;
    }
    const EdtLayout L = edt_layout(width, height);
    if (ws_bytes < L.total) { set_last_error("occgrid_inflate: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(d_ws);
    int* d2 = reinterpret_cast<int*>(ws + L.d2);
    ProfileScope ps(K_DISTANCE_FIELD, st, n_robots > 0 ? 6 : 5);
    edt_run(d_grid, width, height, d2, ws, L, st);
    const long long n = (long long)width * height;
    k_inflate<<<(unsigned int)std::min((n + 255) / 256, (long long)device_sm_count() * 16), 256, 0, st>>>(d_grid, d2, n, max_d2, d_out);
    if (n_robots > 0) {
        // reach: the largest r with r^2 <= max_d2, capped at the grid's longer side
        const long long side = std::max(width, height);
        long long reach = max_d2 >= side * side ? side : (long long)std::sqrt((double)max_d2);
        while (reach * reach > max_d2) --reach;
        while (reach < side && (reach + 1) * (reach + 1) <= max_d2) ++reach;
        const long long box = (2 * reach + 1) * (2 * reach + 1);
        const unsigned int bx = (unsigned int)std::max(1LL, std::min((box + 255) / 256, (long long)device_sm_count() * 4));
        k_inflate_footprint<<<dim3(bx, (unsigned int)n_robots), 256, 0, st>>>(d_grid, width, height, ox, oy, res, d_robot_xy,
                                                                             max_d2, (int)reach, d_out);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
