// Frontier detection and clustering on the device-resident grid (SURVEY §8 row f1).
//
// Reference: OccupancyGrid.get_frontiers / cluster_frontiers / cluster_centroid_world,
// server_nodes/dual_bot_mapper.py:181-237, driven every 3 s from main() (:948-956):
//   * a frontier cell is an interior FREE cell (1 <= x,y <= size-2, :187-190) with at least one
//     UNKNOWN 4-neighbour (:193-196); the list is in row-major scan order;
//   * clusters are the 4-connected components of the frontier set (:214-226), emitted in the
//     order of their first cell in that list (:210), components smaller than
//     FRONTIER_MIN_CLUSTER are dropped (:228-229);
//   * a centroid is grid_to_world(mean x, mean y) (:233-237).
// The reference's BFS also fixes the order of cells INSIDE a cluster; nothing downstream
// depends on it (only the centroid is used, :953), so clusters here list their cells in scan
// order.
//
// Kernels: stencil + ordered compaction (count / single-CTA scan / write), union-find over the
// compact frontier list (neighbours found by index arithmetic and binary search in the sorted
// list, union by smaller index so that a component's root IS its first cell), per-root integer
// sums, ordered compaction of the surviving roots and fp64 centroids.
#include "common.cuh"

namespace occ {

constexpr int kFT = 256;
constexpr int kFCells = 16;                 // cells per thread
constexpr int kFChunk = kFT * kFCells;

// Frontier bits of 16 consecutive cells starting at linear index `base` (x0, y0 = its column/row).
// Fast path: the 16 cells sit in one row and the three rows are 16-byte aligned -> three 16-byte
// loads + two edge bytes, all tests on registers.
__device__ __forceinline__ unsigned int frontier_mask16(const int8_t* __restrict__ g, int w, int h, long long base, long long n) {
    const int y0 = (int)(base / w), x0 = (int)(base - (long long)y0 * w);
    unsigned int mask = 0;
    if (x0 + kFCells <= w && y0 >= 1 && y0 <= h - 2 && ((w & 15) == 0) && ((reinterpret_cast<uintptr_t>(g) & 15) == 0)) {
        const int4 cur4 = __ldg(reinterpret_cast<const int4*>(g + base));
        const int4 up4 = __ldg(reinterpret_cast<const int4*>(g + base - w));
        const int4 dn4 = __ldg(reinterpret_cast<const int4*>(g + base + w));
        const unsigned int cur[4] = {(unsigned)cur4.x, (unsigned)cur4.y, (unsigned)cur4.z, (unsigned)cur4.w};
        const unsigned int up[4] = {(unsigned)up4.x, (unsigned)up4.y, (unsigned)up4.z, (unsigned)up4.w};
        const unsigned int dn[4] = {(unsigned)dn4.x, (unsigned)dn4.y, (unsigned)dn4.z, (unsigned)dn4.w};
        const unsigned int left = x0 > 0 ? (unsigned int)(unsigned char)g[base - 1] : 0u;
        const unsigned int right = x0 + kFCells < w ? (unsigned int)(unsigned char)g[base + kFCells] : 0u;
        // four cells per step on whole words: FREE == 0x00 and UNKNOWN == 0xff are byte-wise compares,
        // the left / right neighbours are the word funnel-shifted by one byte
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const unsigned int c = cur[i];
            const unsigned int l = (c << 8) | (i > 0 ? cur[i - 1] >> 24 : left);
            const unsigned int r = (c >> 8) | ((i < 3 ? cur[i + 1] : right) << 24);
            const unsigned int unk = __vcmpeq4(up[i], 0xffffffffu) | __vcmpeq4(dn[i], 0xffffffffu) |
                                     __vcmpeq4(l, 0xffffffffu) | __vcmpeq4(r, 0xffffffffu);                       // :193-196
            const unsigned int f = __vcmpeq4(c, 0u) & unk & 0x80808080u;                                          // :189
            mask |= ((((f >> 7) * 0x00204081u) >> 21) & 0xfu) << (4 * i);
        }
        if (x0 == 0) mask &= ~1u;                                                                                 // interior columns only (:187-188)
        if (x0 + kFCells == w) mask &= ~(1u << (kFCells - 1));
        return mask;
    }
    int x = x0, y = y0;
    for (int i = 0; i < kFCells; ++i) {
        const long long c = base + i;
        if (c >= n) break;
        if (x >= 1 && y >= 1 && x <= w - 2 && y <= h - 2 && g[c] == OCCGRID_CELL_FREE &&
            (g[c - 1] == OCCGRID_CELL_UNKNOWN || g[c + 1] == OCCGRID_CELL_UNKNOWN ||
             g[c - w] == OCCGRID_CELL_UNKNOWN || g[c + w] == OCCGRID_CELL_UNKNOWN))
            mask |= 1u << i;
        if (++x == w) { x = 0; ++y; }
    }
    return mask;
}

// The grid is read ONCE: the count pass keeps the 16 frontier bits of every thread's cells, the
// write pass expands those bits into (x, y) tuples without touching the grid again.
__global__ void __launch_bounds__(kFT)
k_frontier_count(const int8_t* __restrict__ g, int w, int h, unsigned int* __restrict__ block_counts,
                 unsigned short* __restrict__ masks) {
    __shared__ unsigned int s_warp[33];
    const long long n = (long long)w * h;
    const long long base = ((long long)blockIdx.x * kFT + threadIdx.x) * kFCells;
    const unsigned int m = base < n ? frontier_mask16(g, w, h, base, n) : 0u;
    masks[(size_t)blockIdx.x * kFT + threadIdx.x] = (unsigned short)m;
    unsigned int total;
    block_exclusive_scan(__popc(m), s_warp, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// One CTA, 16 consecutive block counts per thread and round: a 65 536-block grid (16384^2) is
// scanned in four rounds instead of sixty-four.
constexpr int kReserveItems = 16;

__global__ void __launch_bounds__(1024)
k_frontier_reserve(unsigned int* __restrict__ block_counts, int n_blocks, long long capacity,
                   long long* __restrict__ d_count, int* __restrict__ status) {
    const unsigned long long sum = cta_scan_in_place<kReserveItems>(block_counts, n_blocks, 0ull);
    if (threadIdx.x == 0) {
        long long total = (long long)sum;
        if (total > capacity) { atomicOr(status, 1); total = 0; }
        *d_count = total;
    }
}

__global__ void __launch_bounds__(kFT)
k_frontier_write(const unsigned short* __restrict__ masks, int w, int h, const unsigned int* __restrict__ block_offsets,
                 const long long* __restrict__ d_count, int2* __restrict__ xy) {
    __shared__ unsigned int s_warp[33];
    if (*d_count == 0) return;
    const long long base = ((long long)blockIdx.x * kFT + threadIdx.x) * kFCells;
    unsigned int m = masks[(size_t)blockIdx.x * kFT + threadIdx.x];
    unsigned int total;
    long long dst = block_offsets[blockIdx.x] + block_exclusive_scan(__popc(m), s_warp, &total);
    while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        const long long c = base + i;
        const int y = (int)(c / w);
        xy[dst++] = make_int2((int)(c - (long long)y * w), y);                      // (x, y) tuples, :197
    }
}

// ---- union-find over the compact, row-major-sorted frontier list --------------------------

__device__ __forceinline__ unsigned int uf_find(unsigned int* __restrict__ parent, unsigned int i) {
    volatile unsigned int* vp = parent;
    for (;;) {
        const unsigned int p = vp[i];
        if (p == i) return i;
        const unsigned int gp = vp[p];
        if (gp != p) atomicMin(&parent[i], gp);      // path halving; parents only ever decrease
        i = p;
    }
}

__device__ __forceinline__ void uf_union(unsigned int* __restrict__ parent, unsigned int a, unsigned int b) {
    for (;;) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a > b) { const unsigned int t = a; a = b; b = t; }        // smaller index becomes the root
        const unsigned int old = atomicMin(&parent[b], a);
        if (old == b) return;
        b = old;                                                     // somebody else re-parented b: retry
    }
}

// index of linear cell `lin` in the sorted list, or -1
__device__ __forceinline__ long long find_cell(const int2* __restrict__ xy, long long n, int w, long long lin) {
    long long lo = 0, hi = n - 1;
    while (lo <= hi) {
        const long long mid = (lo + hi) >> 1;
        const int2 c = xy[mid];
        const long long v = (long long)c.y * w + c.x;
        if (v == lin) return mid;
        if (v < lin) lo = mid + 1; else hi = mid - 1;
    }
    return -1;
}

__global__ void __launch_bounds__(kFT)
k_cluster_init(const long long* __restrict__ d_count, unsigned int* __restrict__ parent, unsigned int* __restrict__ csize,
               long long* __restrict__ sx, long long* __restrict__ sy) {
    const long long n = *d_count;
    for (long long i = (long long)blockIdx.x * kFT + threadIdx.x; i < n; i += (long long)gridDim.x * kFT) {
        parent[i] = (unsigned int)i; csize[i] = 0u; sx[i] = 0; sy[i] = 0;
    }
}

__global__ void __launch_bounds__(kFT)
k_cluster_union(const int2* __restrict__ xy, const long long* __restrict__ d_count, int w, unsigned int* __restrict__ parent) {
    const long long n = *d_count;
    for (long long i = (long long)blockIdx.x * kFT + threadIdx.x; i < n; i += (long long)gridDim.x * kFT) {
        const int2 c = xy[i];
        if (i > 0) {                                                  // left neighbour is the previous list entry, if present
            const int2 p = xy[i - 1];
            if (p.y == c.y && p.x == c.x - 1) uf_union(parent, (unsigned int)i, (unsigned int)(i - 1));
        }
        const long long up = find_cell(xy, i, w, (long long)(c.y - 1) * w + c.x);   // upper neighbour precedes i
        if (up >= 0) uf_union(parent, (unsigned int)i, (unsigned int)up);
    }
}

__global__ void __launch_bounds__(kFT)
k_cluster_stats(const int2* __restrict__ xy, const long long* __restrict__ d_count, unsigned int* __restrict__ parent,
                int* __restrict__ label, unsigned int* __restrict__ csize, long long* __restrict__ sx, long long* __restrict__ sy) {
    const long long n = *d_count;
    for (long long i = (long long)blockIdx.x * kFT + threadIdx.x; i < n; i += (long long)gridDim.x * kFT) {
        const unsigned int r = uf_find(parent, (unsigned int)i);
        label[i] = (int)r;
        const int2 c = xy[i];
        atomicAdd(&csize[r], 1u);
        atomicAdd(reinterpret_cast<unsigned long long*>(&sx[r]), (unsigned long long)c.x);
        atomicAdd(reinterpret_cast<unsigned long long*>(&sy[r]), (unsigned long long)c.y);
    }
}

// Single CTA: ordered compaction of roots with at least `min_cluster` cells; centroid = :233-237.
constexpr int kEmitItems = 8;
__global__ void __launch_bounds__(1024)
k_cluster_emit(const long long* __restrict__ d_count, const int* __restrict__ label, const unsigned int* __restrict__ csize,
               const long long* __restrict__ sx, const long long* __restrict__ sy, int min_cluster, double ox, double oy,
               double res, int* __restrict__ cluster_root, int* __restrict__ cluster_size, double* __restrict__ centroids,
               long long* __restrict__ n_clusters) {
    __shared__ unsigned int s_warp[33];
    __shared__ unsigned int s_carry;
    const long long n = *d_count;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long start = 0; start < n; start += 1024 * kEmitItems) {          // kEmitItems consecutive candidates per thread
        const long long i0 = start + (long long)threadIdx.x * kEmitItems;
        unsigned int keep = 0;
#pragma unroll
        for (int j = 0; j < kEmitItems; ++j) {
            const long long i = i0 + j;
            if (i < n && label[i] == (int)i && csize[i] >= (unsigned int)min_cluster) keep |= 1u << j;              // :228
        }
        unsigned int total;
        unsigned int pos = s_carry + block_exclusive_scan(__popc(keep), s_warp, &total);
        while (keep) {
            const long long i = i0 + (__ffs(keep) - 1);
            keep &= keep - 1;
            const double cnt = (double)csize[i];
            const double ax = OCC_DDIV((double)sx[i], cnt), ay = OCC_DDIV((double)sy[i], cnt);          // :235-236
            cluster_root[pos] = (int)i;
            cluster_size[pos] = (int)csize[i];
            centroids[2 * pos + 0] = OCC_DADD(ox, OCC_DMUL(OCC_DADD(ax, 0.5), res));                      // grid_to_world, :129
            centroids[2 * pos + 1] = OCC_DADD(oy, OCC_DMUL(OCC_DADD(ay, 0.5), res));
            ++pos;
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_clusters = s_carry;
}

static int fgrid(long long items) {
    long long b = (items + kFT - 1) / kFT;
    if (b < 1) b = 1;
    if (b > device_sm_count() * 16) b = device_sm_count() * 16;
    return (int)b;
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t occgrid_frontier_workspace_bytes(int64_t n_cells, int64_t max_frontiers) {
    const int64_t blocks = (n_cells + kFChunk - 1) / kFChunk;
    return align_up((size_t)blocks * 4, 256) + align_up((size_t)blocks * kFT * 2, 256) +       // block counts | 16 frontier bits per thread
           align_up((size_t)max_frontiers * 4, 256) * 2 + align_up((size_t)max_frontiers * 8, 256) * 2 + 256;
}

int occgrid_frontiers(const int8_t* d_grid, int32_t width, int32_t height, int32_t* d_xy, int64_t capacity,
                      int64_t* d_count, int32_t* d_status, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grid || !d_xy || !d_count || !d_status || !d_ws || width < 3 || height < 3 || capacity <= 0) {
        set_last_error("occgrid_frontiers: bad arguments");
        return OCCGRID_E_ARG;
    }
    const long long n = (long long)width * height;
    if (ws_bytes < occgrid_frontier_workspace_bytes(n, capacity)) { set_last_error("occgrid_frontiers: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)((n + kFChunk - 1) / kFChunk);
    unsigned int* block_counts = reinterpret_cast<unsigned int*>(d_ws);
    ProfileScope ps(K_FRONTIER, st, 3);
    unsigned short* masks = reinterpret_cast<unsigned short*>(reinterpret_cast<char*>(d_ws) + align_up((size_t)blocks * 4, 256));
    k_frontier_count<<<blocks, kFT, 0, st>>>(d_grid, width, height, block_counts, masks);
    k_frontier_reserve<<<1, 1024, 0, st>>>(block_counts, blocks, capacity, (long long*)d_count, d_status);
    k_frontier_write<<<blocks, kFT, 0, st>>>(masks, width, height, block_counts, (const long long*)d_count, reinterpret_cast<int2*>(d_xy));
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int occgrid_frontier_clusters(const int32_t* d_xy, const int64_t* d_count, int64_t capacity, int32_t width, int32_t min_cluster,
                              double ox, double oy, double res, int32_t* d_label, int32_t* d_cluster_root,
                              int32_t* d_cluster_size, double* d_centroids, int64_t* d_n_clusters,
                              void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_xy || !d_count || !d_label || !d_cluster_root || !d_cluster_size || !d_centroids || !d_n_clusters || !d_ws ||
        capacity <= 0 || width < 3) {
        set_last_error("occgrid_frontier_clusters: bad arguments");
        return OCCGRID_E_ARG;
    }
    const size_t a4 = align_up((size_t)capacity * 4, 256), a8 = align_up((size_t)capacity * 8, 256);
    if (ws_bytes < 2 * a4 + 2 * a8) { set_last_error("occgrid_frontier_clusters: workspace too small"); return OCCGRID_E_WORKSPACE; }
    char* ws = reinterpret_cast<char*>(d_ws);
    unsigned int* parent = reinterpret_cast<unsigned int*>(ws);
    unsigned int* csize = reinterpret_cast<unsigned int*>(ws + a4);
    long long* sx = reinterpret_cast<long long*>(ws + 2 * a4);
    long long* sy = reinterpret_cast<long long*>(ws + 2 * a4 + a8);
    cudaStream_t st = (cudaStream_t)stream;
    const int g = fgrid(capacity);
    const int2* xy = reinterpret_cast<const int2*>(d_xy);
    ProfileScope ps(K_FRONTIER_CLUSTER, st, 4);
    k_cluster_init<<<g, kFT, 0, st>>>((const long long*)d_count, parent, csize, sx, sy);
    k_cluster_union<<<g, kFT, 0, st>>>(xy, (const long long*)d_count, width, parent);
    k_cluster_stats<<<g, kFT, 0, st>>>(xy, (const long long*)d_count, parent, d_label, csize, sx, sy);
    k_cluster_emit<<<1, 1024, 0, st>>>((const long long*)d_count, d_label, csize, sx, sy, min_cluster, ox, oy, res,
                                       d_cluster_root, d_cluster_size, d_centroids, (long long*)d_n_clusters);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
