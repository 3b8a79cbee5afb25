// Map-fusion kernels and their C ABI (include/occgrid_b200.h, mapmerge_* entry points).
//
// Reference path replaced: MapMerger.grid_to_pcd / map_callback / publish_global_map,
// server_nodes/map_merger.py:35-127, with the three Open3D calls on it written out
// (PointCloud::Transform :58, operator+= :59, VoxelDownSample :60) and the rigid transform
// supplied by the caller in place of ICP (:45-56, SURVEY §8 a13).
//
// Data layout: a point cloud is two fp64 device arrays (x[], y[]; z == 0 on this path) plus a
// device-resident int64 count, so a whole merge sequence runs stream-ordered without host
// round trips.  All arithmetic that decides a cell or voxel index is fp64 with individually
// rounded operations, in the order the reference evaluates it.
//
// Determinism: Open3D's voxel filter emits voxels in hash-map order (unspecified).  We fix the
// canonical order "first appearance" (voxels in order of their smallest point index, as an
// insertion-ordered map would give) and sum the points of a voxel in ascending point index, so
// results are bit-reproducible and equal to the oracle (oracle/merge_oracle.py).
#include <cstddef>
#include <vector>

#include "common.cuh"

namespace occ {

constexpr int kMT = 256;              // threads per CTA
constexpr int kLoadCells = 16;        // one 16-byte load of int8 cells
constexpr int kCellsPerThread = 64;   // four independent 16-byte loads in flight per thread
constexpr int kChunk = kMT * kCellsPerThread;

// Status word bits (device int32, sticky; checked by the host wrapper at its next sync).
enum { ST_POINT_OVERFLOW = 1, ST_LATTICE_OVERFLOW = 2, ST_CHAIN_ABORTED = 4 };

struct Xform { double m[16]; int identity; };

// ---- a10: occupied-cell extraction (data > 50, map_merger.py:72) --------------------------

__device__ __forceinline__ unsigned int occupied_mask16(const int8_t* __restrict__ grid, long long base, long long n) {
    unsigned int mask = 0;
    if (base + 16 <= n && ((reinterpret_cast<uintptr_t>(grid + base) & 15) == 0)) {
        const int4 v = __ldg(reinterpret_cast<const int4*>(grid + base));
        const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if ((int8_t)((w[i] >> (8 * b)) & 0xff) > 50) mask |= 1u << (4 * i + b);
    } else {
        for (int i = 0; i < 16 && base + i < n; ++i)
            if (grid[base + i] > 50) mask |= 1u << i;
    }
    return mask;
}

// 64 consecutive cells per thread: the four loads are independent, so a thread keeps 64 bytes in flight.
__device__ __forceinline__ unsigned long long occupied_mask64(const int8_t* __restrict__ grid, long long base, long long n) {
    unsigned int m[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) m[q] = occupied_mask16(grid, base + 16 * q, n);
    return (unsigned long long)m[0] | ((unsigned long long)m[1] << 16) | ((unsigned long long)m[2] << 32) |
           ((unsigned long long)m[3] << 48);
}

__global__ void __launch_bounds__(kMT)
k_extract_count(const int8_t* __restrict__ grid, long long n_cells, unsigned int* __restrict__ block_counts) {
    __shared__ unsigned int s_warp[33];
    const long long base = ((long long)blockIdx.x * kMT + threadIdx.x) * kCellsPerThread;
    unsigned int c = base < n_cells ? __popcll(occupied_mask64(grid, base, n_cells)) : 0u;
    unsigned int total;
    block_exclusive_scan(c, s_warp, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// Number of occupied (> 50) cells of a grid, added to *out (device int64).
__global__ void __launch_bounds__(kMT)
k_count_occupied(const int8_t* __restrict__ grid, long long n_cells, long long* __restrict__ out) {
    unsigned int c = 0;
    for (long long base = ((long long)blockIdx.x * kMT + threadIdx.x) * kLoadCells; base < n_cells;
         base += (long long)gridDim.x * kMT * kLoadCells)
        c += __popc(occupied_mask16(grid, base, n_cells));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(reinterpret_cast<unsigned long long*>(out), (unsigned long long)c);
}

// Single-CTA exclusive scan of the per-block counts; also reserves the output range
// [old_count, old_count + total) in the destination cloud.
__global__ void __launch_bounds__(1024)
k_extract_reserve(unsigned int* __restrict__ block_counts, int n_blocks, long long* __restrict__ d_count,
                  long long capacity, long long* __restrict__ ws_base, int* __restrict__ status,
                  long long* __restrict__ d_last_appended) {
    const unsigned long long sum = cta_scan_in_place<1>(block_counts, n_blocks, 0ull);
    if (threadIdx.x == 0) {
        const long long base = *d_count;
        long long total = (long long)sum;
        if (base + total > capacity) { atomicOr(status, ST_POINT_OVERFLOW); total = 0; }
        ws_base[0] = base;
        ws_base[1] = total;
        *d_count = base + total;
        if (d_last_appended) *d_last_appended = total;
    }
}

// grid_to_pcd (:76-77) fused with PointCloud::Transform (:58).
__global__ void __launch_bounds__(kMT)
k_extract_write(const int8_t* __restrict__ grid, long long n_cells, int width, double res, double origin_x,
                double origin_y, Xform T, const unsigned int* __restrict__ block_offsets,
                const long long* __restrict__ ws_base, double* __restrict__ px, double* __restrict__ py) {
    __shared__ unsigned int s_warp[33];
    if (ws_base[1] == 0) return;
    const long long base = ((long long)blockIdx.x * kMT + threadIdx.x) * kCellsPerThread;
    const unsigned long long mask = base < n_cells ? occupied_mask64(grid, base, n_cells) : 0ull;
    unsigned int total;
    unsigned int off = block_exclusive_scan(__popcll(mask), s_warp, &total);
    long long dst = ws_base[0] + block_offsets[blockIdx.x] + off;
    unsigned long long m = mask;
    while (m) {
        const int i = __ffsll((long long)m) - 1;
        m &= m - 1;
        const long long c = base + i;
        const long long row = c / width, col = c - row * width;
        double x = OCC_DADD(OCC_DMUL((double)col, res), origin_x);       // :77
        double y = OCC_DADD(OCC_DMUL((double)row, res), origin_y);       // :76
        if (!T.identity) {
            const double w = OCC_DADD(OCC_DADD(OCC_DMUL(T.m[12], x), OCC_DMUL(T.m[13], y)), T.m[15]);
            const double tx = OCC_DADD(OCC_DADD(OCC_DMUL(T.m[0], x), OCC_DMUL(T.m[1], y)), T.m[3]);
            const double ty = OCC_DADD(OCC_DADD(OCC_DMUL(T.m[4], x), OCC_DMUL(T.m[5], y)), T.m[7]);
            if (w == 1.0) { x = tx; y = ty; }                  // v / 1.0 == v bit for bit
            else { x = OCC_DDIV(tx, w); y = OCC_DDIV(ty, w); }
        }
        px[dst] = x;
        py[dst] = y;
        ++dst;
    }
}

// ---- block-level min/max of (x, y) -----------------------------------------------------------
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Every thread calls with its own values; thread 0 then calls use(min x, min y, max x, max y) of
// the whole block (any block size up to 1024).  Warps fold in a fixed fmin / fmax order, so the
// bounds do not depend on timing, down to the sign of zero.
template <class F>
__device__ __forceinline__ void block_min_max(double mnx, double mny, double mxx, double mxy, F&& use) {
    __shared__ double s_b[4][32];
    mnx = warp_min(mnx); mny = warp_min(mny); mxx = warp_max(mxx); mxy = warp_max(mxy);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_b[0][warp] = mnx; s_b[1][warp] = mny; s_b[2][warp] = mxx; s_b[3][warp] = mxy; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            mnx = fmin(mnx, s_b[0][w]); mny = fmin(mny, s_b[1][w]); mxx = fmax(mxx, s_b[2][w]); mxy = fmax(mxy, s_b[3][w]);
        }
        use(mnx, mny, mxx, mxy);
    }
}

// ---- bounds carried on the device between callbacks ----------------------------------------
// doubles mapped to uint64 keys that sort like the doubles, so min/max become integer atomics;
// benc = {min_x, min_y, max_x, max_y} of the current cloud.
__device__ __forceinline__ unsigned long long enc_double(double d) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double dec_double(unsigned long long k) {
    const unsigned long long u = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)u);
}

// Block-level min/max of (x, y) over the calling threads' values, then 4 atomics per CTA.
__device__ __forceinline__ void block_bounds_atomic(double mnx, double mny, double mxx, double mxy,
                                                    unsigned long long* __restrict__ benc) {
    block_min_max(mnx, mny, mxx, mxy, [&](double x0, double y0, double x1, double y1) {
        if (x0 <= x1) {
            atomicMin(&benc[0], enc_double(x0)); atomicMin(&benc[1], enc_double(y0));
            atomicMax(&benc[2], enc_double(x1)); atomicMax(&benc[3], enc_double(y1));
        }
    });
}

__global__ void k_benc_reset(unsigned long long* __restrict__ benc) {
    benc[0] = benc[1] = enc_double(INFINITY);
    benc[2] = benc[3] = enc_double(-INFINITY);
}

// ---- batched extraction: all agent grids of a merge in one pass ----------------------------
// grids[a] are A device pointers to H x W int8 maps; blockIdx.y = agent.  Output: every agent's
// transformed points, agent after agent (row-major inside an agent), plus per-agent offsets —
// the sequential voxel chain then appends slice a when its turn comes.
struct BatchXform { double m[6]; double w[3]; int identity; int use; };   // rows 0,1 and 3 of the 4x4 (z == 0)

__global__ void __launch_bounds__(kMT)
k_batch_count(const int8_t* const* __restrict__ grids, long long n_cells, int blocks_per_grid,
              unsigned int* __restrict__ block_counts /* [A][blocks_per_grid] */,
              unsigned long long* __restrict__ masks /* [A][blocks_per_grid * kMT]: the write pass reads these, not the grids */) {
    __shared__ unsigned int s_warp[33];
    const int a = blockIdx.y;
    const long long base = ((long long)blockIdx.x * kMT + threadIdx.x) * kCellsPerThread;
    const unsigned long long mask = base < n_cells ? occupied_mask64(grids[a], base, n_cells) : 0ull;
    masks[((size_t)a * blocks_per_grid + blockIdx.x) * kMT + threadIdx.x] = mask;
    unsigned int total;
    block_exclusive_scan(__popcll(mask), s_warp, &total);
    if (threadIdx.x == 0) block_counts[(size_t)a * blocks_per_grid + blockIdx.x] = total;
}

// ---- bulk-copy (TMA) staged scan --------------------------------------------------------------
// The count pass is the one pure HBM stream of the merge path: every agent grid is read once
// (H*W bytes) and leaves one occupancy bit per cell.  Persistent CTAs own a ring of kScanStages
// 16 KiB shared-memory stages; ONE elected thread keeps the ring full with
// cp.async.bulk.shared::cluster.global (the TMA unit's 1-D bulk copy), each stage completing on
// its own mbarrier (complete_tx::bytes), while the 256 threads turn the stage that has landed into
// 64-bit occupancy masks (`data > 50`, map_merger.py:72) — no thread ever waits on a global load.
constexpr int kScanStages = 4;
constexpr int kScanCtasPerSm = 3;            // 3 x 4 x 16 KiB = 192 KiB of bulk loads in flight per SM
constexpr int kScanStageBytes = kChunk;                    // 16 KiB = one chunk of the existing mask layout

// 16 int8 cells (one uint4 from shared memory) -> 16 occupancy bits.
__device__ __forceinline__ unsigned int occupied_bits16(uint4 v) {
    const unsigned int w[4] = {v.x, v.y, v.z, v.w};
    unsigned int bits = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const unsigned int gt = __vcmpgts4(w[i], 0x32323232u) & 0x80808080u;     // per byte: 0x80 where (int8) > 50
        bits |= (((gt >> 7) * 0x00204081u) >> 21 & 0xfu) << (4 * i);             // gather the four flags into 4 bits
    }
    return bits;
}

__global__ void __launch_bounds__(kMT)
k_batch_count_tma(const int8_t* const* __restrict__ grids, long long n_cells, int blocks_per_grid, int n_agents,
                  unsigned int* __restrict__ block_counts, unsigned long long* __restrict__ masks) {
    extern __shared__ __align__(128) unsigned char s_stage[];              // kScanStages x 16 KiB
    __shared__ __align__(8) unsigned long long s_full[kScanStages];
    __shared__ unsigned int s_cnt[kScanStages];
    const long long total = (long long)n_agents * blocks_per_grid;         // chunks, agent-major
    auto chunk_of = [&](long long i) { return (long long)blockIdx.x + i * gridDim.x; };
    auto issue = [&](long long i) {                                        // elected thread only
        const long long c = chunk_of(i);
        if (c >= total) return;
        const int a = (int)(c / blocks_per_grid), blk = (int)(c - (long long)a * blocks_per_grid);
        const long long base = (long long)blk * kChunk;
        const unsigned int bytes = (unsigned int)min((long long)kChunk, n_cells - base);
        const int st = (int)(i % kScanStages);
        mbar_expect_tx(&s_full[st], bytes);
        bulk_load(s_stage + (size_t)st * kScanStageBytes, grids[a] + base, bytes, &s_full[st]);
    };
    if (threadIdx.x == 0) {
        for (int s = 0; s < kScanStages; ++s) mbar_init(&s_full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x < kScanStages) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 0; i < kScanStages; ++i) issue(i);
    for (long long i = 0; chunk_of(i) < total; ++i) {
        const long long c = chunk_of(i);
        const int st = (int)(i % kScanStages);
        const int a = (int)(c / blocks_per_grid), blk = (int)(c - (long long)a * blocks_per_grid);
        const long long base = (long long)blk * kChunk;
        const int valid = (int)min((long long)kChunk, n_cells - base);     // multiple of 16 on this path
        mbar_wait(&s_full[st], (unsigned int)((i / kScanStages) & 1));
        const uint4* src = reinterpret_cast<const uint4*>(s_stage + (size_t)st * kScanStageBytes) + threadIdx.x * 4;
        unsigned long long mask = 0ull;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if ((int)threadIdx.x * kCellsPerThread + 16 * q < valid)
                mask |= (unsigned long long)occupied_bits16(src[q]) << (16 * q);
        masks[((size_t)a * blocks_per_grid + blk) * kMT + threadIdx.x] = mask;
        unsigned int n = __popcll(mask);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if ((threadIdx.x & 31) == 0 && n) atomicAdd(&s_cnt[st], n);
        __syncthreads();                                                   // everyone has read the stage; the count is complete
        if (threadIdx.x == 0) {
            block_counts[(size_t)a * blocks_per_grid + blk] = s_cnt[st];
            s_cnt[st] = 0u;
            issue(i + kScanStages);                                        // refill the stage that was just consumed
        }
    }
}

// One CTA per agent: exclusive scan of its block counts (in place) and its total.
__global__ void __launch_bounds__(1024)
k_batch_scan(unsigned int* __restrict__ block_counts, int blocks_per_grid, long long* __restrict__ agent_total) {
    const unsigned long long total = cta_scan_in_place<1>(block_counts + (size_t)blockIdx.x * blocks_per_grid, blocks_per_grid, 0ull);
    if (threadIdx.x == 0) agent_total[blockIdx.x] = (long long)total;
}

// agent_offset[a] = sum of totals of the agents before a that take part in the merge (one CTA).
__global__ void __launch_bounds__(1024)
k_batch_offsets(const long long* __restrict__ agent_total, const BatchXform* __restrict__ T, int n_agents,
                long long capacity, long long* __restrict__ agent_offset, int* __restrict__ status) {
    __shared__ unsigned long long s_warp[33];
    __shared__ long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int start = 0; start < n_agents; start += blockDim.x) {
        const int a = start + threadIdx.x;
        const unsigned long long v = (a < n_agents && T[a].use) ? (unsigned long long)agent_total[a] : 0ull;
        unsigned long long total;
        const unsigned long long ex = block_exclusive_scan(v, s_warp, &total);
        if (a < n_agents) agent_offset[a] = s_carry + (long long)ex;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += (long long)total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        agent_offset[n_agents] = s_carry;
        if (s_carry > capacity) atomicOr(status, ST_POINT_OVERFLOW);
    }
}

__global__ void __launch_bounds__(kMT)
k_batch_write(const unsigned long long* __restrict__ masks, long long n_cells, int width, double res,
              const double* __restrict__ origins /* [A][2] */, const BatchXform* __restrict__ T, int blocks_per_grid,
              const unsigned int* __restrict__ block_offsets, const long long* __restrict__ agent_offset, long long capacity,
              double* __restrict__ px, double* __restrict__ py) {
    __shared__ unsigned int s_warp[33];
    __shared__ unsigned short s_cell[kChunk];       // occupied cells of this chunk, in cell order
    const int a = blockIdx.y;
    const BatchXform t = T[a];
    if (!t.use || agent_offset[gridDim.y] > capacity) return;
    const long long chunk_base = (long long)blockIdx.x * kChunk;
    const unsigned long long mask = masks[((size_t)a * blocks_per_grid + blockIdx.x) * kMT + threadIdx.x];   // 1 bit per cell, from the count pass
    unsigned int total;
    unsigned int off = block_exclusive_scan(__popcll(mask), s_warp, &total);
    unsigned long long m = mask;
    while (m) {                                      // compact first: walls put many cells in few threads
        const int i = __ffsll((long long)m) - 1;
        m &= m - 1;
        s_cell[off++] = (unsigned short)(threadIdx.x * kCellsPerThread + i);
    }
    __syncthreads();
    const long long dst0 = agent_offset[a] + block_offsets[(size_t)a * blocks_per_grid + blockIdx.x];
    const double ox = origins[2 * a], oy = origins[2 * a + 1];
    for (unsigned int i = threadIdx.x; i < total; i += kMT) {      // then every thread converts its share, coalesced stores
        const long long c = chunk_base + s_cell[i];
        long long row, col;
        if (n_cells <= 0x7fffffffll) { row = (int)c / width; col = (int)c - (int)row * width; }
        else { row = c / width; col = c - row * width; }
        double x = OCC_DADD(OCC_DMUL((double)col, res), ox);       // :77
        double y = OCC_DADD(OCC_DMUL((double)row, res), oy);       // :76
        if (!t.identity) {
            const double w = OCC_DADD(OCC_DADD(OCC_DMUL(t.w[0], x), OCC_DMUL(t.w[1], y)), t.w[2]);
            const double tx = OCC_DADD(OCC_DADD(OCC_DMUL(t.m[0], x), OCC_DMUL(t.m[1], y)), t.m[2]);
            const double ty = OCC_DADD(OCC_DADD(OCC_DMUL(t.m[3], x), OCC_DMUL(t.m[4], y)), t.m[5]);
            if (w == 1.0) { x = tx; y = ty; }                  // rigid transforms: v / 1.0 == v bit for bit, skip two fp64 divisions
            else { x = OCC_DDIV(tx, w); y = OCC_DDIV(ty, w); }
        }
        px[dst0 + i] = x;
        py[dst0 + i] = y;
    }
}

// global_pcd += local_pcd (:59) for agent a of a batched extraction: append its slice.
__global__ void __launch_bounds__(kMT)
k_append_slice(const double* __restrict__ sx, const double* __restrict__ sy, const long long* __restrict__ agent_offset, int a,
               double* __restrict__ px, double* __restrict__ py, long long capacity, long long* __restrict__ d_count,
               int* __restrict__ status, unsigned long long* __restrict__ benc) {
    const long long b = agent_offset[a], e = agent_offset[a + 1];
    const long long n0 = *d_count;                  // read by every thread before the last block bumps it (see below)
    const long long k = e - b;
    if (n0 + k > capacity) { if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(status, ST_POINT_OVERFLOW); return; }
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < k; i += (long long)gridDim.x * kMT) {
        const double x = sx[b + i], y = sy[b + i];
        px[n0 + i] = x;
        py[n0 + i] = y;
        mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
    }
    if (benc) block_bounds_atomic(mnx, mny, mxx, mxy, benc);
}

__global__ void k_bump_count(const long long* __restrict__ agent_offset, int a, long long capacity, long long* __restrict__ d_count) {
    const long long k = agent_offset[a + 1] - agent_offset[a];
    if (*d_count + k <= capacity) *d_count += k;
}

// ---- bounds (GetMinBound/GetMaxBound; publish_global_map :95-98) ---------------------------

__global__ void __launch_bounds__(kMT)
k_bounds_partial(const double* __restrict__ px, const double* __restrict__ py, const long long* __restrict__ d_count,
                 double* __restrict__ partial /* gridDim.x * 4 */) {
    const long long n = *d_count;
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const double x = px[i], y = py[i];
        mnx = fmin(mnx, x); mxx = fmax(mxx, x);
        mny = fmin(mny, y); mxy = fmax(mxy, y);
    }
    block_min_max(mnx, mny, mxx, mxy, [&](double x0, double y0, double x1, double y1) {
        partial[blockIdx.x * 4 + 0] = x0; partial[blockIdx.x * 4 + 1] = y0;
        partial[blockIdx.x * 4 + 2] = x1; partial[blockIdx.x * 4 + 3] = y1;
    });
}

__global__ void __launch_bounds__(kMT)
k_bounds_final(const double* __restrict__ partial, int n_partial, double* __restrict__ bounds) {
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (int i = threadIdx.x; i < n_partial; i += kMT) {
        mnx = fmin(mnx, partial[i * 4 + 0]); mny = fmin(mny, partial[i * 4 + 1]);
        mxx = fmax(mxx, partial[i * 4 + 2]); mxy = fmax(mxy, partial[i * 4 + 3]);
    }
    block_min_max(mnx, mny, mxx, mxy, [&](double x0, double y0, double x1, double y1) {
        bounds[0] = x0; bounds[1] = y0; bounds[2] = x1; bounds[3] = y1;
    });
}

// ---- a11: VoxelDownSample -------------------------------------------------------------------
// O(points) per call.  The dense voxel lattice is only a lookup table (two uint32 planes that are
// all-zero between calls and cleaned by the very threads that dirtied them), never scanned:
//   mark    every point i: key = voxel index; first[key] = max(first[key], ~i) (i.e. the SMALLEST
//           index wins); cnt[key] += 1
//   gather  one lattice read per point -> head[i] (index of the first point of i's voxel) and
//           hcnt[i] (voxel size if i is that head, else 0); the rest streams per-point arrays
//   scan    over the POINTS (3 kernels): exclusive sums of [head] (-> output position: voxels come
//           out in order of first appearance) and of hcnt (-> slot range of the voxel)
//   fill    every point drops its index into its voxel's slot range; cnt counts back to zero and
//           the thread that takes the last ticket clears first[key]
//   reduce  every head visits its voxel's indices in ascending order, accumulates, divides
//           (AccumulatedPoint::GetAveragePoint), writes the mean

struct VoxelHeader {          // lives at the start of the voxel workspace
    double mbx, mby;          // voxel_min_bound = min_bound - 0.5 * voxel
    long long nx, ny, cells;  // lattice extent actually used by this call
    long long n_points;
    unsigned int total_slots, total_voxels;
};

__global__ void k_voxel_setup(const double* __restrict__ bounds_in, unsigned long long* __restrict__ benc,
                              const long long* __restrict__ d_count, double voxel,
                              long long capacity_cells, long long point_capacity, VoxelHeader* __restrict__ hdr,
                              int* __restrict__ status) {
    const long long n = *d_count;
    double bounds[4];
    if (benc) {                              // bounds carried on the device: decode, then reset for this call's output
        for (int j = 0; j < 4; ++j) bounds[j] = dec_double(benc[j]);
        benc[0] = benc[1] = enc_double(INFINITY);
        benc[2] = benc[3] = enc_double(-INFINITY);
    } else {
        for (int j = 0; j < 4; ++j) bounds[j] = bounds_in[j];
    }
    VoxelHeader h;
    h.n_points = n;
    h.total_slots = h.total_voxels = 0;
    h.mbx = OCC_DADD(bounds[0], -OCC_DMUL(voxel, 0.5));
    h.mby = OCC_DADD(bounds[1], -OCC_DMUL(voxel, 0.5));
    if (n <= 0) { h.nx = h.ny = h.cells = 0; h.n_points = 0; *hdr = h; return; }
    h.nx = (long long)floor(OCC_DDIV(OCC_DADD(bounds[2], -h.mbx), voxel)) + 1;
    h.ny = (long long)floor(OCC_DDIV(OCC_DADD(bounds[3], -h.mby), voxel)) + 1;
    h.cells = h.nx * h.ny;
    if (h.nx <= 0 || h.ny <= 0 || h.cells > capacity_cells || h.cells >= 0xffffffffll || n > point_capacity ||
        n >= 0xfffffff0ll) {
        atomicOr(status, n > point_capacity ? ST_POINT_OVERFLOW : ST_LATTICE_OVERFLOW);
        h.cells = 0; h.n_points = 0;        // make every later kernel of this call a no-op
    }
    *hdr = h;
}

constexpr unsigned int kSingle = 0xffffffffu;   // head[] marker: the point is alone in its voxel

// lattice[k] = {first, cnt} share one 8-byte slot (one sector per point per pass)
__global__ void __launch_bounds__(kMT)
k_voxel_mark(const double* __restrict__ px, const double* __restrict__ py, double voxel,
             const VoxelHeader* __restrict__ hdr, uint2* __restrict__ lattice, unsigned int* __restrict__ key) {
    const long long n = hdr->n_points;
    const double mbx = hdr->mbx, mby = hdr->mby;
    const long long nx = hdr->nx;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const long long ix = (long long)floor(OCC_DDIV(OCC_DADD(px[i], -mbx), voxel));
        const long long iy = (long long)floor(OCC_DDIV(OCC_DADD(py[i], -mby), voxel));
        const unsigned int k = (unsigned int)(iy * nx + ix);
        key[i] = k;
        atomicMax(&lattice[k].x, 0xffffffffu - (unsigned int)i);
        atomicAdd(&lattice[k].y, 1u);
    }
}

// One lattice read per point: head[i] = index of the first point of i's voxel; hcnt[i] = size of
// the voxel when i is that head, else 0.  Everything downstream streams these per-point arrays.
__global__ void __launch_bounds__(kMT)
k_voxel_gather(const VoxelHeader* __restrict__ hdr, uint2* __restrict__ lattice, const unsigned int* __restrict__ key,
               unsigned int* __restrict__ head, unsigned int* __restrict__ hcnt) {
    const long long n = hdr->n_points;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const unsigned int k = key[i];
        const uint2 v = lattice[k];
        if (v.y == 1u) {                       // alone in its voxel (the common case): nothing to collect,
            head[i] = kSingle;                 // and nobody else looks at this slot -> clean it right here
            hcnt[i] = 1u;
            lattice[k] = make_uint2(0u, 0u);
            continue;
        }
        const unsigned int h = 0xffffffffu - v.x;
        head[i] = h;
        hcnt[i] = (h == (unsigned int)i) ? v.y : 0u;
    }
}

constexpr int kScanItems = 8;
constexpr int kScanChunk = kMT * kScanItems;

__global__ void __launch_bounds__(kMT)
k_pscan_partial(const VoxelHeader* __restrict__ hdr, const unsigned int* __restrict__ hcnt, uint2* __restrict__ block_sums) {
    __shared__ unsigned int s_warp[33];
    const long long n = hdr->n_points;
    const long long nblocks = (n + kScanChunk - 1) / kScanChunk;
    for (long long b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const long long base = b * kScanChunk + (long long)threadIdx.x * kScanItems;
        unsigned int s = 0, f = 0;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            const unsigned int c = (base + j < n) ? hcnt[base + j] : 0u;
            s += c; f += c ? 1u : 0u;
        }
        unsigned int ts, tf;
        block_exclusive_scan(s, s_warp, &ts);
        block_exclusive_scan(f, s_warp, &tf);
        if (threadIdx.x == 0) block_sums[b] = make_uint2(ts, tf);
    }
}

__global__ void __launch_bounds__(1024)
k_pscan_top(uint2* __restrict__ block_sums, VoxelHeader* __restrict__ hdr) {
    __shared__ unsigned int s_warp[33];
    __shared__ unsigned int s_c0, s_c1;
    const long long n = hdr->n_points;
    const long long nblocks = (n + kScanChunk - 1) / kScanChunk;
    if (threadIdx.x == 0) { s_c0 = 0; s_c1 = 0; }
    __syncthreads();
    for (long long start = 0; start < nblocks; start += blockDim.x) {
        const long long i = start + threadIdx.x;
        const uint2 v = i < nblocks ? block_sums[i] : make_uint2(0u, 0u);
        unsigned int t0, t1;
        const unsigned int e0 = block_exclusive_scan(v.x, s_warp, &t0);
        const unsigned int e1 = block_exclusive_scan(v.y, s_warp, &t1);
        if (i < nblocks) block_sums[i] = make_uint2(s_c0 + e0, s_c1 + e1);
        __syncthreads();
        if (threadIdx.x == 0) { s_c0 += t0; s_c1 += t1; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { hdr->total_slots = s_c0; hdr->total_voxels = s_c1; }
}

// For every head point i: output position vrank[i] and slot offset soff[i].
__global__ void __launch_bounds__(kMT)
k_pscan_apply(const VoxelHeader* __restrict__ hdr, const unsigned int* __restrict__ hcnt,
              const uint2* __restrict__ block_sums, unsigned int* __restrict__ vrank, unsigned int* __restrict__ soff) {
    __shared__ unsigned int s_warp[33];
    const long long n = hdr->n_points;
    const long long nblocks = (n + kScanChunk - 1) / kScanChunk;
    for (long long b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const long long base = b * kScanChunk + (long long)threadIdx.x * kScanItems;
        unsigned int c[kScanItems];
        unsigned int s = 0, f = 0;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            c[j] = (base + j < n) ? hcnt[base + j] : 0u;
            s += c[j]; f += c[j] ? 1u : 0u;
        }
        unsigned int ts, tf;
        unsigned int es = block_exclusive_scan(s, s_warp, &ts);
        unsigned int ef = block_exclusive_scan(f, s_warp, &tf);
        const uint2 carry = block_sums[b];
        es += carry.x;
        ef += carry.y;
#pragma unroll
        for (int j = 0; j < kScanItems; ++j) {
            if (c[j]) { vrank[base + j] = ef; soff[base + j] = es; }
            es += c[j];
            ef += c[j] ? 1u : 0u;
        }
    }
}

// Every point drops its index into its voxel's slot range; the lattice slot is cleared by the
// thread that takes the last ticket (cnt back to 0 -> first := 0), so the table is clean again.
__global__ void __launch_bounds__(kMT)
k_voxel_fill(const VoxelHeader* __restrict__ hdr, const unsigned int* __restrict__ key, uint2* __restrict__ lattice,
             const unsigned int* __restrict__ head, const unsigned int* __restrict__ soff, unsigned int* __restrict__ slots) {
    const long long n = hdr->n_points;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const unsigned int h = head[i];
        if (h == kSingle) continue;                     // already finished (and cleaned) by the gather pass
        const unsigned int k = key[i];
        const unsigned int r = atomicSub(&lattice[k].y, 1u) - 1u;
        if (r == 0u) lattice[k].x = 0u;                 // last ticket: nobody reads first[] any more
        slots[soff[h] + r] = (unsigned int)i;
    }
}

__global__ void __launch_bounds__(kMT)
k_voxel_reduce(const double* __restrict__ px, const double* __restrict__ py, const VoxelHeader* __restrict__ hdr,
               const unsigned int* __restrict__ hcnt, const unsigned int* __restrict__ vrank,
               const unsigned int* __restrict__ soff, const unsigned int* __restrict__ slots,
               double* __restrict__ out_x, double* __restrict__ out_y, long long* __restrict__ out_count,
               unsigned long long* __restrict__ benc) {
    const long long n = hdr->n_points;
    if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = (long long)hdr->total_voxels;
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const unsigned int c = hcnt[i];
        if (c == 0u) continue;                          // not a head
        double sx = px[i], sy = py[i];                  // the head has the smallest index of its voxel
        if (c > 1u) {
            const unsigned int b = soff[i], e = b + c;
            long long last = i;
            for (unsigned int r = b + 1; r < e; ++r) {  // selection by ascending index, O(cnt^2), cnt is tiny
                unsigned int best = 0xffffffffu;
                for (unsigned int q = b; q < e; ++q) {
                    const unsigned int idx = slots[q];
                    if ((long long)idx > last && idx < best) best = idx;
                }
                last = best;
                sx = OCC_DADD(sx, px[best]);
                sy = OCC_DADD(sy, py[best]);
            }
        }
        const double cnt = (double)c;
        const double ox_ = OCC_DDIV(sx, cnt), oy_ = OCC_DDIV(sy, cnt);
        out_x[vrank[i]] = ox_;
        out_y[vrank[i]] = oy_;
        mnx = fmin(mnx, ox_); mxx = fmax(mxx, ox_); mny = fmin(mny, oy_); mxy = fmax(mxy, oy_);
    }
    if (benc) block_bounds_atomic(mnx, mny, mxx, mxy, benc);
}

// ---- incremental voxel chain ---------------------------------------------------------------
// The reference voxel-filters the WHOLE accumulated cloud on every callback (:58-60).  Once a
// cloud G has been filtered under a lattice (anchor = min_bound - voxel/2) it holds one point per
// voxel, and filtering G u S under the SAME lattice only changes the voxels S falls into: every
// other point is alone in its voxel and p / 1.0 == p.  So while the anchor stays bitwise equal a
// callback is three small kernels over the slice:
//   link    every slice point pushes itself on a per-voxel stack hanging off a persistent
//           voxel -> cloud-index map LM (one atomicExch)
//   fold    the point on top of each stack walks it, sums [the cloud point of that voxel, if any]
//           ++ [the slice points in ascending index] and divides: an existing voxel is updated in
//           place, a new one is parked at its first slice index
//   append  ordered compaction of the parked means onto the end of the cloud (order of first
//           appearance), LM and the per-point voxel keys are extended
// When the anchor moves (the cloud's min corner changed) or a mean lands outside the voxel of its
// points, the callback needs the full filter and a rebuilt LM.  Callbacks are enqueued without
// host round trips: the kernels take the next slice from a device cursor and turn into no-ops
// once a callback needs the host (header.stalled), which the host polls every few callbacks.

struct ChainHeader {
    VoxelHeader v;                       // lattice + point count for the full filter of a rebuild
    double mbx, mby;                     // anchor LM / gkey are valid for
    unsigned long long gb_enc[4];        // bounds of the cloud (encoded, see enc_double); min corner exact
    unsigned long long gb2_enc[4];       // scratch of a full recompute
    int have_lattice, force_rebuild, bounds_dirty;
    int stalled;                         // 0 running, else OCC_CHAIN_* reason the host has to deal with
    int cursor;                          // next entry of order[]
    int aborted;                         // a grid barrier timed out (a CTA went missing): the launch gave up
};
enum { CHAIN_RUN = 0, CHAIN_REBUILD = 1, CHAIN_OVERFLOW = 2, CHAIN_REBOUND = 3, CHAIN_ABORTED = 4 };

__device__ __forceinline__ bool voxel_key_of(double x, double y, double mbx, double mby, double voxel, long long W,
                                             long long H, unsigned int* key) {
    const long long ix = (long long)floor(OCC_DDIV(OCC_DADD(x, -mbx), voxel));
    const long long iy = (long long)floor(OCC_DDIV(OCC_DADD(y, -mby), voxel));
    if (ix < 0 || iy < 0 || ix >= W || iy >= H) return false;
    *key = (unsigned int)(iy * W + ix);
    return true;
}

// What the callback for slice `agent` needs; also yields the anchor of cloud u slice.
// Header fields are read with ld.global.cg: other CTAs update them during a launch (atomics and plain
// stores land in L2) and this SM's L1 may still hold an older copy.
__device__ __forceinline__ int chain_decide(const ChainHeader* h, const unsigned long long* sb /* slice bounds */, double voxel,
                                            long long W, long long H, double* nmbx, double* nmby) {
    const unsigned long long g0 = __ldcg(&h->gb_enc[0]), g1 = __ldcg(&h->gb_enc[1]), g2 = __ldcg(&h->gb_enc[2]), g3 = __ldcg(&h->gb_enc[3]);
    const int dirty = __ldcg(&h->bounds_dirty), have = __ldcg(&h->have_lattice), force = __ldcg(&h->force_rebuild);
    const double hmbx = __ldcg(&h->mbx), hmby = __ldcg(&h->mby);
    const double b0 = fmin(dec_double(g0), dec_double(sb[0]));
    const double b1 = fmin(dec_double(g1), dec_double(sb[1]));
    const double b2 = fmax(dec_double(g2), dec_double(sb[2]));
    const double b3 = fmax(dec_double(g3), dec_double(sb[3]));
    *nmbx = OCC_DADD(b0, -OCC_DMUL(voxel, 0.5));
    *nmby = OCC_DADD(b1, -OCC_DMUL(voxel, 0.5));
    if (dirty) return CHAIN_REBOUND;
    const long long nx = (long long)floor(OCC_DDIV(OCC_DADD(b2, -*nmbx), voxel)) + 1;
    const long long ny = (long long)floor(OCC_DDIV(OCC_DADD(b3, -*nmby), voxel)) + 1;
    if (!(nx > 0 && ny > 0 && nx <= W && ny <= H)) return CHAIN_OVERFLOW;
    if (!have || force || *nmbx != hmbx || *nmby != hmby) return CHAIN_REBUILD;
    return CHAIN_RUN;
}

__global__ void k_chain_reset(ChainHeader* __restrict__ h) {
    h->gb_enc[0] = h->gb_enc[1] = h->gb2_enc[0] = h->gb2_enc[1] = enc_double(INFINITY);
    h->gb_enc[2] = h->gb_enc[3] = h->gb2_enc[2] = h->gb2_enc[3] = enc_double(-INFINITY);
    h->have_lattice = h->force_rebuild = 0;
    h->bounds_dirty = 1;                 // k_chain_rebounds + _apply compute the bounds of the adopted cloud
    h->stalled = 0;
    h->cursor = 0;
    h->aborted = 0;
}

// Bounds of every slice of the batch: blockIdx.y = agent, atomics into slice_benc[agent][4]
// (pre-set to +-inf by k_chain_slice_bounds_init).
__global__ void k_chain_slice_bounds_init(unsigned long long* __restrict__ slice_benc, int n_agents) {
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < n_agents; a += gridDim.x * blockDim.x) {
        slice_benc[4 * a + 0] = slice_benc[4 * a + 1] = enc_double(INFINITY);
        slice_benc[4 * a + 2] = slice_benc[4 * a + 3] = enc_double(-INFINITY);
    }
}
__global__ void __launch_bounds__(kMT)
k_chain_slice_bounds(const double* __restrict__ sx, const double* __restrict__ sy, const long long* __restrict__ agent_offset,
                     unsigned long long* __restrict__ slice_benc) {
    const int a = blockIdx.y;
    const long long b = agent_offset[a], e = agent_offset[a + 1];
    if (b + (long long)blockIdx.x * kMT >= e) return;
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (long long i = b + (long long)blockIdx.x * kMT + threadIdx.x; i < e; i += (long long)gridDim.x * kMT) {
        const double x = sx[i], y = sy[i];
        mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
    }
    block_bounds_atomic(mnx, mny, mxx, mxy, slice_benc + 4 * a);
}

// LM[k] = {index + 1 of the cloud point in voxel k (0: none), top of this callback's stack}
//
// The phases of a callback run inside ONE persistent kernel (cooperative launch, every CTA
// resident) separated by grid-wide barriers (two per callback: the next slice is linked while the
// current one is appended), and the kernel loops over up to n_callbacks
// callbacks: a phase is a few microseconds of latency-bound work on ~6e4 points, so kernel
// boundaries would cost as much as the work.  Every CTA keeps its own copy of the cursor and the
// cloud size (they evolve identically everywhere); CTA 0 publishes them for the host.
struct ChainRun {
    ChainHeader* h;
    const int* order;
    int n_order, n_callbacks;
    const long long* agent_offset;
    const unsigned long long* slice_benc;
    const double* sx;
    const double* sy;
    double voxel;
    long long W, H;
    uint2* LM;
    unsigned int *lkey, *next, *gkey, *flag, *blockcount;      // blockcount: two buffers of bc_stride entries
    double *gx, *gy, *resx, *resy;
    long long* d_count;
    long long capacity;
    int* status;
    unsigned int* bar;                                         // {arrivals, exits, release, verdict}; all zero between launches
    int bc_stride;
};

__device__ __forceinline__ void chain_link(const ChainRun& p, long long b, long long n, double mbx, double mby) {
    for (long long j = (long long)blockIdx.x * kMT + threadIdx.x; j < n; j += (long long)gridDim.x * kMT) {
        unsigned int k = 0;
        voxel_key_of(p.sx[b + j], p.sy[b + j], mbx, mby, p.voxel, p.W, p.H, &k);    // in range: the lattice covers cloud u slice
        p.lkey[j] = k;
        p.next[j] = atomicExch(&p.LM[k].y, (unsigned int)j + 1u);
    }
}

__device__ __forceinline__ void chain_fold(const ChainRun& p, long long b, long long n, double mbx, double mby,
                                           unsigned int* bc) {
    ChainHeader* h = p.h;
    const double g0 = dec_double(h->gb_enc[0]), g1 = dec_double(h->gb_enc[1]);
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    const int lane = threadIdx.x & 31;
    for (long long j0 = (long long)blockIdx.x * kMT + (threadIdx.x & ~31); j0 < n; j0 += (long long)gridDim.x * kMT) {
        const long long j = j0 + lane;
        int parked = -1;                                       // append chunk a new voxel of this thread goes to
        unsigned int k = 0;
        uint2 e = make_uint2(0u, 0u);
        if (j < n) { k = p.lkey[j]; e = p.LM[k]; }
        if (j < n && e.y == (unsigned int)j + 1u) {            // top of its voxel's stack: this thread folds it
            unsigned int cnt = 0, head = (unsigned int)j;
            for (unsigned int q = e.y; q; q = p.next[q - 1]) { ++cnt; head = min(head, q - 1u); }
            double ax, ay;
            long long last;
            unsigned int remaining, total;
            if (e.x) { ax = p.gx[e.x - 1]; ay = p.gy[e.x - 1]; last = -1; remaining = cnt; total = cnt + 1u; }
            else     { ax = p.sx[b + head]; ay = p.sy[b + head]; last = head; remaining = cnt - 1u; total = cnt; }
            for (unsigned int r = 0; r < remaining; ++r) {     // ascending slice index; stacks are tiny
                unsigned int best = 0xffffffffu;
                for (unsigned int q = e.y; q; q = p.next[q - 1]) {
                    const unsigned int idx = q - 1u;
                    if ((long long)idx > last && idx < best) best = idx;
                }
                last = best;
                ax = OCC_DADD(ax, p.sx[b + best]);
                ay = OCC_DADD(ay, p.sy[b + best]);
            }
            const double c = (double)total;
            const double x = OCC_DDIV(ax, c), y = OCC_DDIV(ay, c);
            if (e.x) {
                const unsigned int g = e.x - 1u;
                const double oldx = p.gx[g], oldy = p.gy[g];
                // a point on the min corner moving inwards: the bounds need a full pass before the next decision
                if ((oldx <= g0 && x > oldx) || (oldy <= g1 && y > oldy)) h->bounds_dirty = 1;
                p.gx[g] = x; p.gy[g] = y;
                unsigned int k2 = 0;
                if (!voxel_key_of(x, y, mbx, mby, p.voxel, p.W, p.H, &k2) || k2 != k) h->force_rebuild = 1;   // LM no longer describes the cloud
                mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
            } else {
                p.resx[head] = x; p.resy[head] = y;
                p.flag[head] = 1u;
                parked = (int)(head / kMT);
            }
            p.LM[k].y = 0u;
        }
        __syncwarp();
        const unsigned int peers = __match_any_sync(0xffffffffu, parked);      // one atomic per distinct chunk per warp
        if (parked >= 0 && lane == __ffs(peers) - 1) atomicAdd(&bc[parked], (unsigned int)__popc(peers));
    }
    block_bounds_atomic(mnx, mny, mxx, mxy, h->gb_enc);
}

// Ordered compaction of the parked means onto the end of the cloud; returns how many were appended.
__device__ __forceinline__ unsigned int chain_append(const ChainRun& p, long long n, long long n_g, double mbx, double mby,
                                                     const unsigned int* bc, unsigned int* s_warp) {
    ChainHeader* h = p.h;
    const unsigned int nb = (unsigned int)((n + kMT - 1) / kMT);
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    unsigned int all = 0;
    for (unsigned int c0 = 0; c0 < nb; c0 += gridDim.x) {          // uniform trip count: block scans inside
        const unsigned int chunk = c0 + blockIdx.x;
        // chunks in front of this one, and (first round only) every chunk: the appended total
        unsigned int part = 0, whole = 0;
        for (unsigned int q = threadIdx.x; q < nb; q += kMT) {
            const unsigned int v = bc[q];
            if (q < chunk) part += v;
            whole += v;
        }
        unsigned int before;
        block_exclusive_scan(part, s_warp, &before);
        if (c0 == 0) block_exclusive_scan(whole, s_warp, &all);
        const long long j = (long long)chunk * kMT + threadIdx.x;
        const unsigned int f = (chunk < nb && j < n) ? p.flag[j] : 0u;
        unsigned int mine;
        const unsigned int pos = block_exclusive_scan(f, s_warp, &mine);
        if (f) {
            p.flag[j] = 0u;
            const long long idx = n_g + before + pos;
            if (idx >= p.capacity) {
                atomicOr(p.status, ST_POINT_OVERFLOW);
            } else {
                const double x = p.resx[j], y = p.resy[j];
                p.gx[idx] = x; p.gy[idx] = y;
                unsigned int k = 0;
                if (!voxel_key_of(x, y, mbx, mby, p.voxel, p.W, p.H, &k)) { p.gkey[idx] = 0xffffffffu; h->force_rebuild = 1; }
                else {
                    p.gkey[idx] = k;
                    if (atomicExch(&p.LM[k].x, (unsigned int)idx + 1u) != 0u) h->force_rebuild = 1;   // mean drifted into an occupied voxel
                }
                mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
            }
        }
    }
    block_bounds_atomic(mnx, mny, mxx, mxy, h->gb_enc);
    return all;
}

__global__ void __launch_bounds__(kMT)
k_chain_persistent(const ChainRun p) {
    __shared__ unsigned int s_warp[33];
    ChainHeader* h = p.h;
    unsigned int target = 0;
    int done = 0;
    bool alive = true;                                 // false once a barrier timed out: leave without touching shared state
    if (!h->stalled) {
        int cur = h->cursor;
        long long n_g = *p.d_count;
        const double mbx = h->mbx, mby = h->mby;       // the anchor LM is valid for: every callback that runs uses exactly it
        // The first callback of a launch is decided and linked on its own; after that the NEXT
        // slice is linked speculatively (under the unchanged anchor) in the same phase that appends
        // the current one, so a callback costs two grid barriers.  The decision for it is taken by
        // the last CTA to arrive at the second barrier — ONE evaluation of chain_decide on the
        // header as the callback left it — and handed to every CTA with the release; a callback
        // that may not run has its stacks unlinked again.
        bool linked = false;
        if (p.n_callbacks > 0 && cur < p.n_order) {
            const int agent = p.order[cur];
            // nothing has been written since the launch began: all CTAs read the same header here
            double nmbx, nmby;
            const int need = chain_decide(h, p.slice_benc + 4 * agent, p.voxel, p.W, p.H, &nmbx, &nmby);
            if (need != CHAIN_RUN) {
                if (blockIdx.x == 0 && threadIdx.x == 0) {
                    h->stalled = need;
                    if (need == CHAIN_OVERFLOW) atomicOr(p.status, ST_LATTICE_OVERFLOW);
                }
            } else {
                const long long b = p.agent_offset[agent];
                chain_link(p, b, p.agent_offset[agent + 1] - b, mbx, mby);
                // no CTA may start folding (which writes the flags chain_decide reads) before every
                // CTA has taken the decision above
                alive = grid_barrier(p.bar, target, &h->aborted);
                linked = alive;
            }
        }
        for (int it = 0; linked; ++it) {
            const int agent = p.order[cur];
            const long long b = p.agent_offset[agent], n = p.agent_offset[agent + 1] - b;
            unsigned int* bc = p.blockcount + (size_t)(it & 1) * p.bc_stride;
            unsigned int* bc_other = p.blockcount + (size_t)((it & 1) ^ 1) * p.bc_stride;
            if (blockIdx.x == 0 && it > 0)             // the previous callback's counters: its append phase is over
                for (int q = threadIdx.x; q < p.bc_stride; q += kMT) bc_other[q] = 0u;
            chain_fold(p, b, n, mbx, mby, bc);
            if (!(alive = grid_barrier(p.bar, target, &h->aborted))) break;
            const unsigned int added = chain_append(p, n, n_g, mbx, mby, bc, s_warp);
            n_g += added;
            if (n_g > p.capacity) n_g = p.capacity;
            cur += 1;
            done = it + 1;
            if (blockIdx.x == 0 && threadIdx.x == 0) { *p.d_count = n_g; h->cursor = cur; }
            const bool more = it + 1 < p.n_callbacks && cur < p.n_order;
            int next_agent = 0;
            long long nb = 0, nn = 0;
            if (more) {                                // append touches LM[].x, flags and the cloud; link touches LM[].y, lkey, next
                next_agent = p.order[cur];
                nb = p.agent_offset[next_agent];
                nn = p.agent_offset[next_agent + 1] - nb;
                chain_link(p, nb, nn, mbx, mby);
            }
            // bounds / flags of this callback feed the next decision: taken once, by the last arriver
            int need = CHAIN_RUN;
            alive = grid_barrier(p.bar, target, &h->aborted, &need, [&] {
                if (!more) return (int)CHAIN_RUN;
                double ax, ay;
                return chain_decide(h, p.slice_benc + 4 * next_agent, p.voxel, p.W, p.H, &ax, &ay);
            });
            if (!alive || !more) break;
            if (need != CHAIN_RUN) {
                for (long long j = (long long)blockIdx.x * kMT + threadIdx.x; j < nn; j += (long long)gridDim.x * kMT)
                    p.LM[p.lkey[j]].y = 0u;            // unlink: the host deals with this callback
                if (blockIdx.x == 0 && threadIdx.x == 0) {
                    h->stalled = need;
                    if (need == CHAIN_OVERFLOW) atomicOr(p.status, ST_LATTICE_OVERFLOW);
                }
                break;
            }
        }
    }
    if (!alive) {                                      // a barrier timed out: the state is unusable, tell the host
        if (threadIdx.x == 0) { h->stalled = CHAIN_ABORTED; atomicOr(p.status, ST_CHAIN_ABORTED); }
        return;
    }
    // leave the counters and the barrier clean for the next launch
    if (blockIdx.x == 0 && done)
        for (int q = threadIdx.x; q < p.bc_stride; q += kMT) p.blockcount[(size_t)((done - 1) & 1) * p.bc_stride + q] = 0u;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(p.bar + 1, 1u) == gridDim.x - 1) { p.bar[0] = 0u; p.bar[1] = 0u; p.bar[2] = 0u; p.bar[3] = 0u; }
    }
}

// Full min/max pass over the cloud (at start, and when a callback may have moved the min corner inwards).
__global__ void __launch_bounds__(kMT)
k_chain_rebounds(const double* __restrict__ gx, const double* __restrict__ gy, const long long* __restrict__ n_ptr,
                 ChainHeader* __restrict__ h) {
    const long long n = *n_ptr;
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const double x = gx[i], y = gy[i];
        mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
    }
    block_bounds_atomic(mnx, mny, mxx, mxy, h->gb2_enc);
}
__global__ void k_chain_rebounds_apply(ChainHeader* __restrict__ h) {
    h->gb_enc[0] = h->gb2_enc[0]; h->gb_enc[1] = h->gb2_enc[1];
    // max corner: only has to cover the cloud (it sizes the lattice check); keep it monotone
    h->gb_enc[2] = max(h->gb_enc[2], h->gb2_enc[2]); h->gb_enc[3] = max(h->gb_enc[3], h->gb2_enc[3]);
    h->gb2_enc[0] = h->gb2_enc[1] = enc_double(INFINITY);
    h->gb2_enc[2] = h->gb2_enc[3] = enc_double(-INFINITY);
    h->bounds_dirty = 0;
    if (h->stalled == CHAIN_REBOUND) h->stalled = CHAIN_RUN;
}

__global__ void __launch_bounds__(kMT)
k_chain_lm_clear(ChainHeader* __restrict__ h, uint2* __restrict__ LM, const unsigned int* __restrict__ gkey,
                 const long long* __restrict__ d_count) {
    if (!h->have_lattice) return;
    const long long n = *d_count;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const unsigned int k = gkey[i];
        if (k != 0xffffffffu) LM[k] = make_uint2(0u, 0u);
    }
}

// After the slice has been appended: lattice of cloud u slice for the full filter.
__global__ void k_chain_rebuild_hdr(ChainHeader* __restrict__ h, const unsigned long long* __restrict__ slice_benc, int agent,
                                    const long long* __restrict__ d_count, double voxel, long long W, long long H,
                                    long long point_capacity, int* __restrict__ status) {
    double nmbx, nmby;
    const int dirty = h->bounds_dirty;
    h->bounds_dirty = 0;
    int need = chain_decide(h, slice_benc + 4 * agent, voxel, W, H, &nmbx, &nmby);
    h->bounds_dirty = dirty;
    long long n = *d_count;
    if (n > point_capacity || n >= 0x7ffffff0ll) { atomicOr(status, ST_POINT_OVERFLOW); n = 0; }
    if (need == CHAIN_OVERFLOW) { atomicOr(status, ST_LATTICE_OVERFLOW); n = 0; }
    h->v.mbx = nmbx; h->v.mby = nmby;
    h->v.nx = W; h->v.ny = H; h->v.cells = W * H;
    h->v.n_points = n;
    h->v.total_slots = h->v.total_voxels = 0;
    h->force_rebuild = 0;
    h->gb_enc[0] = h->gb_enc[1] = enc_double(INFINITY);     // the filter's reduce pass leaves the new cloud's bounds
    h->gb_enc[2] = h->gb_enc[3] = enc_double(-INFINITY);
}

__global__ void __launch_bounds__(kMT)
k_chain_lm_build(ChainHeader* __restrict__ h, const double* __restrict__ gx, const double* __restrict__ gy,
                 const long long* __restrict__ d_count, double voxel, uint2* __restrict__ LM, unsigned int* __restrict__ gkey) {
    const long long n = *d_count;
    const double mbx = h->v.mbx, mby = h->v.mby;
    const long long W = h->v.nx, H = h->v.ny;
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        unsigned int k;
        if (!voxel_key_of(gx[i], gy[i], mbx, mby, voxel, W, H, &k)) { gkey[i] = 0xffffffffu; h->force_rebuild = 1; continue; }
        gkey[i] = k;
        if (atomicExch(&LM[k].x, (unsigned int)i + 1u) != 0u) h->force_rebuild = 1;   // a mean drifted into a neighbour's voxel
    }
}

__global__ void k_chain_rebuild_done(ChainHeader* __restrict__ h) {
    h->mbx = h->v.mbx; h->mby = h->v.mby;
    h->have_lattice = 1;
    h->bounds_dirty = 0;
    h->stalled = CHAIN_RUN;
    h->cursor += 1;
}

// ---- a12: publish_global_map rasterise (:103-111) -----------------------------------------

__global__ void __launch_bounds__(kMT)
k_raster_fill(int8_t* __restrict__ grid, long long n) {
    const long long n16 = ((reinterpret_cast<uintptr_t>(grid) & 15) == 0) ? n / 16 : 0;
    int4* g4 = reinterpret_cast<int4*>(grid);
    const int4 v = make_int4(-1, -1, -1, -1);
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n16; i += (long long)gridDim.x * kMT) g4[i] = v;
    for (long long i = n16 * 16 + (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) grid[i] = -1;
}

__global__ void __launch_bounds__(kMT)
k_raster_scatter(const double* __restrict__ px, const double* __restrict__ py, const long long* __restrict__ d_count,
                 const double* __restrict__ bounds, double res, int width, int height, int8_t* __restrict__ grid) {
    const long long n = *d_count;
    const double min_x = bounds[0], min_y = bounds[1];
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        long long xi = (long long)OCC_DDIV(OCC_DADD(px[i], -min_x), res);     // :105  astype(int) truncates
        long long yi = (long long)OCC_DDIV(OCC_DADD(py[i], -min_y), res);     // :106
        xi = xi < 0 ? 0 : (xi > width - 1 ? width - 1 : xi);                    // :108
        yi = yi < 0 ? 0 : (yi > height - 1 ? height - 1 : yi);                  // :109
        grid[yi * width + xi] = OCCGRID_CELL_OCCUPIED;                          // :111
    }
}

// Element-wise max of two int8 grids (values {-1, 100}: "occupied wins"), the local half of
// the multi-GPU fuse (the cross-GPU half is ncclMax on int8).
__global__ void __launch_bounds__(kMT)
k_fuse_max(int8_t* __restrict__ dst, const int8_t* __restrict__ src, long long n) {
    for (long long i = (long long)blockIdx.x * kMT + threadIdx.x; i < n; i += (long long)gridDim.x * kMT) {
        const int8_t a = dst[i], b = src[i];
        dst[i] = a > b ? a : b;
    }
}

static int grid_for(long long work_items) {
    long long b = (work_items + kMT - 1) / kMT;
    if (b < 1) b = 1;
    if (b > device_sm_count() * 16) b = device_sm_count() * 16;
    return (int)b;
}

}  // namespace occ

using namespace occ;

extern "C" {

int mapmerge_count_occupied(const int8_t* d_grid, int64_t n_cells, int64_t* d_out, void* stream) {
    if (!d_grid || !d_out) { set_last_error("mapmerge_count_occupied: NULL pointer"); return OCCGRID_E_ARG; }
    if (n_cells < 0) { set_last_error("mapmerge_count_occupied: n_cells %lld < 0", (long long)n_cells); return OCCGRID_E_ARG; }
    if (n_cells == 0) return OCCGRID_OK;
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_MERGE_EXTRACT, st, 1);
    k_count_occupied<<<grid_for(n_cells / kLoadCells + 1), kMT, 0, st>>>(d_grid, n_cells, (long long*)d_out);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

size_t mapmerge_extract_workspace_bytes(int64_t n_cells) {
    const int64_t blocks = (n_cells + kChunk - 1) / kChunk;
    return align_up((size_t)blocks * sizeof(unsigned int), 256) + 256;
}

int mapmerge_extract_transform(const int8_t* d_grid, int32_t width, int32_t height, double res, double origin_x,
                               double origin_y, const double* T_host, double* d_px, double* d_py, int64_t capacity,
                               int64_t* d_count, int64_t* d_last_appended, int32_t* d_status, void* d_ws, size_t ws_bytes,
                               void* stream) {
    if (!d_grid || !d_px || !d_py || !d_count || !d_status || !d_ws || width <= 0 || height <= 0 || !(res > 0.0)) {
        set_last_error("mapmerge_extract_transform: bad arguments");
        return OCCGRID_E_ARG;
    }
    const long long n_cells = (long long)width * height;
    if (ws_bytes < mapmerge_extract_workspace_bytes(n_cells)) { set_last_error("mapmerge_extract_transform: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (int)((n_cells + kChunk - 1) / kChunk);
    long long* ws_base = reinterpret_cast<long long*>(d_ws);
    unsigned int* block_counts = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(d_ws) + 256);
    Xform T;
    T.identity = 1;
    for (int i = 0; i < 16; ++i) T.m[i] = (i % 5 == 0) ? 1.0 : 0.0;
    if (T_host) {
        for (int i = 0; i < 16; ++i) { T.m[i] = T_host[i]; if (T_host[i] != ((i % 5 == 0) ? 1.0 : 0.0)) T.identity = 0; }
    }
    ProfileScope ps(K_MERGE_EXTRACT, st, 3);
    k_extract_count<<<blocks, kMT, 0, st>>>(d_grid, n_cells, block_counts);
    k_extract_reserve<<<1, 1024, 0, st>>>(block_counts, blocks, (long long*)d_count, capacity, ws_base, d_status,
                                           (long long*)d_last_appended);
    k_extract_write<<<blocks, kMT, 0, st>>>(d_grid, n_cells, width, res, origin_x, origin_y, T, block_counts, ws_base, d_px, d_py);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

static size_t batch_counts_bytes(int64_t n_cells, int n_agents) {
    const int64_t blocks = (n_cells + kChunk - 1) / kChunk;
    return align_up((size_t)blocks * (size_t)n_agents * sizeof(unsigned int), 256);
}

// block counts [A][blocks] | occupancy masks [A][blocks * kMT] (one bit per cell)
size_t mapmerge_extract_batch_workspace_bytes(int64_t n_cells, int n_agents) {
    const int64_t blocks = (n_cells + kChunk - 1) / kChunk;
    return batch_counts_bytes(n_cells, n_agents) + align_up((size_t)blocks * kMT * (size_t)n_agents * sizeof(unsigned long long), 256);
}

// Pass 1 of a batched extraction: per-block and per-agent occupied-cell counts.
int mapmerge_extract_batch_count(const int8_t* const* d_grids, int n_agents, int32_t width, int32_t height,
                                 int64_t* d_agent_total, void* d_ws, size_t ws_bytes, int grids_bulk_ok, void* stream) {
    if (!d_grids || !d_agent_total || !d_ws) { set_last_error("mapmerge_extract_batch_count: NULL pointer"); return OCCGRID_E_ARG; }
    if (n_agents <= 0 || n_agents > 65535) {
        set_last_error("mapmerge_extract_batch_count: n_agents %d outside 1..65535", n_agents);
        return OCCGRID_E_ARG;
    }
    if (width <= 0 || height <= 0) {
        set_last_error("mapmerge_extract_batch_count: width x height %d x %d", (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    const long long n_cells = (long long)width * height;
    if (ws_bytes < mapmerge_extract_batch_workspace_bytes(n_cells, n_agents)) { set_last_error("mapmerge_extract_batch_count: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int bpg = (int)((n_cells + kChunk - 1) / kChunk);
    unsigned int* block_counts = reinterpret_cast<unsigned int*>(d_ws);
    ProfileScope ps(K_MERGE_EXTRACT, st, 1);
    dim3 grid((unsigned)bpg, (unsigned)n_agents);
    unsigned long long* masks = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(d_ws) + batch_counts_bytes(n_cells, n_agents));
    {
        // the scan proper, timed on its own: the HBM-bound kernel of the merge path
        ProfileScope scan(K_MERGE_SCAN, st, 1);
        if (grids_bulk_ok && (n_cells % 16) == 0) {
            const int ctas = device_sm_count() * kScanCtasPerSm;
            const size_t smem = (size_t)kScanStages * kScanStageBytes;
            static bool configured = false;
            if (!configured) {
                OCC_CUDA_TRY(cudaFuncSetAttribute(k_batch_count_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                configured = true;
            }
            k_batch_count_tma<<<ctas, kMT, smem, st>>>(d_grids, n_cells, bpg, n_agents, block_counts, masks);
        } else {
            k_batch_count<<<grid, kMT, 0, st>>>(d_grids, n_cells, bpg, block_counts, masks);
        }
    }
    k_batch_scan<<<n_agents, 1024, 0, st>>>(block_counts, bpg, (long long*)d_agent_total);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// Pass 2: the caller has read the totals, decided which agents take part (use_host) and which
// transform each gets (T_host; the first cloud is adopted untransformed, map_merger.py:40-43).
int mapmerge_extract_batch_write(const int8_t* const* d_grids, int n_agents, int32_t width, int32_t height, double res,
                                 const double* d_origins, const double* T_host /* [A][16] row-major or NULL */,
                                 const uint8_t* use_host /* [A] or NULL */, void* d_xforms /* >= A * 96 bytes */,
                                 double* d_px, double* d_py, int64_t capacity, const int64_t* d_agent_total,
                                 int64_t* d_agent_offset, int32_t* d_status, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grids || !d_origins || !d_xforms || !d_px || !d_py || !d_agent_total || !d_agent_offset || !d_status || !d_ws) {
        set_last_error("mapmerge_extract_batch_write: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (n_agents <= 0 || n_agents > 65535) {
        set_last_error("mapmerge_extract_batch_write: n_agents %d outside 1..65535", n_agents);
        return OCCGRID_E_ARG;
    }
    if (width <= 0 || height <= 0) {
        set_last_error("mapmerge_extract_batch_write: width x height %d x %d", (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    if (!(res > 0.0)) { set_last_error("mapmerge_extract_batch_write: res %g must be > 0", res); return OCCGRID_E_ARG; }
    const long long n_cells = (long long)width * height;
    if (ws_bytes < mapmerge_extract_batch_workspace_bytes(n_cells, n_agents)) { set_last_error("mapmerge_extract_batch_write: workspace too small"); return OCCGRID_E_WORKSPACE; }
    static_assert(sizeof(BatchXform) <= 96, "BatchXform must fit the 96-byte slot");
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<BatchXform> hx((size_t)n_agents);
    for (int a = 0; a < n_agents; ++a) {
        BatchXform& t = hx[a];
        t.use = use_host ? (use_host[a] != 0) : 1;
        t.identity = 1;
        const double I[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
        const double* M = T_host ? T_host + 16 * (size_t)a : I;
        for (int i = 0; i < 16; ++i) if (M[i] != I[i]) t.identity = 0;
        t.m[0] = M[0]; t.m[1] = M[1]; t.m[2] = M[3];
        t.m[3] = M[4]; t.m[4] = M[5]; t.m[5] = M[7];
        t.w[0] = M[12]; t.w[1] = M[13]; t.w[2] = M[15];
    }
    OCC_CUDA_TRY(cudaMemcpyAsync(d_xforms, hx.data(), sizeof(BatchXform) * (size_t)n_agents, cudaMemcpyHostToDevice, st));
    OCC_CUDA_TRY(cudaStreamSynchronize(st));        // hx is a local: the copy must have left it
    const int bpg = (int)((n_cells + kChunk - 1) / kChunk);
    unsigned int* block_counts = reinterpret_cast<unsigned int*>(d_ws);
    const BatchXform* dT = reinterpret_cast<const BatchXform*>(d_xforms);
    ProfileScope ps(K_MERGE_EXTRACT, st, 2);
    dim3 grid((unsigned)bpg, (unsigned)n_agents);
    k_batch_offsets<<<1, 1024, 0, st>>>((const long long*)d_agent_total, dT, n_agents, capacity, (long long*)d_agent_offset, d_status);
    const unsigned long long* masks = reinterpret_cast<const unsigned long long*>(reinterpret_cast<const char*>(d_ws) + batch_counts_bytes(n_cells, n_agents));
    k_batch_write<<<grid, kMT, 0, st>>>(masks, n_cells, width, res, d_origins, dT, bpg, block_counts, (const long long*)d_agent_offset,
                                        capacity, d_px, d_py);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_bounds_enc_reset(uint64_t* d_bounds_enc, void* stream) {
    if (!d_bounds_enc) { set_last_error("mapmerge_bounds_enc_reset: NULL"); return OCCGRID_E_ARG; }
    k_benc_reset<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long*)d_bounds_enc);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_append_slice(const double* d_sx, const double* d_sy, const int64_t* d_agent_offset, int agent,
                          double* d_px, double* d_py, int64_t capacity, int64_t* d_count, int32_t* d_status,
                          uint64_t* d_bounds_enc, void* stream) {
    if (!d_sx || !d_sy || !d_agent_offset || !d_px || !d_py || !d_count || !d_status) {
        set_last_error("mapmerge_append_slice: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (agent < 0) { set_last_error("mapmerge_append_slice: agent %d < 0", agent); return OCCGRID_E_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_MERGE_EXTRACT, st, 2);
    k_append_slice<<<device_sm_count(), kMT, 0, st>>>(d_sx, d_sy, (const long long*)d_agent_offset, agent, d_px, d_py, capacity,
                                         (long long*)d_count, d_status, (unsigned long long*)d_bounds_enc);
    k_bump_count<<<1, 1, 0, st>>>((const long long*)d_agent_offset, agent, capacity, (long long*)d_count);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

size_t mapmerge_bounds_workspace_bytes(void) { return (size_t)1024 * 8 * 4 * sizeof(double); }   // room for 8 CTAs on up to 1024 SMs

int mapmerge_bounds(const double* d_px, const double* d_py, const int64_t* d_count, double* d_bounds, void* d_ws,
                    size_t ws_bytes, void* stream) {
    if (!d_px || !d_py || !d_count || !d_bounds || !d_ws) { set_last_error("mapmerge_bounds: NULL pointer"); return OCCGRID_E_ARG; }
    if (ws_bytes < mapmerge_bounds_workspace_bytes()) { set_last_error("mapmerge_bounds: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = device_sm_count() * 8;
    ProfileScope ps(K_MERGE_BOUNDS, st, 2);
    k_bounds_partial<<<blocks, kMT, 0, st>>>(d_px, d_py, (const long long*)d_count, (double*)d_ws);
    k_bounds_final<<<1, kMT, 0, st>>>((const double*)d_ws, blocks, d_bounds);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// Workspace: header | lattice uint2[cells] {first, cnt} | block_sums uint2[...] |
//            key, head, hcnt, vrank, soff, slots: u32[points] each.
// The lattice must be zero on entry (zero the workspace once) and is zero again on exit.
static size_t voxel_layout(int64_t cells, int64_t points, size_t off[9]) {
    size_t o = 0;
    off[0] = o; o += 256;
    off[1] = o; o += align_up((size_t)(cells + 1) * 8, 256);
    off[2] = o; o += align_up((size_t)((points + kScanChunk - 1) / kScanChunk + 1) * 8, 256);
    for (int j = 3; j < 9; ++j) { off[j] = o; o += align_up((size_t)points * 4, 256); }
    return o;
}

size_t mapmerge_voxel_workspace_bytes(int64_t lattice_capacity_cells, int64_t point_capacity) {
    size_t off[9];
    return voxel_layout(lattice_capacity_cells, point_capacity, off);
}

struct VoxelArrays {
    VoxelHeader* hdr;
    uint2* lattice;
    uint2* block_sums;
    unsigned int *key, *head, *hcnt, *vrank, *soff, *slots;
};

static VoxelArrays voxel_arrays(void* d_ws, const size_t off[9]) {
    char* ws = reinterpret_cast<char*>(d_ws);
    VoxelArrays a;
    a.hdr = reinterpret_cast<VoxelHeader*>(ws + off[0]);
    a.lattice = reinterpret_cast<uint2*>(ws + off[1]);
    a.block_sums = reinterpret_cast<uint2*>(ws + off[2]);
    a.key = reinterpret_cast<unsigned int*>(ws + off[3]);
    a.head = reinterpret_cast<unsigned int*>(ws + off[4]);
    a.hcnt = reinterpret_cast<unsigned int*>(ws + off[5]);
    a.vrank = reinterpret_cast<unsigned int*>(ws + off[6]);
    a.soff = reinterpret_cast<unsigned int*>(ws + off[7]);
    a.slots = reinterpret_cast<unsigned int*>(ws + off[8]);
    return a;
}

// mark .. reduce (7 launches) over the points `hdr` describes; `launch_points` sizes the grids.
static void launch_voxel_core(const double* px, const double* py, const VoxelHeader* hdr_c, VoxelHeader* hdr, const VoxelArrays& a,
                              int64_t launch_points, double voxel, double* out_px, double* out_py, long long* out_count,
                              unsigned long long* benc, cudaStream_t st) {
    const int gp = grid_for(launch_points);
    const int gs = grid_for((launch_points + kScanItems - 1) / kScanItems);
    k_voxel_mark<<<gp, kMT, 0, st>>>(px, py, voxel, hdr_c, a.lattice, a.key);
    k_voxel_gather<<<gp, kMT, 0, st>>>(hdr_c, a.lattice, a.key, a.head, a.hcnt);
    k_pscan_partial<<<gs, kMT, 0, st>>>(hdr_c, a.hcnt, a.block_sums);
    k_pscan_top<<<1, 1024, 0, st>>>(a.block_sums, hdr);
    k_pscan_apply<<<gs, kMT, 0, st>>>(hdr_c, a.hcnt, a.block_sums, a.vrank, a.soff);
    k_voxel_fill<<<gp, kMT, 0, st>>>(hdr_c, a.key, a.lattice, a.head, a.soff, a.slots);
    k_voxel_reduce<<<gp, kMT, 0, st>>>(px, py, hdr_c, a.hcnt, a.vrank, a.soff, a.slots, out_px, out_py, out_count, benc);
}

int mapmerge_voxel_downsample(const double* d_px, const double* d_py, const int64_t* d_count, int64_t point_capacity,
                              double voxel, const double* d_bounds, uint64_t* d_bounds_enc, int64_t lattice_capacity_cells,
                              double* d_out_px, double* d_out_py, int64_t* d_out_count, int32_t* d_status,
                              void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_px || !d_py || !d_count || (!d_bounds && !d_bounds_enc) || !d_out_px || !d_out_py || !d_out_count || !d_status || !d_ws) {
        set_last_error("mapmerge_voxel_downsample: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (!(voxel > 0.0)) { set_last_error("mapmerge_voxel_downsample: voxel %g must be > 0", voxel); return OCCGRID_E_ARG; }
    if (lattice_capacity_cells <= 0 || point_capacity <= 0) {
        set_last_error("mapmerge_voxel_downsample: capacity < 1 (lattice %lld cells, %lld points)", (long long)lattice_capacity_cells,
                       (long long)point_capacity);
        return OCCGRID_E_ARG;
    }
    size_t off[9];
    if (ws_bytes < voxel_layout(lattice_capacity_cells, point_capacity, off)) {
        set_last_error("mapmerge_voxel_downsample: workspace too small");
        return OCCGRID_E_WORKSPACE;
    }
    const VoxelArrays a = voxel_arrays(d_ws, off);
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_MERGE_VOXEL, st, 8);
    k_voxel_setup<<<1, 1, 0, st>>>(d_bounds, (unsigned long long*)d_bounds_enc, (const long long*)d_count, voxel,
                                   lattice_capacity_cells, point_capacity, a.hdr, d_status);
    launch_voxel_core(d_px, d_py, a.hdr, a.hdr, a, point_capacity, voxel, d_out_px, d_out_py, (long long*)d_out_count,
                      (unsigned long long*)d_bounds_enc, st);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// ---- incremental voxel chain: entry points --------------------------------------------------
// dims = {lattice_w, lattice_h, point_capacity, slice_capacity} (host array), the same for every
// call on one chain workspace.
struct ChainArrays {
    ChainHeader* h;
    uint2* LM;
    unsigned int *gkey, *lkey, *next, *flag, *blockcount, *bar;
    double *resx, *resy;
    int bc_stride;
    unsigned long long* slice_benc;
    int* order;
};

static size_t chain_layout(const int64_t* dims, int n_agents, ChainArrays* a, void* base) {
    const size_t cells = (size_t)dims[0] * (size_t)dims[1], points = (size_t)dims[2], sl = (size_t)dims[3] + 16;
    char* ws = reinterpret_cast<char*>(base);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t o_h = take(sizeof(ChainHeader)), o_lm = take((cells + 1) * 8), o_gk = take(points * 4);
    const size_t bc_stride = sl / kMT + 2;
    const size_t o_lk = take(sl * 4), o_nx = take(sl * 4), o_fl = take(sl * 4), o_bc = take(2 * bc_stride * 4), o_bar = take(16);
    const size_t o_rx = take(sl * 8), o_ry = take(sl * 8), o_sb = take((size_t)n_agents * 32), o_or = take((size_t)n_agents * 4);
    if (a) {
        a->h = reinterpret_cast<ChainHeader*>(ws + o_h);
        a->LM = reinterpret_cast<uint2*>(ws + o_lm);
        a->gkey = reinterpret_cast<unsigned int*>(ws + o_gk);
        a->lkey = reinterpret_cast<unsigned int*>(ws + o_lk);
        a->next = reinterpret_cast<unsigned int*>(ws + o_nx);
        a->flag = reinterpret_cast<unsigned int*>(ws + o_fl);
        a->blockcount = reinterpret_cast<unsigned int*>(ws + o_bc);
        a->bar = reinterpret_cast<unsigned int*>(ws + o_bar);
        a->bc_stride = (int)bc_stride;
        a->resx = reinterpret_cast<double*>(ws + o_rx);
        a->resy = reinterpret_cast<double*>(ws + o_ry);
        a->slice_benc = reinterpret_cast<unsigned long long*>(ws + o_sb);
        a->order = reinterpret_cast<int*>(ws + o_or);
    }
    return o;
}

static bool chain_dims_ok(const int64_t* dims, int n_agents) {
    return dims && n_agents > 0 && n_agents <= 65535 && dims[0] > 0 && dims[1] > 0 && dims[2] > 0 && dims[3] > 0 &&
           dims[0] * dims[1] < 0x7fffffffll && dims[2] < 0x7ffffff0ll && dims[3] < 0x7ffffff0ll;
}

// chain_dims_ok with a message naming what failed; false -> OCCGRID_E_ARG.
static bool chain_dims_check(const char* fn, const int64_t* dims, int n_agents) {
    if (!dims) { set_last_error("%s: NULL pointer (dims)", fn); return false; }
    if (n_agents <= 0 || n_agents > 65535) { set_last_error("%s: n_agents %d outside 1..65535", fn, n_agents); return false; }
    if (!chain_dims_ok(dims, n_agents)) {
        set_last_error("%s: dims {%lld, %lld, %lld, %lld} out of range", fn, (long long)dims[0], (long long)dims[1],
                       (long long)dims[2], (long long)dims[3]);
        return false;
    }
    return true;
}

size_t mapmerge_chain_workspace_bytes(const int64_t* dims, int n_agents) {
    if (!chain_dims_ok(dims, n_agents)) return 0;
    return chain_layout(dims, n_agents, nullptr, nullptr);
}

int mapmerge_chain_init(void* d_chain, size_t chain_bytes, const int64_t* dims, int n_agents, const double* d_sx,
                        const double* d_sy, const int64_t* d_agent_offset, const int32_t* order_host, int n_order,
                        const double* d_px, const double* d_py, const int64_t* d_count, void* stream) {
    if (!d_chain || !d_sx || !d_sy || !d_agent_offset || !order_host || !d_px || !d_py || !d_count) {
        set_last_error("mapmerge_chain_init: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (!chain_dims_check("mapmerge_chain_init", dims, n_agents)) return OCCGRID_E_ARG;
    if (n_order < 0 || n_order > n_agents) {
        set_last_error("mapmerge_chain_init: n_order %d outside 0..n_agents", n_order);
        return OCCGRID_E_ARG;
    }
    if (chain_bytes < chain_layout(dims, n_agents, nullptr, nullptr)) { set_last_error("mapmerge_chain_init: workspace too small"); return OCCGRID_E_WORKSPACE; }
    for (int i = 0; i < n_order; ++i)
        if (order_host[i] < 0 || order_host[i] >= n_agents) { set_last_error("mapmerge_chain_init: order entry out of range"); return OCCGRID_E_ARG; }
    ChainArrays c;
    chain_layout(dims, n_agents, &c, d_chain);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_order) {
        OCC_CUDA_TRY(cudaMemcpyAsync(c.order, order_host, sizeof(int) * (size_t)n_order, cudaMemcpyHostToDevice, st));
        OCC_CUDA_TRY(cudaStreamSynchronize(st));           // order_host belongs to the caller
    }
    ProfileScope ps(K_CHAIN_PROBE, st, 5);
    k_chain_reset<<<1, 1, 0, st>>>(c.h);
    k_chain_slice_bounds_init<<<(n_agents + 255) / 256, 256, 0, st>>>(c.slice_benc, n_agents);
    dim3 grid((unsigned)grid_for(dims[3]), (unsigned)n_agents);
    if (grid.x > 64) grid.x = 64;
    k_chain_slice_bounds<<<grid, kMT, 0, st>>>(d_sx, d_sy, (const long long*)d_agent_offset, c.slice_benc);
    k_chain_rebounds<<<device_sm_count() * 8, kMT, 0, st>>>(d_px, d_py, (const long long*)d_count, c.h);
    k_chain_rebounds_apply<<<1, 1, 0, st>>>(c.h);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_chain_run(void* d_chain, const int64_t* dims, int n_agents, int n_order, int n_callbacks, const double* d_sx,
                       const double* d_sy, const int64_t* d_agent_offset, double voxel, double* d_px, double* d_py,
                       int64_t capacity, int64_t* d_count, int32_t* d_status, void* stream) {
    if (!d_chain || !d_sx || !d_sy || !d_agent_offset || !d_px || !d_py || !d_count || !d_status) {
        set_last_error("mapmerge_chain_run: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (!chain_dims_check("mapmerge_chain_run", dims, n_agents)) return OCCGRID_E_ARG;
    if (n_order < 0 || n_order > n_agents) { set_last_error("mapmerge_chain_run: n_order %d outside 0..n_agents", n_order); return OCCGRID_E_ARG; }
    if (n_callbacks < 0) { set_last_error("mapmerge_chain_run: n_callbacks %d < 0", n_callbacks); return OCCGRID_E_ARG; }
    if (!(voxel > 0.0)) { set_last_error("mapmerge_chain_run: voxel %g must be > 0", voxel); return OCCGRID_E_ARG; }
    if (capacity > dims[2]) { set_last_error("mapmerge_chain_run: capacity above dims[2]"); return OCCGRID_E_ARG; }
    if (n_callbacks == 0) return OCCGRID_OK;
    ChainArrays c;
    chain_layout(dims, n_agents, &c, d_chain);
    cudaStream_t st = (cudaStream_t)stream;
    static int resident_by_device[64] = {};        // CTAs of the persistent kernel each device can hold at once
    int dev = 0;
    OCC_CUDA_TRY(cudaGetDevice(&dev));
    int resident_ctas = (dev >= 0 && dev < 64) ? resident_by_device[dev] : 0;
    if (resident_ctas == 0) {
        int sms = 0, per_sm = 0;
        OCC_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        OCC_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_chain_persistent, kMT, 0));
        if (sms <= 0 || per_sm <= 0) { set_last_error("mapmerge_chain_run: persistent kernel does not fit the device"); return OCCGRID_E_CUDA; }
        resident_ctas = sms * per_sm;
        if (dev >= 0 && dev < 64) resident_by_device[dev] = resident_ctas;
    }
    int grid = grid_for(dims[3]);
    if (grid > resident_ctas) grid = resident_ctas;
    ChainRun r;
    r.h = c.h; r.order = c.order; r.n_order = n_order; r.n_callbacks = n_callbacks;
    r.agent_offset = (const long long*)d_agent_offset; r.slice_benc = c.slice_benc;
    r.sx = d_sx; r.sy = d_sy; r.voxel = voxel; r.W = dims[0]; r.H = dims[1];
    r.LM = c.LM; r.lkey = c.lkey; r.next = c.next; r.gkey = c.gkey; r.flag = c.flag; r.blockcount = c.blockcount;
    r.gx = d_px; r.gy = d_py; r.resx = c.resx; r.resy = c.resy;
    r.d_count = (long long*)d_count; r.capacity = capacity; r.status = d_status; r.bar = c.bar; r.bc_stride = c.bc_stride;
    void* args[] = {&r};
    ProfileScope ps(K_CHAIN_INCR, st, 1);
    OCC_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_chain_persistent, dim3((unsigned)grid), dim3(kMT), args, 0, st));
    return OCCGRID_OK;
}

// Synchronises the stream; state_out = {cursor, stalled}.
int mapmerge_chain_poll(void* d_chain, const int64_t* dims, int n_agents, int32_t* state_out, void* stream) {
    if (!d_chain || !state_out) { set_last_error("mapmerge_chain_poll: NULL pointer"); return OCCGRID_E_ARG; }
    if (!chain_dims_check("mapmerge_chain_poll", dims, n_agents)) return OCCGRID_E_ARG;
    ChainArrays c;
    chain_layout(dims, n_agents, &c, d_chain);
    cudaStream_t st = (cudaStream_t)stream;
    int two[2] = {0, 0};
    static_assert(offsetof(ChainHeader, cursor) == offsetof(ChainHeader, stalled) + sizeof(int), "stalled and cursor are read as one pair");
    OCC_CUDA_TRY(cudaMemcpyAsync(two, &c.h->stalled, sizeof(two), cudaMemcpyDeviceToHost, st));
    OCC_CUDA_TRY(cudaStreamSynchronize(st));
    state_out[0] = two[1];
    state_out[1] = two[0];
    return OCCGRID_OK;
}

int mapmerge_chain_rebounds(void* d_chain, const int64_t* dims, int n_agents, const double* d_px, const double* d_py,
                            const int64_t* d_count, void* stream) {
    if (!d_chain || !d_px || !d_py || !d_count) { set_last_error("mapmerge_chain_rebounds: NULL pointer"); return OCCGRID_E_ARG; }
    if (!chain_dims_check("mapmerge_chain_rebounds", dims, n_agents)) return OCCGRID_E_ARG;
    ChainArrays c;
    chain_layout(dims, n_agents, &c, d_chain);
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_CHAIN_PROBE, st, 2);
    k_chain_rebounds<<<device_sm_count() * 8, kMT, 0, st>>>(d_px, d_py, (const long long*)d_count, c.h);
    k_chain_rebounds_apply<<<1, 1, 0, st>>>(c.h);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_chain_rebuild(void* d_chain, const int64_t* dims, int n_agents, const double* d_sx, const double* d_sy,
                           const int64_t* d_agent_offset, int agent, double voxel, double* d_px, double* d_py, int64_t capacity,
                           int64_t* d_count, double* d_out_px, double* d_out_py, int64_t* d_out_count, int32_t* d_status,
                           void* d_voxel_ws, size_t voxel_ws_bytes, int64_t lattice_capacity_cells, void* stream) {
    if (!d_chain || !d_sx || !d_sy || !d_agent_offset || !d_px || !d_py || !d_count || !d_out_px || !d_out_py || !d_out_count ||
        !d_status) {
        set_last_error("mapmerge_chain_rebuild: NULL pointer");
        return OCCGRID_E_ARG;
    }
    if (!chain_dims_check("mapmerge_chain_rebuild", dims, n_agents)) return OCCGRID_E_ARG;
    if (agent < 0 || agent >= n_agents) { set_last_error("mapmerge_chain_rebuild: agent %d outside 0..n_agents-1", agent); return OCCGRID_E_ARG; }
    if (!(voxel > 0.0)) { set_last_error("mapmerge_chain_rebuild: voxel %g must be > 0", voxel); return OCCGRID_E_ARG; }
    if (capacity > dims[2]) { set_last_error("mapmerge_chain_rebuild: capacity above dims[2]"); return OCCGRID_E_ARG; }
    size_t off[9];
    if (!d_voxel_ws || lattice_capacity_cells < dims[0] * dims[1] || voxel_ws_bytes < voxel_layout(lattice_capacity_cells, dims[2], off)) {
        set_last_error("mapmerge_chain_rebuild: voxel workspace too small");
        return OCCGRID_E_WORKSPACE;
    }
    const VoxelArrays va = voxel_arrays(d_voxel_ws, off);
    ChainArrays c;
    chain_layout(dims, n_agents, &c, d_chain);
    cudaStream_t st = (cudaStream_t)stream;
    const int gp = grid_for(capacity);
    ProfileScope ps(K_CHAIN_REBUILD, st, 13);
    k_chain_lm_clear<<<gp, kMT, 0, st>>>(c.h, c.LM, c.gkey, (const long long*)d_count);
    k_append_slice<<<device_sm_count(), kMT, 0, st>>>(d_sx, d_sy, (const long long*)d_agent_offset, agent, d_px, d_py, capacity, (long long*)d_count,
                                         d_status, nullptr);
    k_bump_count<<<1, 1, 0, st>>>((const long long*)d_agent_offset, agent, capacity, (long long*)d_count);
    k_chain_rebuild_hdr<<<1, 1, 0, st>>>(c.h, c.slice_benc, agent, (const long long*)d_count, voxel, dims[0], dims[1], dims[2], d_status);
    launch_voxel_core(d_px, d_py, &c.h->v, &c.h->v, va, capacity, voxel, d_out_px, d_out_py, (long long*)d_out_count, c.h->gb_enc, st);
    k_chain_lm_build<<<gp, kMT, 0, st>>>(c.h, d_out_px, d_out_py, (const long long*)d_out_count, voxel, c.LM, c.gkey);
    k_chain_rebuild_done<<<1, 1, 0, st>>>(c.h);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_rasterise(const double* d_px, const double* d_py, const int64_t* d_count, double res, const double* d_bounds,
                       int32_t width, int32_t height, int8_t* d_grid_out, void* stream) {
    if (!d_px || !d_py || !d_count || !d_bounds || !d_grid_out) { set_last_error("mapmerge_rasterise: NULL pointer"); return OCCGRID_E_ARG; }
    if (width <= 0 || height <= 0) {
        set_last_error("mapmerge_rasterise: width x height %d x %d", (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    if (!(res > 0.0)) { set_last_error("mapmerge_rasterise: res %g must be > 0", res); return OCCGRID_E_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    const long long n = (long long)width * height;
    ProfileScope ps(K_MERGE_RASTER, st, 2);
    k_raster_fill<<<grid_for(n / 16 + 1), kMT, 0, st>>>(d_grid_out, n);
    k_raster_scatter<<<device_sm_count() * 8, kMT, 0, st>>>(d_px, d_py, (const long long*)d_count, d_bounds, res, width, height, d_grid_out);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int mapmerge_fuse_max(int8_t* d_dst, const int8_t* d_src, int64_t n, void* stream) {
    if (!d_dst || !d_src) { set_last_error("mapmerge_fuse_max: NULL pointer"); return OCCGRID_E_ARG; }
    if (n < 0) { set_last_error("mapmerge_fuse_max: n %lld < 0", (long long)n); return OCCGRID_E_ARG; }
    if (n == 0) return OCCGRID_OK;
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_MERGE_FUSE, st);
    k_fuse_max<<<grid_for(n), kMT, 0, st>>>(d_dst, d_src, n);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
