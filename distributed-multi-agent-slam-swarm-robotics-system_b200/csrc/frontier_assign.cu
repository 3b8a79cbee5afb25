// Frontier assignment (occgrid_frontier_assign / occgrid_geodesic_field in include/occgrid_b200.h):
// geodesic distances from every robot over the known free space of a grid, the cost of every
// frontier cluster per robot and one cluster per robot by a greedy pass.  EXTENSION: the reference
// computes clusters but its assignment is commented out (dual_bot_mapper.py:958-996).
//
// Distances (DESIGN §6e).  D_a is the 4-connected unit-cost BFS distance from robot a's cell; the
// source gets 0 whatever its value and the search moves only into FREE cells.  D_a is the unique
// fixed point of D(c) = min(seed(c), FREE(c) ? min over 4-neighbours n of D(n) + 1 : inf), so any
// relaxation order that only lowers values gives the same field bit for bit.
//
// Fields are tile-sparse: per (robot, 64 x 64 tile) one 16 KB slot of a pool, handed out from a
// device counter when the robot first reaches the tile; slot[a][tile] = -1 reads as unreachable.
// A label-correcting worklist of (robot, tile) items runs in ONE cooperative kernel, in rounds
// separated by grid_barrier.  An item recomputes its tile from the robot seed and the halo (the
// neighbouring tiles' border values + 1) with a bit-parallel BFS on one warp: 64 rows of 64 bits,
// two rows per lane, dilation by shifts and shuffles, halo seeds joining at their own level.  The
// per-cell levels stay in shared memory and the tile is written once.  Where one of its border
// values dropped, the item enqueues the neighbour behind that border for the next round.  The
// halo only ever decreases, so every recomputation is <= the previous one and the rounds stop at
// the fixed point whatever the order in which items run or read each other's borders.
#include <cmath>

#include "common.cuh"

namespace occ {

constexpr int kGT = 64;                       // tile side; one uint64 per tile row
constexpr int kGCells = kGT * kGT;
constexpr int kGWarps = 4;                    // items in flight per CTA (one per warp)
constexpr int kGThreads = kGWarps * 32;
constexpr int kGInf = 0x7fffffff;             // unreachable inside the pool
constexpr int kGMaxRobots = 65535;

// Control words of one call (zeroed by the host before the seed kernel).
struct GeoCtl {
    unsigned int qcount[2];                   // items queued for the even / odd rounds
    unsigned int alloc;                       // pool slots handed out (may pass the capacity on overflow)
    int abort;                                // grid_barrier's give-up flag
    unsigned int bar[4];                      // grid_barrier words
    unsigned int rounds;
    int overflow;                             // pool or worklist full: the result is incomplete
    unsigned long long items;                 // (robot, tile) items processed
};

struct GeoArgs {
    const unsigned long long* fmask;          // [height][tiles_x]: bit x of word (y, tx) = cell (64 tx + x, y) is FREE
    int width, height, tiles_x, tiles_y, n_tiles;
    int* src;                                 // [A] robot cell y * width + x, or -1
    int* slot;                                // [A][n_tiles] pool slot, -1 = not reached
    int* mark;                                // [A][n_tiles] last round the item was queued for
    unsigned long long* queue0;               // (robot << 32 | tile) items of the even rounds
    unsigned long long* queue1;               // and of the odd rounds
    unsigned int qcap;
    int* pool;                                // [pool_cap][64][64] distances, kGInf = unreachable
    unsigned int pool_cap;
    GeoCtl* ctl;
    int* status;
};

__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ unsigned long long* geo_queue(const GeoArgs& g, int round) { return (round & 1) ? g.queue1 : g.queue0; }

__device__ __forceinline__ void geo_overflow(const GeoArgs& g) {
    atomicExch(&g.ctl->overflow, 1);
    atomicOr(g.status, OCCGRID_ASSIGN_POOL_FULL);
}

__device__ void geo_enqueue(const GeoArgs& g, int a, int t, int round) {
    if (atomicExch(g.mark + (size_t)a * g.n_tiles + t, round) == round) return;      // already queued for that round
    const unsigned int pos = atomicAdd(&g.ctl->qcount[round & 1], 1u);
    if (pos >= g.qcap) { geo_overflow(g); return; }
    geo_queue(g, round)[pos] = ((unsigned long long)a << 32) | (unsigned int)t;
}

// Free bits of every (row, tile column) word: lane l reads columns l and l + 32, two ballots.
__global__ void __launch_bounds__(256)
k_geo_fmask(const int8_t* __restrict__ grid, int width, int height, int tiles_x, unsigned long long* __restrict__ fmask) {
    const int lane = threadIdx.x & 31;
    const long long n_words = (long long)height * tiles_x;
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words;
         w += ((long long)gridDim.x * blockDim.x) >> 5) {
        const long long y = w / tiles_x;
        const int x0 = (int)(w - y * tiles_x) * kGT;
        const int8_t* row = grid + y * width;
        const bool f0 = x0 + lane < width && row[x0 + lane] == OCCGRID_CELL_FREE;
        const bool f1 = x0 + lane + 32 < width && row[x0 + lane + 32] == OCCGRID_CELL_FREE;
        const unsigned int lo = __ballot_sync(0xffffffffu, f0), hi = __ballot_sync(0xffffffffu, f1);
        if (lane == 0) fmask[w] = ((unsigned long long)hi << 32) | lo;
    }
}

// Robot cells (world_to_grid: int((w - o) / res), truncation, fp64 division) and the first items.
__global__ void k_geo_seed(GeoArgs g, const double* __restrict__ robot_xy, int n_robots, double ox, double oy, double res) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_robots) return;
    const double qx = (robot_xy[2 * a] - ox) / res, qy = (robot_xy[2 * a + 1] - oy) / res;
    int cell = -1;
    // int() truncates toward zero, so the cell is inside iff -1 < q < size (false for NaN and inf)
    if (qx > -1.0 && qx < (double)g.width && qy > -1.0 && qy < (double)g.height) {
        const int x = (int)qx, y = (int)qy;
        cell = y * g.width + x;
        geo_enqueue(g, a, (y / kGT) * g.tiles_x + x / kGT, 0);
    }
    g.src[a] = cell;
}

// One (robot, tile) item on one warp.  Lane l owns tile rows 2l and 2l + 1.
__device__ void geo_item(const GeoArgs& g, int a, int t, int round, int* __restrict__ lev) {
    const int lane = threadIdx.x & 31;
    const int r0 = 2 * lane, r1 = 2 * lane + 1;
    const int ty = t / g.tiles_x, tx = t - ty * g.tiles_x;
    const int x0 = tx * kGT, y0 = ty * kGT;
    int* slot_row = g.slot + (size_t)a * g.n_tiles;
    int s = __ldcg(slot_row + t);                 // only this item writes slot_row[t] in this round
    const bool fresh = s < 0;
    if (fresh) {
        if (lane == 0) s = (int)atomicAdd(&g.ctl->alloc, 1u);
        s = __shfl_sync(0xffffffffu, s, 0);
        if ((unsigned int)s >= g.pool_cap) {
            if (lane == 0) geo_overflow(g);
            return;
        }
    }
    const unsigned long long F0 = y0 + r0 < g.height ? __ldg(g.fmask + (size_t)(y0 + r0) * g.tiles_x + tx) : 0ull;
    const unsigned long long F1 = y0 + r1 < g.height ? __ldg(g.fmask + (size_t)(y0 + r1) * g.tiles_x + tx) : 0ull;

    // the robot seed
    const int sc = __ldg(g.src + a);
    int src_row = -1;
    unsigned long long src_bit = 0;
    if (sc >= 0) {
        const int sy = sc / g.width, sx = sc - sy * g.width;
        if (sy - y0 >= 0 && sy - y0 < kGT && sx - x0 >= 0 && sx - x0 < kGT) { src_row = sy - y0; src_bit = 1ull << (sx - x0); }
    }

    // halo seeds: top / bottom at columns lane and lane + 32, left / right at the lane's rows
    auto plus1 = [](int v) { return v == kGInf ? kGInf : v + 1; };
    int sT0 = kGInf, sT1 = kGInf, sB0 = kGInf, sB1 = kGInf, sL0 = kGInf, sL1 = kGInf, sR0 = kGInf, sR1 = kGInf;
    if (ty > 0) {
        const int sn = __ldcg(slot_row + t - g.tiles_x);
        if (sn >= 0) {
            const int* p = g.pool + (size_t)sn * kGCells + (kGT - 1) * kGT;
            sT0 = plus1(__ldcg(p + lane)); sT1 = plus1(__ldcg(p + lane + 32));
        }
    }
    if (ty < g.tiles_y - 1) {
        const int sn = __ldcg(slot_row + t + g.tiles_x);
        if (sn >= 0) {
            const int* p = g.pool + (size_t)sn * kGCells;
            sB0 = plus1(__ldcg(p + lane)); sB1 = plus1(__ldcg(p + lane + 32));
        }
    }
    if (tx > 0) {
        const int sn = __ldcg(slot_row + t - 1);
        if (sn >= 0) {
            const int* p = g.pool + (size_t)sn * kGCells + kGT - 1;
            sL0 = plus1(__ldcg(p + r0 * kGT)); sL1 = plus1(__ldcg(p + r1 * kGT));
        }
    }
    if (tx < g.tiles_x - 1) {
        const int sn = __ldcg(slot_row + t + 1);
        if (sn >= 0) {
            const int* p = g.pool + (size_t)sn * kGCells;
            sR0 = plus1(__ldcg(p + r0 * kGT)); sR1 = plus1(__ldcg(p + r1 * kGT));
        }
    }
    // this tile's previous border, to find the borders that drop
    int oT0 = kGInf, oT1 = kGInf, oB0 = kGInf, oB1 = kGInf, oL0 = kGInf, oL1 = kGInf, oR0 = kGInf, oR1 = kGInf;
    int* dst = g.pool + (size_t)s * kGCells;
    if (!fresh) {
        oT0 = __ldcg(dst + lane); oT1 = __ldcg(dst + lane + 32);
        oB0 = __ldcg(dst + (kGT - 1) * kGT + lane); oB1 = __ldcg(dst + (kGT - 1) * kGT + lane + 32);
        oL0 = __ldcg(dst + r0 * kGT); oL1 = __ldcg(dst + r1 * kGT);
        oR0 = __ldcg(dst + r0 * kGT + kGT - 1); oR1 = __ldcg(dst + r1 * kGT + kGT - 1);
    }

    // level-synchronous BFS; a halo seed joins when the level reaches its value
    unsigned long long V0 = 0, V1 = 0, Fr0 = 0, Fr1 = 0;
    int L = warp_min(min(min(min(sT0, sT1), min(sB0, sB1)), min(min(sL0, sL1), min(sR0, sR1))));
    if (__any_sync(0xffffffffu, src_row >= 0)) L = 0;
    __syncwarp();                                 // the previous item's reads of lev are done
    while (L != kGInf) {
        unsigned long long add0 = (sL0 == L ? 1ull : 0ull) | (sR0 == L ? 1ull << 63 : 0ull);
        unsigned long long add1 = (sL1 == L ? 1ull : 0ull) | (sR1 == L ? 1ull << 63 : 0ull);
        const unsigned int tlo = __ballot_sync(0xffffffffu, sT0 == L), thi = __ballot_sync(0xffffffffu, sT1 == L);
        const unsigned int blo = __ballot_sync(0xffffffffu, sB0 == L), bhi = __ballot_sync(0xffffffffu, sB1 == L);
        if (lane == 0) add0 |= ((unsigned long long)thi << 32) | tlo;
        if (lane == 31) add1 |= ((unsigned long long)bhi << 32) | blo;
        unsigned long long up = __shfl_up_sync(0xffffffffu, Fr1, 1), dn = __shfl_down_sync(0xffffffffu, Fr0, 1);
        if (lane == 0) up = 0;
        if (lane == 31) dn = 0;
        unsigned long long n0 = ((Fr0 << 1) | (Fr0 >> 1) | up | Fr1 | add0) & F0 & ~V0;
        unsigned long long n1 = ((Fr1 << 1) | (Fr1 >> 1) | Fr0 | dn | add1) & F1 & ~V1;
        if (L == 0) {                             // the source is settled whatever its value
            if (src_row == r0) n0 |= src_bit;
            if (src_row == r1) n1 |= src_bit;
        }
        V0 |= n0; V1 |= n1; Fr0 = n0; Fr1 = n1;
        for (unsigned long long m = n0; m; m &= m - 1) lev[r0 * kGT + __ffsll((long long)m) - 1] = L;
        for (unsigned long long m = n1; m; m &= m - 1) lev[r1 * kGT + __ffsll((long long)m) - 1] = L;
        if (__any_sync(0xffffffffu, (n0 | n1) != 0ull)) {
            ++L;
        } else {                                  // the wave died out: jump to the next halo seed, if any
            auto above = [L](int v) { return v > L ? v : kGInf; };
            L = warp_min(min(min(min(above(sT0), above(sT1)), min(above(sB0), above(sB1))),
                             min(min(above(sL0), above(sL1)), min(above(sR0), above(sR1)))));
        }
    }
    __syncwarp();

    // write the tile once, row by row (coalesced); keep the new border
    int nT0 = kGInf, nT1 = kGInf, nB0 = kGInf, nB1 = kGInf;
    for (int y = 0; y < kGT; ++y) {
        const unsigned long long vr = __shfl_sync(0xffffffffu, (y & 1) ? V1 : V0, y >> 1);
        const int v0 = ((vr >> lane) & 1ull) ? lev[y * kGT + lane] : kGInf;
        const int v1 = ((vr >> (lane + 32)) & 1ull) ? lev[y * kGT + lane + 32] : kGInf;
        __stcg(dst + y * kGT + lane, v0);
        __stcg(dst + y * kGT + lane + 32, v1);
        if (y == 0) { nT0 = v0; nT1 = v1; }
        if (y == kGT - 1) { nB0 = v0; nB1 = v1; }
    }
    const int nL0 = (V0 & 1ull) ? lev[r0 * kGT] : kGInf, nL1 = (V1 & 1ull) ? lev[r1 * kGT] : kGInf;
    const int nR0 = (V0 >> 63) ? lev[r0 * kGT + kGT - 1] : kGInf, nR1 = (V1 >> 63) ? lev[r1 * kGT + kGT - 1] : kGInf;
    const bool dT = __any_sync(0xffffffffu, nT0 < oT0 || nT1 < oT1);
    const bool dB = __any_sync(0xffffffffu, nB0 < oB0 || nB1 < oB1);
    const bool dL = __any_sync(0xffffffffu, nL0 < oL0 || nL1 < oL1);
    const bool dR = __any_sync(0xffffffffu, nR0 < oR0 || nR1 < oR1);
    __threadfence();
    __syncwarp();
    if (lane == 0) {
        if (fresh) atomicExch(slot_row + t, s);   // published after the values: a reader never sees an unwritten slot
        if (dT && ty > 0) geo_enqueue(g, a, t - g.tiles_x, round + 1);
        if (dB && ty < g.tiles_y - 1) geo_enqueue(g, a, t + g.tiles_x, round + 1);
        if (dL && tx > 0) geo_enqueue(g, a, t - 1, round + 1);
        if (dR && tx < g.tiles_x - 1) geo_enqueue(g, a, t + 1, round + 1);
        atomicAdd(&g.ctl->items, 1ull);
    }
}

// The worklist: all rounds in one cooperative launch.  The last arriver of each barrier resets the
// count of the round just drained and decides, once for everybody, whether another round runs.
__global__ void __launch_bounds__(kGThreads)
k_geo_rounds(GeoArgs g) {
    extern __shared__ int s_lev[];                // [kGWarps][64 * 64]
    const int warp = threadIdx.x >> 5;
    int* lev = s_lev + warp * kGCells;
    const unsigned int gw = blockIdx.x * kGWarps + warp, nw = gridDim.x * kGWarps;
    unsigned int target = 0;
    for (int round = 0;; ++round) {
        const unsigned int n = min(reinterpret_cast<volatile unsigned int*>(g.ctl->qcount)[round & 1], g.qcap);
        for (unsigned int i = gw; i < n; i += nw) {
            const unsigned long long it = __ldcg(geo_queue(g, round) + i);
            geo_item(g, (int)(it >> 32), (int)(unsigned int)it, round, lev);
        }
        int more = 0;
        const bool ok = grid_barrier(g.ctl->bar, target, &g.ctl->abort, &more, [&] {
            volatile GeoCtl* c = g.ctl;
            const unsigned int next = c->qcount[(round + 1) & 1];
            c->qcount[round & 1] = 0;
            c->rounds = (unsigned int)round + 1;
            return next > 0 && c->overflow == 0 ? 1 : 0;
        });
        if (!ok) {
            if (threadIdx.x == 0) atomicOr(g.status, OCCGRID_ASSIGN_TIMEOUT);
            return;
        }
        if (!more) return;
    }
}

__device__ __forceinline__ bool geo_failed(const GeoCtl* c) {
    return *reinterpret_cast<const volatile int*>(&c->overflow) != 0 || *reinterpret_cast<const volatile int*>(&c->abort) != 0;
}

// D_a of cell (x, y) through the slot table, kGInf when unreached.
__device__ __forceinline__ int geo_dist(const GeoArgs& g, int a, int x, int y) {
    const int s = g.slot[(size_t)a * g.n_tiles + (y / kGT) * g.tiles_x + x / kGT];
    return s < 0 ? kGInf : g.pool[(size_t)s * kGCells + (y % kGT) * kGT + x % kGT];
}

__global__ void __launch_bounds__(256)
k_geo_best_init(unsigned long long* __restrict__ best, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) best[i] = ~0ull;
}

// best[a][k] = min over the cells of cluster k of (D_a << 32 | y * width + x).  Cluster k of a
// frontier cell: its label is the root's list index, found in the ascending cluster_root list.
__global__ void __launch_bounds__(256)
k_geo_cost(GeoArgs g, int n_robots, const int2* __restrict__ xy, const long long* __restrict__ d_count,
           const int* __restrict__ label, const int* __restrict__ cluster_root, const long long* __restrict__ d_n_clusters,
           int max_clusters, unsigned long long* __restrict__ best) {
    if (geo_failed(g.ctl)) return;
    const long long n = *d_count;
    const int K = (int)min(*d_n_clusters, (long long)max_clusters);
    if (n <= 0 || K <= 0) return;
    const long long pairs = n * n_robots;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(p / n);
        const long long i = p - (long long)a * n;
        const int root = label[i];
        int lo = 0, hi = K;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (cluster_root[mid] < root) lo = mid + 1; else hi = mid;
        }
        if (lo == K || cluster_root[lo] != root) continue;            // a dropped (small) cluster
        const int2 c = xy[i];
        const int d = geo_dist(g, a, c.x, c.y);
        if (d == kGInf) continue;
        const unsigned long long key = ((unsigned long long)d << 32) | (unsigned int)(c.y * g.width + c.x);
        atomicMin(best + (size_t)a * max_clusters + lo, key);
    }
}

// One CTA: robot after robot, the unclaimed cluster of least (cost, k).
__global__ void __launch_bounds__(1024)
k_geo_assign(const GeoCtl* __restrict__ ctl, int* __restrict__ status, int n_robots, int width,
             const unsigned long long* __restrict__ best, int max_clusters, const long long* __restrict__ d_n_clusters,
             const double* __restrict__ centroids, unsigned int* __restrict__ claimed, int* __restrict__ cluster,
             int* __restrict__ cost, int* __restrict__ goal, double* __restrict__ target, int* __restrict__ costs) {
    __shared__ unsigned long long s_min[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long ncl = *d_n_clusters;
    int K = (int)min(ncl, (long long)max_clusters);
    if (ncl > max_clusters) {
        if (threadIdx.x == 0) atomicOr(status, OCCGRID_ASSIGN_CLUSTERS_FULL);
        K = 0;
    }
    if (geo_failed(ctl)) K = 0;
    for (int w = threadIdx.x; w < (K + 31) / 32; w += blockDim.x) claimed[w] = 0u;
    __syncthreads();
    for (int a = 0; a < n_robots; ++a) {
        unsigned long long m = ~0ull;
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            const unsigned long long b = best[(size_t)a * max_clusters + k];
            const int c = b == ~0ull ? -1 : (int)(b >> 32);
            costs[(size_t)a * max_clusters + k] = c;
            if (c >= 0 && !((claimed[k >> 5] >> (k & 31)) & 1u)) m = min(m, ((unsigned long long)c << 32) | (unsigned int)k);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) s_min[warp] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = min(m, s_min[w]);
            if (m == ~0ull) {
                cluster[a] = -1; cost[a] = -1; goal[2 * a] = -1; goal[2 * a + 1] = -1;
                target[2 * a] = NAN; target[2 * a + 1] = NAN;
            } else {
                const int k = (int)(unsigned int)m;
                const unsigned int lin = (unsigned int)best[(size_t)a * max_clusters + k];
                claimed[k >> 5] |= 1u << (k & 31);
                cluster[a] = k; cost[a] = (int)(m >> 32);
                goal[2 * a] = (int)(lin % (unsigned int)width); goal[2 * a + 1] = (int)(lin / (unsigned int)width);
                target[2 * a] = centroids[2 * k]; target[2 * a + 1] = centroids[2 * k + 1];
            }
        }
        __syncthreads();
    }
}

// One robot's dense field: -1 where unreached.  Nothing is written when the worklist failed.
__global__ void __launch_bounds__(256)
k_geo_expand(GeoArgs g, int* __restrict__ field) {
    if (geo_failed(g.ctl)) return;
    const long long n = (long long)g.width * g.height;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(c / g.width), x = (int)(c - (long long)y * g.width);
        const int d = geo_dist(g, 0, x, y);
        field[c] = d == kGInf ? -1 : d;
    }
}

__global__ void k_geo_stats(const GeoCtl* __restrict__ ctl, unsigned int pool_cap, long long* __restrict__ stats) {
    stats[0] = ctl->rounds;
    stats[1] = (long long)ctl->items;
    stats[2] = min(ctl->alloc, pool_cap);
}

// Workspace layout of one call; every offset is 256-aligned.  false (and the message key word
// "overflows size_t") when a size does not fit.
struct GeoLayout {
    size_t ctl, src, slot, mark, queue0, queue1, fmask, best, claimed, pool, total;
    int tiles_x, tiles_y, n_tiles;
};

static bool geo_add(size_t& off, size_t& field, size_t count, size_t elem) {
    if (count != 0 && elem > SIZE_MAX / count) return false;
    const size_t bytes = count * elem;
    if (bytes > SIZE_MAX - 512 - off) return false;
    field = off;
    off = align_up(off + bytes, 256);
    return true;
}

static bool geo_layout(int32_t width, int32_t height, int32_t n_robots, int32_t max_clusters, int64_t tile_pool, GeoLayout& L) {
    L.tiles_x = (width + kGT - 1) / kGT;
    L.tiles_y = (height + kGT - 1) / kGT;
    L.n_tiles = L.tiles_x * L.tiles_y;
    size_t off = 0;
    return geo_add(off, L.ctl, 1, sizeof(GeoCtl)) && geo_add(off, L.src, (size_t)n_robots, 4) &&
           geo_add(off, L.slot, (size_t)n_robots * (size_t)L.n_tiles, 4) && geo_add(off, L.mark, (size_t)n_robots * (size_t)L.n_tiles, 4) &&
           geo_add(off, L.queue0, (size_t)tile_pool, 8) && geo_add(off, L.queue1, (size_t)tile_pool, 8) &&
           geo_add(off, L.fmask, (size_t)height * (size_t)L.tiles_x, 8) && geo_add(off, L.best, (size_t)n_robots * (size_t)max_clusters, 8) &&
           geo_add(off, L.claimed, ((size_t)max_clusters + 31) / 32, 4) && geo_add(off, L.pool, (size_t)tile_pool, (size_t)kGCells * 4) &&
           ((L.total = off), true);
}

// The argument checks shared by the workspace query and both entry points; 0 or OCCGRID_E_ARG.
static int geo_check(const char* who, int32_t width, int32_t height, int32_t n_robots, int32_t max_clusters, int64_t tile_pool, GeoLayout& L) {
    if (n_robots < 1 || n_robots > kGMaxRobots) {
        set_last_error("%s: n_robots %d outside 1..%d", who, (int)n_robots, kGMaxRobots);
        return OCCGRID_E_ARG;
    }
    if (width < 3 || height < 3 || (long long)width * height > 0x7ffffffeLL) {
        set_last_error("%s: width x height %d x %d: each must be >= 3 and the grid below 2^31 - 1 cells", who, (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    if (max_clusters < 1 || tile_pool < 1 || tile_pool > 0x7fffffffLL) {
        set_last_error("%s: capacity out of range (max_clusters %d, tile_pool %lld; 1..2^31 - 1)", who, (int)max_clusters, (long long)tile_pool);
        return OCCGRID_E_ARG;
    }
    if (!geo_layout(width, height, n_robots, max_clusters, tile_pool, L)) {
        set_last_error("%s: the workspace (slot table of %d robots x %d x %d cells, pool of %lld tiles) overflows size_t",
                       who, (int)n_robots, (int)width, (int)height, (long long)tile_pool);
        return OCCGRID_E_ARG;
    }
    return OCCGRID_OK;
}

static bool geo_res_ok(double res) { return std::isfinite(res) && res > 0.0; }

// Memsets, the mask and seed kernels and the cooperative worklist: 3 kernels.
static int geo_run(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy, double res,
                   const double* d_robot_xy, int32_t n_robots, int64_t tile_pool, int32_t* d_status,
                   const GeoLayout& L, char* ws, GeoArgs& g, cudaStream_t st) {
    g.width = width; g.height = height; g.tiles_x = L.tiles_x; g.tiles_y = L.tiles_y; g.n_tiles = L.n_tiles;
    g.fmask = reinterpret_cast<unsigned long long*>(ws + L.fmask);
    g.src = reinterpret_cast<int*>(ws + L.src);
    g.slot = reinterpret_cast<int*>(ws + L.slot);
    g.mark = reinterpret_cast<int*>(ws + L.mark);
    g.queue0 = reinterpret_cast<unsigned long long*>(ws + L.queue0);
    g.queue1 = reinterpret_cast<unsigned long long*>(ws + L.queue1);
    g.qcap = (unsigned int)tile_pool;
    g.pool = reinterpret_cast<int*>(ws + L.pool);
    g.pool_cap = (unsigned int)tile_pool;
    g.ctl = reinterpret_cast<GeoCtl*>(ws + L.ctl);
    g.status = d_status;
    OCC_CUDA_TRY(cudaMemsetAsync(ws + L.ctl, 0, sizeof(GeoCtl), st));
    OCC_CUDA_TRY(cudaMemsetAsync(ws + L.slot, 0xff, L.queue0 - L.slot, st));              // slot and mark tables: -1
    const long long words = (long long)height * L.tiles_x;
    const long long fb = (words * 32 + 255) / 256;
    k_geo_fmask<<<(unsigned int)min(fb, (long long)device_sm_count() * 32), 256, 0, st>>>(
        d_grid, width, height, L.tiles_x, const_cast<unsigned long long*>(g.fmask));
    k_geo_seed<<<(n_robots + 127) / 128, 128, 0, st>>>(g, d_robot_xy, n_robots, ox, oy, res);

    const size_t smem = (size_t)kGWarps * kGCells * sizeof(int);
    static int resident_by_device[64] = {};
    int dev = 0;
    OCC_CUDA_TRY(cudaGetDevice(&dev));
    int resident = (dev >= 0 && dev < 64) ? resident_by_device[dev] : 0;
    if (resident == 0) {
        int sms = 0, per_sm = 0;
        OCC_CUDA_TRY(cudaFuncSetAttribute(k_geo_rounds, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OCC_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        OCC_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_geo_rounds, kGThreads, smem));
        if (sms <= 0 || per_sm <= 0) { set_last_error("occgrid_frontier_assign: the worklist kernel does not fit the device"); return OCCGRID_E_CUDA; }
        resident = sms * per_sm;
        if (dev >= 0 && dev < 64) resident_by_device[dev] = resident;
    }
    void* args[] = {&g};
    OCC_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_geo_rounds, dim3((unsigned int)resident), dim3(kGThreads), args, smem, st));
    return OCCGRID_OK;
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t occgrid_frontier_assign_workspace_bytes(int32_t width, int32_t height, int32_t n_robots, int32_t max_clusters, int64_t tile_pool) {
    GeoLayout L;
    if (geo_check("occgrid_frontier_assign_workspace_bytes", width, height, n_robots, max_clusters, tile_pool, L) != OCCGRID_OK) return 0;
    return L.total;
}

int occgrid_frontier_assign(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy, double res,
                            const double* d_robot_xy, int32_t n_robots, const int32_t* d_xy, const int64_t* d_count,
                            const int32_t* d_label, const int32_t* d_cluster_root, const double* d_centroids,
                            const int64_t* d_n_clusters, int32_t max_clusters, int64_t tile_pool,
                            int32_t* d_cluster, int32_t* d_cost, int32_t* d_goal, double* d_target, int32_t* d_costs,
                            int32_t* d_status, int64_t* d_stats, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grid || !d_robot_xy || !d_xy || !d_count || !d_label || !d_cluster_root || !d_centroids || !d_n_clusters ||
        !d_cluster || !d_cost || !d_goal || !d_target || !d_costs || !d_status || !d_ws) {
        set_last_error("occgrid_frontier_assign: NULL pointer");
        return OCCGRID_E_ARG;
    }
    GeoLayout L;
    const int rc = geo_check("occgrid_frontier_assign", width, height, n_robots, max_clusters, tile_pool, L);
    if (rc != OCCGRID_OK) return rc;
    if (!geo_res_ok(res)) {
        set_last_error("occgrid_frontier_assign: resolution must be finite and > 0 (got %g)", res);
        return OCCGRID_E_ARG;
    }
    if (ws_bytes < L.total) { set_last_error("occgrid_frontier_assign: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(d_ws);
    GeoArgs g;
    ProfileScope ps(K_FRONTIER_ASSIGN, st, d_stats ? 7 : 6);
    const int r = geo_run(d_grid, width, height, ox, oy, res, d_robot_xy, n_robots, tile_pool, d_status, L, ws, g, st);
    if (r != OCCGRID_OK) return r;
    unsigned long long* best = reinterpret_cast<unsigned long long*>(ws + L.best);
    const size_t n_best = (size_t)n_robots * (size_t)max_clusters;
    const int gs = device_sm_count() * 8;
    k_geo_best_init<<<(unsigned int)min((n_best + 255) / 256, (size_t)gs), 256, 0, st>>>(best, n_best);
    k_geo_cost<<<gs, 256, 0, st>>>(g, n_robots, reinterpret_cast<const int2*>(d_xy), (const long long*)d_count, d_label,
                                   d_cluster_root, (const long long*)d_n_clusters, max_clusters, best);
    k_geo_assign<<<1, 1024, 0, st>>>(g.ctl, d_status, n_robots, width, best, max_clusters, (const long long*)d_n_clusters,
                                     d_centroids, reinterpret_cast<unsigned int*>(ws + L.claimed), d_cluster, d_cost, d_goal,
                                     d_target, d_costs);
    if (d_stats) k_geo_stats<<<1, 1, 0, st>>>(g.ctl, g.pool_cap, (long long*)d_stats);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int occgrid_geodesic_field(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy, double res,
                           const double* d_robot_xy, int64_t tile_pool, int32_t* d_field, int32_t* d_status,
                           int64_t* d_stats, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grid || !d_robot_xy || !d_field || !d_status || !d_ws) {
        set_last_error("occgrid_geodesic_field: NULL pointer");
        return OCCGRID_E_ARG;
    }
    GeoLayout L;
    const int rc = geo_check("occgrid_geodesic_field", width, height, 1, 1, tile_pool, L);
    if (rc != OCCGRID_OK) return rc;
    if (!geo_res_ok(res)) {
        set_last_error("occgrid_geodesic_field: resolution must be finite and > 0 (got %g)", res);
        return OCCGRID_E_ARG;
    }
    if (ws_bytes < L.total) { set_last_error("occgrid_geodesic_field: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    GeoArgs g;
    ProfileScope ps(K_FRONTIER_ASSIGN, st, d_stats ? 5 : 4);
    const int r = geo_run(d_grid, width, height, ox, oy, res, d_robot_xy, 1, tile_pool, d_status, L, reinterpret_cast<char*>(d_ws), g, st);
    if (r != OCCGRID_OK) return r;
    const long long n = (long long)width * height;
    k_geo_expand<<<(unsigned int)min((n + 255) / 256, (long long)device_sm_count() * 16), 256, 0, st>>>(g, d_field);
    if (d_stats) k_geo_stats<<<1, 1, 0, st>>>(g.ctl, g.pool_cap, (long long*)d_stats);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
