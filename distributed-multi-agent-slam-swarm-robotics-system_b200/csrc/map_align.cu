// Correlative map alignment (mapmerge_align in include/occgrid_b200.h, DESIGN §6h): for every agent
// map, the rotation x translation in a window around its prior that best overlays the reference's
// obstacles, found exactly by a one-level branch and bound.  EXTENSION: the reference starts ICP at
// the identity and has no answer for a prior that ICP cannot recover from.
//
// Candidate (k, dx, dy) moves agent point p (its occupied cell (u, v), rotation k's coefficients) to
// reference cell (j_p + dx, i_p + dy); its score is the sum of the weights w = max_d2 + 1 - d2 (0
// where d2 < 0, d2 > max_d2 or outside the reference) over the points.  The winner is the largest
// 64-bit key score << 32 | (2^32 - 1 - rank): the largest score, ties to the lowest rank.
//
// Kernels, one stream, no host synchronisation:
//   k_align_weights, k_align_rowmax, k_align_colmax: Lw (uint8 weights) on the reference padded by
//     `pad` = 2 Rc + 64 cells on every side, and Ls[y][x] = max of Lw over [y, y + s) x [x, x + s).
//   k_align_cells<false>, k_align_scan_agents, k_align_scan_total, k_align_cells<true>: every agent's
//     occupied cells as (u, v) in row-major order, with 64-bit agent offsets.
//   k_align_score<kBound>: per (agent, rotation, s x s block of offsets at (dx0, dy0)) the bound
//     B = sum_p Ls[i_p + dy0][j_p + dx0] >= the score of every candidate in the block.
//   k_align_pick: per agent, the block with the largest bound.
//   k_align_score<kSeed>: scores exactly the prior candidate (0, 0, 0) and every candidate of the
//     picked block; their best key is the first incumbent.
//   k_align_score<kExact>: scores exactly every other block whose bound key (bound << 32 |
//     (2^32 - 1 - lowest rank in the block)) exceeds the agent's incumbent key, and raises the
//     incumbent with a 64-bit atomicMax.  A block whose bound key does not exceed the incumbent holds
//     no candidate with a larger key, so the incumbent ends as the exhaustive winner whatever the
//     order in which blocks are scored.
//   k_align_finish: the [A][6] rows and the diagnostic counts.
#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"

namespace occ {

constexpr int kAlignThreads = 256;
constexpr int kAlignChunk = 1024;            // points transformed into shared memory per round (4 per thread)
constexpr int kAlignCellsPerCta = 4096;      // cells per CTA of the compaction (16 consecutive per thread)
constexpr int kAlignTile = 16;               // bound positions per tile side: 256 per item
constexpr int kAlignMaxBlock = 64;
constexpr int kAlignDefaultBlock = 8;
constexpr int kAlignMaxCtas = 4096;          // per-CTA counter slots of each scoring kernel
constexpr int kAlignMaxAgents = 65535;
constexpr int kAlignMaxSide = 32768;
constexpr int kAlignMaxOffset = 2048;
constexpr int kAlignMaxAngles = 65535;
constexpr int kAlignMaxD2 = 254;
constexpr double kAlignFar = 1073741824.0;   // 2^30: a point at or beyond it contributes nothing
constexpr double kAlignTol = 1e-9;

static int g_align_block = 0;                // 0: kAlignDefaultBlock
static int align_block() { return g_align_block ? g_align_block : kAlignDefaultBlock; }

enum AlignMode { kBound = 0, kSeed = 1, kExact = 2 };

struct AlignArgs {
    const double* coef;                      // [A][n_angles][6]
    const long long* agent_off;              // [A + 1]
    const int2* pts;                         // (u, v)
    const uint8_t* lw;
    const uint8_t* ls;
    long long pitch;                         // padded row: ref_w + 2 pad
    int pad, wr, hr, rc, d, s, nbx, tiles_x, n_angles, n_agents;
    long long nb;                            // blocks per rotation, nbx^2
    unsigned int* bounds;                    // [A][n_angles][nb]
    unsigned long long* best;                // [A] incumbent keys
    long long* prior_score;                  // [A]
    long long* seed;                         // [A] k * nb + b of the picked block
    const int* flag;                         // nonzero: the points did not fit the workspace
    long long* cta_scored;                   // [2][kAlignMaxCtas]: candidates scored exactly, per CTA
};

// o(v) of the rank: 0, 1, -1, 2, -2, ... -> 0, 1, 2, 3, 4, ...
__host__ __device__ __forceinline__ unsigned int align_o(int v) { return v > 0 ? 2u * v - 1u : (unsigned int)(-2 * v); }

// Lowest o(v) over v in [v0, v1].
__device__ __forceinline__ unsigned int align_o_min(int v0, int v1) {
    return (v0 <= 0 && v1 >= 0) ? 0u : (v0 > 0 ? align_o(v0) : align_o(v1));
}

__device__ __forceinline__ unsigned long long align_key(unsigned int score, unsigned long long rank) {
    return ((unsigned long long)score << 32) | (0xffffffffull - rank);
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// Lw over the padded reference: weight of the reference cell (x - pad, y - pad), 0 outside it.
__global__ void __launch_bounds__(256)
k_align_weights(const int* __restrict__ d2, int wr, int hr, int pad, long long pw, long long n, int max_d2, uint8_t* __restrict__ lw) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        const long long y = c / pw;
        const int ry = (int)(y - pad), rx = (int)(c - y * pw) - pad;
        int w = 0;
        if (rx >= 0 && rx < wr && ry >= 0 && ry < hr) {
            const int v = __ldg(d2 + (size_t)ry * wr + rx);
            if (v >= 0 && v <= max_d2) w = max_d2 + 1 - v;
        }
        lw[c] = (uint8_t)w;
    }
}

// out[y][x] = max of in[y][x .. x + s) (0 past the row's end).
__global__ void __launch_bounds__(256)
k_align_rowmax(const uint8_t* __restrict__ in, long long pw, long long n, int s, uint8_t* __restrict__ out) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        const long long x = c % pw;
        const int m = (int)min((long long)s, pw - x);
        unsigned int v = 0;
        for (int b = 0; b < m; ++b) v = max(v, (unsigned int)__ldg(in + c + b));
        out[c] = (uint8_t)v;
    }
}

// out[y][x] = max of in[y .. y + s)[x] (0 past the last row).
__global__ void __launch_bounds__(256)
k_align_colmax(const uint8_t* __restrict__ in, long long pw, long long ph, long long n, int s, uint8_t* __restrict__ out) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        const long long y = c / pw;
        const int m = (int)min((long long)s, ph - y);
        unsigned int v = 0;
        for (int a = 0; a < m; ++a) v = max(v, (unsigned int)__ldg(in + c + a * pw));
        out[c] = (uint8_t)v;
    }
}

// CTA (c, a) takes cells [4096 c, 4096 (c + 1)) of agent a's map; thread t the 16 consecutive cells
// from 16 t.  kWrite = false: cnt[a][c] = its occupied cells (> 50).  kWrite = true: writes them as
// (u, v) from agent_off[a] + cnt[a][c] (scanned), in row-major order.
template <bool kWrite>
__global__ void __launch_bounds__(kAlignThreads)
k_align_cells(const int8_t* __restrict__ grids, int width, long long cells, long long cpa, unsigned int* __restrict__ cnt,
              const long long* __restrict__ agent_off, int2* __restrict__ pts, const int* __restrict__ flag) {
    __shared__ int8_t s_cells[kAlignCellsPerCta];
    __shared__ unsigned int s_warp[33];
    if (kWrite && *flag) return;
    const int a = blockIdx.y;
    const long long c = blockIdx.x, base = c * kAlignCellsPerCta;
    const int n = (int)min((long long)kAlignCellsPerCta, cells - base);
    const int8_t* g = grids + (size_t)a * (size_t)cells + (size_t)base;
    for (int i = threadIdx.x; i < n; i += kAlignThreads) s_cells[i] = __ldg(g + i);
    __syncthreads();
    const int i0 = threadIdx.x * (kAlignCellsPerCta / kAlignThreads);
    unsigned int mask = 0;
#pragma unroll
    for (int r = 0; r < kAlignCellsPerCta / kAlignThreads; ++r)
        if (i0 + r < n && s_cells[i0 + r] > 50) mask |= 1u << r;
    unsigned int total;
    const unsigned int at = block_exclusive_scan<unsigned int>(__popc(mask), s_warp, &total);
    if (!kWrite) {
        if (threadIdx.x == 0) cnt[(size_t)a * cpa + c] = total;
        return;
    }
    long long pos = agent_off[a] + (long long)cnt[(size_t)a * cpa + c] + at;
    while (mask) {
        const int r = __ffs((int)mask) - 1;
        mask &= mask - 1;
        const long long cell = base + i0 + r;
        const int v = (int)(cell / width);
        pts[pos++] = make_int2((int)(cell - (long long)v * width), v);
    }
}

// CTA a: the exclusive scan of agent a's per-CTA counts in place; its total into agent_off[a + 1].
// An agent has fewer than 2^31 cells, so 32 bits hold its offsets.
__global__ void __launch_bounds__(kAlignThreads)
k_align_scan_agents(unsigned int* cnt, long long cpa, long long* agent_off) {
    const unsigned long long total = cta_scan_in_place<4>(cnt + (size_t)blockIdx.x * cpa, (int)cpa, 0ull);
    if (threadIdx.x == 0) agent_off[blockIdx.x + 1] = (long long)total;
}

// One CTA: agent_off[a + 1] = the points of agents 0..a in 64 bits; *flag = 1 when they exceed capacity.
__global__ void __launch_bounds__(kAlignThreads)
k_align_scan_total(long long* agent_off, int n_agents, long long capacity, int* flag) {
    __shared__ unsigned long long s_warp[33];
    unsigned long long carry = 0;
    for (int b = 0; b < n_agents; b += kAlignThreads) {
        const int a = b + (int)threadIdx.x;
        const unsigned long long v = a < n_agents ? (unsigned long long)agent_off[a + 1] : 0ull;
        unsigned long long total;
        const unsigned long long x = block_exclusive_scan<unsigned long long>(v, s_warp, &total);
        if (a < n_agents) agent_off[a + 1] = (long long)(carry + x + v);
        carry += total;
    }
    if (threadIdx.x == 0) {
        agent_off[0] = 0;
        *flag = carry > (unsigned long long)capacity ? 1 : 0;
    }
}

// Sums T over agent a's points under rotation k for the positions pos0 .. pos0 + n_pos - 1 (n_pos <=
// 256) of an item whose position px + nx py is the offset (x0 + stride px, y0 + stride py).  Thread t
// takes position pos0 + t % n_pos for the points of group t / n_pos (256 / n_pos groups); threads
// t < n_pos return the sum of position pos0 + t.  Every thread of the CTA calls it.
__device__ __forceinline__ unsigned int align_sum(const AlignArgs& p, int a, int k, int x0, int y0, int stride, int nx, int pos0,
                                                  int n_pos, const uint8_t* __restrict__ T, long long* s_pt, unsigned int* s_warp,
                                                  unsigned int* s_part) {
    const int t = threadIdx.x;
    const int groups = kAlignThreads / n_pos, grp = t / n_pos;
    const int pos = pos0 + t % n_pos, py = pos / nx, px = pos - py * nx;
    const int off = py * stride * (int)p.pitch + px * stride;     // < 64 rows of at most 32 768 + 2 * 4160 cells
    const double* e = p.coef + ((size_t)a * p.n_angles + k) * 6;
    const double e0 = e[0], e1 = e[1], e2 = e[2], e3 = e[3], e4 = e[4], e5 = e[5];
    const long long beg = p.agent_off[a], end = p.agent_off[a + 1];
    const long long shift = (long long)(p.pad + y0) * p.pitch + (p.pad + x0) + off;
    constexpr int kPer = kAlignChunk / kAlignThreads;
    unsigned int acc = 0;
    for (long long c0 = beg; c0 < end; c0 += kAlignChunk) {
        long long val[kPer];
        unsigned int ok = 0;
#pragma unroll
        for (int r = 0; r < kPer; ++r) {
            val[r] = 0;
            const long long q = c0 + (long long)t * kPer + r;
            if (q < end) {
                const int2 uv = p.pts[q];
                const double u = (double)uv.x, v = (double)uv.y;
                const double X = __dadd_rn(__dmul_rn(e0, u), __dadd_rn(__dmul_rn(e1, v), e2));
                const double Y = __dadd_rn(__dmul_rn(e3, u), __dadd_rn(__dmul_rn(e4, v), e5));
                if (fabs(X) < kAlignFar && fabs(Y) < kAlignFar) {              // false for NaN
                    const int j = __double2int_rd(X), i = __double2int_rd(Y);
                    // beyond Rc cells outside the reference no candidate reaches a weight
                    if (j >= -p.rc && j < p.wr + p.rc && i >= -p.rc && i < p.hr + p.rc) {
                        val[r] = (long long)i * p.pitch + j;
                        ok |= 1u << r;
                    }
                }
            }
        }
        unsigned int n_valid;
        unsigned int w = block_exclusive_scan<unsigned int>(__popc(ok), s_warp, &n_valid);
#pragma unroll
        for (int r = 0; r < kPer; ++r)
            if (ok & (1u << r)) s_pt[w++] = val[r];
        __syncthreads();
        if (grp < groups) {
            const uint8_t* b = T + shift;
            for (unsigned int q = grp; q < n_valid; q += groups) acc += __ldg(b + s_pt[q]);
        }
        __syncthreads();
    }
    if (groups > 1) {
        s_part[t] = grp < groups ? acc : 0u;
        __syncthreads();
        if (t < n_pos) {
            acc = 0;
            for (int g = 0; g < groups; ++g) acc += s_part[g * n_pos + t];
        }
        __syncthreads();
    }
    return acc;
}

// Scores exactly the nx x ny candidates (k, x0 + px, y0 + py) and raises best[a] to the largest of
// their keys, 256 positions at a time.  Returns the number of candidates scored; the prior's score
// goes to *prior when prior != NULL (thread 0).
__device__ __forceinline__ long long align_exact(const AlignArgs& p, int a, int k, int x0, int y0, int nx, int ny,
                                                 long long* s_pt, unsigned int* s_warp, unsigned int* s_part,
                                                 unsigned long long* s_max, long long* prior) {
    const int t = threadIdx.x, n = nx * ny;
    for (int pos0 = 0; pos0 < n; pos0 += kAlignThreads) {
        const int n_pos = min(kAlignThreads, n - pos0);
        const unsigned int score = align_sum(p, a, k, x0, y0, 1, nx, pos0, n_pos, p.lw, s_pt, s_warp, s_part);
        unsigned long long m = 0;
        if (t < n_pos) {
            const int pos = pos0 + t, py = pos / nx, px = pos - py * nx;
            const unsigned long long rank = ((unsigned long long)k * p.d + align_o(y0 + py)) * p.d + align_o(x0 + px);
            m = align_key(score, rank);
        }
        if (prior && t == 0) *prior = score;
        m = warp_max_u64(m);
        if ((t & 31) == 0) s_max[t >> 5] = m;
        __syncthreads();
        if (t == 0) {
            for (int w = 1; w < kAlignThreads / 32; ++w) m = s_max[w] > m ? s_max[w] : m;
            atomicMax(p.best + a, m);
        }
        __syncthreads();
    }
    return (long long)n;
}

// kBound: items (agent, rotation, 16 x 16 tile of blocks) -> bounds.  kSeed: items 2a (the prior
// candidate) and 2a + 1 (the picked block) -> best, prior_score.  kExact: every (agent, rotation,
// block) whose bound key exceeds the incumbent; CTA x tests the items x + G (256 r + t) of round r
// together, so that the surviving blocks of one agent spread over the CTAs.
template <int kMode>
__global__ void __launch_bounds__(kAlignThreads, 3)
k_align_score(AlignArgs p, long long n_items) {
    __shared__ long long s_pt[kAlignChunk];
    __shared__ unsigned int s_warp[33];
    __shared__ unsigned int s_part[kAlignThreads];
    __shared__ unsigned long long s_max[kAlignThreads / 32];
    __shared__ long long s_items[kAlignThreads];
    __shared__ unsigned long long s_bkey[kAlignThreads];
    __shared__ unsigned long long s_wide[33];
    __shared__ int s_go;
    if (*p.flag) return;
    const int t = threadIdx.x;
    long long scored = 0;
    const long long per_agent = (long long)p.n_angles * p.nb;
    if (kMode == kBound) {
        const long long n_tiles = (long long)p.tiles_x * p.tiles_x;
        for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int a = (int)(item / ((long long)p.n_angles * n_tiles));
            if (p.agent_off[a + 1] == p.agent_off[a]) continue;
            const long long r = item - (long long)a * p.n_angles * n_tiles;
            const int k = (int)(r / n_tiles), tile = (int)(r - (long long)k * n_tiles);
            const int bx0 = (tile % p.tiles_x) * kAlignTile, by0 = (tile / p.tiles_x) * kAlignTile;
            const int nx = min(kAlignTile, p.nbx - bx0), ny = min(kAlignTile, p.nbx - by0);
            const unsigned int bound = align_sum(p, a, k, -p.rc + bx0 * p.s, -p.rc + by0 * p.s, p.s, nx, 0, nx * ny, p.ls,
                                                 s_pt, s_warp, s_part);
            if (t < nx * ny) {
                const int py = t / nx, px = t - py * nx;
                p.bounds[(size_t)a * per_agent + (size_t)k * p.nb + (size_t)(by0 + py) * p.nbx + (bx0 + px)] = bound;
            }
        }
        return;
    }
    if (kMode == kSeed) {
        for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int a = (int)(item >> 1);
            if (p.agent_off[a + 1] == p.agent_off[a]) continue;
            if ((item & 1) == 0) {
                scored += align_exact(p, a, 0, 0, 0, 1, 1, s_pt, s_warp, s_part, s_max, p.prior_score + a);
            } else {
                const long long idx = p.seed[a];
                const int k = (int)(idx / p.nb), b = (int)(idx - (long long)k * p.nb);
                const int x0 = -p.rc + (b % p.nbx) * p.s, y0 = -p.rc + (b / p.nbx) * p.s;
                const int nx = min(p.s, p.rc - x0 + 1), ny = min(p.s, p.rc - y0 + 1);
                scored += align_exact(p, a, k, x0, y0, nx, ny, s_pt, s_warp, s_part, s_max, nullptr);
            }
        }
        if (t == 0) p.cta_scored[blockIdx.x] = scored;
        return;
    }
    const long long G = gridDim.x;
    for (long long round = 0; (long long)blockIdx.x + G * kAlignThreads * round < n_items; ++round) {
        const long long idx = (long long)blockIdx.x + G * (kAlignThreads * round + t);
        bool live = false;
        unsigned long long bkey = 0;
        if (idx < n_items) {
            const int a = (int)(idx / per_agent);
            if (p.agent_off[a + 1] != p.agent_off[a] && idx - (long long)a * per_agent != p.seed[a]) {
                const long long r = idx - (long long)a * per_agent;
                const int k = (int)(r / p.nb), b = (int)(r - (long long)k * p.nb);
                const int x0 = -p.rc + (b % p.nbx) * p.s, y0 = -p.rc + (b / p.nbx) * p.s;
                const int x1 = min(x0 + p.s - 1, p.rc), y1 = min(y0 + p.s - 1, p.rc);
                const unsigned long long low = ((unsigned long long)k * p.d + align_o_min(y0, y1)) * p.d + align_o_min(x0, x1);
                bkey = align_key(p.bounds[idx], low);
                live = bkey > *reinterpret_cast<volatile unsigned long long*>(p.best + a);
            }
        }
        unsigned long long n_live;
        const unsigned long long at = block_exclusive_scan<unsigned long long>(live ? 1u : 0u, s_wide, &n_live);
        if (live) {
            s_items[at] = idx;
            s_bkey[at] = bkey;
        }
        __syncthreads();
        for (unsigned long long q = 0; q < n_live; ++q) {
            const long long it = s_items[q];
            const int a = (int)(it / per_agent);
            const long long r = it - (long long)a * per_agent;
            const int k = (int)(r / p.nb), b = (int)(r - (long long)k * p.nb);
            const int x0 = -p.rc + (b % p.nbx) * p.s, y0 = -p.rc + (b / p.nbx) * p.s;
            // the incumbent may have risen since the test: skip the block if it can no longer win
            if (t == 0) s_go = s_bkey[q] > *reinterpret_cast<volatile unsigned long long*>(p.best + a);
            __syncthreads();
            const bool go = s_go != 0;
            __syncthreads();
            if (!go) continue;
            const int nx = min(p.s, p.rc - x0 + 1), ny = min(p.s, p.rc - y0 + 1);
            scored += align_exact(p, a, k, x0, y0, nx, ny, s_pt, s_warp, s_part, s_max, nullptr);
        }
        __syncthreads();                                       // s_items is rewritten by the next round
    }
    if (t == 0) p.cta_scored[kAlignMaxCtas + blockIdx.x] = scored;
}

// One CTA per agent: seed[a] = the block of the largest bound, ties to the lowest index.
__global__ void __launch_bounds__(kAlignThreads)
k_align_pick(AlignArgs p) {
    __shared__ unsigned long long s_max[kAlignThreads / 32];
    const int a = blockIdx.x;
    if (*p.flag) return;
    const long long n = (long long)p.n_angles * p.nb;        // <= 2^32 - 1
    const unsigned int* bd = p.bounds + (size_t)a * n;
    unsigned long long m = 0;
    for (long long i = threadIdx.x; i < n; i += kAlignThreads) {
        const unsigned long long key = align_key(bd[i], (unsigned long long)i);
        m = key > m ? key : m;
    }
    m = warp_max_u64(m);
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kAlignThreads / 32; ++w) m = s_max[w] > m ? s_max[w] : m;
        p.seed[a] = (long long)(0xffffffffull - (m & 0xffffffffull));
    }
}

__device__ __forceinline__ int align_o_inv(unsigned int o) { return (o & 1u) ? (int)((o + 1u) / 2u) : -(int)(o / 2u); }

// One CTA: the [A][6] rows (score, k, dx, dy, prior_score, n_points) and diag = {candidates searched,
// candidates scored exactly}.
__global__ void __launch_bounds__(kAlignThreads)
k_align_finish(AlignArgs p, int seed_ctas, int exact_ctas, long long* __restrict__ out, long long* __restrict__ diag) {
    __shared__ unsigned long long s_warp[33];
    const int ovf = *p.flag;
    const unsigned long long per_agent = (unsigned long long)p.n_angles * p.d * p.d;
    unsigned long long searched = 0, scored = 0;
    for (int a = threadIdx.x; a < p.n_agents; a += kAlignThreads) {
        long long* row = out + 6 * (size_t)a;
        const long long n = ovf ? 0 : p.agent_off[a + 1] - p.agent_off[a];
        long long v[6] = {ovf ? -2 : 0, 0, 0, 0, 0, n};
        if (n > 0) {
            const unsigned long long key = p.best[a];
            const unsigned long long rank = 0xffffffffull - (key & 0xffffffffull);
            v[0] = (long long)(key >> 32);
            v[2] = align_o_inv((unsigned int)(rank % p.d));
            v[3] = align_o_inv((unsigned int)((rank / p.d) % p.d));
            v[1] = (long long)(rank / p.d / p.d);
            v[4] = p.prior_score[a];
            searched += per_agent;
        }
        for (int c = 0; c < 6; ++c) row[c] = v[c];
    }
    if (!ovf) {
        for (int c = threadIdx.x; c < seed_ctas; c += kAlignThreads) scored += (unsigned long long)p.cta_scored[c];
        for (int c = threadIdx.x; c < exact_ctas; c += kAlignThreads) scored += (unsigned long long)p.cta_scored[kAlignMaxCtas + c];
    }
    unsigned long long tot_searched, tot_scored;
    block_exclusive_scan<unsigned long long>(searched, s_warp, &tot_searched);
    block_exclusive_scan<unsigned long long>(scored, s_warp, &tot_scored);
    if (diag && threadIdx.x == 0) {
        diag[0] = (long long)tot_searched;
        diag[1] = (long long)tot_scored;
    }
}

// Workspace layout; every region is 256-aligned.
struct AlignLayout {
    size_t coef, cnt, agent_off, bounds, best, prior, seed, scored, flag, lw, ls, tmp, pts, fixed;
    long long cpa, nb, pw, ph;
    int pad, nbx;
};

static AlignLayout align_layout(int n_agents, int32_t width, int32_t height, int32_t ref_w, int32_t ref_h, int32_t max_offset,
                                int32_t n_angles, int s) {
    AlignLayout L;
    const size_t A = (size_t)n_agents, n = (size_t)n_angles;
    L.cpa = ((long long)width * height + kAlignCellsPerCta - 1) / kAlignCellsPerCta;
    L.nbx = (2 * max_offset + 1 + s - 1) / s;
    L.nb = (long long)L.nbx * L.nbx;
    L.pad = 2 * max_offset + kAlignMaxBlock;
    L.pw = (long long)ref_w + 2 * L.pad;
    L.ph = (long long)ref_h + 2 * L.pad;
    const size_t np = (size_t)L.pw * (size_t)L.ph;
    L.coef = 0;
    L.cnt = align_up(L.coef + 48 * A * n, 256);
    L.agent_off = align_up(L.cnt + 4 * A * (size_t)L.cpa, 256);
    L.bounds = align_up(L.agent_off + 8 * (A + 1), 256);
    L.best = align_up(L.bounds + 4 * A * n * (size_t)L.nb, 256);
    L.prior = align_up(L.best + 8 * A, 256);
    L.seed = align_up(L.prior + 8 * A, 256);
    L.scored = align_up(L.seed + 8 * A, 256);
    L.flag = align_up(L.scored + 16 * (size_t)kAlignMaxCtas, 256);
    L.lw = L.flag + 256;
    L.ls = align_up(L.lw + np, 256);
    L.tmp = align_up(L.ls + np, 256);
    L.pts = align_up(L.tmp + np, 256);
    L.fixed = L.pts;
    return L;
}

// The size limits shared by the query and the call.  `who` prefixes the message.
static int align_check(const char* who, int n_agents, int32_t width, int32_t height, int32_t ref_w, int32_t ref_h,
                       int32_t max_d2, int32_t max_offset, int32_t n_angles) {
    if (n_agents < 1 || n_agents > kAlignMaxAgents) {
        set_last_error("%s: n_agents %d outside 1..%d", who, n_agents, kAlignMaxAgents);
        return OCCGRID_E_ARG;
    }
    if (max_d2 < 0 || max_d2 > kAlignMaxD2) {
        set_last_error("%s: max_d2 %d outside 0..%d", who, (int)max_d2, kAlignMaxD2);
        return OCCGRID_E_ARG;
    }
    if (width < 1 || height < 1 || (long long)width * height * (max_d2 + 1) > 0x7fffffffLL) {
        set_last_error("%s: width x height %d x %d: each side >= 1 and W*H*(max_d2+1) <= 2^31-1", who, (int)width, (int)height);
        return OCCGRID_E_ARG;
    }
    if (ref_w < 1 || ref_h < 1 || ref_w > kAlignMaxSide || ref_h > kAlignMaxSide) {
        set_last_error("%s: reference size %d x %d: each side in 1..%d", who, (int)ref_w, (int)ref_h, kAlignMaxSide);
        return OCCGRID_E_ARG;
    }
    if (max_offset < 0 || max_offset > kAlignMaxOffset) {
        set_last_error("%s: max_offset %d outside 0..%d", who, (int)max_offset, kAlignMaxOffset);
        return OCCGRID_E_ARG;
    }
    if (n_angles < 1 || n_angles > kAlignMaxAngles) {
        set_last_error("%s: n_angles %d outside 1..%d", who, (int)n_angles, kAlignMaxAngles);
        return OCCGRID_E_ARG;
    }
    const unsigned long long d = 2ull * max_offset + 1;
    if ((unsigned long long)n_angles * d * d > 0xffffffffull) {
        set_last_error("%s: %d angles x (2*%d+1)^2 offsets: more than 2^32-1 candidates", who, (int)n_angles, (int)max_offset);
        return OCCGRID_E_ARG;
    }
    return OCCGRID_OK;
}

static unsigned int align_grid(long long items, int per_sm) {
    const long long cap = std::min((long long)kAlignMaxCtas, (long long)device_sm_count() * per_sm);
    return (unsigned int)std::max(1LL, std::min(items, cap));
}

static unsigned int flat_grid(long long n) {
    return (unsigned int)std::max(1LL, std::min((n + 255) / 256, (long long)device_sm_count() * 16));
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t mapmerge_align_workspace_bytes(int n_agents, int32_t width, int32_t height, int32_t ref_w, int32_t ref_h, int32_t max_d2,
                                      int32_t max_offset, int32_t n_angles, int64_t total_points) {
    if (align_check("mapmerge_align_workspace_bytes", n_agents, width, height, ref_w, ref_h, max_d2, max_offset, n_angles) != OCCGRID_OK)
        return 0;
    if (total_points < 0 || total_points > (int64_t)n_agents * width * height) {
        set_last_error("mapmerge_align_workspace_bytes: total_points %lld outside 0..n_agents*W*H", (long long)total_points);
        return 0;
    }
    const AlignLayout L = align_layout(n_agents, width, height, ref_w, ref_h, max_offset, n_angles, align_block());
    return align_up(L.fixed + 8 * (size_t)total_points, 256);
}

int mapmerge_align_set_block(int s) {
    if (s < 0 || s > kAlignMaxBlock) {
        set_last_error("mapmerge_align_set_block: block %d outside 0..%d", s, kAlignMaxBlock);
        return OCCGRID_E_ARG;
    }
    g_align_block = s;
    return OCCGRID_OK;
}

int mapmerge_align(const int8_t* d_grids, int n_agents, int32_t width, int32_t height, double res, const double* origins_host,
                   const double* priors_host, const int32_t* d_d2, int32_t ref_w, int32_t ref_h, double ref_ox, double ref_oy,
                   double ref_res, const double* rot_host, int32_t n_angles, int32_t max_offset, int32_t max_d2,
                   int64_t* d_out, int64_t* d_diag, void* d_ws, size_t ws_bytes, void* stream) {
    if (!d_grids || !origins_host || !priors_host || !d_d2 || !rot_host || !d_out || !d_ws) {
        set_last_error("mapmerge_align: NULL pointer");
        return OCCGRID_E_ARG;
    }
    int rc = align_check("mapmerge_align", n_agents, width, height, ref_w, ref_h, max_d2, max_offset, n_angles);
    if (rc != OCCGRID_OK) return rc;
    if (!(std::isfinite(res) && res > 0.0) || !(std::isfinite(ref_res) && ref_res > 0.0)) {
        set_last_error("mapmerge_align: resolution must be finite and > 0 (maps %g, reference %g)", res, ref_res);
        return OCCGRID_E_ARG;
    }
    for (int a = 0; a < n_agents; ++a) {
        const double* T = priors_host + 16 * (size_t)a;
        for (int k = 0; k < 16; ++k)
            if (!std::isfinite(T[k])) {
                set_last_error("mapmerge_align: prior %d has a non-finite entry", a);
                return OCCGRID_E_ARG;
            }
        const double R[2][2] = {{T[0], T[1]}, {T[4], T[5]}};
        for (int p = 0; p < 2; ++p)
            for (int q = 0; q < 2; ++q) {
                const double rtr = R[0][p] * R[0][q] + R[1][p] * R[1][q];
                if (!(fabs(rtr - (p == q ? 1.0 : 0.0)) <= kAlignTol)) {
                    set_last_error("mapmerge_align: prior %d is not rigid (|R^T R - I| > 1e-9)", a);
                    return OCCGRID_E_ARG;
                }
            }
    }
    for (int k = 0; k < n_angles; ++k) {
        const double cs = rot_host[2 * (size_t)k], sn = rot_host[2 * (size_t)k + 1];
        if (!(fabs(cs * cs + sn * sn - 1.0) <= kAlignTol)) {
            set_last_error("mapmerge_align: rotation %d (%g, %g) is not a unit (cs, sn) pair", k, cs, sn);
            return OCCGRID_E_ARG;
        }
    }
    const int s = align_block();
    const AlignLayout L = align_layout(n_agents, width, height, ref_w, ref_h, max_offset, n_angles, s);
    if (ws_bytes < L.fixed) {
        set_last_error("mapmerge_align: workspace too small");
        return OCCGRID_E_WORKSPACE;
    }
    const long long capacity = (long long)((ws_bytes - L.fixed) / 8);

    // Coefficients per (agent, rotation), host fp64, each operation rounded on its own.
    std::vector<double> hc((size_t)n_agents * n_angles * 6);
    const double r = res, g = ref_res;
    for (int a = 0; a < n_agents; ++a) {
        const double* P = priors_host + 16 * (size_t)a;
        const double p00 = P[0], p01 = P[1], p03 = P[3], p10 = P[4], p11 = P[5], p13 = P[7];
        const double ox = origins_host[2 * (size_t)a], oy = origins_host[2 * (size_t)a + 1];
        const double mx = ox + ((0.5 * width) * r), my = oy + ((0.5 * height) * r);
        const double ex = -((p00 * mx) + (p01 * my)), ey = -((p10 * mx) + (p11 * my));
        const double bx = ox + 0.5 * r, by = oy + 0.5 * r;
        for (int k = 0; k < n_angles; ++k) {
            const double cs = rot_host[2 * (size_t)k], sn = rot_host[2 * (size_t)k + 1];
            const double m00 = (cs * p00) - (sn * p10), m01 = (cs * p01) - (sn * p11);
            const double m10 = (sn * p00) + (cs * p10), m11 = (sn * p01) + (cs * p11);
            const double tx = p03 + (((cs - 1.0) * ex) - (sn * ey)), ty = p13 + ((sn * ex) + ((cs - 1.0) * ey));
            double* e = hc.data() + ((size_t)a * n_angles + k) * 6;
            e[0] = (m00 * r) / g;
            e[1] = (m01 * r) / g;
            e[2] = ((((m00 * bx) + (m01 * by)) + tx) - ref_ox) / g;
            e[3] = (m10 * r) / g;
            e[4] = (m11 * r) / g;
            e[5] = ((((m10 * bx) + (m11 * by)) + ty) - ref_oy) / g;
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(d_ws);
    // A copy from pageable memory has been staged by the driver when cudaMemcpyAsync returns, so hc
    // may go out of scope without a stream synchronisation.
    OCC_CUDA_TRY(cudaMemcpyAsync(ws + L.coef, hc.data(), sizeof(double) * hc.size(), cudaMemcpyHostToDevice, st));
    OCC_CUDA_TRY(cudaMemsetAsync(ws + L.best, 0, 8 * (size_t)n_agents, st));

    AlignArgs p;
    p.coef = reinterpret_cast<const double*>(ws + L.coef);
    p.agent_off = reinterpret_cast<const long long*>(ws + L.agent_off);
    p.pts = reinterpret_cast<const int2*>(ws + L.pts);
    p.lw = reinterpret_cast<const uint8_t*>(ws + L.lw);
    p.ls = s == 1 ? p.lw : reinterpret_cast<const uint8_t*>(ws + L.ls);
    p.pitch = L.pw;
    p.pad = L.pad;
    p.wr = ref_w;
    p.hr = ref_h;
    p.rc = max_offset;
    p.d = 2 * max_offset + 1;
    p.s = s;
    p.nbx = L.nbx;
    p.tiles_x = (L.nbx + kAlignTile - 1) / kAlignTile;
    p.n_angles = n_angles;
    p.n_agents = n_agents;
    p.nb = L.nb;
    p.bounds = reinterpret_cast<unsigned int*>(ws + L.bounds);
    p.best = reinterpret_cast<unsigned long long*>(ws + L.best);
    p.prior_score = reinterpret_cast<long long*>(ws + L.prior);
    p.seed = reinterpret_cast<long long*>(ws + L.seed);
    int* flag = reinterpret_cast<int*>(ws + L.flag);
    p.flag = flag;
    p.cta_scored = reinterpret_cast<long long*>(ws + L.scored);

    const long long np = L.pw * L.ph, cells = (long long)width * height;
    const long long n_bound = (long long)n_agents * n_angles * p.tiles_x * p.tiles_x;
    const long long n_exact = (long long)n_agents * n_angles * L.nb;
    const unsigned int g_bound = align_grid(n_bound, 8), g_seed = align_grid(2LL * n_agents, 8), g_exact = align_grid(n_exact, 8);
    unsigned int* cnt = reinterpret_cast<unsigned int*>(ws + L.cnt);
    long long* agent_off = reinterpret_cast<long long*>(ws + L.agent_off);
    int2* pts = reinterpret_cast<int2*>(ws + L.pts);
    uint8_t* lw = reinterpret_cast<uint8_t*>(ws + L.lw);
    {
        ProfileScope ps(K_MAP_ALIGN, st, s == 1 ? 10 : 12);
        k_align_weights<<<flat_grid(np), 256, 0, st>>>(d_d2, ref_w, ref_h, L.pad, L.pw, np, max_d2, lw);
        if (s > 1) {
            uint8_t* tmp = reinterpret_cast<uint8_t*>(ws + L.tmp);
            k_align_rowmax<<<flat_grid(np), 256, 0, st>>>(lw, L.pw, np, s, tmp);
            k_align_colmax<<<flat_grid(np), 256, 0, st>>>(tmp, L.pw, L.ph, np, s, reinterpret_cast<uint8_t*>(ws + L.ls));
        }
        const dim3 cg((unsigned int)L.cpa, (unsigned int)n_agents);
        k_align_cells<false><<<cg, kAlignThreads, 0, st>>>(d_grids, width, cells, L.cpa, cnt, agent_off, pts, flag);
        k_align_scan_agents<<<n_agents, kAlignThreads, 0, st>>>(cnt, L.cpa, agent_off);
        k_align_scan_total<<<1, kAlignThreads, 0, st>>>(agent_off, n_agents, capacity, flag);
        k_align_cells<true><<<cg, kAlignThreads, 0, st>>>(d_grids, width, cells, L.cpa, cnt, agent_off, pts, flag);
        k_align_score<kBound><<<g_bound, kAlignThreads, 0, st>>>(p, n_bound);
        k_align_pick<<<n_agents, kAlignThreads, 0, st>>>(p);
        k_align_score<kSeed><<<g_seed, kAlignThreads, 0, st>>>(p, 2LL * n_agents);
        k_align_score<kExact><<<g_exact, kAlignThreads, 0, st>>>(p, n_exact);
        k_align_finish<<<1, kAlignThreads, 0, st>>>(p, (int)g_seed, (int)g_exact, reinterpret_cast<long long*>(d_out),
                                                   reinterpret_cast<long long*>(d_diag));
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
