// Occupancy-grid integration kernels and their C ABI (include/occgrid_b200.h).
//
// Reference path replaced: the per-packet loop body of main()
// (server_nodes/dual_bot_mapper.py:826-903) and OccupancyGrid.update_ray/_bresenham
// (:136-179).  The reference is a sequential overwrite ("last writer wins" across beams in
// stream order, SURVEY.md App. A.7).  On the GPU the order is carried explicitly: every
// beam has an ordinal (record index * 4 + sensor index), each touched cell keeps the
// largest  (ordinal + 1) << 1 | is_occupied  stamp, and the stamp's low bit is the cell value
// the sequential loop would have left behind.
//
// Strategy GLOBAL_ATOMIC (this file): one thread per packet decodes, expands and walks its
// four beams, issuing one red.global.max.u32 per cell on a window-sized stamp plane; a
// streaming resolve pass folds the stamps into the int8 grid and re-zeroes the plane.
// Strategy TILED lives in occgrid_tiled.cu.
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace occ {

static thread_local std::string g_last_error;

void set_last_error(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

bool cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    set_last_error("CUDA error %s (%d) in %s", cudaGetErrorString(e), (int)e, what);
    return false;
}

// ---- per-kernel profiling hook -----------------------------------------------------------
struct ProfileState {
    std::mutex mu;
    bool on = false;
    std::vector<cudaEvent_t> ev[K_N_KERNELS];   // begin/end pairs
    long long kernels[K_N_KERNELS] = {};         // kernels launched inside the scopes
};
static ProfileState g_prof;

bool profile_enabled() { return g_prof.on; }

void profile_mark(int id, cudaStream_t st, bool begin, int n_kernels) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    if (begin) g_prof.kernels[id] += n_kernels;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    g_prof.ev[id].push_back(e);
}

int validate_geom(const occgrid_geom* g) {
    if (!g) { set_last_error("geom is NULL"); return OCCGRID_E_ARG; }
    if (!(g->res > 0.0) || !isfinite(g->res) || !isfinite(g->ox) || !isfinite(g->oy)) {
        set_last_error("geom: res must be > 0 and origin finite");
        return OCCGRID_E_ARG;
    }
    if (g->size_x <= 0 || g->size_y <= 0 || g->size_x > (1 << 30) || g->size_y > (1 << 30)) {
        set_last_error("geom: grid size must be in 1..2^30");
        return OCCGRID_E_ARG;
    }
    if (g->win_w <= 0 || g->win_h <= 0 || g->win_x0 < 0 || g->win_y0 < 0 ||
        (int64_t)g->win_x0 + g->win_w > g->size_x || (int64_t)g->win_y0 + g->win_h > g->size_y) {
        set_last_error("geom: window must be a non-empty sub-rectangle of the grid");
        return OCCGRID_E_ARG;
    }
    if (OCC_MAX_DIST_M / g->res > 16000.0) {
        set_last_error("geom: res %.3g gives rays longer than 16000 cells", g->res);
        return OCCGRID_E_RANGE;
    }
    return OCCGRID_OK;
}

// ------------------------------------------------------------------------------------------
//  Strategy GLOBAL_ATOMIC
// ------------------------------------------------------------------------------------------

constexpr int kThreads = 256;          // threads (= packets) per CTA

// Walk one beam (exact reference Bresenham, :158-179) and raise the stamp of every cell the
// sequential update_ray (:148-156) would have stored to: all cells but the last -> FREE,
// the last -> OCCUPIED when hit_valid, untouched otherwise.  `skip_first` drops the write
// to the start cell when a later beam of the same packet overwrites it anyway.
__device__ __forceinline__ void draw_beam_global(const Geom& g, unsigned int* __restrict__ stamps,
                                                 const Beam& b, unsigned int ord1, bool skip_first) {
    if (!b.valid) return;
    const int wx1 = g.win_x0 + g.win_w, wy1 = g.win_y0 + g.win_h;
    const int bx0 = min(b.x0, b.x1), bx1 = max(b.x0, b.x1);
    const int by0 = min(b.y0, b.y1), by1 = max(b.y0, b.y1);
    if (bx1 < g.win_x0 || bx0 >= wx1 || by1 < g.win_y0 || by0 >= wy1) return;   // per-cell clip would reject all
    const bool inside = bx0 >= g.win_x0 && bx1 < wx1 && by0 >= g.win_y0 && by1 < wy1;
    int x = b.x0, y = b.y0;
    const int dx = bx1 - bx0, dy = by1 - by0;
    const int sx = b.x0 < b.x1 ? 1 : -1, sy = b.y0 < b.y1 ? 1 : -1;
    int err = dx - dy;
    const int n = max(dx, dy);
    const unsigned int free_stamp = ord1 << 1;
    for (int i = 0; i < n; ++i) {
        if (!(i == 0 && skip_first) && (inside || (x >= g.win_x0 && x < wx1 && y >= g.win_y0 && y < wy1)))
            atomicMax(&stamps[(size_t)(y - g.win_y0) * g.win_w + (x - g.win_x0)], free_stamp);
        const int e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x += sx; }
        if (e2 < dx)  { err += dx; y += sy; }
    }
    if (b.hit && !(n == 0 && skip_first) && (inside || (x >= g.win_x0 && x < wx1 && y >= g.win_y0 && y < wy1)))
        atomicMax(&stamps[(size_t)(y - g.win_y0) * g.win_w + (x - g.win_x0)], free_stamp | 1u);
}

// Hit/miss COUNT mode (extension): counts = int32 [win_h][win_w][2] = {miss, hit} per cell.  Every
// cell update_ray would have stored FREE to counts a miss, the OCCUPIED end cell of a valid hit
// counts a hit; integer adds commute, so the planes equal np.add.at over the reference's cells.
__device__ __forceinline__ void count_beam_global(const Geom& g, int* __restrict__ counts, const Beam& b) {
    if (!b.valid) return;
    const int wx1 = g.win_x0 + g.win_w, wy1 = g.win_y0 + g.win_h;
    const int bx0 = min(b.x0, b.x1), bx1 = max(b.x0, b.x1);
    const int by0 = min(b.y0, b.y1), by1 = max(b.y0, b.y1);
    if (bx1 < g.win_x0 || bx0 >= wx1 || by1 < g.win_y0 || by0 >= wy1) return;
    int x = b.x0, y = b.y0;
    const int dx = bx1 - bx0, dy = by1 - by0;
    const int sx = b.x0 < b.x1 ? 1 : -1, sy = b.y0 < b.y1 ? 1 : -1;
    int err = dx - dy;
    const int n = max(dx, dy);
    for (int i = 0; i < n; ++i) {
        if (x >= g.win_x0 && x < wx1 && y >= g.win_y0 && y < wy1)
            atomicAdd(&counts[2 * ((size_t)(y - g.win_y0) * g.win_w + (x - g.win_x0))], 1);
        const int e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x += sx; }
        if (e2 < dx)  { err += dx; y += sy; }
    }
    if (b.hit && x >= g.win_x0 && x < wx1 && y >= g.win_y0 && y < wy1)
        atomicAdd(&counts[2 * ((size_t)(y - g.win_y0) * g.win_w + (x - g.win_x0)) + 1], 1);
}

__device__ __forceinline__ bool start_in_window(const Geom& g, const Beam& b) {
    return b.valid && b.x0 >= g.win_x0 && b.x0 < g.win_x0 + g.win_w && b.y0 >= g.win_y0 && b.y0 < g.win_y0 + g.win_h;
}

// kMaps: one stamp plane per agent (occgrid_integrate_packets_agent_maps); a record of agent a
// draws into plane a - 1, `map_cells` words after plane a - 2.
template <bool kCounts, bool kMaps = false>
__global__ void __launch_bounds__(kThreads)
k_integrate_global(Geom g, const uint8_t* __restrict__ pkts, long long n, int stride,
                   const int32_t* __restrict__ agent_idx, const double* __restrict__ drift,
                   const double* __restrict__ agent_off, int n_agents,
                   unsigned int* __restrict__ stamps, uint64_t* counters, size_t map_cells = 0) {
    __shared__ __align__(16) uint8_t s_rec[kThreads * kMaxRecStride];
    __shared__ unsigned long long s_acc[(OCCGRID_C_OWNED_UPDATES + 1) * 32];
    const long long first = (long long)blockIdx.x * kThreads;
    const int count = (int)min((long long)kThreads, n - first);
    stage_records(pkts + (size_t)first * stride, (size_t)count * stride, s_rec);
    __syncthreads();

    unsigned long long c[OCCGRID_C_OWNED_UPDATES + 1] = {};
    if ((int)threadIdx.x < count) {
        const long long k = first + threadIdx.x;
        double rx, ry, ryaw;
        float dist[4];
        int agent = 1;
        c[OCCGRID_C_PACKETS] = 1;
        const int st = decode_packet(s_rec + threadIdx.x * stride, k, agent_idx, drift, agent_off, n_agents,
                                     &rx, &ry, &ryaw, dist, kMaps ? &agent : nullptr);
        if (st == PKT_DROPPED) c[OCCGRID_C_DROPPED] = 1;
        else if (st == PKT_BAD_POSE) c[OCCGRID_C_BAD_POSE] = 1;
        else {
            c[OCCGRID_C_ACCEPTED] = 1;
            if (kMaps) stamps += (size_t)(agent - 1) * map_cells;
            Beam b[4];
            expand_packet(g, rx, ry, ryaw, dist, LibSinCos(), b);
            bool later_writes_first = false;
#pragma unroll
            for (int s = 3; s >= 0; --s) {
                const int cells = b[s].valid ? beam_cells(b[s]) : 0;
                c[OCCGRID_C_BEAMS] += 1;
                c[OCCGRID_C_HITS] += b[s].hit;
                c[OCCGRID_C_UPDATES] += cells;
                c[OCCGRID_C_SLOWPATH] += b[s].slow;
                if (start_in_window(g, b[s])) c[OCCGRID_C_OWNED_UPDATES] += cells;
                if (kCounts) count_beam_global(g, reinterpret_cast<int*>(stamps), b[s]);
                else draw_beam_global(g, stamps, b[s], (unsigned int)(k * 4 + s + 1), later_writes_first);
                later_writes_first = later_writes_first || (b[s].valid && (cells > 1 || b[s].hit));
            }
        }
    }
    block_add_counters(c, s_acc, counters);
}

// Decoded input (routed pose records): same as k_integrate_global minus the decode.
__global__ void __launch_bounds__(kThreads)
k_integrate_poses_global(Geom g, const PoseRec* __restrict__ recs, long long n, int ordinals_in_records,
                         unsigned int* __restrict__ stamps, uint64_t* counters) {
    __shared__ unsigned long long s_acc[(OCCGRID_C_OWNED_UPDATES + 1) * 32];
    const long long k = (long long)blockIdx.x * kThreads + threadIdx.x;
    unsigned long long c[OCCGRID_C_OWNED_UPDATES + 1] = {};
    if (k < n) {
        const PoseRec r = recs[k];
        c[OCCGRID_C_PACKETS] = 1;
        if (!(isfinite(r.rx) && isfinite(r.ry) && isfinite(r.yaw))) c[OCCGRID_C_BAD_POSE] = 1;
        else {
            c[OCCGRID_C_ACCEPTED] = 1;
            const float dist[4] = {r.d[0], r.d[1], r.d[2], r.d[3]};
            Beam b[4];
            expand_packet(g, r.rx, r.ry, (double)r.yaw, dist, LibSinCos(), b);
            bool later_writes_first = false;
#pragma unroll
            for (int s = 3; s >= 0; --s) {
                const int cells = b[s].valid ? beam_cells(b[s]) : 0;
                c[OCCGRID_C_BEAMS] += 1;
                c[OCCGRID_C_HITS] += b[s].hit;
                c[OCCGRID_C_UPDATES] += cells;
                c[OCCGRID_C_SLOWPATH] += b[s].slow;
                if (start_in_window(g, b[s])) c[OCCGRID_C_OWNED_UPDATES] += cells;
                const unsigned int ord = ordinals_in_records ? r.k : (unsigned int)k;
                draw_beam_global(g, stamps, b[s], ord * 4u + (unsigned int)s + 1u, later_writes_first);
                later_writes_first = later_writes_first || (b[s].valid && (cells > 1 || b[s].hit));
            }
        }
    }
    block_add_counters(c, s_acc, counters);
}

__global__ void __launch_bounds__(kThreads)
k_update_rays_global(Geom g, const double* __restrict__ rays, const uint8_t* __restrict__ hit, long long n,
                     unsigned int* __restrict__ stamps, uint64_t* counters) {
    __shared__ unsigned long long s_acc[(OCCGRID_C_OWNED_UPDATES + 1) * 32];
    const long long k = (long long)blockIdx.x * kThreads + threadIdx.x;
    unsigned long long c[OCCGRID_C_OWNED_UPDATES + 1] = {};
    if (k < n) {
        const double2 r0 = __ldg(reinterpret_cast<const double2*>(rays) + 2 * k);
        const double2 r1 = __ldg(reinterpret_cast<const double2*>(rays) + 2 * k + 1);
        Beam b;
        ray_to_beam(g, r0.x, r0.y, r1.x, r1.y, hit[k] != 0, &b);
        const int cells = b.valid ? beam_cells(b) : 0;
        c[OCCGRID_C_BEAMS] = 1;
        c[OCCGRID_C_HITS] = b.hit;
        c[OCCGRID_C_UPDATES] = cells;
        if (start_in_window(g, b)) c[OCCGRID_C_OWNED_UPDATES] = cells;
        draw_beam_global(g, stamps, b, (unsigned int)(k + 1), false);
    }
    block_add_counters(c, s_acc, counters);
}

// Fold stamps into the grid and re-zero them: 4 cells per thread per step, 16-byte stamp
// loads, 4-byte grid read-modify-write only where something was touched.
__global__ void __launch_bounds__(kThreads)
k_resolve(unsigned int* __restrict__ stamps, int8_t* __restrict__ grid, size_t n_cells, int vec_ok) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    size_t tail_begin = 0;
    if (vec_ok) {
        const size_t n4 = n_cells / 4;
        uint4* s4 = reinterpret_cast<uint4*>(stamps);
        char4* g4 = reinterpret_cast<char4*>(grid);
        for (size_t i = tid; i < n4; i += nthreads) {
            const uint4 s = s4[i];
            if (s.x | s.y | s.z | s.w) {
                char4 v = g4[i];
                if (s.x) v.x = (s.x & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
                if (s.y) v.y = (s.y & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
                if (s.z) v.z = (s.z & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
                if (s.w) v.w = (s.w & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
                g4[i] = v;
                s4[i] = make_uint4(0u, 0u, 0u, 0u);
            }
        }
        tail_begin = n4 * 4;
    }
    for (size_t i = tail_begin + tid; i < n_cells; i += nthreads) {
        const unsigned int s = stamps[i];
        if (s) {
            grid[i] = (s & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
            stamps[i] = 0u;
        }
    }
}

int device_sm_count() {
    static int by_device[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (by_device[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        by_device[dev] = n;
    }
    return by_device[dev];
}

// n_maps > 1: the planes and grids of an agent-map stack are contiguous, so one pass streams them all.
static int launch_resolve(const occgrid_geom* geom, unsigned int* stamps, int8_t* grid, cudaStream_t st, int n_maps = 1) {
    const size_t n_cells = (size_t)geom->win_w * geom->win_h * (size_t)n_maps;
    const int vec_ok = ((reinterpret_cast<uintptr_t>(stamps) & 15) == 0 && (reinterpret_cast<uintptr_t>(grid) & 3) == 0) ? 1 : 0;
    size_t want = (n_cells / 4 + kThreads - 1) / kThreads;
    if (want < 1) want = 1;
    const size_t cap = (size_t)device_sm_count() * 8;
    const int blocks = (int)(want < cap ? want : cap);
    ProfileScope ps(K_RESOLVE, st);
    k_resolve<<<blocks, kThreads, 0, st>>>(stamps, grid, n_cells, vec_ok);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// One stamp plane per map, each the size of the window (agent maps: the whole grid).
static size_t global_workspace_bytes(const occgrid_geom* geom, int n_maps) {
    return align_up((size_t)geom->win_w * geom->win_h * (size_t)n_maps * sizeof(unsigned int), 256);
}

// Count planes take the beams' adds directly: no stamp plane, no workspace, no resolve.
static int integrate_packets_global(const occgrid_geom* geom, const PacketBatch& b, Output kind, void* d_out, void* d_ws,
                                    size_t ws_bytes, uint64_t* d_counters, cudaStream_t st) {
    const int n_maps = kind == Output::kAgentMaps ? b.n_agents : 1;
    const size_t need = global_workspace_bytes(geom, n_maps);
    if (kind != Output::kCounts && ws_bytes < need) {
        set_last_error("workspace %zu B < %zu B needed by GLOBAL_ATOMIC for %d map(s)", ws_bytes, need, n_maps);
        return OCCGRID_E_WORKSPACE;
    }
    unsigned int* stamps = reinterpret_cast<unsigned int*>(kind == Output::kCounts ? d_out : d_ws);
    const Geom g = to_geom(geom);
    const unsigned int blocks = (unsigned int)((b.n + kThreads - 1) / kThreads);
    {
        ProfileScope ps(K_INTEGRATE_GLOBAL, st);
        if (kind == Output::kCounts)
            k_integrate_global<true><<<blocks, kThreads, 0, st>>>(g, b.pkts, b.n, b.stride, b.agent_idx, b.drift, b.agent_off,
                                                                  b.n_agents, stamps, d_counters);
        else if (kind == Output::kAgentMaps)
            k_integrate_global<false, true><<<blocks, kThreads, 0, st>>>(g, b.pkts, b.n, b.stride, b.agent_idx, b.drift, b.agent_off,
                                                                         b.n_agents, stamps, d_counters, (size_t)geom->win_w * geom->win_h);
        else
            k_integrate_global<false><<<blocks, kThreads, 0, st>>>(g, b.pkts, b.n, b.stride, b.agent_idx, b.drift, b.agent_off,
                                                                   b.n_agents, stamps, d_counters);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    if (kind == Output::kCounts) return OCCGRID_OK;
    return launch_resolve(geom, stamps, reinterpret_cast<int8_t*>(d_out), st, n_maps);
}

// L = clamp(hits * l_occ + misses * l_free, l_min, l_max), derived from the integer planes so
// that it does not depend on the order the beams arrived in (no float atomics anywhere).
__global__ void __launch_bounds__(kThreads)
k_counts_to_logodds(const int32_t* __restrict__ counts, long long n_cells, double l_occ, double l_free, double l_min, double l_max,
                    float* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n_cells; i += (long long)gridDim.x * kThreads) {
        const int2 c = reinterpret_cast<const int2*>(counts)[i];          // {miss, hit}
        const double l = OCC_DADD(OCC_DMUL((double)c.y, l_occ), OCC_DMUL((double)c.x, l_free));
        out[i] = (float)fmin(fmax(l, l_min), l_max);
    }
}

// ------------------------------------------------------------------------------------------
//  Scatter-roofline probes (SURVEY §8d)
// ------------------------------------------------------------------------------------------

__device__ __forceinline__ unsigned int mix32(unsigned int x) {   // lowbias32
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}

__global__ void __launch_bounds__(kThreads)
k_probe_global_atomic(unsigned int* plane, unsigned long long cells, int iters, unsigned int seed) {
    unsigned int h = mix32(seed ^ (blockIdx.x * kThreads + threadIdx.x));
    for (int i = 0; i < iters; ++i) {
        h = mix32(h + 0x9e3779b9U);
        const unsigned long long idx = ((unsigned long long)h * cells) >> 32;
        atomicMax(&plane[idx], h | 1u);
    }
}

__global__ void __launch_bounds__(kThreads)
k_probe_global_store8(uint8_t* plane, unsigned long long cells, int iters, unsigned int seed) {
    unsigned int h = mix32(seed ^ (blockIdx.x * kThreads + threadIdx.x));
    for (int i = 0; i < iters; ++i) {
        h = mix32(h + 0x9e3779b9U);
        const unsigned long long idx = ((unsigned long long)h * cells) >> 32;
        plane[idx] = (uint8_t)h;
    }
}

template <bool kReturn>
__global__ void __launch_bounds__(kThreads)
k_probe_hot_add(unsigned int* plane, unsigned long long cells, int iters, unsigned int seed) {
    unsigned int h = mix32(seed ^ (blockIdx.x * kThreads + threadIdx.x));
    unsigned int acc = 0;
    for (int i = 0; i < iters; ++i) {
        h = mix32(h + 0x9e3779b9U);
        const unsigned long long idx = (((unsigned long long)h * cells) >> 32) * 64ull;   // one hot word per 256 B
        if (kReturn) acc += atomicAdd(&plane[idx], 1u);
        else atomicAdd(&plane[idx], 1u);
    }
    if (kReturn && acc == 0x12345678u) plane[0] = acc;
}

template <bool kAtomic>
__global__ void __launch_bounds__(kThreads)
k_probe_smem(unsigned int* out, unsigned int cells, int iters, unsigned int seed) {
    extern __shared__ unsigned int s_tile[];
    for (unsigned int i = threadIdx.x; i < cells; i += blockDim.x) s_tile[i] = 0;
    __syncthreads();
    unsigned int h = mix32(seed ^ (blockIdx.x * kThreads + threadIdx.x));
    for (int i = 0; i < iters; ++i) {
        h = mix32(h + 0x9e3779b9U);
        const unsigned int idx = (unsigned int)(((unsigned long long)h * cells) >> 32);
        if (kAtomic) atomicMax(&s_tile[idx], h | 1u);
        else reinterpret_cast<volatile unsigned int*>(s_tile)[idx] = h;
    }
    __syncthreads();
    unsigned int acc = 0;
    for (unsigned int i = threadIdx.x; i < cells; i += blockDim.x) acc ^= s_tile[i];
    if (acc == 0x12345678u) out[blockIdx.x] = acc;   // keep the stores alive
}

}  // namespace occ

// ------------------------------------------------------------------------------------------
//  C ABI
// ------------------------------------------------------------------------------------------
using namespace occ;

namespace occ {

int check_packet_batch(const PacketBatch& b, int rec_len, const char* who) {
    if (b.n < 0 || b.n > (1ll << 29) - 1) {
        set_last_error("%sn=%lld outside 0..2^29-1 records per call", who, (long long)b.n);
        return OCCGRID_E_ARG;
    }
    if (rec_len != OCCGRID_PACKET_SIZE && rec_len != OCCGRID_PACKET_SIZE_V1) {
        set_last_error("%srec_len must be 42 or 41, got %d", who, rec_len);
        return OCCGRID_E_ARG;
    }
    if (b.stride < rec_len || b.stride > kMaxRecStride) {
        set_last_error("%sstride %d outside %d..%d", who, b.stride, rec_len, kMaxRecStride);
        return OCCGRID_E_ARG;
    }
    if (b.n_agents < 1 || !b.agent_off) { set_last_error("%sneed n_agents >= 1 and an agent offset table", who); return OCCGRID_E_ARG; }
    if (b.n > 0 && !b.pkts) { set_last_error("%spackets is NULL", who); return OCCGRID_E_ARG; }
    return OCCGRID_OK;
}

// Geometry of an agent-map stack: a valid geometry whose window is the whole grid, n_agents >= 1,
// and a stack (of 4-byte stamps: the larger of the two) whose size fits size_t.
static int validate_agent_maps(const occgrid_geom* geom, int n_agents) {
    int rc = validate_geom(geom);
    if (rc != OCCGRID_OK) return rc;
    if (geom->win_x0 != 0 || geom->win_y0 != 0 || geom->win_w != geom->size_x || geom->win_h != geom->size_y) {
        set_last_error("agent maps: the window must be the whole grid");
        return OCCGRID_E_ARG;
    }
    if (n_agents < 1) { set_last_error("agent maps: n_agents=%d, need >= 1", n_agents); return OCCGRID_E_ARG; }
    const size_t cells = (size_t)geom->size_x * (size_t)geom->size_y;
    if (cells > SIZE_MAX / sizeof(unsigned int) / (size_t)n_agents) {
        set_last_error("agent maps: %d maps of %d x %d cells overflow size_t", n_agents, geom->size_x, geom->size_y);
        return OCCGRID_E_ARG;
    }
    return OCCGRID_OK;
}

// AUTO takes TILED wherever it supports the geometry and the number of maps.  An explicit TILED
// that does not is E_RANGE; an unknown strategy is E_ARG.
static int pick_strategy(const occgrid_geom* geom, int n_maps, int strategy, int* picked) {
    if (strategy == OCCGRID_STRATEGY_AUTO) {
        strategy = tiled_supported(geom, n_maps) ? OCCGRID_STRATEGY_TILED : OCCGRID_STRATEGY_GLOBAL_ATOMIC;
    } else if (strategy == OCCGRID_STRATEGY_TILED && !tiled_supported(geom, n_maps)) {
        set_last_error("TILED strategy does not support this geometry%s", n_maps > 1 ? " and agent count" : "");
        return OCCGRID_E_RANGE;
    } else if (strategy != OCCGRID_STRATEGY_TILED && strategy != OCCGRID_STRATEGY_GLOBAL_ATOMIC) {
        set_last_error("unknown strategy %d", strategy);
        return OCCGRID_E_ARG;
    }
    *picked = strategy;
    return OCCGRID_OK;
}

static size_t workspace_bytes(const occgrid_geom* geom, int n_maps, int64_t max_packets, int strategy) {
    if (max_packets < 0) { set_last_error("max_packets < 0"); return 0; }
    int s;
    if (pick_strategy(geom, n_maps, strategy, &s) != OCCGRID_OK) return 0;
    return s == OCCGRID_STRATEGY_TILED ? tiled_workspace_bytes(geom, n_maps, max_packets) : global_workspace_bytes(geom, n_maps);
}

// The packet entry points once the batch and their output have been checked.
static int integrate_packets(const occgrid_geom* geom, const PacketBatch& b, Output kind, void* d_out, void* d_ws, size_t ws_bytes,
                             uint64_t* d_counters, int strategy, void* stream) {
    if (b.n == 0) return OCCGRID_OK;
    int s;
    const int rc = pick_strategy(geom, kind == Output::kAgentMaps ? b.n_agents : 1, strategy, &s);
    if (rc != OCCGRID_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (s == OCCGRID_STRATEGY_TILED) return integrate_tiled(geom, b, nullptr, 0, kind, d_out, d_ws, ws_bytes, d_counters, st);
    return integrate_packets_global(geom, b, kind, d_out, d_ws, ws_bytes, d_counters, st);
}
}

extern "C" {

int occgrid_abi_version(void) { return OCCGRID_ABI_VERSION; }

const char* occgrid_last_error(void) { return g_last_error.c_str(); }

size_t occgrid_workspace_bytes(const occgrid_geom* geom, int64_t max_packets, int strategy) {
    if (validate_geom(geom) != OCCGRID_OK) return 0;
    return workspace_bytes(geom, 1, max_packets, strategy);
}

size_t occgrid_agent_maps_workspace_bytes(const occgrid_geom* geom, int n_agents, int64_t max_packets, int strategy) {
    if (validate_agent_maps(geom, n_agents) != OCCGRID_OK) return 0;
    return workspace_bytes(geom, n_agents, max_packets, strategy);
}

int occgrid_workspace_reset(void* d_workspace, size_t workspace_bytes, void* stream) {
    if (!d_workspace && workspace_bytes) { set_last_error("workspace is NULL"); return OCCGRID_E_ARG; }
    OCC_CUDA_TRY(cudaMemsetAsync(d_workspace, 0, workspace_bytes, (cudaStream_t)stream));
    return OCCGRID_OK;
}

int occgrid_integrate_packets(const occgrid_geom* geom, const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                              const int32_t* d_agent_idx, const double* d_drift, const double* d_agent_off,
                              int n_agents, int8_t* d_grid, void* d_workspace, size_t workspace_bytes,
                              uint64_t* d_counters, int strategy, void* stream) {
    const PacketBatch b = {d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents};
    int rc = validate_geom(geom);
    if (rc == OCCGRID_OK) rc = check_packet_batch(b, rec_len, "");
    if (rc != OCCGRID_OK) return rc;
    if (!d_grid || !d_workspace) { set_last_error("grid/workspace is NULL"); return OCCGRID_E_ARG; }
    return integrate_packets(geom, b, Output::kGrid, d_grid, d_workspace, workspace_bytes, d_counters, strategy, stream);
}

int occgrid_integrate_packets_agent_maps(const occgrid_geom* geom, const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                                         const int32_t* d_agent_idx, const double* d_drift, const double* d_agent_off,
                                         int n_agents, int8_t* d_grids, void* d_workspace, size_t workspace_bytes,
                                         uint64_t* d_counters, int strategy, void* stream) {
    const PacketBatch b = {d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents};
    int rc = validate_agent_maps(geom, n_agents);
    if (rc == OCCGRID_OK) rc = check_packet_batch(b, rec_len, "");
    if (rc != OCCGRID_OK) return rc;
    if (!d_grids || !d_workspace) { set_last_error("grids/workspace is NULL"); return OCCGRID_E_ARG; }
    return integrate_packets(geom, b, Output::kAgentMaps, d_grids, d_workspace, workspace_bytes, d_counters, strategy, stream);
}

int occgrid_accumulate_packets(const occgrid_geom* geom, const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                               const int32_t* d_agent_idx, const double* d_drift, const double* d_agent_off,
                               int n_agents, int32_t* d_counts, void* d_workspace, size_t workspace_bytes,
                               uint64_t* d_counters, int strategy, void* stream) {
    const PacketBatch b = {d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents};
    int rc = validate_geom(geom);
    if (rc == OCCGRID_OK) rc = check_packet_batch(b, rec_len, "");
    if (rc != OCCGRID_OK) return rc;
    if (!d_counts || (reinterpret_cast<uintptr_t>(d_counts) & 7) || !d_workspace) { set_last_error("counts (8-byte aligned) / workspace is NULL"); return OCCGRID_E_ARG; }
    return integrate_packets(geom, b, Output::kCounts, d_counts, d_workspace, workspace_bytes, d_counters, strategy, stream);
}

int occgrid_counts_to_logodds(const int32_t* d_counts, int64_t n_cells, double l_occ, double l_free, double l_min, double l_max,
                              float* d_logodds, void* stream) {
    if (!d_counts || !d_logodds || n_cells < 0 || !(l_min <= l_max)) { set_last_error("occgrid_counts_to_logodds: bad arguments"); return OCCGRID_E_ARG; }
    if (n_cells == 0) return OCCGRID_OK;
    cudaStream_t st = (cudaStream_t)stream;
    long long blocks = (n_cells + kThreads - 1) / kThreads;
    if (blocks > device_sm_count() * 16) blocks = device_sm_count() * 16;
    ProfileScope ps(K_RESOLVE, st);
    k_counts_to_logodds<<<(unsigned int)blocks, kThreads, 0, st>>>(d_counts, n_cells, l_occ, l_free, l_min, l_max, d_logodds);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

int occgrid_integrate_poses(const occgrid_geom* geom, const void* d_pose_recs, int64_t n, int ordinals_in_records,
                            int8_t* d_grid, void* d_workspace, size_t workspace_bytes, uint64_t* d_counters, int strategy,
                            void* stream) {
    int rc = validate_geom(geom);
    if (rc != OCCGRID_OK) return rc;
    if (n < 0 || n > (1ll << 29) - 1) { set_last_error("n=%lld outside 0..2^29-1 records per call", (long long)n); return OCCGRID_E_ARG; }
    if (!d_grid || !d_workspace) { set_last_error("grid/workspace is NULL"); return OCCGRID_E_ARG; }
    if (n == 0) return OCCGRID_OK;
    if (!d_pose_recs || (reinterpret_cast<uintptr_t>(d_pose_recs) & 15)) { set_last_error("pose records must be non-NULL and 16-byte aligned"); return OCCGRID_E_ARG; }
    int s;
    rc = pick_strategy(geom, 1, strategy, &s);
    if (rc != OCCGRID_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (s == OCCGRID_STRATEGY_TILED) {
        PacketBatch b = {};
        b.n = n;
        return integrate_tiled(geom, b, reinterpret_cast<const PoseRec*>(d_pose_recs), ordinals_in_records, Output::kGrid, d_grid,
                               d_workspace, workspace_bytes, d_counters, st);
    }
    if (workspace_bytes < global_workspace_bytes(geom, 1)) {
        set_last_error("workspace %zu B < %zu B needed by GLOBAL_ATOMIC", workspace_bytes, global_workspace_bytes(geom, 1));
        return OCCGRID_E_WORKSPACE;
    }
    unsigned int* stamps = reinterpret_cast<unsigned int*>(d_workspace);
    const long long blocks = (n + kThreads - 1) / kThreads;
    {
        ProfileScope ps(K_INTEGRATE_GLOBAL, st);
        k_integrate_poses_global<<<(unsigned int)blocks, kThreads, 0, st>>>(to_geom(geom), reinterpret_cast<const PoseRec*>(d_pose_recs),
                                                                            n, ordinals_in_records, stamps, d_counters);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return launch_resolve(geom, stamps, d_grid, st);
}

int occgrid_update_rays(const occgrid_geom* geom, const double* d_rays, const uint8_t* d_hit, int64_t n,
                        int8_t* d_grid, void* d_workspace, size_t workspace_bytes, uint64_t* d_counters,
                        int strategy, void* stream) {
    (void)strategy;   // explicit rays always use the stamp plane
    int rc = validate_geom(geom);
    if (rc != OCCGRID_OK) return rc;
    if (n < 0 || n > (1ll << 31) - 2) { set_last_error("n=%lld outside 0..2^31-2 rays per call", (long long)n); return OCCGRID_E_ARG; }
    if (!d_grid || !d_workspace) { set_last_error("grid/workspace is NULL"); return OCCGRID_E_ARG; }
    if (n == 0) return OCCGRID_OK;
    if (!d_rays || !d_hit) { set_last_error("rays/hit is NULL"); return OCCGRID_E_ARG; }
    if (reinterpret_cast<uintptr_t>(d_rays) & 15) { set_last_error("rays must be 16-byte aligned"); return OCCGRID_E_ARG; }
    if (workspace_bytes < global_workspace_bytes(geom, 1)) {
        set_last_error("workspace %zu B < %zu B needed by update_rays", workspace_bytes, global_workspace_bytes(geom, 1));
        return OCCGRID_E_WORKSPACE;
    }
    unsigned int* stamps = reinterpret_cast<unsigned int*>(d_workspace);
    cudaStream_t st = (cudaStream_t)stream;
    const long long blocks = (n + kThreads - 1) / kThreads;
    {
        ProfileScope ps(K_UPDATE_RAYS, st);
        k_update_rays_global<<<(unsigned int)blocks, kThreads, 0, st>>>(to_geom(geom), d_rays, d_hit, n, stamps, d_counters);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return launch_resolve(geom, stamps, d_grid, st);
}

int occgrid_set_raycast_ctas_per_sm(int cap) {
    set_raycast_cta_cap(cap);
    return OCCGRID_OK;
}

int occgrid_profile_begin(void) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    for (auto& v : g_prof.ev) { for (auto e : v) cudaEventDestroy(e); v.clear(); }
    for (auto& k : g_prof.kernels) k = 0;
    g_prof.on = true;
    return OCCGRID_OK;
}

int occgrid_profile_end(double* ms_by_kernel, int64_t* launches_by_kernel, int n_slots) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.on = false;
    int rc = OCCGRID_OK;
    for (int k = 0; k < K_N_KERNELS; ++k) {
        double ms = 0.0;
        auto& v = g_prof.ev[k];
        for (size_t i = 0; i + 1 < v.size(); i += 2) {
            float t = 0.f;
            if (cudaEventSynchronize(v[i + 1]) != cudaSuccess || cudaEventElapsedTime(&t, v[i], v[i + 1]) != cudaSuccess) rc = OCCGRID_E_CUDA;
            ms += t;
        }
        if (k < n_slots) {
            if (ms_by_kernel) ms_by_kernel[k] = ms;
            if (launches_by_kernel) launches_by_kernel[k] = (int64_t)g_prof.kernels[k];
        }
        for (auto e : v) cudaEventDestroy(e);
        v.clear();
    }
    if (rc != OCCGRID_OK) set_last_error("profile_end: event query failed");
    return rc;
}

int occgrid_scatter_probe(int kind, void* d_plane, int64_t plane_cells, int64_t n_ops, uint32_t seed, void* stream) {
    if (!d_plane || plane_cells <= 0 || n_ops <= 0) { set_last_error("probe: bad arguments"); return OCCGRID_E_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    const int iters = kind == 6 ? 4096 : 64;       // kind 6: long runs, so that the tile set-up does not dilute the rate
    long long threads = (n_ops + iters - 1) / iters;
    long long blocks = (threads + kThreads - 1) / kThreads;
    if (blocks < 1) blocks = 1;
    if (blocks > 0x7fffffffll) { set_last_error("probe: n_ops too large"); return OCCGRID_E_ARG; }
    switch (kind) {
        case 0:
            k_probe_global_atomic<<<(unsigned int)blocks, kThreads, 0, st>>>((unsigned int*)d_plane, (unsigned long long)plane_cells, iters, seed);
            break;
        case 1:
            k_probe_global_store8<<<(unsigned int)blocks, kThreads, 0, st>>>((uint8_t*)d_plane, (unsigned long long)plane_cells, iters, seed);
            break;
        case 2:
        case 3:
        case 6: {
            if (plane_cells > 56 * 1024) { set_last_error("probe: smem tile limited to 56Ki words"); return OCCGRID_E_ARG; }
            const size_t smem = (size_t)plane_cells * 4;
            if (kind != 3) {
                OCC_CUDA_TRY(cudaFuncSetAttribute(k_probe_smem<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_probe_smem<true><<<(unsigned int)blocks, kThreads, smem, st>>>((unsigned int*)d_plane, (unsigned int)plane_cells, iters, seed);
            } else {
                OCC_CUDA_TRY(cudaFuncSetAttribute(k_probe_smem<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_probe_smem<false><<<(unsigned int)blocks, kThreads, smem, st>>>((unsigned int*)d_plane, (unsigned int)plane_cells, iters, seed);
            }
            break;
        }
        case 4:
            k_probe_hot_add<false><<<(unsigned int)blocks, kThreads, 0, st>>>((unsigned int*)d_plane, (unsigned long long)plane_cells, iters, seed);
            break;
        case 5:
            k_probe_hot_add<true><<<(unsigned int)blocks, kThreads, 0, st>>>((unsigned int*)d_plane, (unsigned long long)plane_cells, iters, seed);
            break;
        default:
            set_last_error("probe: unknown kind %d", kind);
            return OCCGRID_E_ARG;
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
