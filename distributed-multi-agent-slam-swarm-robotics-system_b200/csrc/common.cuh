// Shared host-side helpers of the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/occgrid_b200.h"
#include "beam_expand.cuh"
#include "block_ops.cuh"

namespace occ {

void set_last_error(const char* fmt, ...);
bool cuda_ok(cudaError_t e, const char* what);

#define OCC_CUDA_TRY(call)                                  \
    do {                                                    \
        if (!occ::cuda_ok((call), #call)) return OCCGRID_E_CUDA; \
    } while (0)

inline Geom to_geom(const occgrid_geom* g) {
    Geom o;
    o.ox = g->ox; o.oy = g->oy; o.res = g->res; o.inv_res = 1.0 / g->res;
    o.size_x = g->size_x; o.size_y = g->size_y;
    o.win_x0 = g->win_x0; o.win_y0 = g->win_y0; o.win_w = g->win_w; o.win_h = g->win_h;
    return o;
}

int validate_geom(const occgrid_geom* g);

// SM count of the CURRENT device (cached per device ordinal; 148 on a B200).
int device_sm_count();

// A decoded, pose-corrected packet (struct occgrid_pose_rec in the public header): what the
// TILED strategy bins, and what travels between GPUs after routing.
struct __align__(16) PoseRec {       // 48 bytes
    double rx, ry;                   // corrected pose (dual_bot_mapper.py:851-857)
    float yaw;
    float d[4];                      // front, left, back, right (:882-885)
    unsigned int k;                  // ordinal of the source record in the canonical stream
    int tile;                        // home tile in the RECEIVER's window (filled by the fused router; else unused)
    unsigned int pad;
};
static_assert(sizeof(PoseRec) == 48, "PoseRec must be 48 bytes");

// Optional per-kernel timing (occgrid_profile_begin/_end): when enabled, every launch of one
// of our kernels is bracketed by cudaEventRecord on its stream, so bench.py can report the
// dominant kernel's own duration and the exact number of launches.
enum KernelId { K_INTEGRATE_GLOBAL = 0, K_RESOLVE, K_UPDATE_RAYS, K_TILE_COUNT, K_TILE_SCAN, K_TILE_SCATTER,
                K_TILE_RAYCAST, K_TILE_RESOLVE, K_MERGE_EXTRACT, K_MERGE_BOUNDS, K_MERGE_VOXEL, K_MERGE_RASTER,
                K_MERGE_FUSE, K_PROBE, K_ROUTE, K_FRONTIER, K_FRONTIER_CLUSTER, K_CHAIN_PROBE, K_CHAIN_INCR,
                K_CHAIN_REBUILD, K_ICP, K_BAND_BARRIER, K_RENDER, K_MERGE_SCAN, K_MERGE_WARP_FUSE, K_FRONTIER_ASSIGN,
                K_ICP_BATCH, K_N_KERNELS };
bool profile_enabled();
void profile_mark(int kernel_id, cudaStream_t st, bool begin, int n_kernels);

struct ProfileScope {
    int id; cudaStream_t st; bool on; int nk;
    ProfileScope(int id_, cudaStream_t st_, int n_kernels = 1) : id(id_), st(st_), on(profile_enabled()), nk(n_kernels) {
        if (on) profile_mark(id, st, true, nk);
    }
    ~ProfileScope() { if (on) profile_mark(id, st, false, nk); }
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- packet batches -------------------------------------------------------------------------------
constexpr int kMaxRecStride = 64;            // bytes per packet record slot staged in shared memory

// One batch of wire records as the packet entry points receive it (include/occgrid_b200.h).
struct PacketBatch {
    const uint8_t* pkts; int64_t n; int stride;
    const int32_t* agent_idx; const double* drift; const double* agent_off; int n_agents;
};

// What a packet batch is integrated into: one int8 grid, a stack of n_agents grids (agent a's at
// a - 1), or the int32 {miss, hit} count planes of one grid.
enum class Output { kGrid, kAgentMaps, kCounts };

// The record checks every packet entry point shares: n in 0..2^29-1, rec_len 42 or 41, stride in
// rec_len..kMaxRecStride, n_agents >= 1 with an agent offset table, packets non-NULL when n > 0.
// `who` prefixes the error message.
int check_packet_batch(const PacketBatch& b, int rec_len, const char* who);

// Cooperative copy of a CTA's records into shared memory with 16-byte loads.
__device__ __forceinline__ void stage_records(const uint8_t* __restrict__ src, size_t bytes, uint8_t* smem) {
    const size_t nvec = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) ? bytes / 16 : 0;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(smem);
    for (size_t i = threadIdx.x; i < nvec; i += blockDim.x) d4[i] = __ldg(s4 + i);
    for (size_t i = nvec * 16 + threadIdx.x; i < bytes; i += blockDim.x) smem[i] = __ldg(src + i);
}

// ---- tiles of the TILED strategy (occgrid_tiled.cu) ------------------------------------------------
constexpr int kTile = 64;            // home-tile side in cells
constexpr int kTileShift = 6;

// Cells a beam can reach from the robot cell: R = ceil(MAX_DIST_M / res) + 2 (:57, :900).
__host__ __device__ __forceinline__ int reach_cells(double res) { return (int)ceil(OCC_MAX_DIST_M / res) + 2; }

struct TileGeom {
    int reach;            // R
    int pad;              // cells added around the window so that every home tile is >= 0
    int tiles_x, tiles_y, n_tiles;
    int win_side;         // smem window side = kTile + 2R
    int pitch;            // smem row pitch (odd)
};

inline TileGeom tile_geom(double res, int win_w, int win_h) {
    TileGeom t;
    t.reach = reach_cells(res);
    t.pad = ((t.reach + kTile - 1) / kTile) * kTile;
    t.tiles_x = (win_w + 2 * t.pad + kTile - 1) >> kTileShift;
    t.tiles_y = (win_h + 2 * t.pad + kTile - 1) >> kTileShift;
    t.n_tiles = t.tiles_x * t.tiles_y;
    t.win_side = kTile + 2 * t.reach;
    t.pitch = t.win_side | 1;
    return t;
}
inline TileGeom tile_geom(const occgrid_geom* g) { return tile_geom(g->res, g->win_w, g->win_h); }

// ---- band exchange (multi-GPU row bands, SURVEY §8e) -----------------------------------------
// Records of a batch arrive in per-source segments of a receive slot: segment s occupies record
// addresses [s * seg_cap, s * seg_cap + count[s]).  count[] lives on the device (written by the
// sources before the cross-GPU barrier) — the host never reads it.
constexpr int kSegChunk = 2048;              // seg_cap is a multiple of this: a chunk never straddles two segments
constexpr int kRouteItemPk = 512;            // packets per route sub-batch of the fused kernel (two per thread)
constexpr int kRouteSubsPerItem = 2;         // sub-batches per route work item
constexpr int kMaxBands = 32;

struct SegInfo {
    int n_segs;
    unsigned int seg_cap;
    const unsigned int* d_counts;            // [n_segs] or NULL: one segment of host_count records
    unsigned int host_count;
};

// One batch to decode and push to the band owners, executed by the persistent raycast CTAs in
// between their raycast work items (occgrid_tiled.cu: k_home_raycast<kCounts, true>).
struct RouteJob {
    const uint8_t* pkts; long long n; int stride;
    const int32_t* agent_idx; const double* drift; const double* agent_off; int n_agents;
    unsigned int ordinal_base;
    double ox, oy, res, inv_res;             // global grid geometry
    int size_x;                              // bands are full-width rows: window x0 = 0, w = size_x
    int reach, pad, tiles_x;                 // tile geometry of a band window (the same for every band)
    int n_bands, src_rank;
    int band_y0[kMaxBands + 1];
    PoseRec* const* peer_recs;               // device array [n_bands]: band owner's receive slot (its segment 0)
    int* const* peer_tiles;                  // device array [n_bands]: the slot's compact tile ids (same addressing)
    unsigned int seg_cap;
    unsigned int* resv;                      // LOCAL reservation counters [n_bands]; zero when the batch starts
    int* status;                             // bit 1: a segment overflowed
    uint64_t* counters;                      // optional: packets / accepted / dropped / bad_pose of the routed share
    unsigned int n_route_items;              // work items of kRouteItemPk * kRouteSubs packets
};

// TILED entry points.  n_maps: grids the call writes (n_agents for Output::kAgentMaps, else 1);
// their tile keys, map * n_tiles + tile, must stay below 2^24.
bool tiled_supported(const occgrid_geom* geom, int n_maps);
size_t tiled_workspace_bytes(const occgrid_geom* geom, int n_maps, int64_t max_packets);
// Integrates a packet batch, or (d_poses != NULL) batch.n decoded pose records, into d_out.
int integrate_tiled(const occgrid_geom* geom, const PacketBatch& batch, const PoseRec* d_poses, int ordinals_in_records, Output kind,
                    void* d_out, void* d_ws, size_t ws_bytes, uint64_t* d_counters, cudaStream_t st);
void set_raycast_cta_cap(int cap);
size_t tiled_band_workspace_bytes(const occgrid_geom* geom, int n_segs, int64_t seg_cap);
int tiled_prepare_poses(const occgrid_geom* geom, const PoseRec* d_recs, const int* d_tiles, const SegInfo& seg, int tiles_in_records,
                        void* d_ws, size_t ws_bytes, uint64_t* d_counters, cudaStream_t st);
int tiled_raycast_route(const occgrid_geom* geom, const PoseRec* d_recs, int have_items, const RouteJob* job,
                        int8_t* d_grid, void* d_ws, size_t ws_bytes, int64_t max_records, uint64_t* d_counters, cudaStream_t st,
                        cudaEvent_t after_fused = nullptr);

// Block-wide accumulation of the first N uint64 counter slots: per-thread values -> warp
// shuffle -> per-warp partials in shared memory -> one global atomic per slot per CTA.
// All threads must call.  smem_acc needs N * 32 entries.
template <int N>
__device__ __forceinline__ void block_add_counters(const unsigned long long (&v)[N],
                                                   unsigned long long* smem_acc /* >= N * 32 */, uint64_t* d_counters) {
    if (d_counters == nullptr) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        unsigned long long x = v[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) smem_acc[i * 32 + warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        unsigned long long t = 0;
        for (int w = 0; w < nwarps; ++w) t += smem_acc[threadIdx.x * 32 + w];
        if (t) atomicAdd(reinterpret_cast<unsigned long long*>(d_counters) + threadIdx.x, t);
    }
}

}  // namespace occ
