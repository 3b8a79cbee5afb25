/*
 * occgrid_b200 — C ABI of the B200-native occupancy-grid integration and map-fusion engine.
 *
 * This is the drop-in boundary for the ONE hot path of
 * deevinandu/Distributed-Multi-Agent-SLAM-Swarm-Robotics-System (SURVEY.md §8):
 *
 *   QuasarPacket batch -> pose correction -> 4 beams -> integer Bresenham -> int8 grid scatter
 *       (server_nodes/dual_bot_mapper.py:41-46, 826-903, 110-179)
 *   agent grids -> occupied-cell extraction -> rigid transform -> voxel fuse -> rasterise
 *       (server_nodes/map_merger.py:35-127)
 *
 * The reference is pure Python and has no FFI of its own; the entry points below are what a
 * ctypes binding in dual_bot_mapper.py / map_merger.py would call (INTEGRATION.md shows the
 * stub).  Conventions:
 *   - plain pointers and sizes only; every `d_` pointer is DEVICE memory owned by the caller
 *     (torch in our Python host layer); the library allocates nothing and keeps no global
 *     state except a thread-local last-error string;
 *   - every call is asynchronous on the given CUDA stream (`stream` is a cudaStream_t passed
 *     as void*; NULL = the legacy default stream);
 *   - return value 0 = ok, <0 = error (see occgrid_last_error()).  Malformed packets are
 *     counted and skipped, never fatal (dual_bot_mapper.py:838-843 `continue`s);
 *   - one host thread per stream (the reference path is single-threaded: :797, map_merger.py:132).
 */
#ifndef OCCGRID_B200_H
#define OCCGRID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCCGRID_ABI_VERSION 2

/* Cell values — dual_bot_mapper.py:92-94 (same convention as nav_msgs/OccupancyGrid.data). */
#define OCCGRID_CELL_UNKNOWN  (-1)
#define OCCGRID_CELL_FREE       0
#define OCCGRID_CELL_OCCUPIED 100

/* Wire format — dual_bot_mapper.py:41-46; firmware struct AgentFirmware_Bot1.ino:172-185.
 * '<4sBfffiIffffB': magic@0 'QSRL', agent_id u8@4, x f32@5, y f32@9, yaw f32@13,
 * encoder i32@17, v2v u32@21, front/left/back/right f32@25/29/33/37 (metres), landmark u8@41. */
#define OCCGRID_PACKET_SIZE    42
#define OCCGRID_PACKET_SIZE_V1 41

/* Error codes */
#define OCCGRID_OK             0
#define OCCGRID_E_ARG        (-1)   /* bad argument (null pointer, size, alignment)            */
#define OCCGRID_E_WORKSPACE  (-2)   /* workspace too small for this call                        */
#define OCCGRID_E_CUDA       (-3)   /* a CUDA runtime call failed; see occgrid_last_error()      */
#define OCCGRID_E_RANGE      (-4)   /* geometry outside supported range (ray longer than limit)  */

/* Integration strategies (both hand-written sm_100a kernels; results are identical). */
#define OCCGRID_STRATEGY_AUTO          (-1)
#define OCCGRID_STRATEGY_GLOBAL_ATOMIC   0  /* per-cell atomicMax on a global order-stamp plane     */
#define OCCGRID_STRATEGY_TILED           1  /* beams binned by tile; order stamps resolved in smem  */

/* Grid geometry.  Mirrors OccupancyGrid.__init__ (dual_bot_mapper.py:113-119) plus a window:
 * `d_grid` holds rows [win_y0, win_y0+win_h) x columns [win_x0, win_x0+win_w) of the global
 * size_y x size_x grid, row-major ([gy][gx], :150), row stride win_w.  The reference case
 * is win = whole grid; a spatial tile of a multi-GPU map uses a proper sub-window.  Cells
 * are clipped one by one (:149,:155), never geometrically. */
typedef struct occgrid_geom {
    double  ox, oy;          /* world coordinates of the lower-left corner of cell (0,0) */
    double  res;             /* metres per cell                                          */
    int32_t size_x, size_y;  /* global grid extent in cells                              */
    int32_t win_x0, win_y0;  /* window origin in global cells                            */
    int32_t win_w, win_h;    /* window extent in cells                                   */
} occgrid_geom;

/* A decoded, pose-corrected packet: 48 bytes, 16-byte aligned. */
typedef struct occgrid_pose_rec {
    double   rx, ry;      /* pose after `+ agent offset` (:851-852) and `+ drift` (:855-857) */
    float    yaw;         /* wire field, unchanged                                            */
    float    d[4];        /* front, left, back, right ranges in metres (:882-885)            */
    uint32_t k;           /* ordinal of the source record in the canonical stream            */
    int32_t  tile;        /* home tile in the receiver's window (set by the fused router)    */
    uint32_t pad;
} occgrid_pose_rec;

/* Counter slots (uint64 each, device memory, accumulated with atomics; caller zeroes). */
enum {
    OCCGRID_C_PACKETS = 0,   /* records seen                                              */
    OCCGRID_C_ACCEPTED,      /* passed magic/agent filter and pose is finite               */
    OCCGRID_C_DROPPED,       /* bad magic or agent id outside 1..n_agents (:840-843)       */
    OCCGRID_C_BAD_POSE,      /* NaN/Inf pose: skipped (the reference would crash, :123)     */
    OCCGRID_C_BEAMS,         /* beams expanded (4 per accepted packet)                     */
    OCCGRID_C_HITS,          /* beams with MIN_DIST < d <= MAX_DIST (:888)                 */
    OCCGRID_C_UPDATES,       /* beam-cell updates = sum of max(|dx|,|dy|)+1 (SURVEY §8d)   */
    OCCGRID_C_SLOWPATH,      /* beams re-evaluated with double-double sin/cos               */
    OCCGRID_C_OWNED_UPDATES, /* updates of beams whose start cell lies in this window       */
    OCCGRID_C_RECORDS,       /* (tile, beam) records binned by the tiled strategy           */
    OCCGRID_N_COUNTERS = 16
};

int         occgrid_abi_version(void);
const char* occgrid_last_error(void);

/* Bytes of device workspace occgrid_integrate_packets / occgrid_update_rays need for up to
 * `max_packets` records per call under `strategy`.  0 on error. */
size_t occgrid_workspace_bytes(const occgrid_geom* geom, int64_t max_packets, int strategy);

/* Zero the workspace (once after allocation, and after any failed call). */
int occgrid_workspace_reset(void* d_workspace, size_t workspace_bytes, void* stream);

/*
 * Batched replacement of the per-packet loop body, dual_bot_mapper.py:826-903:
 * for each record in buffer order: decode (:828-838), filter (:840-843), pose correction
 * (:851-857), and for front,left,back,right (:882-886): hit test (:888), endpoint
 * (:890-891 | :900-902), OccupancyGrid.update_ray (:136-156) with last-writer-wins in
 * record order, then sensor order.
 *
 *   d_packets    n records `stride` bytes apart (stride >= rec_len); 16-byte aligned base
 *   rec_len      42 (v2) or 41 (v1, no landmark byte) — the landmark is not read on this path
 *   d_agent_idx  NULL, or int32[n]: out-of-band agent index replacing the wire byte
 *                (extension for > 255 agents)
 *   d_drift      NULL, or double[n][2]: SLAM drift (cdx, cdy) in force when record k arrived
 *                (:855-857; produced sequentially by PoseGraphSLAM on the host, :908-914)
 *   d_agent_off  double[n_agents+1][2]: start offset of agent a at [a]; ids 1..n_agents are
 *                accepted.  Reference mode: n_agents = 2, {(0,0),(0,0),(separation,0)} (:851-852)
 *   d_grid       int8 window (see occgrid_geom), updated in place
 *   d_counters   NULL or uint64[OCCGRID_N_COUNTERS]
 */
int occgrid_integrate_packets(const occgrid_geom* geom,
                              const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                              const int32_t* d_agent_idx, const double* d_drift,
                              const double* d_agent_off, int n_agents,
                              int8_t* d_grid,
                              void* d_workspace, size_t workspace_bytes,
                              uint64_t* d_counters, int strategy, void* stream);

/*
 * Per-agent maps (EXTENSION): the same batch integrated into a stack of n_agents grids, one per
 * agent, the input map_merger.py's MapMerger fuses (/agent_{id}/map).  Grid a - 1 of the stack
 * ends equal to occgrid_integrate_packets run over only the records whose agent (wire byte, or
 * d_agent_idx[k]) is a, in buffer order: decode, filter, offsets, drift, beams, per-cell clipping
 * and last-writer-wins are unchanged, and records of different agents never interact.  The
 * counters equal those of occgrid_integrate_packets on the same batch, geometry and strategy.
 *
 *   geom     shared by every map; the window must be the whole grid
 *   d_grids  int8 [n_agents][size_y][size_x], agent a at index a - 1, updated in place
 *   other arguments as occgrid_integrate_packets
 * AUTO picks TILED when the geometry supports it and n_agents * (tiles of the grid) <= 2^24, else
 * GLOBAL_ATOMIC.  The workspace holds n_agents stamp planes (0 bytes on error).
 */
size_t occgrid_agent_maps_workspace_bytes(const occgrid_geom* geom, int n_agents, int64_t max_packets, int strategy);
int occgrid_integrate_packets_agent_maps(const occgrid_geom* geom,
                                         const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                                         const int32_t* d_agent_idx, const double* d_drift,
                                         const double* d_agent_off, int n_agents,
                                         int8_t* d_grids,
                                         void* d_workspace, size_t workspace_bytes,
                                         uint64_t* d_counters, int strategy, void* stream);

/*
 * Batched OccupancyGrid.update_ray (dual_bot_mapper.py:136-156) on explicit world-space rays:
 * d_rays = double[n][4] (robot_x, robot_y, hit_x, hit_y), d_hit = uint8[n] (hit_valid),
 * applied in index order with last-writer-wins.
 */
int occgrid_update_rays(const occgrid_geom* geom,
                        const double* d_rays, const uint8_t* d_hit, int64_t n,
                        int8_t* d_grid,
                        void* d_workspace, size_t workspace_bytes,
                        uint64_t* d_counters, int strategy, void* stream);

/*
 * Scatter-roofline microkernels (SURVEY §8d): `n_ops` operations to uniformly random cells.
 *   kind 0: atomicMax(u32) on a global plane of `plane_cells` words   (red.global.max.u32)
 *   kind 1: plain 1-byte stores to a global plane of `plane_cells` bytes
 *   kind 2: atomicMax(u32) on a per-CTA shared-memory tile of `plane_cells` words
 *   kind 3: plain 4-byte stores to a per-CTA shared-memory tile
 *   kind 4: atomicAdd without return (red.global.add) spread over only `plane_cells` HOT words,
 *           one per 256 B (plane must hold plane_cells*64 words) — contended-address rate
 *   kind 5: as 4 but using the returned value (atom.global.add)
 * Used by bench.py to put a measured ceiling beside the integrate kernels.
 */
int occgrid_scatter_probe(int kind, void* d_plane, int64_t plane_cells, int64_t n_ops,
                          uint32_t seed, void* stream);

/*
 * Multi-GPU routing (SURVEY §8e): the global grid is cut into `n_bands` row bands
 * (band b = rows [band_y0[b], band_y0[b+1]), host array of n_bands+1 boundaries).  Every
 * accepted record is decoded (:828-857) and written as an occgrid_pose_rec, in stable order, to
 * the segment of `d_send` of each band its rays can reach (robot row +- ceil(MAX_DIST_M/res)+2
 * cells); d_band_counts[b] receives the segment lengths (segments are laid out in band order).
 * d_status bit 0 = send buffer too small (nothing written).  The caller then exchanges the
 * segments (NCCL all-to-all) and feeds what it receives to occgrid_integrate_poses with its own
 * window.
 */
size_t occgrid_route_workspace_bytes(int64_t n, int n_bands);
int occgrid_route_packets(const occgrid_geom* geom, int n_bands, const int32_t* band_y0_host,
                          const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                          const int32_t* d_agent_idx, const double* d_drift,
                          const double* d_agent_off, int n_agents,
                          void* d_send /* occgrid_pose_rec[send_capacity] */,
                          int64_t send_capacity, int64_t* d_band_counts, int32_t* d_status,
                          uint64_t* d_counters, void* d_ws, size_t ws_bytes, void* stream);

/* Integrate n decoded records (occgrid_pose_rec, 16-byte aligned) in index order: the second half
 * of occgrid_integrate_packets (beam expansion :881-903 + update_ray :136-156) for input whose
 * decode/filter/pose correction (:826-857) already happened — on another GPU, in the router. */
int occgrid_integrate_poses(const occgrid_geom* geom, const void* d_pose_recs, int64_t n,
                            int ordinals_in_records /* 0: order = index; 1: order = rec.k */,
                            int8_t* d_grid, void* d_workspace, size_t workspace_bytes,
                            uint64_t* d_counters, int strategy, void* stream);

/* ---- Multi-GPU row-band step: fused raycast + route over NVLink peer memory (SURVEY §8e) ------
 *
 * One GPU per row band of the global grid.  Every rank ingests ITS share of the packet stream
 * (the reference's ingest loop, dual_bot_mapper.py:816-843, once per server socket); a record has
 * to reach the owner of every band its rays can touch (robot row +- ceil(MAX_DIST_M/res)+2).
 * Receive buffers live in peer-mapped memory: each rank owns, per slot (2 slots), `n_bands`
 * per-SOURCE segments of `seg_capacity` occgrid_pose_rec (a multiple of 2048), the same number of
 * int32 tile ids (a compact copy of rec.tile, so that binning reads 4 bytes per record) plus uint32
 * seg_counts[n_bands]; a source reserves slots in ITS segment with a local atomic, so no remote
 * atomics and no counts exchange are needed.  One step on every rank, all stream-ordered:
 *
 *   occgrid_band_prepare(slot j-1)          bin the records that arrived during the last step
 *   occgrid_band_raycast_route(slot j-1, job -> peers' slot j)
 *                                           ONE persistent kernel: raycast batch j-1 and, between
 *                                           its work items, decode batch j and store the records
 *                                           straight into the band owners' segments (compute and
 *                                           NVLink traffic overlap); then stamps -> int8 band
 *   occgrid_band_publish(slot j, epoch j+1) seg_counts to the owners + cross-GPU barrier
 *
 * Records carry rec.k = ordinal_base + index (canonical stream = rank 0's share, then rank 1's,
 * ...; last writer wins exactly as on one GPU) and rec.tile = home tile in the owner's window.
 * d_status bits: 2 = a segment overflowed (records dropped), 4 = the barrier timed out. */
typedef struct occgrid_route_job {
    const uint8_t* d_packets;      /* this rank's share of the NEXT batch: n records, `stride` apart */
    int64_t        n;
    int32_t        stride, rec_len;
    const int32_t* d_agent_idx;    /* optional, as in occgrid_integrate_packets                      */
    const double*  d_drift;        /* optional [n][2]                                                */
    const double*  d_agent_off;    /* [n_agents + 1][2]                                              */
    int32_t        n_agents;
    uint32_t       ordinal_base;   /* ordinal of record 0 in the canonical stream                    */
    double         ox, oy, res;    /* GLOBAL grid geometry                                           */
    int32_t        size_x;         /* global width in cells (bands are full rows)                    */
    int32_t        n_bands, src_rank;
    int32_t        band_y0[33];    /* band b = rows [band_y0[b], band_y0[b+1])                       */
    void* const*   d_peer_recs;    /* DEVICE array [n_bands]: owner b's receive slot (segment 0)     */
    int32_t* const* d_peer_tiles;  /* DEVICE array [n_bands]: owner b's tile ids of that slot        */
    int64_t        seg_capacity;
    uint32_t*      d_resv;         /* LOCAL uint32[n_bands], zero before the batch's first item      */
    int32_t*       d_status;
    uint64_t*      d_counters;     /* optional: packets/accepted/dropped/bad_pose of this share      */
} occgrid_route_job;

size_t occgrid_band_workspace_bytes(const occgrid_geom* band_geom, int n_segs, int64_t seg_capacity);
int occgrid_band_prepare(const occgrid_geom* band_geom /* window = my band */, const void* d_recv_slot,
                         const int32_t* d_recv_tiles /* int32[n_segs * seg_capacity] of the slot, or NULL: read rec.tile */, int n_segs,
                         int64_t seg_capacity, const uint32_t* d_seg_counts, void* d_workspace,
                         size_t workspace_bytes, uint64_t* d_counters, void* stream);
int occgrid_band_raycast_route(const occgrid_geom* band_geom, const void* d_recv_slot, int n_segs,
                               int64_t seg_capacity, int have_prepared /* 0: nothing to raycast yet */,
                               const occgrid_route_job* job /* NULL: nothing to route */, int8_t* d_grid,
                               void* d_workspace, size_t workspace_bytes, uint64_t* d_counters, void* stream);
/* Everything a rank's steps share (all DEVICE pointers; [2] = the two receive slots). */
typedef struct occgrid_band_ctx {
    occgrid_geom     band_geom;            /* window = my band                                        */
    int32_t          n_bands, rank;
    int64_t          seg_capacity;
    void*            d_recv[2];            /* my receive slots: occgrid_pose_rec[n_bands][seg_capacity] */
    int32_t*         d_recv_tiles[2];      /* int32[n_bands][seg_capacity]                             */
    uint32_t*        d_seg_counts[2];      /* uint32[n_bands]                                          */
    void* const*     d_peer_recs[2];       /* device arrays [n_bands] of the owners' slot pointers     */
    int32_t* const*  d_peer_tiles[2];
    uint32_t* const* d_peer_seg_counts[2];
    uint32_t* const* d_peer_flags;
    const uint32_t*  d_my_flags;
    uint32_t*        d_resv;
    int32_t*         d_status;
    int8_t*          d_grid;
    void*            d_workspace;
    size_t           workspace_bytes;
    uint64_t*        d_counters;
    void*            ev_fused;             /* library-owned (created on first use with a side stream); start as NULL */
    void*            ev_published;
    int32_t          published_pending;    /* start as 0 */
} occgrid_band_ctx;

/* prepare (when a batch is pending) + raycast_route + publish (when `job` != NULL; job->n may be 0)
 * for step `step_index` (slot = step_index & 1, epoch = step_index + 1) in one host call; the job's
 * n_bands / src_rank / seg_capacity / peer pointers / d_resv / d_status are taken from `ctx`.
 * `side_stream` != NULL: publish + barrier run there, right after the fused kernel and concurrently
 * with the resolve pass on `stream`; the next step (or occgrid_band_join) waits for them. */
int occgrid_band_step(occgrid_band_ctx* ctx, int64_t step_index, int have_pending,
                      const occgrid_route_job* job /* NULL: flush only */, int wait, void* stream, void* side_stream);
int occgrid_band_join(occgrid_band_ctx* ctx, void* stream);

int occgrid_band_publish(int n_bands, int rank, uint32_t* d_resv, int64_t seg_capacity,
                         uint32_t* const* d_peer_seg_counts /* DEVICE array: owner b's seg_counts of the slot */,
                         uint32_t* const* d_peer_flags /* DEVICE array: owner b's uint32 flags[n_bands] */,
                         const uint32_t* d_my_flags, uint32_t epoch, int wait /* 0: publish only */,
                         int32_t* d_status, void* stream);

/* Occupancy overlay of the reference's dashboard as a headless RGB image (SURVEY §8 row f4):
 * MapRenderer._draw_occupancy (dual_bot_mapper.py:492-527) with world_to_screen (:404-408): the
 * `width` x `height` image (uint8 [height][width][3], device) is filled with `bg_rgb` and every
 * visible cell of the WHOLE grid `d_grid` (size_y x size_x) that is neither UNKNOWN nor OCCUPIED is
 * painted `fg_rgb` (CELL_COLOR_FREE) as a cell_px = max(1, int(res * scale)) square centred on its
 * screen position (a single pixel when cell_px == 2; nothing when cell_px < 2).  `scale` = pixels
 * per metre, `offset_x/_y` = screen position of the world origin (y flipped). */
int occgrid_render_overlay(const int8_t* d_grid, int32_t size_x, int32_t size_y, double ox, double oy, double res,
                           double scale, double offset_x, double offset_y, int32_t width, int32_t height,
                           const uint8_t* bg_rgb_host, const uint8_t* fg_rgb_host, uint8_t* d_rgb, void* stream);

/* ------------------------------------------------------------------------------------------
 *  Map fusion — server_nodes/map_merger.py:35-127
 *
 *  A point cloud is two fp64 device arrays x[], y[] (z == 0 on this path) of `capacity`
 *  elements and a DEVICE-resident int64 count, so a merge sequence runs stream-ordered with
 *  no host round trip.  `d_status` is a sticky device int32: bit 0 = point capacity exceeded,
 *  bit 1 = voxel lattice capacity exceeded (the offending call becomes a no-op; the host
 *  wrapper checks the word at its next synchronisation and raises).
 *  The rigid transform replaces Open3D ICP (:45-56), which is outside this path (SURVEY §8 a13).
 * ---------------------------------------------------------------------------------------- */

/* grid_to_pcd (:64-85) fused with PointCloud::Transform (:58): scan an int8 occupancy grid
 * (row-major, height x width), keep cells with value > 50 (:72), emit the cell-corner
 * coordinates x = col*res + origin_x, y = row*res + origin_y (:76-77) in row-major (argwhere)
 * order, apply the 4x4 row-major transform `T_host` (HOST pointer; NULL = identity), and
 * append to the cloud at [*d_count, ...) (= `global_pcd += local_pcd`, :59).
 * *d_last_appended (optional) receives the number of points of this grid. */
/* *d_out += number of cells with value > 50 (:72) — lets a batched merge size its cloud once. */
int mapmerge_count_occupied(const int8_t* d_grid, int64_t n_cells, int64_t* d_out, void* stream);

size_t mapmerge_extract_workspace_bytes(int64_t n_cells);
int mapmerge_extract_transform(const int8_t* d_grid, int32_t width, int32_t height, double res,
                               double origin_x, double origin_y, const double* T_host,
                               double* d_px, double* d_py, int64_t capacity,
                               int64_t* d_count, int64_t* d_last_appended, int32_t* d_status,
                               void* d_ws, size_t ws_bytes, void* stream);

/* Batched form of mapmerge_extract_transform for one merge() of A same-sized grids, in two
 * passes over all grids at once (blockIdx.y = agent).  d_grids is a DEVICE array of A grid
 * pointers.  _count: d_agent_total[a] = occupied cells of grid a (the caller reads them to size
 * the cloud and to find the first non-empty grid, which is adopted untransformed, :40-43).
 * _write: T_host (HOST, [A][16] row-major or NULL) and use_host (HOST, [A] or NULL: 0 = skip the
 * agent) describe the callbacks; the transformed points land in d_px/d_py agent after agent and
 * d_agent_offset[a] = start of agent a's slice (d_agent_offset[A] = total).  d_xforms is scratch
 * (A * 96 bytes); the workspace must be the one _count filled, untouched: it carries the block
 * counts and one occupancy bit per cell, so _write does not read the grids again.  The sequential chain appends
 * slice a with mapmerge_append_slice when callback a's turn comes (:59).
 * Argument errors of the older merge entry points (this one, mapmerge_count_occupied,
 * mapmerge_append_slice, mapmerge_bounds, mapmerge_voxel_downsample, mapmerge_chain_*,
 * mapmerge_rasterise, mapmerge_fuse_max) return OCCGRID_E_ARG before anything is launched, with the
 * message key word in quotes: a "NULL pointer", "n_agents" outside 1..65 535, "width x height"
 * below 1, a "res" or "voxel" that is not > 0 (NaN included), a negative "n_cells" / "n", an
 * "agent" out of range, "dims" out of range, "n_order" outside 0..n_agents, "n_callbacks" < 0, a
 * "capacity" below 1 (voxel filter) or above dims[2] (chain), an "order entry" out of range.  A
 * workspace below its *_workspace_bytes returns OCCGRID_E_WORKSPACE ("workspace"). */
size_t mapmerge_extract_batch_workspace_bytes(int64_t n_cells, int n_agents);
int mapmerge_extract_batch_count(const int8_t* const* d_grids, int n_agents, int32_t width, int32_t height,
                                 int64_t* d_agent_total, void* d_ws, size_t ws_bytes,
                                 int grids_bulk_ok /* 1: every grid pointer is 16-byte aligned -> the scan runs on
                                                      cp.async.bulk + mbarrier staged shared memory (TMA) */,
                                 void* stream);
int mapmerge_extract_batch_write(const int8_t* const* d_grids, int n_agents, int32_t width, int32_t height,
                                 double res, const double* d_origins, const double* T_host,
                                 const uint8_t* use_host, void* d_xforms,
                                 double* d_px, double* d_py, int64_t capacity,
                                 const int64_t* d_agent_total, int64_t* d_agent_offset, int32_t* d_status,
                                 void* d_ws, size_t ws_bytes, void* stream);
int mapmerge_append_slice(const double* d_sx, const double* d_sy, const int64_t* d_agent_offset,
                          int agent, double* d_px, double* d_py, int64_t capacity,
                          int64_t* d_count, int32_t* d_status, uint64_t* d_bounds_enc, void* stream);

/* Bounds carried on the device across the callbacks of a batched merge (no min/max pass, no host
 * read): d_bounds_enc = uint64[4], order-preserving encodings of {min_x, min_y, max_x, max_y} of
 * the current cloud.  _reset empties it; mapmerge_append_slice widens it by the appended points;
 * mapmerge_voxel_downsample (when given it instead of d_bounds) consumes it as the bounds of its
 * input and leaves the bounds of its output in it. */
int mapmerge_bounds_enc_reset(uint64_t* d_bounds_enc, void* stream);

/* GetMinBound/GetMaxBound of a cloud, also publish_global_map's bbox (:95-98):
 * d_bounds = {min_x, min_y, max_x, max_y}. */
size_t mapmerge_bounds_workspace_bytes(void);
int mapmerge_bounds(const double* d_px, const double* d_py, const int64_t* d_count,
                    double* d_bounds, void* d_ws, size_t ws_bytes, void* stream);

/* PointCloud::VoxelDownSample(voxel) (:60): voxel_min_bound = min_bound - 0.5*voxel, index =
 * floor((p - voxel_min_bound)/voxel), one output point per non-empty voxel = mean of its
 * points (summed in ascending point index), emitted in order of first appearance (by smallest
 * point index).  O(points): the lattice planes in the workspace are a lookup table that must be
 * ZERO on entry (zero the workspace once) and is zero again on exit.
 * `d_bounds` must hold the bounds of the input cloud; the lattice of this call must fit
 * `lattice_capacity_cells`.  Output arrays must not alias the input. */
size_t mapmerge_voxel_workspace_bytes(int64_t lattice_capacity_cells, int64_t point_capacity);
int mapmerge_voxel_downsample(const double* d_px, const double* d_py, const int64_t* d_count,
                              int64_t point_capacity, double voxel, const double* d_bounds,
                              uint64_t* d_bounds_enc /* NULL: use d_bounds */,
                              int64_t lattice_capacity_cells,
                              double* d_out_px, double* d_out_py, int64_t* d_out_count,
                              int32_t* d_status, void* d_ws, size_t ws_bytes, void* stream);

/* Incremental form of the callback chain `global_pcd += local; global_pcd =
 * global_pcd.voxel_down_sample(v)` (map_merger.py:58-60) over the slices of a batched extraction.
 * A filtered cloud holds one point per voxel, so while the lattice anchor (min_bound - v/2) is
 * bitwise unchanged a callback only touches the voxels its slice falls into: the chain keeps a
 * voxel -> cloud-index map, re-averages the touched voxels in place and appends the new voxels in
 * order of first appearance (three kernels over the slice).  A callback whose anchor moved, or
 * whose means left their voxels, needs the full filter (_rebuild).  Results are bitwise those of
 * mapmerge_append_slice + mapmerge_voxel_downsample per callback.
 *   dims (host) = {lattice_w, lattice_h, point_capacity, slice_capacity}: a lattice that covers
 *   every cloud of the chain, the largest cloud, the largest slice.
 *   order_host[n_order]: the agents (slice indices) to merge, in callback order.
 *   _init      d_chain must be all-zero; takes the bounds of every slice and of the adopted cloud.
 *   _run       enqueues n_callbacks incremental callbacks; each takes the next agent from a device
 *              cursor; once a callback needs the host, it and all later ones are no-ops.
 *   _poll      synchronises; state_out = {cursor, stalled}: stalled 0 = running, 1 = callback
 *              order[cursor] needs _rebuild, 2 = lattice does not fit dims (status word set),
 *              3 = the cloud's min corner may have moved inwards: call _rebounds, then go on.
 *   _rebuild   appends slice `agent`, filters the whole cloud into (d_out_*), rebuilds the map and
 *              advances the cursor (the caller swaps the clouds, as after
 *              mapmerge_voxel_downsample).  d_voxel_ws: a mapmerge_voxel_downsample workspace with
 *              lattice capacity >= lattice_w * lattice_h and point capacity dims[2]. */
size_t mapmerge_chain_workspace_bytes(const int64_t* dims, int n_agents);
int mapmerge_chain_init(void* d_chain, size_t chain_bytes, const int64_t* dims, int n_agents,
                        const double* d_sx, const double* d_sy, const int64_t* d_agent_offset,
                        const int32_t* order_host, int n_order, const double* d_px, const double* d_py,
                        const int64_t* d_count, void* stream);
int mapmerge_chain_run(void* d_chain, const int64_t* dims, int n_agents, int n_order, int n_callbacks,
                       const double* d_sx, const double* d_sy, const int64_t* d_agent_offset,
                       double voxel, double* d_px, double* d_py, int64_t capacity, int64_t* d_count,
                       int32_t* d_status, void* stream);
int mapmerge_chain_poll(void* d_chain, const int64_t* dims, int n_agents, int32_t* state_out,
                        void* stream);
int mapmerge_chain_rebounds(void* d_chain, const int64_t* dims, int n_agents, const double* d_px,
                            const double* d_py, const int64_t* d_count, void* stream);
int mapmerge_chain_rebuild(void* d_chain, const int64_t* dims, int n_agents, const double* d_sx,
                           const double* d_sy, const int64_t* d_agent_offset, int agent, double voxel,
                           double* d_px, double* d_py, int64_t capacity, int64_t* d_count,
                           double* d_out_px, double* d_out_py, int64_t* d_out_count,
                           int32_t* d_status, void* d_voxel_ws, size_t voxel_ws_bytes,
                           int64_t lattice_capacity_cells, void* stream);

/* registration_icp(local, global, max_correspondence_distance, identity,
 * TransformationEstimationPointToPoint(), ICPConvergenceCriteria(max_iteration)) as called at
 * map_merger.py:45-52 (Open3D, absent and un-pinned here: follows its published algorithm, see
 * oracle/icp_oracle.py).  Source = local cloud (n_source points), target = global cloud
 * (n_target points), both planar fp64 device arrays.  The target is binned into a uniform cell
 * list: cells of size `cell` (use max_correspondence_distance / 4) starting at (min_x, min_y),
 * cells_w x cells_h of them covering the target's bounds.  Exact nearest neighbours (squared
 * distance < max^2, ties by lowest target index), rigid fit in closed form, sums reduced in a
 * fixed order.  Runs stream-ordered without host round trips: the iteration loop is one
 * cooperative kernel (the device must support cooperative launch).
 * d_result (20 doubles): [0..15] transformation row-major, [16] fitness, [17] inlier_rmse,
 * [18] iterations run (-1: the loop kernel was aborted by a grid-barrier time-out),
 * [19] number of correspondences of the last evaluation. */
size_t mapmerge_icp_workspace_bytes(int64_t target_points, int64_t source_points, int32_t cells_w,
                                    int32_t cells_h);
int mapmerge_icp_register(const double* d_sx, const double* d_sy, int64_t n_source,
                          const double* d_tx, const double* d_ty, int64_t n_target, double min_x,
                          double min_y, double cell, int32_t cells_w, int32_t cells_h,
                          double max_correspondence_distance, int32_t max_iteration,
                          double relative_fitness, double relative_rmse, double* d_result,
                          void* d_ws, size_t ws_bytes, void* stream);

/* EXTENSION (no reference counterpart): batched map registration (DESIGN §6f).  Refines A
 * agent->global transforms against ONE reference cloud in one stream-ordered call.
 * Inputs:
 *   d_sx, d_sy: the A source clouds back to back, agent a's points at [d_offsets[a], d_offsets[a + 1]);
 *     d_offsets int64 [n_agents + 1] on the device, d_offsets[0] = 0, non-decreasing.  The
 *     Python layer passes every agent's occupied cells (> 50) at cell corners transformed by its
 *     prior, in row-major order: what mapmerge_extract_batch_count / mapmerge_extract_batch_write
 *     produce.
 *   d_tx, d_ty: the reference cloud of n_target points (1 <= n_target < 2^32 - 1), binned into the
 *     cell list of mapmerge_icp_register: cells of size `cell` from (min_x, min_y), cells_w x cells_h.
 *   max_correspondence_distance (the threshold), max_iteration, relative_fitness, relative_rmse:
 *     as mapmerge_icp_register.
 * Per agent a, row d_results[a][0..19] has the layout of mapmerge_icp_register's d_result and
 * equals, bit for bit, mapmerge_icp_register(source_a, reference, the same cell list and
 * parameters): the 16 doubles of the refinement U_a, fitness, inlier_rmse, iterations and
 * correspondences, with the same iteration count and convergence step.  An agent with no points
 * gets an identity U_a, fitness 0, RMSE 0, iterations 0 and 0 correspondences and is never
 * launched (the single call rejects n_source <= 0; this is the batched call's own rule).
 * Iterations -1: a grid barrier of the loop kernel timed out before the agent finished.
 * Iterations -2 in every row (identity, zeros otherwise): the offset table is not valid, or its
 * d_offsets[n_agents] points do not fit the workspace.
 * The cell list is built once; the loops of all agents run in one cooperative launch of
 * k_icp_loop_batch (a converged agent is skipped in later rounds); the result does not depend on
 * the grid size.  No host round trip, no atomics in the sums.
 * Workspace: mapmerge_icp_register_batch_workspace_bytes(n_target, total_source_points, n_agents,
 * cells_w, cells_h), regions aligned to 256 bytes: three cell tables of (cells + 1) * 4 bytes, the
 * sorted target (n_target * (8 + 8 + 4)), the scan's block sums ((ceil(cells / 16384) + 1) * 4),
 * 328 bytes of state per agent, (n_agents + 1) * 4 of block offsets and 256 of barrier words; then
 * per point 8 + 8 + 4 bytes of working copy and per virtual block (ceil(points / 256) + n_agents of
 * them) 48 + 16 + 4 bytes.  The call holds as many points as ws_bytes allows.
 * OCCGRID_E_ARG (message key word in quotes) for a "NULL pointer", "n_agents" outside 1..65 535,
 * "n_target" outside 1..2^32 - 2, a "cell" or "threshold" that is not finite and > 0,
 * "max_iteration" below 0, "cells" below 1 and a cell list that "overflows size_t" (the workspace
 * query also rejects "total_source_points" outside 0..2^39 and returns 0 for every argument
 * error); OCCGRID_E_WORKSPACE for ws_bytes below the workspace of zero points. */
size_t mapmerge_icp_register_batch_workspace_bytes(int64_t n_target, int64_t total_source_points,
                                                   int n_agents, int32_t cells_w, int32_t cells_h);
int mapmerge_icp_register_batch(const double* d_sx, const double* d_sy, const int64_t* d_offsets,
                                int n_agents, const double* d_tx, const double* d_ty, int64_t n_target,
                                double min_x, double min_y, double cell, int32_t cells_w,
                                int32_t cells_h, double max_correspondence_distance,
                                int32_t max_iteration, double relative_fitness, double relative_rmse,
                                double* d_results /* [n_agents][20] */, void* d_ws, size_t ws_bytes,
                                void* stream);
/* Testing and tuning knob: cap the CTAs of k_icp_loop_batch (0 = every resident CTA, the default).
 * Results do not depend on it.  Process-wide; OCCGRID_E_ARG for ctas < 0. */
int mapmerge_icp_batch_set_max_ctas(int ctas);

/* publish_global_map's rasterisation (:103-111): fill width x height with -1, then
 * grid[int((y-min_y)/res)][int((x-min_x)/res)] = 100 with index clipping (:108-109).
 * width/height follow :100-101 and are computed by the caller from the bounds. */
int mapmerge_rasterise(const double* d_px, const double* d_py, const int64_t* d_count, double res,
                       const double* d_bounds, int32_t width, int32_t height,
                       int8_t* d_grid_out, void* stream);

/* dst = max(dst, src) element-wise on int8 grids ({-1,100}: occupied wins) — the local half
 * of the multi-GPU fuse; the cross-GPU half is an NCCL max-reduction on int8. */
int mapmerge_fuse_max(int8_t* d_dst, const int8_t* d_src, int64_t n, void* stream);

/* EXTENSION (no reference counterpart): fused occupancy map.  Resamples every map of a stack
 * d_maps int8 [n_agents][height][width] (row-major [gy][gx], agent a's origin origins_host[a] =
 * (ox_a, oy_a), resolution res for all) into one target grid d_out int8 [out_h][out_w] with origin
 * (out_ox, out_oy) and resolution out_res, and keeps free space: out = max(-1, max over the agents
 * covering a cell of their cell value), so with -1/0/100 maps occupied beats free beats unknown and
 * the result does not depend on agent order.  Every target cell is written (-1 where no agent
 * covers it); the previous contents do not matter.
 *   T_host [n_agents][16]: agent->global 4x4 row-major, R = T[0:2,0:2], t = (T[0][3], T[1][3]), each
 *   applied as given (nothing is adopted).  Rejected unless every entry is finite and every entry of
 *   R^T R - I is within 1e-9; the inverse used is R^T.
 * Coefficients (host fp64, each operation rounded on its own, as bracketed):
 *   bx = (out_ox + 0.5*g) - tx        by = (out_oy + 0.5*g) - ty        (g = out_res, r = res)
 *   c0 = (R00*g)/r   c1 = (R10*g)/r   c2 = ((R00*bx + R10*by) - ox_a)/r
 *   c3 = (R01*g)/r   c4 = (R11*g)/r   c5 = ((R01*bx + R11*by) - oy_a)/r
 * Per target cell, column j and row i (device fp64, no contraction):
 *   u = (c0*j) + ((c1*i) + c2)        v = (c3*j) + ((c4*i) + c5)
 *   agent a covers the cell iff 0 <= u < width and 0 <= v < height (NaN never covers), and then
 *   contributes map_a[(int)v][(int)u].
 * An identity transform into a target of the maps' geometry returns the map bit for bit.
 * n_agents 1..65535; the stack and the target may exceed 2^31 bytes.  OCCGRID_E_ARG for NULL
 * pointers, n_agents or a size out of range, a resolution that is not finite and > 0, a stack whose
 * size overflows size_t and a non-finite or non-rigid transform; OCCGRID_E_WORKSPACE for d_ws
 * smaller than mapmerge_warp_fuse_workspace_bytes (64 bytes per agent, which returns 0 for
 * n_agents or a target size out of range).  Stream-ordered: no atomics and no host
 * synchronisation; the per-agent coefficients are copied into d_ws with cudaMemcpyAsync. */
size_t mapmerge_warp_fuse_workspace_bytes(int n_agents, int32_t out_w, int32_t out_h);
int mapmerge_warp_fuse(const int8_t* d_maps, int n_agents, int32_t width, int32_t height, double res,
                       const double* origins_host /* [A][2] */, const double* T_host /* [A][16] */,
                       double out_ox, double out_oy, double out_res, int32_t out_w, int32_t out_h,
                       int8_t* d_out, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 *  Frontier detection and clustering (SURVEY §8 row f1) — dual_bot_mapper.py:181-237, :948-956
 * ---------------------------------------------------------------------------------------- */

/* OccupancyGrid.get_frontiers (:181-197) on a full height x width int8 grid: interior FREE cells
 * with an UNKNOWN 4-neighbour, written as (x, y) int32 pairs in row-major scan order.
 * *d_count receives the number found; d_status bit 0 = more than `capacity`. */
size_t occgrid_frontier_workspace_bytes(int64_t n_cells, int64_t max_frontiers);
int occgrid_frontiers(const int8_t* d_grid, int32_t width, int32_t height, int32_t* d_xy,
                      int64_t capacity, int64_t* d_count, int32_t* d_status,
                      void* d_ws, size_t ws_bytes, void* stream);

/* cluster_frontiers (:199-231) + cluster_centroid_world (:233-237) on the list produced above:
 * 4-connected components; d_label[i] = list index of the first cell of i's component; clusters
 * with at least `min_cluster` cells (FRONTIER_MIN_CLUSTER = 3, :102) are emitted in order of
 * their first cell: d_cluster_root (list index), d_cluster_size, d_centroids (world x, y).
 * Workspace: occgrid_frontier_workspace_bytes. */
int occgrid_frontier_clusters(const int32_t* d_xy, const int64_t* d_count, int64_t capacity,
                              int32_t width, int32_t min_cluster, double ox, double oy, double res,
                              int32_t* d_label, int32_t* d_cluster_root, int32_t* d_cluster_size,
                              double* d_centroids, int64_t* d_n_clusters,
                              void* d_ws, size_t ws_bytes, void* stream);

/* EXTENSION (no reference counterpart; the reference's assignment is commented out,
 * dual_bot_mapper.py:958-996): frontier assignment by geodesic distance (DESIGN §6e).
 * Inputs:
 *   a grid int8 [H][W] (-1 / 0 / 100, [gy][gx]), origin (ox, oy) and resolution res;
 *   robot positions in world metres, d_robot_xy double [A][2], 1 <= A <= 65 535;
 *   the frontier clusters as occgrid_frontier_clusters leaves them on the device: the xy list,
 *   d_count, d_label, d_cluster_root, d_centroids and d_n_clusters (cluster membership is read
 *   from the labels and the ascending root list, so min_cluster is the one the clusters used).
 * Rules:
 *   Robot cell: the reference's world_to_grid, int((w - o) / res) with true fp64 division and
 *     truncation.  A robot whose cell lies outside the grid, or whose position is not finite, has
 *     no source: its row of costs is all -1 and it gets no target.
 *   Geodesic distance: D_a(c) is the 4-connected, unit-cost BFS distance from robot a's cell.  The
 *     source gets 0 whatever its value; the search moves only into FREE (0) cells.  Unreachable
 *     cells are -1; values are int32.  D is the unique fixed point of
 *     D(c) = min(seed(c), c FREE ? min over 4-neighbours n of D(n) + 1 : unreachable),
 *     so any correct relaxation order gives the same field bit for bit.
 *   Cost: cost[a][k] = min over the cells c of cluster k of D_a(c), or -1 when none is reachable;
 *     the goal cell attains it, ties to the lowest linear index y*W + x.  Clusters are numbered in
 *     frontier_centroids() order.
 *   Assignment: a greedy pass in robot order.  For a = 0..A-1, robot a takes the unclaimed
 *     cluster with the smallest non-negative cost[a][k], ties to the lowest k, and claims it.  A
 *     robot left with no reachable unclaimed cluster gets -1.
 * Outputs (device): d_cluster int32 [A], d_cost int32 [A], d_goal int32 [A][2] (x, y), d_target
 * double [A][2] (the assigned cluster's centroid copied from d_centroids, NaN when none; cluster,
 * cost and goal are -1 then) and d_costs int32 [A][max_clusters], of which columns
 * 0..n_clusters-1 are written.  d_stats (optional, int64 [3]) receives the worklist rounds, the
 * (robot, tile) items processed and the pool slots used.
 * Fields are stored per (robot, 64 x 64 tile) in a pool of tile_pool slots of 16 KB inside d_ws.
 * d_status bits are OR-ed in (zero it first):
 *   OCCGRID_ASSIGN_POOL_FULL      the tile pool (or the worklist, which holds tile_pool items) ran
 *                                 out; nothing is written outside the workspace and the outputs
 *                                 are all "no target".  Grow tile_pool and call again.
 *   OCCGRID_ASSIGN_TIMEOUT        a grid barrier of the worklist kernel timed out (an error).
 *   OCCGRID_ASSIGN_CLUSTERS_FULL  n_clusters > max_clusters; the outputs are all "no target".
 * OCCGRID_E_ARG (message key word in quotes) for a "NULL pointer", "n_robots" outside 1..65 535,
 * "width x height" below 3 or a grid of 2^31 - 1 cells or more, a "resolution" that is not finite
 * and > 0, a "capacity" (max_clusters, tile_pool) outside 1..2^31 - 1 and a workspace that
 * "overflows size_t" (the [A][n_tiles] slot tables); OCCGRID_E_WORKSPACE for ws_bytes below
 * occgrid_frontier_assign_workspace_bytes (which returns 0 for the same argument errors).
 * Stream-ordered: the robots are read on the device, and the worklist runs as one cooperative
 * launch with no host round trip.
 * d_grid may be a navigation grid from occgrid_inflate of the grid the clusters came from; the costs
 * are then path lengths over its FREE cells. */
#define OCCGRID_ASSIGN_POOL_FULL     1
#define OCCGRID_ASSIGN_TIMEOUT       2
#define OCCGRID_ASSIGN_CLUSTERS_FULL 4
size_t occgrid_frontier_assign_workspace_bytes(int32_t width, int32_t height, int32_t n_robots,
                                               int32_t max_clusters, int64_t tile_pool);
int occgrid_frontier_assign(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy,
                            double res, const double* d_robot_xy, int32_t n_robots,
                            const int32_t* d_xy, const int64_t* d_count, const int32_t* d_label,
                            const int32_t* d_cluster_root, const double* d_centroids,
                            const int64_t* d_n_clusters, int32_t max_clusters, int64_t tile_pool,
                            int32_t* d_cluster, int32_t* d_cost, int32_t* d_goal, double* d_target,
                            int32_t* d_costs, int32_t* d_status, int64_t* d_stats,
                            void* d_ws, size_t ws_bytes, void* stream);

/* One robot's dense geodesic field d_field int32 [H][W] (the D_a above, -1 where unreachable),
 * for navigation (descend the field to the goal).  The same worklist run for the one robot at
 * d_robot_xy double [2], then its tiles expanded.  Workspace:
 * occgrid_frontier_assign_workspace_bytes(width, height, 1, 1, tile_pool).  Status bits, stats and
 * argument errors as occgrid_frontier_assign; d_field is not written when the pool ran out. */
int occgrid_geodesic_field(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy,
                           double res, const double* d_robot_xy, int64_t tile_pool, int32_t* d_field,
                           int32_t* d_status, int64_t* d_stats, void* d_ws, size_t ws_bytes, void* stream);

/* EXTENSION (no reference counterpart): obstacle clearance (DESIGN §6g).
 * occgrid_distance_field: the exact squared Euclidean distance transform of a grid int8 [H][W]
 * ([gy][gx]), 1 <= W, H <= 32 768.  Obstacles are the cells > 50 (the occupied rule of grid_to_pcd).
 * d_d2 int32 [H][W] receives d2[y][x] = min over obstacles (x', y') of (x - x')^2 + (y - y')^2, the
 * squared distance between cell centres in cells (0 on obstacles, at most 2 * 32 767^2, which fits
 * int32), or -1 in every cell when the grid has no obstacle.  Integer arithmetic, no atomics: the
 * result depends on the input alone.
 * occgrid_inflate: the navigation grid of a robot radius.  d_out int8 [H][W] (must not overlap
 * d_grid) is OCCUPIED (100) where grid[c] == 0 (FREE), 0 <= d2[c] <= max_d2 and c lies in no robot's
 * footprint, else grid[c].  Robot a's footprint is the cells (x, y) with (x - rx)^2 + (y - ry)^2 <=
 * max_d2 around its cell (rx, ry) = (int((x_a - ox) / res), int((y_a - oy) / res)) (fp64 division,
 * truncation, as occgrid_frontier_assign); a robot outside the grid or at a non-finite position has no
 * footprint.  d_robot_xy double [A][2] world metres, 0 <= A <= 65 535 (NULL allowed when A == 0).  The
 * footprint lets a robot that stands closer than its radius to a wall leave it.  The EDT is computed
 * in the workspace.
 * Both take one workspace of occgrid_distance_field_workspace_bytes(W, H) bytes; with
 * n_bands = ceil(H / 32) and a(v) = v rounded up to a multiple of 256 it is exactly
 *   a(4 W n_bands) + a(8 W n_bands) + a(4 W H) + a(8 W H)
 * (band masks, band links, the inflation's d2, the envelope stacks).
 * OCCGRID_E_ARG (message key word in quotes) for a "NULL pointer" (d_robot_xy too when A > 0), a
 * "width x height" side outside 1..32 768, "max_d2" < 0, "n_robots" outside 0..65 535 and a
 * "resolution" that is not finite and > 0; OCCGRID_E_WORKSPACE for a short workspace (the query
 * returns 0 for a bad side).  Stream-ordered, no host synchronisation. */
size_t occgrid_distance_field_workspace_bytes(int32_t width, int32_t height);
int occgrid_distance_field(const int8_t* d_grid, int32_t width, int32_t height,
                           int32_t* d_d2, void* d_ws, size_t ws_bytes, void* stream);
int occgrid_inflate(const int8_t* d_grid, int32_t width, int32_t height, double ox, double oy, double res,
                    int64_t max_d2, const double* d_robot_xy /* [A][2] or NULL when A == 0 */, int32_t n_robots,
                    int8_t* d_out, void* d_ws, size_t ws_bytes, void* stream);

/* EXTENSION (no reference counterpart): correlative map alignment (DESIGN §6h).  For every agent map,
 * the rotation x translation in a window around its prior that best overlays the reference's
 * obstacles, exactly the winner of the exhaustive search, in one stream-ordered call.  Its transform
 * is the prior for mapmerge_icp_register_batch when the prior is too far off for ICP.
 * Inputs:
 *   d_grids int8 [A][H][W] on the device (W = width, H = height); origins_host [A][2] = (ox_a, oy_a)
 *     and one resolution r = res for all.
 *   priors_host [A][16]: agent->global, 4x4 row-major.  Rejected unless every entry is finite and
 *     |R^T R - I| <= 1e-9, the rule of mapmerge_warp_fuse.
 *   The reference as its squared distance field d_d2 int32 [Hr][Wr] on the device (Wr = ref_w, Hr =
 *     ref_h), exactly what occgrid_distance_field writes (-1 everywhere when the grid has no
 *     obstacle), its origin (gox, goy) = (ref_ox, ref_oy) and resolution g = ref_res (g need not
 *     equal r).
 *   rot_host [n_angles][2]: the rotation table (cs_k, sn_k), each |cs^2 + sn^2 - 1| <= 1e-9.  The
 *     caller orders it by preference, entry 0 normally the identity (1, 0).
 *   max_offset = Rc, the translation half-width in reference cells, and max_d2.
 * Occupied cells: agent a's cells > 50 (the rule of grid_to_pcd, the extraction and ICP).  Cell (u, v)
 * is column u, row v.
 * Coefficients per (agent, rotation), host fp64, each operation rounded on its own as bracketed (the
 * library is built with -ffp-contract=off); p = the prior:
 *   mx = ox_a + ((0.5*W)*r)          my = oy_a + ((0.5*H)*r)            (map centre, agent frame)
 *   ex = -((p00*mx) + (p01*my))      ey = -((p10*mx) + (p11*my))        (t_p - c, where c is the centre placed by the prior)
 *   m00 = (cs*p00) - (sn*p10)        m01 = (cs*p01) - (sn*p11)
 *   m10 = (sn*p00) + (cs*p10)        m11 = (sn*p01) + (cs*p11)
 *   tx = p03 + (((cs - 1)*ex) - (sn*ey))      ty = p13 + ((sn*ex) + ((cs - 1)*ey))
 *   bx = ox_a + 0.5*r                by = oy_a + 0.5*r                  (centre of agent cell (0, 0))
 *   e0 = (m00*r)/g   e1 = (m01*r)/g   e2 = ((((m00*bx) + (m01*by)) + tx) - gox)/g
 *   e3 = (m10*r)/g   e4 = (m11*r)/g   e5 = ((((m10*bx) + (m11*by)) + ty) - goy)/g
 * Together these rotate the map about its own centre, as placed by the prior.  With (cs, sn) = (1, 0),
 * m and t are the prior's own entries, bit for bit up to the sign of a zero.
 * Per occupied cell, on the device (fp64, no contraction, __dmul_rn / __dadd_rn as in §4):
 *   X = (e0*u) + ((e1*v) + e2)       Y = (e3*u) + ((e4*v) + e5)         j = floor(X), i = floor(Y)
 *   A point with |X| or |Y| >= 2^30, or NaN, contributes 0 to every candidate.
 * Candidates: (k, dx, dy) with -Rc <= dx, dy <= Rc moves every point of rotation k to cell
 *   (j + dx, i + dy).  A point contributes w = max_d2 + 1 - d2[i+dy][j+dx] when that cell lies inside
 *   the reference and 0 <= d2 <= max_d2, and 0 otherwise.  score = the integer sum of these; with
 *   max_d2 = 0 it is the number of points that land on reference obstacles.
 * Winner: the largest score, ties to the lowest rank, where
 *   o(v) = 2v - 1 if v > 0, else -2v          rank = (k*(2Rc+1) + o(dy))*(2Rc+1) + o(dx)
 *   so candidate (0, 0, 0), the prior, wins every tie and an agent that matches nothing keeps its
 *   prior.  The key (uint64)score << 32 | (2^32 - 1 - rank) makes this a plain 64-bit integer max,
 *   independent of order.
 * Output d_out int64 [A][6]: score, k, dx, dy, prior_score (the score of (0, 0, 0)), n_points.  An agent
 *   with no occupied cells gets all zeros.  If the occupied cells do not fit the workspace, every row
 *   is -2, 0, 0, 0, 0, 0 (as mapmerge_icp_register_batch).  d_diag int64 [2] (may be NULL): the
 *   candidates searched (A' * n_angles * (2Rc+1)^2 over the A' agents with points) and the
 *   candidates scored exactly; these depend on the block size and are not part of the contract.
 * Transform of candidate (k, dx, dy): [[m00, m01, 0, tx + dx*g], [m10, m11, 0, ty + dy*g], [0, 0, 1, 0],
 *   [0, 0, 0, 1]], computed in host fp64.
 * Limits: OCCGRID_E_ARG (message key word in quotes) for a "NULL pointer" (d_diag may be NULL),
 * "n_agents" outside 1..65 535, "width x height" with a side < 1 or W*H*(max_d2+1) > 2^31 - 1 (so a
 * score fits 31 bits), a "reference size" side outside 1..32 768 (the range of
 * occgrid_distance_field), "max_d2" outside 0..254, "max_offset" (Rc) outside 0..2048, "n_angles"
 * outside 1..65 535, more than 2^32 - 1 "candidates" (n_angles*(2Rc+1)^2), a "resolution" that is not
 * finite and > 0, a "prior" that is not finite or not rigid and a "rotation" that is not a unit
 * (cs, sn) pair.  OCCGRID_E_WORKSPACE for ws_bytes below the workspace of zero points.
 * Workspace: mapmerge_align_workspace_bytes(n_agents, W, H, Wr, Hr, max_d2, Rc, n_angles,
 * total_points) returns 0 for any of the size errors above and for total_points outside
 * 0..A*W*H; otherwise, with a(v) = v rounded up to a multiple of 256, s the block size in effect
 * (mapmerge_align_set_block), cpa = ceil(W*H / 4096), nb = ceil((2Rc+1) / s)^2, pad = 2Rc + 64 and
 * np = (Wr + 2 pad)(Hr + 2 pad), it is exactly
 *   a(48 A n_angles) + a(4 A cpa) + a(8 (A + 1)) + a(4 A n_angles nb) + 3 a(8 A) + a(65 536) + 256
 *   + a(np) + a(np) + a(np) + a(8 total_points)
 * (coefficients, compaction counts, agent offsets, block bounds, best keys / prior scores / picked
 * blocks, per-CTA counts, status, the weight table Lw, its s x s maximum Ls and the row maxima, the
 * (u, v) points).  Every size is below 2^51, so nothing overflows.  The call holds as many points as
 * ws_bytes allows.
 * Stream-ordered: no host synchronisation and no atomics except the 64-bit key max; the per-(agent,
 * rotation) coefficients reach the device by cudaMemcpyAsync into the workspace. */
size_t mapmerge_align_workspace_bytes(int n_agents, int32_t width, int32_t height, int32_t ref_w, int32_t ref_h,
                                      int32_t max_d2, int32_t max_offset, int32_t n_angles, int64_t total_points);
int mapmerge_align(const int8_t* d_grids, int n_agents, int32_t width, int32_t height, double res,
                   const double* origins_host /* [A][2] */, const double* priors_host /* [A][16] */,
                   const int32_t* d_d2, int32_t ref_w, int32_t ref_h, double ref_ox, double ref_oy, double ref_res,
                   const double* rot_host /* [n_angles][2] */, int32_t n_angles, int32_t max_offset, int32_t max_d2,
                   int64_t* d_out /* [A][6] */, int64_t* d_diag /* [2] or NULL */, void* d_ws, size_t ws_bytes,
                   void* stream);
/* Testing knob: the pruning block size s (0 = the default, 8; 1..64 allowed).  Results do not depend
 * on it; the workspace does (nb above).  Process-wide; OCCGRID_E_ARG ("block") outside 0..64. */
int mapmerge_align_set_block(int s);

/* Tuning knob of the TILED strategy: cap the persistent raycast CTAs per SM (0 = as many as fit,
 * the default).  A pipelined multi-GPU ingest lowers it to 2 so that the routing kernel of the
 * next batch finds room on every SM and runs concurrently.  Process-wide. */
int occgrid_set_raycast_ctas_per_sm(int cap);

/* EXTENSION beyond the reference (north-star wording "hit/miss log-odds", SURVEY §8c): instead of
 * the last-writer-wins int8 grid, accumulate per-cell COUNTS over the same beams, cells and
 * per-cell clipping: d_counts = int32 [win_h][win_w][2] = {misses, hits}; every cell update_ray
 * (dual_bot_mapper.py:148-156) would have stored FREE to counts one miss, the OCCUPIED end cell of
 * a valid hit one hit (a missed beam's end cell counts nothing, :153).  Integer adds commute: the
 * planes are exactly np.add.at over the reference's _bresenham cells, whatever the order.
 * Arguments as occgrid_integrate_packets; the counts accumulate across calls (zero them to reset).
 * occgrid_counts_to_logodds: L = clamp(hits*l_occ + misses*l_free, l_min, l_max) as float32,
 * evaluated in fp64 from the integer planes (no float atomics: order-independent). */
int occgrid_accumulate_packets(const occgrid_geom* geom, const uint8_t* d_packets, int64_t n_records,
                               int rec_stride, int rec_len, const int32_t* d_agent_idx,
                               const double* d_drift_xy, const double* d_agent_offset_xy, int n_agents,
                               int32_t* d_counts, void* d_workspace, size_t workspace_bytes,
                               uint64_t* d_counters, int strategy, void* stream);
int occgrid_counts_to_logodds(const int32_t* d_counts, int64_t n_cells, double l_occ, double l_free,
                              double l_min, double l_max, float* d_logodds, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Host-side producer of the per-packet drift table (no GPU involved): the sequential half of
 * the ingest loop, dual_bot_mapper.py:826-857 + :908-914 with PoseGraphSLAM.add_pose /
 * _check_closure (:261-322).  For every record k of a HOST buffer, in order: drift_out[k] =
 * (cdx, cdy) in force for that packet ((0, 0) for dropped records) — the table
 * occgrid_integrate_packets takes as d_drift_xy.  State (pose count, landmarks, closures,
 * per-agent drift) lives in the handle and carries over from batch to batch.
 * rec_sizes: per-record datagram sizes (42 = v2, 41 = v1, anything else is dropped, :828-838),
 * or NULL when every record has rec_size bytes.  Bit-identical to the reference's arithmetic.
 * ------------------------------------------------------------------------------------------- */
typedef struct occgrid_slam occgrid_slam;
occgrid_slam* occgrid_slam_create(void);
void occgrid_slam_destroy(occgrid_slam* slam);
int occgrid_slam_drift_table(occgrid_slam* slam, const uint8_t* packets_host, int64_t n_records,
                             int32_t rec_stride, int32_t rec_size, const int32_t* rec_sizes,
                             double separation, double* drift_out_xy);
int occgrid_slam_counts(const occgrid_slam* slam, int64_t* n_nodes, int64_t* n_landmarks,
                        int64_t* n_closures);
/* closures in the order they were found: (landmark's node index, closing node index, correction) */
int occgrid_slam_closures(const occgrid_slam* slam, int64_t capacity, int64_t* lm_node,
                          int64_t* node, double* corr_xy, int32_t* agent);
/* PoseGraphSLAM.get_correction_for_agent (:324-332) */
int occgrid_slam_correction_for_agent(const occgrid_slam* slam, int32_t agent_id, double* out_xy);

/*
 * Measurement hook (bench.py): between _begin and _end every kernel this library launches is
 * bracketed by CUDA events on its stream.  _end synchronises those events and returns, per
 * kernel id (OCCGRID_K_*), the summed device time in ms and the number of launches.
 */
enum {
    OCCGRID_K_INTEGRATE_GLOBAL = 0, OCCGRID_K_RESOLVE, OCCGRID_K_UPDATE_RAYS, OCCGRID_K_TILE_COUNT,
    OCCGRID_K_TILE_SCAN, OCCGRID_K_TILE_SCATTER, OCCGRID_K_TILE_RAYCAST, OCCGRID_K_TILE_RESOLVE,
    OCCGRID_K_MERGE_EXTRACT, OCCGRID_K_MERGE_BOUNDS, OCCGRID_K_MERGE_VOXEL, OCCGRID_K_MERGE_RASTER,
    OCCGRID_K_MERGE_FUSE, OCCGRID_K_PROBE, OCCGRID_K_ROUTE, OCCGRID_K_FRONTIER, OCCGRID_K_FRONTIER_CLUSTER,
    OCCGRID_K_CHAIN_PROBE, OCCGRID_K_CHAIN_INCR, OCCGRID_K_CHAIN_REBUILD, OCCGRID_K_ICP,
    OCCGRID_K_N_KERNELS
};
int occgrid_profile_begin(void);
int occgrid_profile_end(double* ms_by_kernel, int64_t* launches_by_kernel, int n_slots);

#ifdef __cplusplus
}
#endif
#endif /* OCCGRID_B200_H */
