// Multi-GPU row-band step of the occupancy-grid integration (SURVEY §8e "Integration"), C ABI
// occgrid_band_* of include/occgrid_b200.h.
//
// The global grid is cut into row bands, one per GPU.  Every GPU ingests its own share of the
// QuasarPacket stream (server_nodes/dual_bot_mapper.py:816-843), and a packet's rays (<=
// MAX_DIST_M / res cells, :57, :900) can only touch rows within `reach` of its robot cell, so a
// decoded record has to reach one band owner (two next to a band edge).  One step is
//
//   occgrid_band_prepare        count -> plan -> scatter of the batch that ARRIVED last step
//                               (per-source segments of a receive slot, fill counts on the device)
//   occgrid_band_raycast_route  ONE persistent kernel: raycasts that batch (shared-memory stamp
//                               windows, occgrid_tiled.cu) and, in between its work items, decodes
//                               the NEXT batch and stores the 48-byte records straight into the
//                               band owners' receive buffers over NVLink peer memory — compute and
//                               exchange overlap item by item, nothing is staged, no all-to-all
//   occgrid_band_publish        tells every owner how many records this rank sent it, then a
//                               cross-GPU barrier (release/acquire flags in peer memory)
//
// all stream-ordered, no host read-back anywhere.  Last-writer-wins stays exact because every
// record carries its ordinal in the canonical stream ("rank 0's share, then rank 1's, ...").
#include "common.cuh"

namespace occ {

constexpr unsigned long long kBandBarrierTimeoutNs = 10000000000ull;      // 10 s: a peer died; give up instead of hanging

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Thread b talks to band owner b: seg_counts[b][rank] = what I reserved in my segment there, my
// reservation counter goes back to zero, then flag[b][rank] = epoch with release semantics (every
// record store of the preceding kernels on this stream happens-before it).  With `wait` the thread
// then spins until owner b's flag for THIS rank's buffers shows the same epoch.
__global__ void k_band_publish(int n_bands, int rank, unsigned int* __restrict__ resv, unsigned int seg_cap,
                               unsigned int* const* __restrict__ peer_seg_counts, unsigned int* const* __restrict__ peer_flags,
                               const unsigned int* __restrict__ my_flags, unsigned int epoch, int wait, int* __restrict__ status) {
    const int b = threadIdx.x;
    if (b >= n_bands) return;
    unsigned int n = resv[b];
    if (n > seg_cap) n = seg_cap;
    resv[b] = 0u;
    peer_seg_counts[b][rank] = n;
    __threadfence_system();
    st_release_sys(peer_flags[b] + rank, epoch);
    if (!wait) return;
    const unsigned long long t0 = global_ns();
    unsigned int spins = 0;
    while ((int)(ld_acquire_sys(my_flags + b) - epoch) < 0) {
        if (((++spins) & 255u) == 0u && global_ns() - t0 > kBandBarrierTimeoutNs) { atomicOr(status, 4); return; }
    }
}

}  // namespace occ

using namespace occ;

// event occgrid_band_step wants recorded between the fused kernel and the resolve (per host thread)
static thread_local cudaEvent_t g_after_fused = nullptr;

extern "C" {

size_t occgrid_band_workspace_bytes(const occgrid_geom* band_geom, int n_segs, int64_t seg_capacity) {
    if (validate_geom(band_geom) != OCCGRID_OK) return 0;
    if (n_segs < 1 || n_segs > kMaxBands || seg_capacity < kSegChunk || seg_capacity % kSegChunk ||
        (int64_t)n_segs * seg_capacity >= (1ll << 32)) {
        set_last_error("band: need 1..32 segments of a multiple of %d records, < 2^32 addresses in total", kSegChunk);
        return 0;
    }
    return tiled_band_workspace_bytes(band_geom, n_segs, seg_capacity);
}

int occgrid_band_prepare(const occgrid_geom* band_geom, const void* d_recv_slot, const int32_t* d_recv_tiles, int n_segs, int64_t seg_capacity,
                         const uint32_t* d_seg_counts, void* d_workspace, size_t workspace_bytes, uint64_t* d_counters,
                         void* stream) {
    int rc = validate_geom(band_geom);
    if (rc != OCCGRID_OK) return rc;
    if (!d_recv_slot || (reinterpret_cast<uintptr_t>(d_recv_slot) & 15) || !d_seg_counts || !d_workspace) {
        set_last_error("band_prepare: NULL / misaligned argument");
        return OCCGRID_E_ARG;
    }
    if (occgrid_band_workspace_bytes(band_geom, n_segs, seg_capacity) == 0) return OCCGRID_E_ARG;
    SegInfo seg;
    seg.n_segs = n_segs; seg.seg_cap = (unsigned int)seg_capacity; seg.d_counts = d_seg_counts; seg.host_count = 0;
    return tiled_prepare_poses(band_geom, reinterpret_cast<const PoseRec*>(d_recv_slot), d_recv_tiles, seg, 1, d_workspace, workspace_bytes,
                               d_counters, (cudaStream_t)stream);
}

int occgrid_band_raycast_route(const occgrid_geom* band_geom, const void* d_recv_slot, int n_segs, int64_t seg_capacity,
                               int have_prepared, const occgrid_route_job* job, int8_t* d_grid, void* d_workspace,
                               size_t workspace_bytes, uint64_t* d_counters, void* stream) {
    int rc = validate_geom(band_geom);
    if (rc != OCCGRID_OK) return rc;
    if (!d_grid || !d_workspace || (have_prepared && !d_recv_slot)) { set_last_error("band_raycast_route: NULL argument"); return OCCGRID_E_ARG; }
    if (occgrid_band_workspace_bytes(band_geom, n_segs, seg_capacity) == 0) return OCCGRID_E_ARG;
    RouteJob J = {};
    if (job && job->n > 0) {
        const PacketBatch batch = {job->d_packets, job->n, job->stride, job->d_agent_idx, job->d_drift, job->d_agent_off, job->n_agents};
        rc = check_packet_batch(batch, job->rec_len, "band_raycast_route: ");
        if (rc != OCCGRID_OK) return rc;
        if (!job->d_peer_recs || !job->d_peer_tiles || !job->d_resv || !job->d_status) {
            set_last_error("band_raycast_route: NULL pointer in the route job");
            return OCCGRID_E_ARG;
        }
        if (job->n_bands < 1 || job->n_bands > kMaxBands || job->src_rank < 0 || job->src_rank >= job->n_bands) {
            set_last_error("band_raycast_route: n_bands must be 1..32 and src_rank one of them");
            return OCCGRID_E_ARG;
        }
        if ((uint64_t)job->ordinal_base + (uint64_t)job->n > (1ull << 29) - 1) { set_last_error("band_raycast_route: ordinals must stay below 2^29-1"); return OCCGRID_E_ARG; }
        if (job->seg_capacity != seg_capacity) { set_last_error("band_raycast_route: the job's segment capacity differs from the slot's"); return OCCGRID_E_ARG; }
        const TileGeom tg = tile_geom(job->res, job->size_x, 0);      // bands are full-width rows: only reach, pad and tiles_x are used
        const int reach = tg.reach;
        for (int b = 0; b < job->n_bands; ++b)
            if (job->band_y0[b + 1] - job->band_y0[b] < 2 * reach + 1 && job->n_bands > 1) {
                set_last_error("band_raycast_route: band %d is thinner than 2 * reach + 1 = %d rows (a packet may reach at most two bands)", b, 2 * reach + 1);
                return OCCGRID_E_RANGE;
            }
        J.pkts = job->d_packets; J.n = job->n; J.stride = job->stride;
        J.agent_idx = job->d_agent_idx; J.drift = job->d_drift; J.agent_off = job->d_agent_off; J.n_agents = job->n_agents;
        J.ordinal_base = job->ordinal_base;
        J.ox = job->ox; J.oy = job->oy; J.res = job->res; J.inv_res = 1.0 / job->res; J.size_x = job->size_x;
        J.reach = tg.reach; J.pad = tg.pad; J.tiles_x = tg.tiles_x;
        J.n_bands = job->n_bands; J.src_rank = job->src_rank;
        for (int b = 0; b <= kMaxBands; ++b) J.band_y0[b] = job->band_y0[b <= job->n_bands ? b : job->n_bands];
        J.peer_recs = reinterpret_cast<PoseRec* const*>(job->d_peer_recs);
        J.peer_tiles = reinterpret_cast<int* const*>(job->d_peer_tiles);
        J.seg_cap = (unsigned int)seg_capacity;
        J.resv = job->d_resv; J.status = job->d_status; J.counters = job->d_counters;
        J.n_route_items = (unsigned int)((job->n + kRouteItemPk * kRouteSubsPerItem - 1) / (kRouteItemPk * kRouteSubsPerItem));
    }
    return tiled_raycast_route(band_geom, reinterpret_cast<const PoseRec*>(d_recv_slot), have_prepared ? 1 : 0,
                               J.n_route_items ? &J : nullptr, d_grid, d_workspace, workspace_bytes,
                               (int64_t)n_segs * seg_capacity, d_counters, (cudaStream_t)stream, g_after_fused);
}

int occgrid_band_publish(int n_bands, int rank, uint32_t* d_resv, int64_t seg_capacity, uint32_t* const* d_peer_seg_counts,
                         uint32_t* const* d_peer_flags, const uint32_t* d_my_flags, uint32_t epoch, int wait,
                         int32_t* d_status, void* stream) {
    if (n_bands < 1 || n_bands > kMaxBands || rank < 0 || rank >= n_bands || !d_resv || !d_peer_seg_counts || !d_peer_flags ||
        !d_my_flags || !d_status || seg_capacity <= 0) {
        set_last_error("band_publish: bad arguments");
        return OCCGRID_E_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ProfileScope ps(K_BAND_BARRIER, st);
    k_band_publish<<<1, 32, 0, st>>>(n_bands, rank, d_resv, (unsigned int)seg_capacity, d_peer_seg_counts, d_peer_flags, d_my_flags,
                                     epoch, wait, d_status);
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// One whole step from ONE host call (the per-step host cost decides how far ahead of the GPUs the
// launch queue runs, and with it how much of every rank's jitter ends up inside the barrier).
// With a `side_stream` the publish + barrier of this step's routed batch run THERE, right after the
// fused kernel and concurrently with the resolve pass; the next step's prepare waits for them.
int occgrid_band_step(occgrid_band_ctx* ctx, int64_t step_index, int have_pending, const occgrid_route_job* job,
                      int wait, void* stream, void* side_stream) {
    if (!ctx) { set_last_error("band_step: NULL context"); return OCCGRID_E_ARG; }
    const int prev = (int)((step_index + 1) & 1), slot = (int)(step_index & 1);
    cudaStream_t st = (cudaStream_t)stream, side = (cudaStream_t)side_stream;
    int rc;
    if (side && !ctx->ev_fused) {
        cudaEvent_t a = nullptr, p = nullptr;
        OCC_CUDA_TRY(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        OCC_CUDA_TRY(cudaEventCreateWithFlags(&p, cudaEventDisableTiming));
        ctx->ev_fused = a; ctx->ev_published = p;
    }
    if (side && ctx->published_pending) {            // the batch about to be binned must have arrived from every rank
        OCC_CUDA_TRY(cudaStreamWaitEvent(st, (cudaEvent_t)ctx->ev_published, 0));
        ctx->published_pending = 0;
    }
    if (have_pending) {
        rc = occgrid_band_prepare(&ctx->band_geom, ctx->d_recv[prev], ctx->d_recv_tiles[prev], ctx->n_bands, ctx->seg_capacity,
                                  ctx->d_seg_counts[prev], ctx->d_workspace, ctx->workspace_bytes, ctx->d_counters, stream);
        if (rc != OCCGRID_OK) return rc;
    }
    occgrid_route_job j;
    if (job) {
        j = *job;
        j.n_bands = ctx->n_bands; j.src_rank = ctx->rank; j.seg_capacity = ctx->seg_capacity;
        j.d_peer_recs = ctx->d_peer_recs[slot]; j.d_peer_tiles = ctx->d_peer_tiles[slot];
        j.d_resv = ctx->d_resv; j.d_status = ctx->d_status;
    }
    g_after_fused = (side && job) ? (cudaEvent_t)ctx->ev_fused : nullptr;
    rc = occgrid_band_raycast_route(&ctx->band_geom, ctx->d_recv[prev], ctx->n_bands, ctx->seg_capacity, have_pending,
                                    job ? &j : nullptr, ctx->d_grid, ctx->d_workspace, ctx->workspace_bytes, ctx->d_counters, stream);
    g_after_fused = nullptr;
    if (rc != OCCGRID_OK) return rc;
    if (!job) return OCCGRID_OK;
    if (side) {
        OCC_CUDA_TRY(cudaStreamWaitEvent(side, (cudaEvent_t)ctx->ev_fused, 0));
        rc = occgrid_band_publish(ctx->n_bands, ctx->rank, ctx->d_resv, ctx->seg_capacity, ctx->d_peer_seg_counts[slot],
                                  ctx->d_peer_flags, ctx->d_my_flags, (uint32_t)(step_index + 1), wait, ctx->d_status, side_stream);
        if (rc != OCCGRID_OK) return rc;
        OCC_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->ev_published, side));
        ctx->published_pending = 1;
        return OCCGRID_OK;
    }
    return occgrid_band_publish(ctx->n_bands, ctx->rank, ctx->d_resv, ctx->seg_capacity, ctx->d_peer_seg_counts[slot],
                                ctx->d_peer_flags, ctx->d_my_flags, (uint32_t)(step_index + 1), wait, ctx->d_status, stream);
}

// Make `stream` wait for the last publish + barrier issued on the side stream (before reading the map).
int occgrid_band_join(occgrid_band_ctx* ctx, void* stream) {
    if (!ctx) { set_last_error("band_join: NULL context"); return OCCGRID_E_ARG; }
    if (ctx->published_pending) {
        OCC_CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)ctx->ev_published, 0));
        ctx->published_pending = 0;
    }
    return OCCGRID_OK;
}

}  // extern "C"
