// Packet routing for the spatially tiled multi-GPU map (SURVEY §8e "Integration").
//
// The global grid is cut into row bands, one per GPU.  A beam is at most MAX_DIST_M / res cells
// long (server_nodes/dual_bot_mapper.py:57, :900), so a packet can only touch rows within
// `reach` cells of its robot cell; it is sent to every band that interval intersects (one band
// almost always, two near a boundary).  The receiving GPU walks the SAME global Bresenham
// lines and masks cells outside its window (per-cell clipping, :149/:155), so the assembled
// map is identical to the single-GPU one.
//
// Last-writer-wins needs a global order: the canonical stream is "rank 0's share, then rank
// 1's, ..." and this routing is STABLE within a share, so after an all-to-all (which
// concatenates by source rank) the record index on the receiving side is consistent with the
// canonical order and no sequence numbers have to travel.
//
// This file is the NCCL variant (records grouped in a send buffer, exchanged with all-to-all); the
// default path is the fused raycast + route kernel over peer memory (occgrid_band.cu).
//
// Three kernels: per-CTA band histograms -> single-CTA scan (band-major) -> stable scatter into
// a send buffer grouped by band.  What travels is the DECODED record (48-byte PoseRec: pose
// already corrected by the agent offset and the SLAM drift), so no side arrays follow it and the
// receiver integrates with occgrid_integrate_poses.
#include "common.cuh"

namespace occ {

constexpr int kRT = 256;

struct RouteParams {
    double oy, res;
    int size_y;
    int reach;                       // cells
    int n_bands;
    int band_y0[kMaxBands + 1];      // row boundaries, band b = [band_y0[b], band_y0[b+1])
};

// Bands whose rows intersect [gy - reach, gy + reach]; 0 for packets that are dropped, have a
// non-finite pose, or cannot touch the grid.
__device__ __forceinline__ unsigned int band_mask(const RouteParams& P, const uint8_t* rec, long long k,
                                                  const int32_t* agent_idx, const double* drift,
                                                  const double* agent_off, int n_agents, int* status, PoseRec* out) {
    double rx, ry, ryaw;
    float dist[4];
    const int st = decode_packet(rec, k, agent_idx, drift, agent_off, n_agents, &rx, &ry, &ryaw, dist);
    *status = st;
    if (st != PKT_OK) return 0u;
    out->rx = rx; out->ry = ry; out->yaw = (float)ryaw;            // ryaw came from an fp32 field: exact
    out->d[0] = dist[0]; out->d[1] = dist[1]; out->d[2] = dist[2]; out->d[3] = dist[3];
    out->k = (unsigned int)k; out->tile = -1; out->pad = 0;
    const double q = cell_quotient(ry, P.oy, P.res);
    if (!quotient_in_range(q)) return 0u;
    const int gy = trunc_cell(q);
    const int lo = gy - P.reach, hi = gy + P.reach;
    unsigned int m = 0;
    for (int b = 0; b < P.n_bands; ++b)
        if (hi >= P.band_y0[b] && lo < P.band_y0[b + 1]) m |= 1u << b;
    return m;
}

__global__ void __launch_bounds__(kRT)
k_route_count(RouteParams P, const uint8_t* __restrict__ pkts, long long n, int stride,
              const int32_t* __restrict__ agent_idx, const double* __restrict__ drift,
              const double* __restrict__ agent_off, int n_agents,
              unsigned int* __restrict__ hist /* [n_bands][n_blocks] */, int n_blocks, uint64_t* counters) {
    __shared__ __align__(16) uint8_t s_rec[kRT * kMaxRecStride];
    __shared__ unsigned int s_hist[kMaxBands];
    __shared__ unsigned long long s_acc[4 * 32];
    const long long first = (long long)blockIdx.x * kRT;
    const int count = (int)min((long long)kRT, n - first);
    if (threadIdx.x < kMaxBands) s_hist[threadIdx.x] = 0;
    stage_records(pkts + (size_t)first * stride, (size_t)count * stride, s_rec);
    __syncthreads();
    unsigned int m = 0;
    int st = -1;
    PoseRec unused;
    if ((int)threadIdx.x < count)
        m = band_mask(P, s_rec + threadIdx.x * stride, first + threadIdx.x, agent_idx, drift, agent_off, n_agents, &st, &unused);
    for (int b = 0; b < P.n_bands; ++b) {
        const unsigned int bal = __ballot_sync(0xffffffffu, (m >> b) & 1u);
        if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&s_hist[b], __popc(bal));
    }
    unsigned long long c[4] = {(unsigned long long)(st >= 0), (unsigned long long)(st == PKT_OK),
                               (unsigned long long)(st == PKT_DROPPED), (unsigned long long)(st == PKT_BAD_POSE)};
    __syncthreads();
    if ((int)threadIdx.x < P.n_bands) hist[(size_t)threadIdx.x * n_blocks + blockIdx.x] = s_hist[threadIdx.x];
    block_add_counters(c, s_acc, counters);
}

// Exclusive scan of hist in band-major order; band_counts[b] = records routed to band b.
__global__ void __launch_bounds__(1024)
k_route_scan(unsigned int* __restrict__ hist, int n_bands, int n_blocks, long long* __restrict__ band_counts,
             long long capacity, int* __restrict__ status) {
    unsigned long long carry = 0;
    for (int b = 0; b < n_bands; ++b) {                        // offsets < 2^32 (checked by host)
        const unsigned long long next = cta_scan_in_place<1>(hist + (size_t)b * n_blocks, n_blocks, carry);
        if (threadIdx.x == 0) band_counts[b] = (long long)(next - carry);
        carry = next;
    }
    if (threadIdx.x == 0 && (long long)carry > capacity) atomicOr(status, 1);
}

__global__ void __launch_bounds__(kRT)
k_route_scatter(RouteParams P, const uint8_t* __restrict__ pkts, long long n, int stride,
                const int32_t* __restrict__ agent_idx, const double* __restrict__ drift,
                const double* __restrict__ agent_off, int n_agents,
                const unsigned int* __restrict__ hist, int n_blocks, const int* __restrict__ status,
                PoseRec* __restrict__ send) {
    __shared__ __align__(16) uint8_t s_rec[kRT * kMaxRecStride];
    __shared__ unsigned int s_woff[kRT / 32];
    if (*status & 1) return;                                   // send buffer too small: nothing is written
    const long long first = (long long)blockIdx.x * kRT;
    const int count = (int)min((long long)kRT, n - first);
    stage_records(pkts + (size_t)first * stride, (size_t)count * stride, s_rec);
    __syncthreads();
    unsigned int m = 0;
    int st;
    PoseRec rec;
    const long long k = first + threadIdx.x;
    if ((int)threadIdx.x < count) m = band_mask(P, s_rec + threadIdx.x * stride, k, agent_idx, drift, agent_off, n_agents, &st, &rec);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = 0; b < P.n_bands; ++b) {
        const unsigned int bit = (m >> b) & 1u;
        const unsigned int bal = __ballot_sync(0xffffffffu, bit);
        if (lane == 0) s_woff[warp] = __popc(bal);
        __syncthreads();
        unsigned int woff = 0;
        for (int w = 0; w < warp; ++w) woff += s_woff[w];
        __syncthreads();
        if (bit) {
            const size_t dst = (size_t)hist[(size_t)b * n_blocks + blockIdx.x] + woff + __popc(bal & ((1u << lane) - 1u));
            send[dst] = rec;                                   // three 16-byte stores
        }
    }
}

}  // namespace occ

using namespace occ;

extern "C" {

size_t occgrid_route_workspace_bytes(int64_t n, int n_bands) {
    const int64_t blocks = (n + kRT - 1) / kRT;
    return align_up((size_t)blocks * (size_t)n_bands * sizeof(unsigned int), 256) + 256;
}

int occgrid_route_packets(const occgrid_geom* geom, int n_bands, const int32_t* band_y0_host,
                          const uint8_t* d_packets, int64_t n, int stride, int rec_len,
                          const int32_t* d_agent_idx, const double* d_drift, const double* d_agent_off, int n_agents,
                          void* d_send, int64_t send_capacity,
                          int64_t* d_band_counts, int32_t* d_status, uint64_t* d_counters,
                          void* d_ws, size_t ws_bytes, void* stream) {
    int rc = validate_geom(geom);
    if (rc != OCCGRID_OK) return rc;
    if (n_bands < 1 || n_bands > kMaxBands || !band_y0_host) { set_last_error("route: n_bands must be 1..32"); return OCCGRID_E_ARG; }
    rc = check_packet_batch(PacketBatch{d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents}, rec_len, "route: ");
    if (rc != OCCGRID_OK) return rc;
    if (!d_send || !d_band_counts || !d_status || !d_ws) { set_last_error("route: NULL argument"); return OCCGRID_E_ARG; }
    if (reinterpret_cast<uintptr_t>(d_send) & 15) { set_last_error("route: send buffer must be 16-byte aligned"); return OCCGRID_E_ARG; }
    if (send_capacity >= (1ll << 32)) { set_last_error("route: send capacity must be < 2^32 records"); return OCCGRID_E_ARG; }
    if (ws_bytes < occgrid_route_workspace_bytes(n, n_bands)) { set_last_error("route: workspace too small"); return OCCGRID_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    RouteParams P;
    P.oy = geom->oy; P.res = geom->res; P.size_y = geom->size_y;
    P.reach = reach_cells(geom->res);
    P.n_bands = n_bands;
    for (int b = 0; b <= n_bands; ++b) P.band_y0[b] = band_y0_host[b];
    for (int b = n_bands + 1; b <= kMaxBands; ++b) P.band_y0[b] = band_y0_host[n_bands];
    const int blocks = (int)((n + kRT - 1) / kRT);
    unsigned int* hist = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(d_ws) + 256);
    if (n == 0) {
        OCC_CUDA_TRY(cudaMemsetAsync(d_band_counts, 0, sizeof(int64_t) * n_bands, st));
        return OCCGRID_OK;
    }
    ProfileScope ps(K_ROUTE, st, 3);
    k_route_count<<<blocks, kRT, 0, st>>>(P, d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents, hist, blocks, d_counters);
    k_route_scan<<<1, 1024, 0, st>>>(hist, n_bands, blocks, (long long*)d_band_counts, send_capacity, d_status);
    k_route_scatter<<<blocks, kRT, 0, st>>>(P, d_packets, n, stride, d_agent_idx, d_drift, d_agent_off, n_agents, hist, blocks,
                                            d_status, reinterpret_cast<PoseRec*>(d_send));
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // extern "C"
