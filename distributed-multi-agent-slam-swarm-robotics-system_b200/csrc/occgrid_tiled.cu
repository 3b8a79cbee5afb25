// Strategy TILED of occgrid_integrate_packets: packets binned by the HOME TILE of the robot
// cell, last-writer-wins resolved with SHARED-MEMORY atomics.
//
// Same reference semantics as occgrid_integrate.cu (server_nodes/dual_bot_mapper.py:826-903,
// :136-179; every cell keeps the largest  (beam ordinal + 1) << 1 | occupied  stamp), but the
// per-cell atomicMax runs on a stamp window in shared memory, where B200 sustains
// ~1.0-1.5e12 atomics/s (measured, occgrid_scatter_probe kind 2) against ~2.2e11/s for
// red.global (kind 0).  Only the surviving stamp of each touched cell goes to L2.
//
// All four beams of a packet start at the robot cell (:142) and are at most
// R = ceil(MAX_DIST_M / res) + 2 cells long (:57, :900), so they lie inside the robot's 64x64
// home tile grown by R on every side.  Binning therefore needs only the robot cell — no
// trigonometry, one record per packet, no duplicates:
//
//   k_home_bin      thread/packet: decode (:828-843), pose correction (:851-857), robot cell
//                   (:142) -> 48-byte pose record (packet order) + packets per home tile, and each
//                   CTA's packet indices grouped by tile with its rank inside every tile's bin
//   k_tile_plan     one CTA over the active tiles (listed by the bin pass): exclusive scan of
//                   their counts -> bin offsets, (tile, chunk) work items of <= kChunkPk packets
//   k_place_runs    thread/packet: copy the grouped indices to their tile's bin
//   k_home_raycast  persistent CTAs pull work items: zero the (64+2R)^2 smem window, expand
//                   each record into its 4 beams (fp64 endpoints, :887-902) and walk the exact
//                   reference Bresenham (:158-179) with atomicMax in shared memory; then flush
//                   the non-zero stamps with coalesced red.global.max to the stamp plane
//   k_home_resolve  persistent CTAs over the active tiles' windows: stamps -> int8 grid, := 0
//
// Windows of neighbouring tiles overlap; the global atomicMax merges them, and chunks of one
// tile likewise, so the result is independent of how work was cut.
#include "common.cuh"

namespace occ {

constexpr int kTT = 256;             // threads per CTA
// Packets per work item: chosen per batch by k_tile_plan so that the persistent raycast CTAs get
// ~kItemsPerCta items each: a small batch cut into 2 048-packet items would leave most CTAs without
// work, while many small items cost more than they balance (every item re-reads and flushes its
// tile's hot cells).
constexpr int kChunkPk = 2048;       // largest work item
constexpr int kChunkMin = 256;       // smallest: one packet per thread
constexpr int kItemsPerCta = 3;       // raycast of configs[1]: 3 -> 0.202 ms, 5 -> 0.220, 8 -> 0.235, 12 -> 0.263; cutting only the
                                      // last quarter of the queue 4x / 8x finer: 0.201 / 0.215 against 0.198
constexpr int kMaxWindowBytes = 100 * 1024;   // smem window budget (two CTAs per SM at least)

struct TilePlanHeader {
    unsigned int n_items, n_active, total_records, work_counter, resolve_counter, overflow;
    unsigned int active_count;   // tiles appended to the active list by the count pass of the current call
    unsigned int pad;
};

// Home tile of a corrected pose, or -1 when no beam of the packet can reach the window.
__device__ __forceinline__ int home_tile(const Geom& g, const TileGeom& tg, double rx, double ry) {
    const double qx = cell_quotient(rx, g.ox, g.res), qy = cell_quotient(ry, g.oy, g.res);
    if (!quotient_in_range(qx) || !quotient_in_range(qy)) return -1;
    const int px = trunc_cell(qx) - g.win_x0 + tg.pad, py = trunc_cell(qy) - g.win_y0 + tg.pad;
    if (px < tg.pad - tg.reach || py < tg.pad - tg.reach || px >= tg.pad + g.win_w + tg.reach ||
        py >= tg.pad + g.win_h + tg.reach)
        return -1;
    return (py >> kTileShift) * tg.tiles_x + (px >> kTileShift);
}

// ---- binning passes ------------------------------------------------------------------------
// The hot tiles of a swarm are few (two robots per room), so per-packet global atomics on the
// tile counters serialise on a handful of L2 addresses.  Each CTA therefore bins kPkPerCta
// packets in a shared-memory hash table first and touches every distinct tile once.
constexpr int kPkPerCta = 2048;
constexpr int kSub = kPkPerCta / kTT;           // packets per thread
constexpr int kHash = 4096;                     // >= 2 * kPkPerCta would be ideal; distinct tiles <= kPkPerCta
constexpr unsigned int kEmpty = 0xffffffffu;
static_assert(kHash >= 2 * kPkPerCta, "hash table must stay at most half full");

__device__ __forceinline__ int hash_insert(unsigned int* keys, unsigned int tile) {
    unsigned int h = (tile * 2654435761u) >> 20;             // 12 bits
    for (;;) {
        const unsigned int old = atomicCAS(&keys[h], kEmpty, tile);
        if (old == kEmpty || old == tile) return (int)h;
        h = (h + 1) & (kHash - 1);
    }
}

// End of a binning CTA: every distinct tile of the shared-memory hash goes to the global counters
// with ONE atomic.  The 16 slots a thread owns are handled in two unrolled phases so that all its
// atomics are in flight together (the first-toucher test needs their return values; waiting for
// each one in turn made these kernels pure L2 round-trip latency).
constexpr int kHashPerThread = kHash / kTT;

__device__ __forceinline__ void flush_tile_counts(const unsigned int* s_keys, const unsigned int* s_vals,
                                                  unsigned int* __restrict__ tile_count, unsigned int* __restrict__ active,
                                                  TilePlanHeader* __restrict__ hdr) {
    unsigned int key[kHashPerThread], old[kHashPerThread];
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j) {
        const int i = j * kTT + threadIdx.x;
        key[j] = s_keys[i];
        old[j] = 1u;
        if (key[j] != kEmpty) old[j] = atomicAdd(&tile_count[key[j]], s_vals[i]);
    }
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j)
        if (key[j] != kEmpty && old[j] == 0u) active[atomicAdd(&hdr->active_count, 1u)] = key[j];      // first toucher lists the tile
}

// Scatter side: one range reservation per distinct tile; s_vals[slot] becomes the first bin slot.
__device__ __forceinline__ void reserve_tile_ranges(const unsigned int* s_keys, unsigned int* s_vals,
                                                    const unsigned int* __restrict__ tile_offset, unsigned int* __restrict__ tile_cursor) {
    unsigned int key[kHashPerThread], base[kHashPerThread], off[kHashPerThread];
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j) {
        const int i = j * kTT + threadIdx.x;
        key[j] = s_keys[i];
        base[j] = off[j] = 0u;
        if (key[j] != kEmpty) { off[j] = tile_offset[key[j]]; base[j] = atomicAdd(&tile_cursor[key[j]], s_vals[i]); }
    }
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j)
        if (key[j] != kEmpty) s_vals[j * kTT + threadIdx.x] = off[j] + base[j];
}

// Packet path: the bin pass does the whole binning but the final placement.  Binning CTA b owns
// the segment [b * kPkPerCta, (b + 1) * kPkPerCta) of the batch and of the arrays below:
//   local_bins  its accepted packets grouped by home tile: (run << 16) | packet index in the segment
//   runs        one per distinct tile of the segment, in local_bins order: (tile, tile_rank - local
//               begin), where tile_rank is the CTA's position inside the tile's bin (the return
//               value of its one atomic on tile_count) and local begin the run's first position
//   seg_count   number of local_bins entries
// Once k_tile_plan has the bin offsets, k_place_runs moves entry j of run r to
// bins[tile_offset[tile] + tile_rank + (j - local begin)].  The decoded 48-byte pose record of
// every binned packet is stored in packet order for the raycast: decoding the 42-byte wire record
// again in the raycast instead was measured slower (DESIGN §3).
//
// kMaps (occgrid_integrate_packets_agent_maps): the map is folded into the tile KEY, (agent - 1) *
// n_tiles + home tile.  Everything below and the plan and placement passes work on keys unchanged.
constexpr size_t kBinSmem = (size_t)kTT * kMaxRecStride + 2 * kHash * sizeof(unsigned int) + kPkPerCta * sizeof(unsigned short);
constexpr unsigned int kNoSlot = 0xffffu;

template <bool kMaps = false>
__global__ void __launch_bounds__(kTT)
k_home_bin(Geom g, TileGeom tg, const uint8_t* __restrict__ pkts, long long n, int stride,
           const int32_t* __restrict__ agent_idx, const double* __restrict__ drift,
           const double* __restrict__ agent_off, int n_agents,
           unsigned int* __restrict__ tile_count, PoseRec* __restrict__ recs, unsigned int* __restrict__ local_bins, uint2* __restrict__ runs,
           unsigned int* __restrict__ seg_count, unsigned int* __restrict__ active, TilePlanHeader* __restrict__ hdr,
           uint64_t* counters) {
    extern __shared__ __align__(16) uint8_t s_bin[];                                  // kBinSmem
    uint8_t* const s_rec = s_bin;                                                     // staged records, later the local bin list
    unsigned int* const s_keys = reinterpret_cast<unsigned int*>(s_bin + kTT * kMaxRecStride);
    unsigned int* const s_vals = s_keys + kHash;
    unsigned short* const s_slot = reinterpret_cast<unsigned short*>(s_vals + kHash);   // hash slot of every packet, or kNoSlot
    __shared__ unsigned int s_wsum[kTT / 32];
    for (int i = threadIdx.x; i < kHash; i += kTT) { s_keys[i] = kEmpty; s_vals[i] = 0u; }
    unsigned long long c[OCCGRID_C_HITS + 1] = {};
    const long long cta_first = (long long)blockIdx.x * kPkPerCta;
    // Software-pipelined staging: the 16-byte loads of sub-batch s+1 are in flight while
    // sub-batch s is decoded out of shared memory.
    constexpr int kVec = (kTT * kMaxRecStride / 16 + kTT - 1) / kTT;      // uint4 per thread per sub-batch (<= 4)
    uint4 pre[kVec];
    auto prefetch = [&](int sub) {
        const long long first = cta_first + (long long)sub * kTT;
        const long long left = n - first;
        const size_t bytes = left <= 0 ? 0 : (size_t)min((long long)kTT, left) * stride;
        const uint4* s4 = reinterpret_cast<const uint4*>(pkts + (size_t)first * stride);
#pragma unroll
        for (int j = 0; j < kVec; ++j) {
            const size_t i = (size_t)j * kTT + threadIdx.x;
            pre[j] = (i * 16 + 16 <= bytes) ? __ldg(s4 + i) : make_uint4(0u, 0u, 0u, 0u);
        }
    };
    const bool vec_ok = (reinterpret_cast<uintptr_t>(pkts) & 15) == 0 && ((kTT * stride) & 15) == 0;
    if (vec_ok) prefetch(0);
    for (int sub = 0; sub < kSub; ++sub) {
        const long long first = cta_first + (long long)sub * kTT;
        if (first >= n) break;
        const int count = (int)min((long long)kTT, n - first);
        __syncthreads();
        if (vec_ok) {
            const size_t bytes = (size_t)count * stride;
            uint4* d4 = reinterpret_cast<uint4*>(s_rec);
#pragma unroll
            for (int j = 0; j < kVec; ++j) {
                const size_t i = (size_t)j * kTT + threadIdx.x;
                if (i * 16 + 16 <= bytes) d4[i] = pre[j];
            }
            for (size_t i = (bytes / 16) * 16 + threadIdx.x; i < bytes; i += kTT) s_rec[i] = __ldg(pkts + (size_t)first * stride + i);
            if (sub + 1 < kSub) prefetch(sub + 1);
        } else {
            stage_records(pkts + (size_t)first * stride, (size_t)count * stride, s_rec);
        }
        __syncthreads();
        if ((int)threadIdx.x < count) {
            const long long k = first + threadIdx.x;
            double rx, ry, ryaw;
            float dist[4];
            c[OCCGRID_C_PACKETS] += 1;
            unsigned int slot = kNoSlot;
            int agent = 1;
            const int st = decode_packet(s_rec + threadIdx.x * stride, k, agent_idx, drift, agent_off, n_agents, &rx, &ry, &ryaw, dist,
                                         kMaps ? &agent : nullptr);
            if (st == PKT_DROPPED) c[OCCGRID_C_DROPPED] += 1;
            else if (st == PKT_BAD_POSE) c[OCCGRID_C_BAD_POSE] += 1;
            else {
                c[OCCGRID_C_ACCEPTED] += 1;
                c[OCCGRID_C_BEAMS] += 4;
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const double d = (double)dist[s];
                    c[OCCGRID_C_HITS] += (OCC_MIN_DIST_M < d && d <= OCC_MAX_DIST_M) ? 1 : 0;     // :888
                }
                int tile = home_tile(g, tg, rx, ry);
                if (kMaps && tile >= 0) tile += (agent - 1) * tg.n_tiles;
                if (tile >= 0) {
                    slot = (unsigned int)hash_insert(s_keys, (unsigned int)tile);
                    atomicAdd(&s_vals[slot], 1u);
                    PoseRec r;
                    r.rx = rx; r.ry = ry; r.yaw = (float)ryaw;      // ryaw came from an fp32 field: exact
                    r.d[0] = dist[0]; r.d[1] = dist[1]; r.d[2] = dist[2]; r.d[3] = dist[3];
                    r.k = (unsigned int)k;
                    r.tile = tile; r.pad = 0;
                    recs[k] = r;                                    // packet order: coalesced 48-byte stores
                }
            }
            s_slot[sub * kTT + threadIdx.x] = (unsigned short)slot;
        }
    }
    __syncthreads();
    // One global atomic per distinct tile, as in flush_tile_counts; its return value is this CTA's
    // rank inside the tile's bin.
    unsigned int key[kHashPerThread], rank[kHashPerThread];
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j) {
        const int i = j * kTT + threadIdx.x;
        key[j] = s_keys[i];
        rank[j] = 0u;
        if (key[j] != kEmpty) rank[j] = atomicAdd(&tile_count[key[j]], s_vals[i]);
    }
    // Exclusive scan of (count | 1 << 16) over the occupied slots in (thread, j) order: the low half
    // is the slot's first local position, the high half its run index (both < kPkPerCta).  An empty
    // slot has count 0.
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int mine = 0u;
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j) mine += key[j] != kEmpty ? s_vals[j * kTT + threadIdx.x] + 0x10000u : 0u;
    unsigned int inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned int u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
    if (lane == 31) s_wsum[warp] = inc;
    __syncthreads();
    unsigned int pos = inc - mine, n_local = 0u;
#pragma unroll
    for (int w = 0; w < kTT / 32; ++w) {
        pos += w < warp ? s_wsum[w] : 0u;
        n_local += s_wsum[w];
    }
    n_local &= 0xffffu;
    if (threadIdx.x == 0) seg_count[blockIdx.x] = n_local;
    const size_t seg0 = (size_t)blockIdx.x * kPkPerCta;
    // run descriptors; each slot (owned by this thread alone) now holds its run index and its next
    // free local position
#pragma unroll
    for (int j = 0; j < kHashPerThread; ++j) {
        if (key[j] == kEmpty) continue;
        const int i = j * kTT + threadIdx.x;
        const unsigned int run = pos >> 16, begin = pos & 0xffffu;
        runs[seg0 + run] = make_uint2(key[j], rank[j] - begin);
        pos += s_vals[i] + 0x10000u;
        s_keys[i] = run;
        s_vals[i] = begin;
        if (rank[j] == 0u) active[atomicAdd(&hdr->active_count, 1u)] = key[j];     // first toucher lists the tile
    }
    __syncthreads();
    // the packet indices grouped by tile, assembled in the (now free) staging buffer, then stored
    // coalesced
    unsigned int* const s_local = reinterpret_cast<unsigned int*>(s_rec);
    const int n_seg = (int)min((long long)kPkPerCta, n - (long long)seg0);
    for (int j = threadIdx.x; j < n_seg; j += kTT) {
        const unsigned int slot = s_slot[j];
        if (slot != kNoSlot) s_local[atomicAdd(&s_vals[slot], 1u)] = (s_keys[slot] << 16) | (unsigned int)j;
    }
    __syncthreads();
    for (unsigned int j = threadIdx.x; j < n_local; j += kTT) local_bins[seg0 + j] = s_local[j];
    __syncthreads();
    block_add_counters(c, reinterpret_cast<unsigned long long*>(s_rec), counters);
}

// Thread per local_bins entry of one binning CTA's segment (see k_home_bin): no hash and no atomics,
// and the stores of a run are contiguous.
__global__ void __launch_bounds__(kTT)
k_place_runs(const unsigned int* __restrict__ local_bins, const uint2* __restrict__ runs, const unsigned int* __restrict__ seg_count,
             const unsigned int* __restrict__ tile_offset, const TilePlanHeader* __restrict__ hdr, unsigned int* __restrict__ bins) {
    if (hdr->overflow) return;
    const size_t seg0 = (size_t)blockIdx.x * kPkPerCta;
    const int n_local = (int)seg_count[blockIdx.x];
    // three dependent gathers per entry: each phase has all of the thread's loads in flight
    unsigned int e[kSub], off[kSub];
    uint2 d[kSub];
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub) {
        const int j = sub * kTT + threadIdx.x;
        e[sub] = j < n_local ? local_bins[seg0 + j] : kEmpty;
    }
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub) d[sub] = e[sub] != kEmpty ? runs[seg0 + (e[sub] >> 16)] : make_uint2(0u, 0u);
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub) off[sub] = e[sub] != kEmpty ? tile_offset[d[sub].x] : 0u;
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub)
        if (e[sub] != kEmpty) bins[off[sub] + d[sub].y + (unsigned int)(sub * kTT + threadIdx.x)] = (unsigned int)(seg0 + (e[sub] & 0xffffu));
}

// Segment / validity of one 2048-address chunk of a (possibly segmented) record buffer.
__device__ __forceinline__ int chunk_valid(const SegInfo& seg, long long chunk, long long* addr0) {
    const long long a0 = chunk * kSegChunk;
    *addr0 = a0;
    const unsigned int sg = (unsigned int)(a0 / seg.seg_cap);
    const unsigned int j0 = (unsigned int)(a0 - (long long)sg * seg.seg_cap);
    unsigned int cnt = seg.d_counts ? seg.d_counts[sg] : seg.host_count;
    if (cnt > seg.seg_cap) cnt = seg.seg_cap;                       // a segment that overflowed was truncated by its writer
    return cnt > j0 ? (int)min((unsigned int)kSegChunk, cnt - j0) : 0;
}

// The count pass for input that is already decoded (routed pose records, binned in place).
// The buffer is a set of per-source segments whose fill counts live on the device; persistent
// CTAs stride over 2048-address chunks and skip the empty ones.  `tiles_in_records`: the router
// already computed the home tile for THIS window (rec.tile), nothing is re-derived here.
__global__ void __launch_bounds__(kTT)
k_home_count_poses(Geom g, TileGeom tg, const PoseRec* __restrict__ recs, const int* __restrict__ in_tiles, SegInfo seg, long long n_chunks,
                   int tiles_in_records,
                   unsigned int* __restrict__ tile_count, int* __restrict__ tile_ids,
                   unsigned int* __restrict__ active, TilePlanHeader* __restrict__ hdr, uint64_t* counters) {
    __shared__ unsigned int s_keys[kHash];
    __shared__ unsigned int s_vals[kHash];
    __shared__ unsigned long long s_acc[(OCCGRID_C_HITS + 1) * 32];
    unsigned long long c[OCCGRID_C_HITS + 1] = {};
    for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        long long addr0;
        const int valid = chunk_valid(seg, chunk, &addr0);
        if (valid == 0) continue;                                   // uniform across the CTA
        for (int i = threadIdx.x; i < kHash; i += kTT) { s_keys[i] = kEmpty; s_vals[i] = 0u; }
        __syncthreads();
        if (tiles_in_records) {
            int tl[kSub];
#pragma unroll
            for (int sub = 0; sub < kSub; ++sub) {              // all loads of the thread in flight together
                const int j = sub * kTT + threadIdx.x;
                tl[sub] = -1;
                if (j < valid) tl[sub] = in_tiles ? in_tiles[addr0 + j] : recs[addr0 + j].tile;
            }
#pragma unroll
            for (int sub = 0; sub < kSub; ++sub) {
                const int j = sub * kTT + threadIdx.x;
                if (j >= valid) continue;
                int tile = tl[sub];                             // packets / beams / hits were counted by the source rank
                if (tile >= tg.n_tiles) tile = -1;              // never trust a tile id that came over the wire
                if (tile >= 0) atomicAdd(&s_vals[hash_insert(s_keys, (unsigned int)tile)], 1u);
                tile_ids[addr0 + j] = tile;
            }
        } else {
            for (int sub = 0; sub < kSub; ++sub) {
                const int j = sub * kTT + threadIdx.x;
                if (j >= valid) break;
                const long long k = addr0 + j;
                int tile = -1;
                const PoseRec r = recs[k];
                c[OCCGRID_C_PACKETS] += 1;
                if (!(isfinite(r.rx) && isfinite(r.ry) && isfinite(r.yaw))) c[OCCGRID_C_BAD_POSE] += 1;
                else {
                    c[OCCGRID_C_ACCEPTED] += 1;
                    c[OCCGRID_C_BEAMS] += 4;
#pragma unroll
                    for (int s2 = 0; s2 < 4; ++s2) {
                        const double dd = (double)r.d[s2];
                        c[OCCGRID_C_HITS] += (OCC_MIN_DIST_M < dd && dd <= OCC_MAX_DIST_M) ? 1 : 0;
                    }
                    tile = home_tile(g, tg, r.rx, r.ry);
                }
                if (tile >= 0) atomicAdd(&s_vals[hash_insert(s_keys, (unsigned int)tile)], 1u);
                tile_ids[k] = tile;
            }
        }
        __syncthreads();
        flush_tile_counts(s_keys, s_vals, tile_count, active, hdr);
        __syncthreads();
    }
    block_add_counters(c, s_acc, counters);
}

// Scatter for segmented record buffers: bins hold record ADDRESSES (segment * seg_cap + index).
__global__ void __launch_bounds__(kTT)
k_home_scatter_segs(SegInfo seg, long long n_chunks, const int* __restrict__ tile_ids, const unsigned int* __restrict__ tile_offset,
                    unsigned int* __restrict__ tile_cursor, const TilePlanHeader* __restrict__ hdr, unsigned int* __restrict__ bins) {
    __shared__ unsigned int s_keys[kHash];
    __shared__ unsigned int s_vals[kHash];
    if (hdr->overflow) return;
    for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        long long addr0;
        const int valid = chunk_valid(seg, chunk, &addr0);
        if (valid == 0) continue;
        for (int i = threadIdx.x; i < kHash; i += kTT) { s_keys[i] = kEmpty; s_vals[i] = 0u; }
        __syncthreads();
        unsigned int where[kSub];
        int tl[kSub];
#pragma unroll
        for (int sub = 0; sub < kSub; ++sub) {
            const int j = sub * kTT + threadIdx.x;
            tl[sub] = j < valid ? tile_ids[addr0 + j] : -1;
        }
#pragma unroll
        for (int sub = 0; sub < kSub; ++sub) {
            const int j = sub * kTT + threadIdx.x;
            where[sub] = kEmpty;
            if (j < valid) {
                const int tile = tl[sub];
                if (tile >= 0) {
                    const int h = hash_insert(s_keys, (unsigned int)tile);
                    where[sub] = ((unsigned int)h << 16) | atomicAdd(&s_vals[h], 1u);
                }
            }
        }
        __syncthreads();
        reserve_tile_ranges(s_keys, s_vals, tile_offset, tile_cursor);
        __syncthreads();
#pragma unroll
        for (int sub = 0; sub < kSub; ++sub)
            if (where[sub] != kEmpty)
                bins[s_vals[where[sub] >> 16] + (where[sub] & 0xffffu)] = (unsigned int)(addr0 + sub * kTT + threadIdx.x);
        __syncthreads();
    }
}

// One CTA over the ACTIVE tiles only (listed by the count pass, in arbitrary order — nothing
// downstream depends on the order): exclusive scan of their counts -> bin offsets, cursors
// zeroed, (tile, chunk) work items built.  tile_count is re-zeroed for the next call.
__global__ void __launch_bounds__(1024)
k_tile_plan(unsigned int* __restrict__ tile_count, unsigned int* __restrict__ tile_offset,
            unsigned int* __restrict__ tile_cursor, uint4* __restrict__ items, unsigned int max_items,
            const unsigned int* __restrict__ active, unsigned long long max_records, TilePlanHeader* __restrict__ hdr,
            uint64_t* counters, unsigned int target_items) {
    __shared__ unsigned int s_warp[2][33];
    __shared__ unsigned int s_carry[2];
    __shared__ unsigned int s_total;
    if (threadIdx.x < 2) s_carry[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_total = 0;
    __syncthreads();
    const int n_active = (int)hdr->active_count;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // records of this batch -> packets per work item (a multiple of kChunkMin)
    {
        unsigned int mine = 0;
        for (int i = threadIdx.x; i < n_active; i += blockDim.x) mine += tile_count[active[i]];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
        if (lane == 0 && mine) atomicAdd(&s_total, mine);
    }
    __syncthreads();
    unsigned int chunk_pk = (s_total / target_items + kChunkMin) / kChunkMin * kChunkMin;
    chunk_pk = chunk_pk > (unsigned int)kChunkPk ? (unsigned int)kChunkPk : chunk_pk;
    for (int start = 0; start < n_active; start += blockDim.x) {
        const int i = start + threadIdx.x;
        const unsigned int t = i < n_active ? active[i] : 0u;
        const unsigned int cnt = i < n_active ? tile_count[t] : 0u;
        unsigned int v[2] = {cnt, (cnt + chunk_pk - 1) / chunk_pk};
        unsigned int ex[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            unsigned int inc = v[j];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { unsigned int u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
            if (lane == 31) s_warp[j][warp] = inc;
            ex[j] = inc - v[j];
        }
        __syncthreads();
        if (warp < 2) {
            unsigned int w = s_warp[warp][lane], winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { unsigned int u = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += u; }
            s_warp[warp][lane] = winc - w;
            if (lane == 31) s_warp[warp][32] = winc;
        }
        __syncthreads();
        const unsigned int off = s_carry[0] + s_warp[0][warp] + ex[0];
        const unsigned int item0 = s_carry[1] + s_warp[1][warp] + ex[1];
        if (i < n_active) {
            tile_offset[t] = off;
            tile_cursor[t] = 0u;
            tile_count[t] = 0u;
            for (unsigned int j = 0; j < v[1]; ++j) {
                const unsigned int b = off + j * chunk_pk;
                const unsigned int e = min(off + cnt, b + chunk_pk);
                if (item0 + j < max_items) items[item0 + j] = make_uint4(t, b, e, 0u);
            }
        }
        __syncthreads();
        if (threadIdx.x < 2) s_carry[threadIdx.x] += s_warp[threadIdx.x][32];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        TilePlanHeader h;
        h.total_records = s_carry[0];
        h.n_items = s_carry[1];
        h.n_active = (unsigned int)n_active;
        h.work_counter = 0;
        h.resolve_counter = 0;
        h.active_count = 0;                  // ready for the next call's count pass
        h.overflow = (s_carry[0] > max_records || s_carry[1] > max_items) ? 1u : 0u;
        if (h.overflow) { h.n_items = 0; h.n_active = 0; }
        h.pad = 0;
        *hdr = h;
        if (counters) atomicAdd(reinterpret_cast<unsigned long long*>(counters) + OCCGRID_C_RECORDS, (unsigned long long)s_carry[0]);
    }
}

// Walk one beam into the shared-memory window (exact reference Bresenham, :158-179: strict
// `e2 > -dy` / `e2 < dx`, both may fire, sx = -1 when x0 == x1).  (x, y) are window-local.
// Both end points inside the (convex) window => every cell is inside, so the hot loop carries
// no bounds test and steps a running shared-memory offset instead of recomputing y*pitch+x.
__device__ __noinline__ void draw_beam_smem(unsigned int* __restrict__ s_win, int side, int pitch, int x, int y,
                                               int ddx, int ddy, unsigned int free_stamp, bool hit, bool skip_first) {
    const int dx = abs(ddx), dy = abs(ddy);
    int err = dx - dy;
    const int n = max(dx, dy);
    const unsigned int us = (unsigned int)side;
    if ((unsigned int)x < us && (unsigned int)y < us && (unsigned int)(x + ddx) < us && (unsigned int)(y + ddy) < us) {
        // Major/minor form of the same recurrence.  With err = dx - dy the reference steps the
        // major axis on EVERY iteration (for dx > dy: 2*err > -dy always holds; for dy > dx:
        // 2*err < dx always holds; both step when dx == dy), and the minor axis steps iff
        //   x-major: 2*err < dx        y-major: 2*err > -dy  <=>  2*(-err) < dy
        // i.e. with E = |err-form| = dmaj - dmin initially:  minor iff 2*E < dmaj (strict, like
        // the reference), then E += (minor ? dmaj : 0) - dmin.  Branch-free across octants, so
        // lanes walking different octants do not diverge.  (Exhaustive KAT on device:
        // tests/test_gpu_integrate.py::test_bresenham_exhaustive_on_device.)
        const int sxo = ddx > 0 ? 1 : -1;
        const int syo = ddy > 0 ? pitch : -pitch;
        const bool xmajor = dx >= dy;
        const int dmaj = xmajor ? dx : dy, dmin = xmajor ? dy : dx;
        const int step_maj = xmajor ? sxo : syo;
        const int step_both = sxo + syo;
        const int e_minor = dmaj - dmin;         // E change when the minor axis steps too
        int E = dmaj - dmin;
        int off = y * pitch + x;
        int i = 0;
        if (skip_first) {                     // the start cell is overwritten by a later beam of the packet
            if (n == 0) return;
            const bool minor = 2 * E < dmaj;
            off += minor ? step_both : step_maj;
            E += minor ? e_minor : -dmin;
            i = 1;
        }
        for (; i < n; ++i) {
            atomicMax(&s_win[off], free_stamp);
            const bool minor = 2 * E < dmaj;
            off += minor ? step_both : step_maj;
            E += minor ? e_minor : -dmin;
        }
        if (hit) atomicMax(&s_win[off], free_stamp | 1u);
        return;
    }
    // guarded path (cannot happen while the reach bound holds): per-cell window test
    const int sx = ddx > 0 ? 1 : -1, sy = ddy > 0 ? 1 : -1;
    for (int i = 0; i < n; ++i) {
        if (!(i == 0 && skip_first) && (unsigned int)x < us && (unsigned int)y < us) atomicMax(&s_win[y * pitch + x], free_stamp);
        const int e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x += sx; }
        if (e2 < dx)  { err += dx; y += sy; }
    }
    if (hit && !(n == 0 && skip_first) && (unsigned int)x < us && (unsigned int)y < us) atomicMax(&s_win[y * pitch + x], free_stamp | 1u);
}

// Hit/miss COUNT mode (extension, SURVEY §8c): the same walk, but every cell update_ray (:148-156)
// would have stored FREE to counts one miss (low half of the window word) and the OCCUPIED end
// cell of a valid hit counts one hit (high half).  A work item holds <= 4 * kChunkPk beams and a
// beam visits a cell once, so 16 bits per half cannot overflow.
__device__ __noinline__ void count_beam_smem(unsigned int* __restrict__ s_win, int side, int pitch, int x, int y,
                                                int ddx, int ddy, bool hit) {
    const int dx = abs(ddx), dy = abs(ddy);
    const int n = max(dx, dy);
    const unsigned int us = (unsigned int)side;
    if ((unsigned int)x < us && (unsigned int)y < us && (unsigned int)(x + ddx) < us && (unsigned int)(y + ddy) < us) {
        const int sxo = ddx > 0 ? 1 : -1;
        const int syo = ddy > 0 ? pitch : -pitch;
        const bool xmajor = dx >= dy;
        const int dmaj = xmajor ? dx : dy, dmin = xmajor ? dy : dx;
        const int step_maj = xmajor ? sxo : syo;
        const int step_both = sxo + syo;
        const int e_minor = dmaj - dmin;
        int E = dmaj - dmin;
        int off = y * pitch + x;
        for (int i = 0; i < n; ++i) {
            atomicAdd(&s_win[off], 1u);
            const bool minor = 2 * E < dmaj;
            off += minor ? step_both : step_maj;
            E += minor ? e_minor : -dmin;
        }
        if (hit) atomicAdd(&s_win[off], 0x10000u);
        return;
    }
    int err = dx - dy;
    const int sx = ddx > 0 ? 1 : -1, sy = ddy > 0 ? 1 : -1;
    for (int i = 0; i < n; ++i) {
        if ((unsigned int)x < us && (unsigned int)y < us) atomicAdd(&s_win[y * pitch + x], 1u);
        const int e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x += sx; }
        if (e2 < dx)  { err += dx; y += sy; }
    }
    if (hit && (unsigned int)x < us && (unsigned int)y < us) atomicAdd(&s_win[y * pitch + x], 0x10000u);
}



// ---- table-driven walk -------------------------------------------------------------------------
// The minor-axis steps of the reference's Bresenham (:158-179) depend only on (dmaj, dmin): bit i of
// walk_mask(dmaj, dmin) says whether step i also moves the minor axis — the very recurrence of
// draw_beam_smem (E = dmaj - dmin; minor iff 2E < dmaj; E += minor ? dmaj - dmin : -dmin), run once
// per (dmaj, dmin) pair when the CTA starts instead of once per cell.  561 pairs for dmaj <= 32
// (a 1.2 m ray at 5 cm is <= 26 cells); longer beams take the recurrence.  The walk itself is
// then: one shared-memory reduction per cell on a running BYTE address, one bit test, one add.
constexpr int kMaskMaxLen = 32;
constexpr int kMaskEntries = (kMaskMaxLen + 1) * (kMaskMaxLen + 2) / 2;

__device__ __forceinline__ unsigned int walk_mask_of(int dmaj, int dmin) {
    unsigned int m = 0u;
    int E = dmaj - dmin;
    for (int i = 0; i < dmaj; ++i) {
        const bool minor = 2 * E < dmaj;
        m |= (minor ? 1u : 0u) << i;
        E += minor ? (dmaj - dmin) : -dmin;
    }
    return m;
}

__device__ __forceinline__ void build_walk_masks(unsigned int* s_mask) {
    for (int e = threadIdx.x; e < kMaskEntries; e += blockDim.x) {
        int dmaj = 0;
        while ((dmaj + 1) * (dmaj + 2) / 2 <= e) ++dmaj;
        s_mask[e] = walk_mask_of(dmaj, e - dmaj * (dmaj + 1) / 2);
    }
}

template <bool kAdd>
__device__ __forceinline__ void smem_red(unsigned int addr, unsigned int v) {
    if (kAdd) asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
    else      asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Fast path of draw_beam_smem / count_beam_smem: both end points inside the window, dmaj <= 32.
// win = 32-bit shared-space address of the window; (x, y) window-local start cell.
//   kAdd = false: atomicMax of `v_free` on every cell but the last, `v_free | 1` on the last if hit
//   kAdd = true : += 1 on every cell but the last, += 0x10000 on the last if hit (count mode)
template <bool kAdd>
__device__ __forceinline__ void walk_beam_masked(unsigned int win, int pitch, int x, int y, int ddx, int ddy,
                                                 unsigned int v_free, bool hit, bool skip_first, const unsigned int* s_mask) {
    const int dx = abs(ddx), dy = abs(ddy);
    const bool xmajor = dx >= dy;
    const int dmaj = xmajor ? dx : dy, dmin = xmajor ? dy : dx;
    const int sx4 = ddx > 0 ? 4 : -4;
    const int sy4 = (ddy > 0 ? pitch : -pitch) * 4;
    const int step_maj = xmajor ? sx4 : sy4, step_min = xmajor ? sy4 : sx4;
    unsigned int mask = s_mask[dmaj * (dmaj + 1) / 2 + dmin];
    unsigned int a = win + (unsigned int)(y * pitch + x) * 4u;
    const unsigned int a_end = a + (unsigned int)((ddy * pitch + ddx) * 4);
    int rem = dmaj;                                   // cells still to mark FREE (the end cell is not one of them)
    if (rem > 0) {
        if (!skip_first) smem_red<kAdd>(a, v_free);   // the start cell is overwritten by a later beam of the packet otherwise
        a += step_maj + ((mask & 1u) ? step_min : 0);
        mask >>= 1;
        --rem;
    }
    // straight-line groups of 8 and 4 cells (no guard per cell: ptxas turns a guarded ATOMS into a
    // branch), then at most 3 single cells
    while (rem >= 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            smem_red<kAdd>(a, v_free);
            a += step_maj + ((mask & (1u << j)) ? step_min : 0);
        }
        mask >>= 8;
        rem -= 8;
    }
    if (rem >= 4) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            smem_red<kAdd>(a, v_free);
            a += step_maj + ((mask & (1u << j)) ? step_min : 0);
        }
        mask >>= 4;
        rem -= 4;
    }
    for (; rem > 0; --rem) {
        smem_red<kAdd>(a, v_free);
        a += step_maj + ((mask & 1u) ? step_min : 0);
        mask >>= 1;
    }
    if (hit && !(dmaj == 0 && skip_first && !kAdd)) smem_red<kAdd>(a_end, kAdd ? 0x10000u : (v_free | 1u));
}

// ---- route work item (multi-GPU row bands, fused into the persistent raycast kernel) -----------
// One item = kRouteItemPk packets of the NEXT batch, one per thread: decode (:828-843), pose
// correction (:851-857), robot cell (:142) -> the band(s) whose rows the packet's rays can reach
// and its home tile IN THAT BAND'S WINDOW; the 48-byte records are sorted by band in shared
// memory (the raycast window, free between two raycast items), a slot range is reserved in this
// rank's segment of every destination with a LOCAL atomic, and the runs are copied into the band
// owners' receive buffers over NVLink with fully coalesced 16-byte stores.  The stores are fire and
// forget: they drain while the CTA is already walking the next raycast item.
struct RouteSmem {
    unsigned int cnt[kMaxBands];        // entries per band of this item
    unsigned int off[kMaxBands + 1];    // exclusive offsets in the sorted buffer
    unsigned int base[kMaxBands];       // reserved first slot in my segment of band b (0xffffffff: overflow)
};

// 32-bit little-endian field at byte offset `byte_off` (any alignment) of a buffer staged in shared
// memory: two aligned word loads and a funnel shift instead of four byte loads.
__device__ __forceinline__ unsigned int lds_u32_at(const unsigned int* __restrict__ words, unsigned int byte_off) {
    const unsigned int w = byte_off >> 2, sh = (byte_off & 3u) * 8u;
    return __funnelshift_r(words[w], words[w + 1], sh);
}

// Same result as decode_packet (beam_expand.cuh) for a record staged in shared memory.
__device__ __forceinline__ int decode_packet_smem(const unsigned int* __restrict__ words, unsigned int byte_off, long long k,
                                                  const int32_t* agent_idx, const double* drift, const double* agent_off,
                                                  int n_agents, double* rx, double* ry, float* yaw, float dist[4]) {
    if (lds_u32_at(words, byte_off) != 0x4c525351u) return PKT_DROPPED;                      // 'QSRL' (:840)
    const unsigned int b4 = lds_u32_at(words, byte_off + 4);                                 // agent id, x[0..2]
    const long long agent = agent_idx ? (long long)agent_idx[k] : (long long)(b4 & 0xffu);
    if (agent < 1 || agent > n_agents) return PKT_DROPPED;                                   // :842
    const unsigned int b8 = lds_u32_at(words, byte_off + 8), b12 = lds_u32_at(words, byte_off + 12),
                       b16 = lds_u32_at(words, byte_off + 16);
    double x = (double)__uint_as_float(__funnelshift_r(b4, b8, 8));                          // bytes 5..8
    double y = (double)__uint_as_float(__funnelshift_r(b8, b12, 8));                         // bytes 9..12
    const float fyaw = __uint_as_float(__funnelshift_r(b12, b16, 8));                        // bytes 13..16
    x = OCC_DADD(x, agent_off[2 * agent + 0]);                                               // :851-852
    y = OCC_DADD(y, agent_off[2 * agent + 1]);
    if (drift) {                                                                             // :855-857
        const double2 dv = *reinterpret_cast<const double2*>(drift + 2 * k);
        x = OCC_DADD(x, dv.x);
        y = OCC_DADD(y, dv.y);
    }
    if (!(isfinite(x) && isfinite(y) && isfinite(fyaw))) return PKT_BAD_POSE;
    *rx = x; *ry = y; *yaw = fyaw;
    const unsigned int c24 = lds_u32_at(words, byte_off + 24), c28 = lds_u32_at(words, byte_off + 28),
                       c32 = lds_u32_at(words, byte_off + 32), c36 = lds_u32_at(words, byte_off + 36),
                       c40 = lds_u32_at(words, byte_off + 40);
    dist[0] = __uint_as_float(__funnelshift_r(c24, c28, 8));                                 // bytes 25..28
    dist[1] = __uint_as_float(__funnelshift_r(c28, c32, 8));
    dist[2] = __uint_as_float(__funnelshift_r(c32, c36, 8));
    dist[3] = __uint_as_float(__funnelshift_r(c36, c40, 8));                                 // bytes 37..40
    return PKT_OK;
}

// Robot cell along one axis: the screened quotient (r - o) * (1 / res) decides unless it lies within
// the tolerance of an integer, where the reference's true division (:123-124) is evaluated.
__device__ __forceinline__ bool robot_cell(double r, double o, double res, double inv_res, int* cell) {
    double q = OCC_DMUL(OCC_DADD(r, -o), inv_res);
    const double tol = OCC_DMUL(OCC_DMUL(fabs(r) + fabs(o) + 11.0, inv_res), 0x1p-47);
    if (near_cell_boundary(q, tol)) q = cell_quotient(r, o, res);
    if (!quotient_in_range(q)) return false;
    *cell = trunc_cell(q);
    return true;
}

// Statistics of the routed share, packed per thread (16 bits each, folded into the 64-bit counters
// when the kernel ends): a = packets | accepted << 16, b = dropped | hits << 16.
struct RouteStats { unsigned int a, b; };

constexpr int kRouteSubs = kRouteSubsPerItem;
constexpr int kRoutePerThread = kRouteItemPk / kTT;      // packets per thread and sub-batch
static_assert(kRouteItemPk % kTT == 0 && kRoutePerThread >= 1 && kRoutePerThread <= 4, "route sub-batch = 1..4 packets per thread");

// One decoded packet on its way to (at most) two band owners.
struct RoutePk {
    double rx, ry;
    float yaw, d[4];
    int band0, nb, tile0, tile1;        // bands are contiguous rows: the second band is band0 + 1
    unsigned int rank0, rank1;
};

__device__ __forceinline__ void route_decode(const RouteJob& J, const unsigned int* s_buf, int slot, long long k, RoutePk& P,
                                             RouteStats& st_acc) {
    P.band0 = -1; P.nb = 0; P.tile0 = P.tile1 = -1; P.rank0 = P.rank1 = 0u;
    const int st = decode_packet_smem(s_buf, (unsigned int)slot * (unsigned int)J.stride, k, J.agent_idx, J.drift, J.agent_off,
                                      J.n_agents, &P.rx, &P.ry, &P.yaw, P.d);
    st_acc.a += 1u + (st == PKT_OK ? 0x10000u : 0u);
    st_acc.b += st == PKT_DROPPED ? 1u : 0u;
    if (st != PKT_OK) return;
    unsigned int hits = 0;
#pragma unroll
    for (int s2 = 0; s2 < 4; ++s2) {
        const double dd = (double)P.d[s2];
        hits += (OCC_MIN_DIST_M < dd && dd <= OCC_MAX_DIST_M) ? 1u : 0u;                 // :888
    }
    st_acc.b += hits << 16;
    int gx, gy;
    if (!(robot_cell(P.rx, J.ox, J.res, J.inv_res, &gx) && robot_cell(P.ry, J.oy, J.res, J.inv_res, &gy))) return;
    const int reach = J.reach;
    if (gx < -reach || gx >= J.size_x + reach) return;
    const int tcol = (gx + J.pad) >> kTileShift;
    for (int b = 0; b < J.n_bands; ++b) {
        if (gy - reach < J.band_y0[b + 1]) {                                 // first band whose rows end above the reach interval
            const int py = gy - J.band_y0[b];
            if (py >= -reach) {
                P.band0 = b; P.nb = 1;
                P.tile0 = ((py + J.pad) >> kTileShift) * J.tiles_x + tcol;
                if (b + 1 < J.n_bands && gy + reach >= J.band_y0[b + 1]) {
                    P.nb = 2;
                    P.tile1 = ((gy - J.band_y0[b + 1] + J.pad) >> kTileShift) * J.tiles_x + tcol;
                }
            }
            break;
        }
    }
}

// rank of every entry inside its band's run (arrival order is free: ordinals travel in the records)
__device__ __forceinline__ void route_rank(RouteSmem& S, RoutePk& P, int lane, unsigned int lt) {
    const unsigned int p0 = __match_any_sync(0xffffffffu, P.band0);
    if (P.band0 >= 0) {
        const int leader = __ffs(p0) - 1;
        unsigned int b0 = 0;
        if (lane == leader) b0 = atomicAdd(&S.cnt[P.band0], (unsigned int)__popc(p0));
        P.rank0 = __shfl_sync(p0, b0, leader) + __popc(p0 & lt);
    }
    if (__any_sync(0xffffffffu, P.nb == 2)) {                            // rare: only next to a band edge
        const unsigned int p1 = __match_any_sync(0xffffffffu, P.nb == 2 ? P.band0 + 1 : -1);
        if (P.nb == 2) {
            const int leader = __ffs(p1) - 1;
            unsigned int b1 = 0;
            if (lane == leader) b1 = atomicAdd(&S.cnt[P.band0 + 1], (unsigned int)__popc(p1));
            P.rank1 = __shfl_sync(p1, b1, leader) + __popc(p1 & lt);
        }
    }
}

__device__ __forceinline__ void route_store(const RouteJob& J, uint4* s16, const RoutePk& P, unsigned int my_off, long long k) {
    const unsigned int o0 = __shfl_sync(0xffffffffu, my_off, P.band0 < 0 ? 0 : P.band0);
    const unsigned long long ux = (unsigned long long)__double_as_longlong(P.rx), uy = (unsigned long long)__double_as_longlong(P.ry);
    const uint4 w0 = make_uint4((unsigned int)ux, (unsigned int)(ux >> 32), (unsigned int)uy, (unsigned int)(uy >> 32));
    const uint4 w1 = make_uint4(__float_as_uint(P.yaw), __float_as_uint(P.d[0]), __float_as_uint(P.d[1]), __float_as_uint(P.d[2]));
    const unsigned int ord = J.ordinal_base + (unsigned int)k;
    if (P.band0 >= 0) {                                                  // struct occgrid_pose_rec, 3 x 16 bytes
        uint4* dst = s16 + (size_t)(o0 + P.rank0) * 3;
        dst[0] = w0; dst[1] = w1; dst[2] = make_uint4(__float_as_uint(P.d[3]), ord, (unsigned int)P.tile0, 0u);
    }
    if (__any_sync(0xffffffffu, P.nb == 2)) {
        const unsigned int o1 = __shfl_sync(0xffffffffu, my_off, P.nb == 2 ? P.band0 + 1 : 0);
        if (P.nb == 2) {
            uint4* dst = s16 + (size_t)(o1 + P.rank1) * 3;
            dst[0] = w0; dst[1] = w1; dst[2] = make_uint4(__float_as_uint(P.d[3]), ord, (unsigned int)P.tile1, 0u);
        }
    }
}

__device__ __noinline__ RouteStats route_item(const RouteJob& J, unsigned int item, unsigned int* s_buf /* >= kRouteItemPk * 96 B */,
                                              RouteSmem& S, RouteStats st_in) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned int lt = (1u << lane) - 1u;
    long long first = (long long)item * (kRouteItemPk * kRouteSubs);
    for (int sub = 0; sub < kRouteSubs; ++sub, first += kRouteItemPk) {
        const int count = (int)max(0ll, min((long long)kRouteItemPk, J.n - first));
        if (count == 0) break;                                           // uniform across the CTA
        __syncthreads();                                                 // the previous sub-batch's copy-out has left the buffer
        if (threadIdx.x < kMaxBands) S.cnt[threadIdx.x] = 0u;
        {   // staging with every load of the thread in flight before the first store (a load-store loop
            // would pay one DRAM latency per iteration)
            const uint8_t* src = J.pkts + (size_t)first * J.stride;
            const size_t bytes = (size_t)count * J.stride;
            constexpr int kVec = kRouteItemPk * kMaxRecStride / 16 / kTT;         // <= 8 chunks of 16 bytes per thread
            if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                const uint4* s4 = reinterpret_cast<const uint4*>(src);
                uint4* d4 = reinterpret_cast<uint4*>(s_buf);
                const size_t nvec = bytes / 16;
                uint4 v[kVec];
#pragma unroll
                for (int j = 0; j < kVec; ++j) {
                    const size_t i = (size_t)j * kTT + threadIdx.x;
                    if (i < nvec) v[j] = __ldg(s4 + i);
                }
#pragma unroll
                for (int j = 0; j < kVec; ++j) {
                    const size_t i = (size_t)j * kTT + threadIdx.x;
                    if (i < nvec) d4[i] = v[j];
                }
                for (size_t i = nvec * 16 + threadIdx.x; i < bytes; i += kTT) reinterpret_cast<uint8_t*>(s_buf)[i] = __ldg(src + i);
            } else {
                stage_records(src, bytes, reinterpret_cast<uint8_t*>(s_buf));
            }
        }
        {   // pull the NEXT sub-batch towards L2 while this one is decoded, sorted and copied out
            const long long nf = first + kRouteItemPk;
            const long long nbytes = max(0ll, min((long long)kRouteItemPk, J.n - nf)) * J.stride;
            const long long o = (long long)threadIdx.x * 128;
            if (sub + 1 < kRouteSubs && o < nbytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(J.pkts + (size_t)nf * J.stride + o));
        }
        __syncthreads();
        RoutePk P[kRoutePerThread];
#pragma unroll
        for (int u = 0; u < kRoutePerThread; ++u) {                      // decode first (the table loads of all packets overlap) ...
            const int slot = u * kTT + threadIdx.x;
            P[u].band0 = -1; P[u].nb = 0;
            if (slot < count) route_decode(J, s_buf, slot, first + slot, P[u], st_in);
        }
#pragma unroll
        for (int u = 0; u < kRoutePerThread; ++u) route_rank(S, P[u], lane, lt);   // ... then the warp-level ranking
        __syncthreads();                                                 // counts complete; raw packets decoded: the buffer is free
        // every warp scans the <= 32 band counts in registers (lane b holds band b)
        const unsigned int n_b = lane < J.n_bands ? S.cnt[lane] : 0u;
        unsigned int inc = n_b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const unsigned int my_off = inc - n_b;                           // exclusive offset of band `lane` in the sorted buffer
        if (warp == 0) {                                                 // one reservation per band and sub-batch, on a LOCAL counter
            unsigned int base = 0u;
            if (n_b) {
                base = atomicAdd(&J.resv[lane], n_b);
                if (base + n_b > J.seg_cap) { atomicOr(J.status, 2); base = 0xffffffffu; }
            }
            S.base[lane] = base;                                         // (its latency overlaps the record stores below)
            S.off[lane] = my_off;
            if (lane == 31) S.off[32] = inc;
        }
        uint4* s16 = reinterpret_cast<uint4*>(s_buf);
#pragma unroll
        for (int u = 0; u < kRoutePerThread; ++u) route_store(J, s16, P[u], my_off, first + u * kTT + threadIdx.x);
        __syncthreads();
        // copy-out: one contiguous run per band, all threads on it: consecutive threads -> consecutive
        // 16-byte chunks in the owner's segment (full NVLink / HBM write transactions)
        for (int b = 0; b < J.n_bands; ++b) {
            const unsigned int base = S.base[b];
            const unsigned int n_rec = S.off[b + 1] - S.off[b];
            if (n_rec == 0u || base == 0xffffffffu) continue;                // uniform across the CTA
            const size_t slot0 = (size_t)J.src_rank * J.seg_cap + base;
            uint4* out = reinterpret_cast<uint4*>(J.peer_recs[b] + slot0);
            const uint4* in = s16 + (size_t)S.off[b] * 3;
            for (unsigned int q = threadIdx.x; q < n_rec * 3u; q += kTT) out[q] = in[q];
            // compact copy of the tile ids (word 10 of every record): the owner bins from 4 bytes per record
            int* tout = J.peer_tiles[b] + slot0;
            const unsigned int* tin = s_buf + (size_t)S.off[b] * 12 + 10;
            for (unsigned int q = threadIdx.x; q < n_rec; q += kTT) tout[q] = (int)tin[(size_t)q * 12];
        }
    }
    return st_in;
}

// Route items that precede position i of the unified work queue (see k_home_raycast): half of them
// are interleaved with the raycast items, half close the queue.  Measured (fused kernel, bit-exact
// throughout): all interleaved 0.343 ms at N = 2 / 0.396 at N = 8; a quarter at the end 0.323 / -;
// half 0.315 / 0.386; all at the end 0.311 / 0.409 (the route-only phase is NVLink-bound at N = 8).
#define OCC_ROUTE_TAIL_DIV 2
__device__ __forceinline__ unsigned int route_items_before(unsigned int i, unsigned int n_items, unsigned int n_route) {
    const unsigned int tail = n_items ? n_route / OCC_ROUTE_TAIL_DIV : 0u;      // route items kept for the end of the queue
    const unsigned int n_body = n_route - tail, n_head = n_items + n_body;
    if (i >= n_head) return n_body + (i - n_head);
    return (unsigned int)(((unsigned long long)i * n_body) / n_head);
}

// Three CTAs per SM (80 registers): measured 0.204 ms against 0.248 (two CTAs, <= 128 registers)
// and 0.256 (four CTAs, 64 registers with spills) on BASELINE configs[1].
// kMaps: item.x is a key (map * n_tiles + tile, see k_home_bin); the map selects the stamp plane.
template <bool kCounts, bool kRoute, bool kMaps = false>
__global__ void __launch_bounds__(kTT, 3)
k_home_raycast(Geom g, TileGeom tg, const uint4* __restrict__ items, TilePlanHeader* __restrict__ hdr,
               const unsigned int* __restrict__ bins, const PoseRec* __restrict__ recs, int ordinals_in_records,
               unsigned int* __restrict__ stamps, uint64_t* counters, int have_items, const RouteJob job) {
    extern __shared__ __align__(16) unsigned int s_win[];
    unsigned long long* const s_acc = reinterpret_cast<unsigned long long*>(s_win);   // [6 * 32], used once the window is dead
    __shared__ RouteSmem s_route;
    __shared__ unsigned int s_mask[kMaskEntries];
    __shared__ RouteJob s_job;                     // the route path reads the job from shared memory, not from a stack copy
    if (kRoute && threadIdx.x == 0) s_job = job;
    build_walk_masks(s_mask);                      // both visible after the first __syncthreads of the loop below
    const unsigned int win_addr = (unsigned int)__cvta_generic_to_shared(s_win);
    const unsigned int n_items = have_items ? hdr->n_items : 0u;
    // Unified queue: raycast items of THIS batch and route items of the NEXT one, interleaved in
    // proportion, so the NVLink traffic is spread over the whole kernel and overlaps the walks.
    const unsigned int n_route = kRoute ? job.n_route_items : 0u;
    const unsigned int n_total = n_items + n_route;
    const int side = tg.win_side, pitch = tg.pitch, words = side * pitch;
    unsigned long long c[3] = {0, 0, 0};     // updates, slowpath, owned updates
    RouteStats rs = {0u, 0u};                // routed share, packed (see RouteStats)
    // Work queue: the position of the next item is claimed while the current one is flushed (the
    // atomic's round trip to L2 is off the critical path), and without route items the flush
    // itself leaves the window clean: an item costs two CTA barriers and no clearing pass.
    __shared__ unsigned int s_next[2];
    if (threadIdx.x == 0) s_next[0] = atomicAdd(&hdr->work_counter, 1u);
    for (int i = threadIdx.x; i < words; i += kTT) s_win[i] = 0u;
    __syncthreads();
    for (int turn = 0;; turn ^= 1) {
        unsigned int it = s_next[turn];
        if (it >= n_total) break;
        if (kRoute) {
            // Route items precede queue position i: r(i) = floor(i * n_body / n_head) in the head of the
            // queue (all raycast items + n_body route items, interleaved in proportion), then the
            // remaining route items on their own: the queue ends with SHORT items, so no CTA starts
            // a 2 048-packet raycast item while the others run dry.
            const unsigned int r0 = route_items_before(it, n_items, n_route), r1 = route_items_before(it + 1u, n_items, n_route);
            if (r1 > r0) {
                if (threadIdx.x == 0) s_next[turn ^ 1] = atomicAdd(&hdr->work_counter, 1u);   // a route item is short
                rs = route_item(s_job, r0, s_win, s_route, rs);
                __syncthreads();
                continue;
            }
            it -= r0;
            // route items use the window as scratch and outnumber the raycast items: clear it here,
            // in full, and let the flush below leave it alone
            for (int i = threadIdx.x; i < words; i += kTT) s_win[i] = 0u;
            __syncthreads();
        }
        const uint4 item = items[it];
        const unsigned int map = kMaps ? item.x / (unsigned int)tg.n_tiles : 0u;
        const unsigned int tile = item.x - map * (unsigned int)tg.n_tiles;
        unsigned int* __restrict__ const plane = kMaps ? stamps + (size_t)map * ((size_t)g.win_w * g.win_h) : stamps;
        const int ttx = tile % tg.tiles_x, tty = tile / tg.tiles_x;
        // global cell of window-local (0, 0)
        const int wx0 = g.win_x0 - tg.pad + (ttx << kTileShift) - tg.reach;
        const int wy0 = g.win_y0 - tg.pad + (tty << kTileShift) - tg.reach;
        for (unsigned int r = item.y + threadIdx.x; r < item.z; r += kTT) {
            const unsigned int idx = bins[r];
            const PoseRec rec = recs[idx];
            const unsigned int k = ordinals_in_records ? rec.k : idx;   // packet ordinal in this batch
            PacketFrame F;
            packet_frame(g, rec.rx, rec.ry, (double)rec.yaw, LibSinCos(), &F);
            const bool owned = F.x0 >= g.win_x0 && F.x0 < g.win_x0 + g.win_w && F.y0 >= g.win_y0 && F.y0 < g.win_y0 + g.win_h;
            const int lx = F.x0 - wx0, ly = F.y0 - wy0;
            const unsigned int us = (unsigned int)side;
            bool later_writes_first = false;
            // ONE copy of the expansion + walk code, looped over the four sensors (last sensor first:
            // only the last beam that writes the shared start cell has to touch it).  Unrolling it
            // four times made the kernel 110 KB of SASS and instruction-fetch bound.
#pragma unroll 1
            for (int s = 3; s >= 0; --s) {
                Beam b;
                expand_beam_of(g, F, s, s == 0 ? rec.d[0] : (s == 1 ? rec.d[1] : (s == 2 ? rec.d[2] : rec.d[3])), LibSinCos(), &b);
                if (!b.valid) continue;
                const int cells = beam_cells(b);
                c[0] += cells;
                c[1] += b.slow;
                if (owned) c[2] += cells;
                const int ddx = b.x1 - b.x0, ddy = b.y1 - b.y0;
                const bool fast = (unsigned int)lx < us && (unsigned int)ly < us && (unsigned int)(lx + ddx) < us &&
                                  (unsigned int)(ly + ddy) < us && cells <= kMaskMaxLen + 1;
                if (kCounts) {
                    if (fast) walk_beam_masked<true>(win_addr, pitch, lx, ly, ddx, ddy, 1u, b.hit != 0, false, s_mask);
                    else count_beam_smem(s_win, side, pitch, lx, ly, ddx, ddy, b.hit != 0);
                } else {
                    const unsigned int stamp = (k * 4u + (unsigned int)s + 1u) << 1;
                    if (fast) walk_beam_masked<false>(win_addr, pitch, lx, ly, ddx, ddy, stamp, b.hit != 0, later_writes_first, s_mask);
                    else draw_beam_smem(s_win, side, pitch, lx, ly, ddx, ddy, stamp, b.hit != 0, later_writes_first);
                }
                later_writes_first = later_writes_first || (cells > 1 || b.hit);
            }
        }
        // Bind the next queue position late — a raycast item is long, and an item claimed early
        // waits for this CTA while others idle at the end of the queue — but keep the atomic's round
        // trip off the critical path: it is issued here and consumed after the flush.
        unsigned int next_pos = 0u;
        if (threadIdx.x == 0) next_pos = atomicAdd(&hdr->work_counter, 1u);
        __syncthreads();
        // flush + clear: window rows are contiguous in the stamp plane -> coalesced reductions.  Every
        // touched word is zeroed on the way out (cells outside the grid window included: they are
        // dropped, not flushed), so the next item finds a clean window.
        {
            const int lx_lo = max(0, g.win_x0 - wx0), lx_hi = min(side, g.win_x0 + g.win_w - wx0);
            const int ly_lo = max(0, g.win_y0 - wy0), ly_hi = min(side, g.win_y0 + g.win_h - wy0);
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            for (int ly = warp; ly < side; ly += kTT / 32) {                   // one warp per window row
                unsigned int* row = s_win + ly * pitch;
                const bool row_in = ly >= ly_lo && ly < ly_hi;
                unsigned int* out = plane + (size_t)(wy0 + ly - g.win_y0) * g.win_w + (wx0 - g.win_x0);
                for (int lx = lane; lx < side; lx += 32) {
                    const unsigned int v = row[lx];
                    if (!v) continue;
                    if (!kRoute) row[lx] = 0u;
                    if (!(row_in && lx >= lx_lo && lx < lx_hi)) continue;
                    if (kCounts)     // {miss, hit} int32 pair of the cell: one 64-bit add (the halves cannot carry into each other)
                        atomicAdd(reinterpret_cast<unsigned long long*>(plane) + ((size_t)(wy0 + ly - g.win_y0) * g.win_w + (wx0 - g.win_x0) + lx),
                                  ((unsigned long long)(v >> 16) << 32) | (unsigned long long)(v & 0xffffu));
                    else
                        atomicMax(out + lx, v);
                }
            }
        }
        if (threadIdx.x == 0) s_next[turn ^ 1] = next_pos;
        __syncthreads();
    }
    if (kRoute && job.counters) {
        __syncthreads();
        const unsigned long long pk = rs.a & 0xffffu, acc = rs.a >> 16, drp = rs.b & 0xffffu, hits = rs.b >> 16;
        const unsigned long long rc[6] = {pk, acc, drp, pk - acc - drp, 4ull * acc, hits};
        block_add_counters(rc, s_acc, job.counters);            // slots OCCGRID_C_PACKETS .. OCCGRID_C_HITS
    }
    if (counters) {
        __syncthreads();
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            unsigned long long x = c[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if (lane == 0) s_acc[i * 32 + warp] = x;
        }
        __syncthreads();
        if (threadIdx.x < 3) {
            unsigned long long t = 0;
            for (int w = 0; w < kTT / 32; ++w) t += s_acc[threadIdx.x * 32 + w];
            const int slot = threadIdx.x == 0 ? OCCGRID_C_UPDATES : (threadIdx.x == 1 ? OCCGRID_C_SLOWPATH : OCCGRID_C_OWNED_UPDATES);
            if (t) atomicAdd(reinterpret_cast<unsigned long long*>(counters) + slot, t);
        }
    }
}

constexpr int kResolveSplit = 8;      // CTAs per active window (row slices) — few tiles are active, keep all SMs busy

// kMaps: the active list holds keys (see k_home_bin); the map selects the stamp plane and the grid.
template <bool kMaps = false>
__global__ void __launch_bounds__(kTT)
k_home_resolve(Geom g, TileGeom tg, const unsigned int* __restrict__ active, TilePlanHeader* __restrict__ hdr,
               unsigned int* __restrict__ stamps, int8_t* __restrict__ grid) {
    __shared__ unsigned int s_item;
    const unsigned int n_work = hdr->n_active * kResolveSplit;
    const int side = tg.win_side;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_item = atomicAdd(&hdr->resolve_counter, 1u);
        __syncthreads();
        const unsigned int it = s_item;
        if (it >= n_work) break;
        const unsigned int key = active[it / kResolveSplit];
        const unsigned int map = kMaps ? key / (unsigned int)tg.n_tiles : 0u;
        const unsigned int t = key - map * (unsigned int)tg.n_tiles;
        const size_t map_off = kMaps ? (size_t)map * ((size_t)g.win_w * g.win_h) : 0;
        unsigned int* __restrict__ const plane = stamps + map_off;
        int8_t* __restrict__ const map_grid = grid + map_off;
        const int part = (int)(it % kResolveSplit);
        const int ttx = t % tg.tiles_x, tty = t / tg.tiles_x;
        const int wx0 = -tg.pad + (ttx << kTileShift) - tg.reach;      // window-relative
        const int wy0 = -tg.pad + (tty << kTileShift) - tg.reach;
        const int lx_lo = max(0, -wx0), lx_hi = min(side, g.win_w - wx0);
        const int ly_lo = max(0, -wy0), ly_hi = min(side, g.win_h - wy0);
        if (lx_hi <= lx_lo) continue;
        for (int ly = ly_lo + part * (kTT / 32) + warp; ly < ly_hi; ly += kResolveSplit * (kTT / 32)) {   // one warp per row
            const size_t row = (size_t)(wy0 + ly) * g.win_w + wx0;
            for (int lx = lx_lo + lane; lx < lx_hi; lx += 32) {
                const unsigned int s = plane[row + lx];
                if (s) {
                    map_grid[row + lx] = (s & 1u) ? OCCGRID_CELL_OCCUPIED : OCCGRID_CELL_FREE;
                    plane[row + lx] = 0u;
                }
            }
        }
    }
}

// ---- host side ----------------------------------------------------------------------------

// Persistent raycast CTAs per SM (0 = as many as fit).  A multi-GPU pipeline lowers it so that
// the routing kernel of the next batch can be co-resident (occgrid_set_raycast_ctas_per_sm).
static int g_raycast_cta_cap = 0;
void set_raycast_cta_cap(int cap) { g_raycast_cta_cap = cap < 0 ? 0 : cap; }

struct TiledLayout {
    size_t off_stamps, off_count, off_offset, off_cursor, off_active, off_hdr, off_items, off_ids, off_bins, off_local, off_runs,
        off_segs, off_recs, total;
    unsigned long long max_records;
    unsigned int max_items;
};

// max_records = record ADDRESSES the bins must cover.  packets: the arrays of k_home_bin for a
// packet batch (local bins, runs, segment counts, decoded records); else the tile ids that
// k_home_count_poses hands to the scatter (input that arrives decoded brings its own records).
// n_maps > 1 (agent maps, packets only): one stamp plane per map and per-key tile arrays, key =
// map * n_tiles + tile.
static TiledLayout tiled_layout(const occgrid_geom* geom, int64_t max_records, bool packets, int n_maps = 1) {
    TiledLayout L;
    const TileGeom tg = tile_geom(geom);
    const size_t n_keys = (size_t)n_maps * tg.n_tiles;
    L.max_records = (unsigned long long)max_records;
    unsigned long long items = L.max_records / kChunkMin + (unsigned long long)n_keys + 1;
    if (items > L.max_records + 1) items = L.max_records + 1;
    L.max_items = (unsigned int)items;
    size_t o = 0;
    L.off_stamps = o; o += align_up((size_t)geom->win_w * geom->win_h * 4 * (size_t)n_maps, 256);
    L.off_count = o;  o += align_up((n_keys + 1) * 4, 256);
    L.off_offset = o; o += align_up((n_keys + 1) * 4, 256);
    L.off_cursor = o; o += align_up((n_keys + 1) * 4, 256);
    L.off_active = o; o += align_up((n_keys + 1) * 4, 256);
    L.off_hdr = o;    o += 256;
    L.off_items = o;  o += align_up((size_t)L.max_items * sizeof(uint4), 256);
    L.off_ids = o;    o += packets ? 0 : align_up((size_t)L.max_records * sizeof(int), 256);
    L.off_bins = o;   o += align_up((size_t)L.max_records * sizeof(unsigned int), 256);
    L.off_local = o;  o += packets ? align_up((size_t)L.max_records * sizeof(unsigned int), 256) : 0;
    L.off_runs = o;   o += packets ? align_up((size_t)L.max_records * sizeof(uint2), 256) : 0;     // worst case: a run per packet
    L.off_segs = o;   o += packets ? align_up((size_t)(L.max_records + kPkPerCta - 1) / kPkPerCta * sizeof(unsigned int), 256) : 0;
    L.off_recs = o;   o += packets ? align_up((size_t)L.max_records * sizeof(PoseRec), 256) : 0;
    L.total = o;
    return L;
}

bool tiled_supported(const occgrid_geom* geom, int n_maps) {
    const TileGeom tg = tile_geom(geom);
    return (size_t)tg.win_side * tg.pitch * 4 <= (size_t)kMaxWindowBytes && (long long)n_maps * tg.n_tiles <= (1ll << 24);
}

size_t tiled_workspace_bytes(const occgrid_geom* geom, int n_maps, int64_t max_packets) {
    return tiled_layout(geom, max_packets < 1 ? 1 : max_packets, true, n_maps).total;
}

size_t tiled_band_workspace_bytes(const occgrid_geom* geom, int n_segs, int64_t seg_cap) {
    return tiled_layout(geom, (int64_t)n_segs * seg_cap, false).total;
}

struct TiledPtrs {
    unsigned int *stamps, *tile_count, *tile_offset, *tile_cursor, *active, *bins, *local_bins, *seg_count;
    TilePlanHeader* hdr;
    uint4* items;
    int* tile_ids;
    uint2* runs;
    PoseRec* recs;
};

static TiledPtrs tiled_ptrs(const TiledLayout& L, void* d_ws) {
    char* ws = reinterpret_cast<char*>(d_ws);
    TiledPtrs p;
    p.stamps = reinterpret_cast<unsigned int*>(ws + L.off_stamps);
    p.tile_count = reinterpret_cast<unsigned int*>(ws + L.off_count);
    p.tile_offset = reinterpret_cast<unsigned int*>(ws + L.off_offset);
    p.tile_cursor = reinterpret_cast<unsigned int*>(ws + L.off_cursor);
    p.active = reinterpret_cast<unsigned int*>(ws + L.off_active);
    p.hdr = reinterpret_cast<TilePlanHeader*>(ws + L.off_hdr);
    p.items = reinterpret_cast<uint4*>(ws + L.off_items);
    p.bins = reinterpret_cast<unsigned int*>(ws + L.off_bins);
    p.tile_ids = reinterpret_cast<int*>(ws + L.off_ids);
    p.local_bins = reinterpret_cast<unsigned int*>(ws + L.off_local);
    p.runs = reinterpret_cast<uint2*>(ws + L.off_runs);
    p.seg_count = reinterpret_cast<unsigned int*>(ws + L.off_segs);
    p.recs = reinterpret_cast<PoseRec*>(ws + L.off_recs);
    return p;
}

// Dynamic shared memory of the raycast kernel: the stamp window, or the route item's staging
// buffer (raw packets, then <= 2 records per packet) when that is larger.
static size_t raycast_smem(const TileGeom& tg, bool route) {
    size_t b = (size_t)tg.win_side * tg.pitch * 4;
    const size_t r = (size_t)kRouteItemPk * 2 * sizeof(PoseRec);   // every packet may go to two bands
    const size_t raw = (size_t)kRouteItemPk * kMaxRecStride;
    if (route) b = b > r ? b : r;
    if (route) b = b > raw ? b : raw;
    return b;
}

template <bool kCounts, bool kRoute, bool kMaps = false>
static int launch_raycast(const Geom& g, const TileGeom& tg, const TiledPtrs& P, const PoseRec* recs, int ordinals_in_records,
                          unsigned int* plane, uint64_t* d_counters, int have_items, const RouteJob& job, cudaStream_t st) {
    const size_t smem = raycast_smem(tg, kRoute);
    static thread_local size_t configured = 0;
    if (smem > configured) {
        OCC_CUDA_TRY(cudaFuncSetAttribute(k_home_raycast<kCounts, kRoute, kMaps>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    int ctas_per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, k_home_raycast<kCounts, kRoute, kMaps>, kTT, smem) != cudaSuccess || ctas_per_sm < 1)
        ctas_per_sm = 1;
    if (g_raycast_cta_cap > 0 && ctas_per_sm > g_raycast_cta_cap) ctas_per_sm = g_raycast_cta_cap;
    ProfileScope ps(K_TILE_RAYCAST, st);
    k_home_raycast<kCounts, kRoute, kMaps><<<device_sm_count() * ctas_per_sm, kTT, smem, st>>>(g, tg, P.items, P.hdr, P.bins, recs,
                                                                                               ordinals_in_records, plane, d_counters,
                                                                                               have_items, job);
    return OCCGRID_OK;
}

// Work items the plan aims for: kItemsPerCta per persistent raycast CTA (three CTAs per SM).
static unsigned int plan_target_items() { return (unsigned int)device_sm_count() * 3u * (unsigned int)kItemsPerCta; }

static int grid_chunks(long long n_chunks) {
    long long b = n_chunks < 1 ? 1 : n_chunks;
    const long long cap = (long long)device_sm_count() * 8;
    return (int)(b < cap ? b : cap);
}

// Pose records are binned like a band's receive slot of one segment: count, plan and scatter run
// over 2048-record chunks of it.
int integrate_tiled(const occgrid_geom* geom, const PacketBatch& batch, const PoseRec* d_poses, int ordinals_in_records, Output kind,
                    void* d_out, void* d_ws, size_t ws_bytes, uint64_t* d_counters, cudaStream_t st) {
    const int64_t n = batch.n;
    const bool maps = kind == Output::kAgentMaps;
    const TiledLayout L = tiled_layout(geom, n, d_poses == nullptr, maps ? batch.n_agents : 1);
    if (ws_bytes < L.total) {
        set_last_error("workspace %zu B < %zu B needed by TILED for %lld records", ws_bytes, L.total, (long long)n);
        return OCCGRID_E_WORKSPACE;
    }
    const TiledPtrs P = tiled_ptrs(L, d_ws);
    const PoseRec* recs = d_poses ? d_poses : P.recs;
    const Geom g = to_geom(geom);
    const TileGeom tg = tile_geom(geom);
    const unsigned int blocks = (unsigned int)((n + kPkPerCta - 1) / kPkPerCta);
    SegInfo seg;
    seg.n_segs = 1; seg.seg_cap = (unsigned int)align_up((size_t)n, kSegChunk); seg.d_counts = nullptr; seg.host_count = (unsigned int)n;
    const long long n_chunks = (n + kSegChunk - 1) / kSegChunk;
    {
        ProfileScope ps(K_TILE_COUNT, st);
        if (d_poses) {
            k_home_count_poses<<<grid_chunks(n_chunks), kTT, 0, st>>>(g, tg, d_poses, nullptr, seg, n_chunks, 0, P.tile_count, P.tile_ids, P.active,
                                                                      P.hdr, d_counters);
        } else {
            const auto bin = maps ? k_home_bin<true> : k_home_bin<false>;
            OCC_CUDA_TRY(cudaFuncSetAttribute(bin, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBinSmem));
            bin<<<blocks, kTT, kBinSmem, st>>>(g, tg, batch.pkts, n, batch.stride, batch.agent_idx, batch.drift, batch.agent_off, batch.n_agents,
                                               P.tile_count, P.recs, P.local_bins, P.runs, P.seg_count, P.active, P.hdr, d_counters);
        }
    }
    {
        ProfileScope ps(K_TILE_SCAN, st);
        k_tile_plan<<<1, 1024, 0, st>>>(P.tile_count, P.tile_offset, P.tile_cursor, P.items, L.max_items, P.active, L.max_records, P.hdr,
                                        d_counters, plan_target_items());
    }
    {
        ProfileScope ps(K_TILE_SCATTER, st);
        if (d_poses) k_home_scatter_segs<<<grid_chunks(n_chunks), kTT, 0, st>>>(seg, n_chunks, P.tile_ids, P.tile_offset, P.tile_cursor, P.hdr, P.bins);
        else         k_place_runs<<<blocks, kTT, 0, st>>>(P.local_bins, P.runs, P.seg_count, P.tile_offset, P.hdr, P.bins);
    }
    RouteJob none = {};
    unsigned int* const plane = kind == Output::kCounts ? reinterpret_cast<unsigned int*>(d_out) : P.stamps;
    if (kind == Output::kCounts) launch_raycast<true, false>(g, tg, P, recs, ordinals_in_records, plane, d_counters, 1, none, st);
    else if (maps)               launch_raycast<false, false, true>(g, tg, P, recs, ordinals_in_records, plane, d_counters, 1, none, st);
    else                         launch_raycast<false, false>(g, tg, P, recs, ordinals_in_records, plane, d_counters, 1, none, st);
    if (kind != Output::kCounts) {
        ProfileScope ps(K_TILE_RESOLVE, st);
        const auto resolve = maps ? k_home_resolve<true> : k_home_resolve<false>;
        resolve<<<device_sm_count() * 8, kTT, 0, st>>>(g, tg, P.active, P.hdr, P.stamps, reinterpret_cast<int8_t*>(d_out));
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// ---- multi-GPU band step (include/occgrid_b200.h: occgrid_band_*) ---------------------------
// count -> plan -> scatter over the per-source segments of a receive slot.
int tiled_prepare_poses(const occgrid_geom* geom, const PoseRec* d_recs, const int* d_tiles, const SegInfo& seg, int tiles_in_records,
                        void* d_ws, size_t ws_bytes, uint64_t* d_counters, cudaStream_t st) {
    const int64_t max_records = (int64_t)seg.n_segs * seg.seg_cap;
    const TiledLayout L = tiled_layout(geom, max_records, false);
    if (ws_bytes < L.total) {
        set_last_error("workspace %zu B < %zu B needed by the band step for %lld record addresses", ws_bytes, L.total, (long long)max_records);
        return OCCGRID_E_WORKSPACE;
    }
    const TiledPtrs P = tiled_ptrs(L, d_ws);
    const Geom g = to_geom(geom);
    const TileGeom tg = tile_geom(geom);
    const long long n_chunks = max_records / kSegChunk;
    {
        ProfileScope ps(K_TILE_COUNT, st);
        k_home_count_poses<<<grid_chunks(n_chunks), kTT, 0, st>>>(g, tg, d_recs, d_tiles, seg, n_chunks, tiles_in_records, P.tile_count, P.tile_ids,
                                                                  P.active, P.hdr, d_counters);
    }
    {
        ProfileScope ps(K_TILE_SCAN, st);
        k_tile_plan<<<1, 1024, 0, st>>>(P.tile_count, P.tile_offset, P.tile_cursor, P.items, L.max_items, P.active, L.max_records, P.hdr,
                                        d_counters, plan_target_items());
    }
    {
        ProfileScope ps(K_TILE_SCATTER, st);
        k_home_scatter_segs<<<grid_chunks(n_chunks), kTT, 0, st>>>(seg, n_chunks, P.tile_ids, P.tile_offset, P.tile_cursor, P.hdr, P.bins);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

// The fused kernel: raycast the prepared batch (have_items) and, in between its work items, decode
// and push the NEXT batch to the band owners (job != NULL); then resolve.
int tiled_raycast_route(const occgrid_geom* geom, const PoseRec* d_recs, int have_items, const RouteJob* job,
                        int8_t* d_grid, void* d_ws, size_t ws_bytes, int64_t max_records, uint64_t* d_counters, cudaStream_t st,
                        cudaEvent_t after_fused) {
    const TiledLayout L = tiled_layout(geom, max_records, false);
    if (ws_bytes < L.total) { set_last_error("workspace too small for the band step"); return OCCGRID_E_WORKSPACE; }
    const TiledPtrs P = tiled_ptrs(L, d_ws);
    const Geom g = to_geom(geom);
    const TileGeom tg = tile_geom(geom);
    if (!have_items) {
        // nothing prepared (first step of a stream): the header still has to carry a clean queue
        OCC_CUDA_TRY(cudaMemsetAsync(P.hdr, 0, sizeof(TilePlanHeader), st));
    }
    if (job) {
        launch_raycast<false, true>(g, tg, P, d_recs, 1, P.stamps, d_counters, have_items, *job, st);
    } else {
        RouteJob none = {};
        launch_raycast<false, false>(g, tg, P, d_recs, 1, P.stamps, d_counters, have_items, none, st);
    }
    if (after_fused) OCC_CUDA_TRY(cudaEventRecord(after_fused, st));      // the routed batch is out: publishing may overlap the resolve
    if (have_items) {
        ProfileScope ps(K_TILE_RESOLVE, st);
        k_home_resolve<false><<<device_sm_count() * 8, kTT, 0, st>>>(g, tg, P.active, P.hdr, P.stamps, d_grid);
    }
    OCC_CUDA_TRY(cudaGetLastError());
    return OCCGRID_OK;
}

}  // namespace occ
