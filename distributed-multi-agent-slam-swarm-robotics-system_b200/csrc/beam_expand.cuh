// Packet decode, pose correction and beam expansion — the arithmetic of
// server_nodes/dual_bot_mapper.py:826-903 and OccupancyGrid.world_to_grid (:121-125),
// written once for host and device (the CPU test-suite compiles this header with g++ and
// checks it against the oracle; the CUDA kernels include the same code).
//
// Parity rules (SURVEY.md Appendix A): fp32 wire fields widen to fp64 before any
// arithmetic; every fp64 operation is individually rounded (no FMA contraction:
// `rx + dist * cos(a)` is a multiply then an add in CPython); cells = trunc((w - o) / res)
// with a true division and truncation toward zero.
#pragma once
#include "sincos_dd.cuh"

namespace occ {

struct Geom {
    double ox, oy, res;
    double inv_res;          // 1.0 / res, used only by the screened fast path
    int size_x, size_y;
    int win_x0, win_y0, win_w, win_h;
};

// One expanded beam in global cell coordinates.
struct Beam {
    int x0, y0, x1, y1;
    int hit;     // hit_valid (:888)
    int valid;   // 0 -> nothing to draw (coordinates outside the +-2^30 cell range)
    int slow;    // endpoint was re-evaluated with double-double sin/cos
};

// dual_bot_mapper.py:57-58
#define OCC_MAX_DIST_M 1.20
#define OCC_MIN_DIST_M 0.05
// Cells beyond +-2^30 cannot intersect any grid (size <= 2^30 enforced) and a ray is at
// most OCC_MAX_DIST_M / res cells long, so such beams have no effect in the reference
// either; they are skipped instead of walked.
#define OCC_CELL_LIMIT 1073741824.0

OCC_HD float load_f32_unaligned(const uint8_t* p) {
    uint32_t v = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
#if defined(__CUDA_ARCH__)
    return __uint_as_float(v);
#else
    float f;
    __builtin_memcpy(&f, &v, 4);
    return f;
#endif
}

// world_to_grid quotient, :123-124 — (w - o) / res, both operations rounded separately.
OCC_HD double cell_quotient(double w, double o, double res) { return OCC_DDIV(OCC_DADD(w, -o), res); }

OCC_HD bool quotient_in_range(double q) { return fabs(q) < OCC_CELL_LIMIT; }   // false for NaN

OCC_HD int trunc_cell(double q) {
#if defined(__CUDA_ARCH__)
    return __double2int_rz(q);
#else
    return (int)q;
#endif
}

// Screening tolerance of the fast path.  The fast path evaluates ONE library sincos per packet
// (the other three sensor directions are quarter turns of it) and multiplies by 1/res instead
// of dividing; a cell index can differ from the reference's only if the approximate quotient
// lies within `tol` of an integer, in which case the beam is re-evaluated exactly (true angle
// yaw + ANG[s], double-double sin/cos, true division).  Error budget (DESIGN.md "fp64 parity"):
//   |dq| <= 2^-52 * (3.5 * S + 0.65 * (|yaw| + 9) / res),  S = (|r| + |o| + 2) / res
// (2-ulp library sincos, the rounding of yaw + ANG[s], 1/res and every rounded operation);
// tol = 2^-47 * (S + (|yaw| + 9) / res) leaves a 9x margin on the first term, 49x on the second.
OCC_HD double screening_tolerance(double r, double o, double yaw, double inv_res) {
    return OCC_DMUL(OCC_DMUL(fabs(r) + fabs(o) + fabs(yaw) + 11.0, inv_res), 0x1p-47);
}

OCC_HD bool near_cell_boundary(double q, double tol) { return !(fabs(q - rint(q)) > tol); }   // true for NaN/inf too

// Library sincos: CUDA's on the device, glibc's on the host.  FastSinCos is a hook so the
// CPU tests can substitute a deliberately perturbed routine and exercise the slow path.
struct LibSinCos {
    OCC_HD_MEMBER void operator()(double a, double* s, double* c) const {
#if defined(__CUDA_ARCH__)
        sincos(a, s, c);
#else
        *s = sin(a);
        *c = cos(a);
#endif
    }
};

// The four sensor angles, :61-66: 0, math.pi/2, math.pi, -math.pi/2.
OCC_HD double sensor_angle(int s) {
    const double h = 0x1.921fb54442d18p+0;
    return s == 0 ? 0.0 : (s == 1 ? h : (s == 2 ? 0x1.921fb54442d18p+1 : -h));
}

// Endpoint cell of one beam (:887-891 | :898-902, :143).  (sn, cs) is the screened estimate of
// sin/cos of the beam direction; the exact path recomputes everything the way the reference does.
template <class FastSinCos>
OCC_HD void expand_beam(const Geom& g, double rx, double ry, double ryaw, int x0, int y0, bool origin_ok,
                        int sensor, float dist_f32, double sn, double cs, double tolx, double toly,
                        const FastSinCos& fsc, Beam* b) {
    double dist = (double)dist_f32;
    bool hit = (OCC_MIN_DIST_M < dist) && (dist <= OCC_MAX_DIST_M);     // :888 (false for NaN)
    double range = hit ? dist : OCC_MAX_DIST_M;                          // :900 reduces to MAX for every non-hit
    double qx = OCC_DMUL(OCC_DADD(OCC_DADD(rx, OCC_DMUL(range, cs)), -g.ox), g.inv_res);
    double qy = OCC_DMUL(OCC_DADD(OCC_DADD(ry, OCC_DMUL(range, sn)), -g.oy), g.inv_res);
    int slow = 0;
    if (near_cell_boundary(qx, tolx) || near_cell_boundary(qy, toly)) {
        double ang = OCC_DADD(ryaw, sensor_angle(sensor));              // :887
        double s2, c2;
        if (!sincos_dd(ang, &s2, &c2)) fsc(ang, &s2, &c2);
        qx = cell_quotient(OCC_DADD(rx, OCC_DMUL(range, c2)), g.ox, g.res);   // :890 | :901, :143
        qy = cell_quotient(OCC_DADD(ry, OCC_DMUL(range, s2)), g.oy, g.res);   // :891 | :902
        slow = 1;
    }
    b->hit = hit ? 1 : 0;
    b->slow = slow;
    b->x0 = x0;
    b->y0 = y0;
    bool ok = origin_ok && quotient_in_range(qx) && quotient_in_range(qy);
    b->valid = ok ? 1 : 0;
    b->x1 = ok ? trunc_cell(qx) : 0;
    b->y1 = ok ? trunc_cell(qy) : 0;
}

// Packet status codes
enum { PKT_OK = 0, PKT_DROPPED = 1, PKT_BAD_POSE = 2 };

// Decode + filter + pose correction for one record (:828-857).  `p` points at the record
// (any alignment).  Returns PKT_*; on PKT_OK fills the corrected pose and the 4 ranges, and
// `agent_out` (when given) with the accepted agent id 1..n_agents.
OCC_HD int decode_packet(const uint8_t* p, long long k, const int32_t* agent_idx, const double* drift,
                         const double* agent_off, int n_agents,
                         double* rx, double* ry, double* ryaw, float dist[4], int* agent_out = nullptr) {
    if (!(p[0] == 'Q' && p[1] == 'S' && p[2] == 'R' && p[3] == 'L')) return PKT_DROPPED;   // :840
    long long agent = agent_idx ? (long long)agent_idx[k] : (long long)p[4];
    if (agent < 1 || agent > n_agents) return PKT_DROPPED;                                  // :842
    if (agent_out) *agent_out = (int)agent;
    double x = (double)load_f32_unaligned(p + 5);
    double y = (double)load_f32_unaligned(p + 9);
    double yaw = (double)load_f32_unaligned(p + 13);
    x = OCC_DADD(x, agent_off[2 * agent + 0]);                                              // :851-852
    y = OCC_DADD(y, agent_off[2 * agent + 1]);
    if (drift) {                                                                            // :855-857
        x = OCC_DADD(x, drift[2 * k + 0]);
        y = OCC_DADD(y, drift[2 * k + 1]);
    }
    if (!(isfinite(x) && isfinite(y) && isfinite(yaw))) return PKT_BAD_POSE;
    *rx = x;
    *ry = y;
    *ryaw = yaw;
    dist[0] = load_f32_unaligned(p + 25);
    dist[1] = load_f32_unaligned(p + 29);
    dist[2] = load_f32_unaligned(p + 33);
    dist[3] = load_f32_unaligned(p + 37);
    return PKT_OK;
}

// All four beams of an accepted packet.
template <class FastSinCos>
OCC_HD void expand_packet(const Geom& g, double rx, double ry, double ryaw, const float dist[4],
                          const FastSinCos& fsc, Beam out[4]) {
    const double tolx = screening_tolerance(rx, g.ox, ryaw, g.inv_res);
    const double toly = screening_tolerance(ry, g.oy, ryaw, g.inv_res);
    double q0x = OCC_DMUL(OCC_DADD(rx, -g.ox), g.inv_res);
    double q0y = OCC_DMUL(OCC_DADD(ry, -g.oy), g.inv_res);
    if (near_cell_boundary(q0x, tolx)) q0x = cell_quotient(rx, g.ox, g.res);               // :142
    if (near_cell_boundary(q0y, toly)) q0y = cell_quotient(ry, g.oy, g.res);
    bool origin_ok = quotient_in_range(q0x) && quotient_in_range(q0y);
    int x0 = origin_ok ? trunc_cell(q0x) : 0;
    int y0 = origin_ok ? trunc_cell(q0y) : 0;
    double s0, c0;
    fsc(ryaw, &s0, &c0);
    // front: yaw, left: yaw + pi/2, back: yaw + pi, right: yaw - pi/2 (:61-66) as quarter turns
    expand_beam(g, rx, ry, ryaw, x0, y0, origin_ok, 0, dist[0], s0, c0, tolx, toly, fsc, &out[0]);
    expand_beam(g, rx, ry, ryaw, x0, y0, origin_ok, 1, dist[1], c0, -s0, tolx, toly, fsc, &out[1]);
    expand_beam(g, rx, ry, ryaw, x0, y0, origin_ok, 2, dist[2], -s0, -c0, tolx, toly, fsc, &out[2]);
    expand_beam(g, rx, ry, ryaw, x0, y0, origin_ok, 3, dist[3], -c0, s0, tolx, toly, fsc, &out[3]);
}

// Per-packet part of expand_packet, for kernels that loop over the four sensors instead of
// unrolling them: start cell (:142), screening tolerances and ONE library sincos of the yaw.
struct PacketFrame {
    double rx, ry, ryaw, tolx, toly, s0, c0;
    int x0, y0;
    bool origin_ok;
};

template <class FastSinCos>
OCC_HD void packet_frame(const Geom& g, double rx, double ry, double ryaw, const FastSinCos& fsc, PacketFrame* F) {
    F->rx = rx; F->ry = ry; F->ryaw = ryaw;
    F->tolx = screening_tolerance(rx, g.ox, ryaw, g.inv_res);
    F->toly = screening_tolerance(ry, g.oy, ryaw, g.inv_res);
    double q0x = OCC_DMUL(OCC_DADD(rx, -g.ox), g.inv_res);
    double q0y = OCC_DMUL(OCC_DADD(ry, -g.oy), g.inv_res);
    if (near_cell_boundary(q0x, F->tolx)) q0x = cell_quotient(rx, g.ox, g.res);               // :142
    if (near_cell_boundary(q0y, F->toly)) q0y = cell_quotient(ry, g.oy, g.res);
    F->origin_ok = quotient_in_range(q0x) && quotient_in_range(q0y);
    F->x0 = F->origin_ok ? trunc_cell(q0x) : 0;
    F->y0 = F->origin_ok ? trunc_cell(q0y) : 0;
    fsc(ryaw, &F->s0, &F->c0);
}

// Beam of sensor s (0 front, 1 left, 2 back, 3 right; :61-66) as a quarter turn of the frame's
// sincos — the same values expand_packet hands to expand_beam.
template <class FastSinCos>
OCC_HD void expand_beam_of(const Geom& g, const PacketFrame& F, int s, float dist, const FastSinCos& fsc, Beam* out) {
    const double sn = s == 0 ? F.s0 : (s == 1 ? F.c0 : (s == 2 ? -F.s0 : -F.c0));
    const double cs = s == 0 ? F.c0 : (s == 1 ? -F.s0 : (s == 2 ? -F.c0 : F.s0));
    expand_beam(g, F.rx, F.ry, F.ryaw, F.x0, F.y0, F.origin_ok, s, dist, sn, cs, F.tolx, F.toly, fsc, out);
}

// Explicit world-space ray -> beam (OccupancyGrid.update_ray's two world_to_grid calls, :142-143).
OCC_HD void ray_to_beam(const Geom& g, double x0w, double y0w, double x1w, double y1w, int hit, Beam* b) {
    double q0x = cell_quotient(x0w, g.ox, g.res), q0y = cell_quotient(y0w, g.oy, g.res);
    double q1x = cell_quotient(x1w, g.ox, g.res), q1y = cell_quotient(y1w, g.oy, g.res);
    bool ok = quotient_in_range(q0x) && quotient_in_range(q0y) && quotient_in_range(q1x) && quotient_in_range(q1y);
    b->valid = ok ? 1 : 0;
    b->hit = hit ? 1 : 0;
    b->slow = 0;
    b->x0 = ok ? trunc_cell(q0x) : 0;
    b->y0 = ok ? trunc_cell(q0y) : 0;
    b->x1 = ok ? trunc_cell(q1x) : 0;
    b->y1 = ok ? trunc_cell(q1y) : 0;
}

// Number of cells _bresenham (:158-179) produces for a beam: max(|dx|,|dy|) + 1.
OCC_HD int beam_cells(const Beam& b) {
    int dx = b.x1 > b.x0 ? b.x1 - b.x0 : b.x0 - b.x1;
    int dy = b.y1 > b.y0 ? b.y1 - b.y0 : b.y0 - b.y1;
    return (dx > dy ? dx : dy) + 1;
}

// Integer Bresenham walk with the reference's exact tie-breaks (:158-179): strict
// `e2 > -dy` and `e2 < dx`, both may fire in one step, sx = -1 when x0 == x1.  Calls
// visit(x, y, is_last) for every cell in order.
template <class Visit>
OCC_HD void bresenham_walk(int x0, int y0, int x1, int y1, Visit&& visit) {
    int dx = x1 > x0 ? x1 - x0 : x0 - x1;
    int dy = y1 > y0 ? y1 - y0 : y0 - y1;
    int sx = x0 < x1 ? 1 : -1;
    int sy = y0 < y1 ? 1 : -1;
    int err = dx - dy;
    int n = dx > dy ? dx : dy;
    for (int i = 0; i < n; ++i) {
        visit(x0, y0, false);
        int e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x0 += sx; }
        if (e2 < dx)  { err += dx; y0 += sy; }
    }
    visit(x0, y0, true);
}

}  // namespace occ
