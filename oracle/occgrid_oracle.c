/*
 * ORACLE — TEST INFRASTRUCTURE ONLY.  Not product code.
 *
 * Plain-C, single-threaded restatement of the reference's occupancy-grid integration
 * path (server_nodes/dual_bot_mapper.py, cited per function).  It exists so that parity
 * tests and the cpu_baseline leg can replay 1e5..1e7-beam batches in seconds; the
 * line-for-line Python restatement (oracle/occgrid_oracle.py) pins it on small inputs
 * and both are pinned on fixtures produced by the unmodified reference
 * (oracle/make_golden.py -> tests/golden/).
 *
 * Built by oracle/build.py with  gcc -O2 -ffp-contract=off  (no FMA contraction: Python
 * evaluates  rx + dist*cos(a)  as a rounded multiply followed by a rounded add).
 * cos()/sin() are glibc's, i.e. the very functions CPython's math.cos/math.sin call.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define CELL_FREE 0
#define CELL_OCCUPIED 100

/* dual_bot_mapper.py:57-58 */
static const double MAX_DIST_M = 1.20;
static const double MIN_DIST_M = 0.05;

enum { C_PACKETS = 0, C_ACCEPTED, C_DROPPED, C_BAD_POSE, C_BEAMS, C_HITS, C_UPDATES, C_SPARE };

static float rd_f32(const uint8_t* p) { float v; memcpy(&v, p, 4); return v; }

/* int() of a finite double: truncation toward zero (dual_bot_mapper.py:123-124).  Values
 * beyond +-2^62 cannot be cells of any grid we allocate; saturate so the C cast is defined. */
static int64_t trunc_i64(double q) {
    if (q >= 4.0e18) return INT64_MAX / 2;
    if (q <= -4.0e18) return -(INT64_MAX / 2);
    return (int64_t)q;
}

/* Where update_ray's stores go: the int8 grid (last writer wins, :148-156) or, when `counts` is
 * set, int32 {miss, hit} pairs per cell (count mode: every FREE store counts one miss, every
 * OCCUPIED store one hit).  Exactly one of the two pointers is set. */
typedef struct { int8_t* grid; int32_t* counts; } Plane;

static void store_cell(Plane out, int64_t i, int occupied) {
    if (out.counts) out.counts[2 * i + (occupied ? 1 : 0)]++;
    else out.grid[i] = occupied ? CELL_OCCUPIED : CELL_FREE;
}

/* OccupancyGrid.update_ray + _bresenham + in_bounds — dual_bot_mapper.py:133-179.
 * The window (win_x0, win_y0, win_w, win_h) is the part of the global grid that `out`
 * holds (row stride win_w): the full grid for the reference case, a spatial tile for the
 * multi-GPU tests.  Cells are generated on the unclipped global line and masked one by
 * one, exactly like the per-cell in_bounds test at :149,:155. */
static int64_t update_ray_cells(Plane out, int64_t size_x, int64_t size_y,
                                int64_t win_x0, int64_t win_y0, int64_t win_w, int64_t win_h,
                                int64_t x0, int64_t y0, int64_t x1, int64_t y1, int hit_valid) {
    int64_t dx = x1 > x0 ? x1 - x0 : x0 - x1;
    int64_t dy = y1 > y0 ? y1 - y0 : y0 - y1;
    int64_t sx = x0 < x1 ? 1 : -1;
    int64_t sy = y0 < y1 ? 1 : -1;
    int64_t err = dx - dy;
    int64_t n = 0;
    for (;;) {
        int last = (x0 == x1 && y0 == y1);
        n++;
        if ((!last || hit_valid) && x0 >= 0 && x0 < size_x && y0 >= 0 && y0 < size_y) {
            int64_t lx = x0 - win_x0, ly = y0 - win_y0;
            if (lx >= 0 && lx < win_w && ly >= 0 && ly < win_h)
                store_cell(out, ly * win_w + lx, last);
        }
        if (last) break;
        int64_t e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x0 += sx; }
        if (e2 < dx)  { err += dx; y0 += sy; }
    }
    return n;
}

/* Per-packet loop of main() — dual_bot_mapper.py:826-903 (SLAM's output enters as the
 * per-packet drift table; see oracle/occgrid_oracle.py:replay for the coupled version).
 *
 *  pkts       n records, `stride` bytes apart, each `rec_len` (41 = v1, 42 = v2) bytes valid
 *  agent_idx  optional out-of-band agent index per packet (EXTENSION for >255 agents);
 *             NULL -> the wire byte at offset 4
 *  agent_off  (n_agents+1) x 2 doubles; ids 1..n_agents accepted (:842), offset added to
 *             the pose (:851-852; reference mode = {(0,0),(0,0),(separation,0)})
 *  drift      n x 2 doubles or NULL (:855-857)
 */
static int packets_into(const uint8_t* pkts, int64_t n, int stride, int rec_len,
                        const int32_t* agent_idx, const double* drift,
                        const double* agent_off, int n_agents,
                        double ox, double oy, double res,
                        int64_t size_x, int64_t size_y,
                        int64_t win_x0, int64_t win_y0, int64_t win_w, int64_t win_h,
                        Plane out, uint64_t* counters) {
    /* :61-66 — math.pi/2, math.pi, -math.pi/2 as doubles (hex literals: exact) */
    static const double ANG[4] = { 0.0, 0x1.921fb54442d18p+0, 0x1.921fb54442d18p+1,
                                   -0x1.921fb54442d18p+0 };
    if (rec_len != 41 && rec_len != 42) return -1;
    for (int64_t k = 0; k < n; k++) {
        const uint8_t* p = pkts + k * (int64_t)stride;
        counters[C_PACKETS]++;
        if (memcmp(p, "QSRL", 4) != 0) { counters[C_DROPPED]++; continue; }   /* :840 */
        int64_t agent = agent_idx ? agent_idx[k] : p[4];
        if (agent < 1 || agent > n_agents) { counters[C_DROPPED]++; continue; }  /* :842 */
        double rx = (double)rd_f32(p + 5);
        double ry = (double)rd_f32(p + 9);
        double ryaw = (double)rd_f32(p + 13);
        rx += agent_off[2 * agent + 0];                                   /* :851-852 */
        ry += agent_off[2 * agent + 1];
        if (drift) { rx += drift[2 * k + 0]; ry += drift[2 * k + 1]; }       /* :855-857 */
        if (!isfinite(rx) || !isfinite(ry) || !isfinite(ryaw)) { counters[C_BAD_POSE]++; continue; }
        counters[C_ACCEPTED]++;
        int64_t x0 = trunc_i64((rx - ox) / res);                            /* :142 */
        int64_t y0 = trunc_i64((ry - oy) / res);
        for (int s = 0; s < 4; s++) {                                       /* :886 */
            double dist = (double)rd_f32(p + 25 + 4 * s);
            double ray_angle = ryaw + ANG[s];                               /* :887 */
            int hit_valid = (MIN_DIST_M < dist) && (dist <= MAX_DIST_M);    /* :888 */
            double range = hit_valid ? dist : MAX_DIST_M;                   /* :900 */
            double wx = rx + range * cos(ray_angle);                        /* :890 / :901 */
            double wy = ry + range * sin(ray_angle);                        /* :891 / :902 */
            int64_t x1 = trunc_i64((wx - ox) / res);                        /* :143 */
            int64_t y1 = trunc_i64((wy - oy) / res);
            counters[C_BEAMS]++;
            counters[C_HITS] += (uint64_t)hit_valid;
            counters[C_UPDATES] += (uint64_t)update_ray_cells(out, size_x, size_y, win_x0, win_y0,
                                                              win_w, win_h, x0, y0, x1, y1, hit_valid);
        }
    }
    return 0;
}

/* The loop body into the int8 grid `grid` [win_h][win_w]. */
int oracle_integrate_packets(const uint8_t* pkts, int64_t n, int stride, int rec_len,
                             const int32_t* agent_idx, const double* drift,
                             const double* agent_off, int n_agents,
                             double ox, double oy, double res,
                             int64_t size_x, int64_t size_y,
                             int64_t win_x0, int64_t win_y0, int64_t win_w, int64_t win_h,
                             int8_t* grid, uint64_t* counters) {
    const Plane out = { grid, NULL };
    return packets_into(pkts, n, stride, rec_len, agent_idx, drift, agent_off, n_agents, ox, oy, res,
                        size_x, size_y, win_x0, win_y0, win_w, win_h, out, counters);
}

/* Count mode: the same loop body, adding into `counts` [win_h][win_w][2] = {miss, hit}. */
int oracle_accumulate_packets(const uint8_t* pkts, int64_t n, int stride, int rec_len,
                              const int32_t* agent_idx, const double* drift,
                              const double* agent_off, int n_agents,
                              double ox, double oy, double res,
                              int64_t size_x, int64_t size_y,
                              int64_t win_x0, int64_t win_y0, int64_t win_w, int64_t win_h,
                              int32_t* counts, uint64_t* counters) {
    const Plane out = { NULL, counts };
    return packets_into(pkts, n, stride, rec_len, agent_idx, drift, agent_off, n_agents, ox, oy, res,
                        size_x, size_y, win_x0, win_y0, win_w, win_h, out, counters);
}

/* OccupancyGrid.update_ray on explicit world-space rays (the per-ray API, :136-156). */
int oracle_update_rays(const double* rays /* n x 4: x0 y0 x1 y1 */, const uint8_t* hit, int64_t n,
                       double ox, double oy, double res, int64_t size_x, int64_t size_y,
                       int8_t* grid, uint64_t* counters) {
    for (int64_t k = 0; k < n; k++) {
        int64_t x0 = trunc_i64((rays[4 * k + 0] - ox) / res);
        int64_t y0 = trunc_i64((rays[4 * k + 1] - oy) / res);
        int64_t x1 = trunc_i64((rays[4 * k + 2] - ox) / res);
        int64_t y1 = trunc_i64((rays[4 * k + 3] - oy) / res);
        counters[C_BEAMS]++;
        counters[C_HITS] += hit[k] != 0;
        const Plane out = { grid, NULL };
        counters[C_UPDATES] += (uint64_t)update_ray_cells(out, size_x, size_y, 0, 0, size_x, size_y,
                                                          x0, y0, x1, y1, hit[k] != 0);
    }
    return 0;
}

/* _bresenham (:158-179) into caller buffers; returns the cell count. */
int64_t oracle_bresenham(int64_t x0, int64_t y0, int64_t x1, int64_t y1,
                         int32_t* xs, int32_t* ys, int64_t cap) {
    int64_t dx = x1 > x0 ? x1 - x0 : x0 - x1;
    int64_t dy = y1 > y0 ? y1 - y0 : y0 - y1;
    int64_t sx = x0 < x1 ? 1 : -1, sy = y0 < y1 ? 1 : -1, err = dx - dy, n = 0;
    for (;;) {
        if (n < cap) { xs[n] = (int32_t)x0; ys[n] = (int32_t)y0; }
        n++;
        if (x0 == x1 && y0 == y1) break;
        int64_t e2 = 2 * err;
        if (e2 > -dy) { err -= dy; x0 += sx; }
        if (e2 < dx)  { err += dx; y0 += sy; }
    }
    return n;
}
