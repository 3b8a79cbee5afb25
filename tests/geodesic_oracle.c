/*
 * TEST INFRASTRUCTURE ONLY.  Reference geodesic field for the frontier-assignment tests: a plain
 * FIFO-queue BFS from cell (sx, sy) of an int8 grid [h][w], 4-connected, unit cost, moving only
 * into FREE (0) cells; the source gets 0 whatever its value, unreachable cells -1.  A source
 * outside the grid leaves every cell -1.  Built by tests/frontier_assign_util.py with gcc.
 */
#include <stdint.h>
#include <stdlib.h>

int oracle_geodesic(const int8_t* grid, int64_t w, int64_t h, int64_t sx, int64_t sy, int32_t* dist) {
    for (int64_t i = 0; i < w * h; i++) dist[i] = -1;
    if (sx < 0 || sy < 0 || sx >= w || sy >= h) return 0;
    int64_t* queue = malloc(sizeof(int64_t) * (size_t)(w * h));
    if (!queue) return -1;
    int64_t head = 0, tail = 0;
    dist[sy * w + sx] = 0;
    queue[tail++] = sy * w + sx;
    while (head < tail) {
        const int64_t c = queue[head++], x = c % w, y = c / w;
        const int64_t nb[4] = {x > 0 ? c - 1 : -1, x < w - 1 ? c + 1 : -1, y > 0 ? c - w : -1, y < h - 1 ? c + w : -1};
        for (int k = 0; k < 4; k++) {
            if (nb[k] >= 0 && grid[nb[k]] == 0 && dist[nb[k]] < 0) {
                dist[nb[k]] = dist[c] + 1;
                queue[tail++] = nb[k];
            }
        }
    }
    free(queue);
    return 0;
}
