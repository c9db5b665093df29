// astar4.cuh — the reference's astar_4 (astar_4.py:21-109, restated as episode_io.astar_path) as a level-synchronous
// wavefront: one warp finds one path, bit-exact with the heap version, tie-breaking included.
//
// astar_path pops heap entries (f, g, cell, parent), skips closed cells, and overwrites a neighbour's parent when the
// neighbour's cost is equal or better.  Four facts make it parallel without changing a path (tests/test_astar_level_model.py
// checks a NumPy statement of this algorithm against astar_path):
//  1. One live key per cell.  Only an entry carrying a cell's current best g can pop before the cell closes (a worse one
//     has a larger f, the h being the same), so an open cell has exactly one key that matters: (g + h, g, r*Wd + c).
//     The parent in the tuple only orders entries of the same cell.  The start's entry has f = 0, but it is alone.
//  2. Only two f values are open at a time.  h is the Manhattan distance and every step costs 1, so h is consistent:
//     popped f never decreases and every open key has f in {f*, f* + 2}.
//  3. A level expands at once.  The cells sharing the minimum (f, g) — a level — pop in cell-index order.  A neighbour
//     reached from the level gets g + 1 and so a key after the whole level; a member proposes g + 1 > g to another member,
//     which changes nothing.  So the level expands in parallel: a free, in-bounds, not-closed neighbour n with g[n] unset
//     or g[n] >= g + 1 gets g[n] = g + 1, and its parent is the HIGHEST-index member of the level adjacent to n (a later
//     pop overwrites on equal cost).  The left / up / right / down order of the reference cannot change a result.
//  4. Stop at the goal.  In the level that holds the goal, the members before it propose g + 1 to cells that are not the
//     goal's ancestors, and parents of closed cells never change: the goal's parent chain at that point is the path.
// Row-major cell indices keep the (r, c) tuple order, so padding a map with walls changes no path.
//
// Shared state per warp: g as int16 per cell, open / closed / level bit sets, the parent as a 2-bit direction per cell.
#pragma once
#include "common.cuh"

namespace mapf {

// parent direction, from a cell to its parent: 0 up (c - Wd), 1 left (c - 1), 2 right (c + 1), 3 down (c + Wd) — the
// order of the neighbours' cell indices
struct Astar4Smem {
    int16_t *g;         // [cells] best g, -1 = not reached
    uint32_t *open;     // [words] reached, not closed
    uint32_t *closed;   // [words]
    uint32_t *lvl;      // [words] members of the level being expanded
    uint32_t *par;      // [ceil(cells / 16)] 2-bit parent directions
};

__host__ __device__ constexpr int astar4_words(int cells) { return (cells + 31) >> 5; }

__device__ __forceinline__ int astar4_parent(const Astar4Smem &s, int Wd, int c) {
    const int d = (s.par[c >> 4] >> ((c & 15) * 2)) & 3;
    return d == 0 ? c - Wd : d == 1 ? c - 1 : d == 2 ? c + 1 : c + Wd;
}

// g of the goal (>= 1) when a path exists, -1 otherwise; start != goal, both inside the H x Wd map.  free(c) says whether
// cell c may be entered; a blocked start is still expanded (astar_path does).  Every lane returns the same value; the
// path is then goal, parent(goal), ... back to start, and g of the k-th cell from the start is k.
template <class Free>
__device__ int astar4_search(const Astar4Smem &s, int H, int Wd, int start, int goal, const Free &free) {
    const int lane = threadIdx.x & 31, cells = H * Wd, words = astar4_words(cells);
    const int gr = goal / Wd, gcol = goal - gr * Wd;
    auto key = [&](int c) -> uint32_t {         // (f, g) packed; f < cells + H + Wd < 2^16
        const int r = c / Wd, col = c - r * Wd, g = s.g[c];
        return ((uint32_t)(g + abs(r - gr) + abs(col - gcol)) << 16) | (uint32_t)g;
    };
    auto bit = [](const uint32_t *set, int c) { return (set[c >> 5] >> (c & 31)) & 1u; };
    for (int c = lane; c < cells; c += 32) s.g[c] = -1;
    for (int k = lane; k < words; k += 32) { s.open[k] = 0; s.closed[k] = 0; }
    __syncwarp();
    if (lane == 0) { s.g[start] = 0; s.open[start >> 5] = 1u << (start & 31); }
    __syncwarp();
    for (;;) {
        uint32_t best = 0xFFFFFFFFu;            // the minimum (f, g) over the open set (facts 1, 2)
        for (int k = lane; k < words; k += 32)
            for (uint32_t b = s.open[k]; b; b &= b - 1) best = min(best, key(32 * k + __ffs(b) - 1));
        best = __reduce_min_sync(FULL, best);
        if (best == 0xFFFFFFFFu) return -1;     // the heap ran empty
        const int gl = (int)(best & 0xFFFFu);
        if (bit(s.open, goal) && key(goal) == best) return gl;   // the goal pops in this level (fact 4)
        for (int k = lane; k < words; k += 32) {                 // close the level
            const uint32_t o = s.open[k];
            uint32_t m = 0;
            for (uint32_t b = o; b; b &= b - 1) {
                const int j = __ffs(b) - 1;
                if (key(32 * k + j) == best) m |= 1u << j;
            }
            s.lvl[k] = m; s.open[k] = o & ~m; s.closed[k] |= m;
        }
        __syncwarp();
        const int16_t ng = (int16_t)(gl + 1);
        for (int k = lane; k < words; k += 32) {                 // expand it (fact 3)
            for (uint32_t b = s.lvl[k]; b; b &= b - 1) {
                const int m = 32 * k + __ffs(b) - 1, r = m / Wd, col = m - r * Wd;
                // n = neighbour of m; dir = direction from n back to m
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    int n, dir;
                    if (t == 0) { if (col == 0) continue; n = m - 1; dir = 2; }
                    else if (t == 1) { if (r == 0) continue; n = m - Wd; dir = 3; }
                    else if (t == 2) { if (col + 1 >= Wd) continue; n = m + 1; dir = 1; }
                    else { if (r + 1 >= H) continue; n = m + Wd; dir = 0; }
                    if (!free(n) || bit(s.closed, n)) continue;
                    const int gn = s.g[n];
                    if (gn >= 0 && gn < ng) continue;
                    // the highest-index member adjacent to n is its parent; only that member writes n
                    const int nr = r + (t == 1 ? -1 : t == 3 ? 1 : 0), ncol = col + (t == 0 ? -1 : t == 2 ? 1 : 0);
                    const int p = (nr + 1 < H && bit(s.lvl, n + Wd)) ? 3
                                : (ncol + 1 < Wd && bit(s.lvl, n + 1)) ? 2
                                : (ncol > 0 && bit(s.lvl, n - 1)) ? 1 : 0;
                    if (p != dir) continue;
                    s.g[n] = ng;
                    atomicOr(&s.open[n >> 5], 1u << (n & 31));
                    const int sh = (n & 15) * 2;
                    atomicAnd(&s.par[n >> 4], ~(3u << sh));
                    atomicOr(&s.par[n >> 4], (uint32_t)p << sh);
                }
            }
        }
        __syncwarp();
    }
}

}  // namespace mapf
