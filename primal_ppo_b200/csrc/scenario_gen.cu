// scenario_gen.cu — on-device generation of the exogenous inputs of a batch of worlds (SURVEY.md §8 f1 + f2).
//
// The reference draws all of this on the host, one world per process, from the global NumPy stream:
//   map        generateWarehouse (map_generator.py:127-138, the training env: MapfGym.__init__ mapf_gym.py:166) or the
//              PRIMAL density map `-(rand(size,size) < prob)` (map_generator.py:13-28)
//   human      entrance = rejection-sampled free cell on row 0 / column 0 (mapf_gym.py:18-23), goal = free cell
//              (util.py:67-76), path = astar_4 out and back (mapf_gym.py:33-37), walked one cell per jointStep
//   agents     starts and first goals: sequential rejection sampling on a scratch map that marks the human, earlier
//              starts and earlier goals (populateMap, mapf_gym.py:175-190); later goals: free cells (mapf_gym.py:626)
// Here one warp builds one world with Philox4x32-10 keyed by (seed; global world index, stream, draw).  The results are
// EQUAL IN DISTRIBUTION to the reference's, not in bits (different generator; later goals are drawn at reset, so they
// avoid obstacles and the previous goal but cannot avoid the agents' future cells).  The walk between the drawn cells
// depends on human_path: 1 is astar_4's path itself, bit-exact with its tie-breaking (astar4.cuh), so for the same map,
// entrance and goals the walk is the reference's; 0 (the default) descends the BFS field with a fixed neighbour order,
// another shortest path.  Both have the same length, so every draw and the trace's timing are the same in both modes.  The warehouse layout itself is a
// deterministic function of the drawn length and is bit-identical to generateWarehouse (tests/golden/warehouse_maps.npz).
// Output arrays are exactly the MapfScenario arrays of include/mapf_b200.h, written in HBM, so mapf_reset consumes
// them without a host round trip.
#include "astar4.cuh"
#include "common.cuh"

namespace mapf {

namespace {

struct GenView {
    int W, H, Wd, N, Q, L;
    int kind, density_mode, size_lo, size_hi, human_loops, human_path;
    float dlo, dhi;
    unsigned long long seed;
    int world_offset;
    uint8_t *obst;
    int16_t *dims, *starts, *goal_queue, *htrace, *hp5;
    int32_t *hlen;
    uint32_t *gen_err;
};

constexpr uint32_t TAG = 0x47454E53u;   // "GENS"
struct U4 { uint32_t x, y, z, w; };
__device__ __forceinline__ U4 philox4(unsigned long long seed, uint32_t world, uint32_t stream, uint32_t idx) {
    uint32_t c0 = world, c1 = stream, c2 = idx, c3 = TAG;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}
__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-08f; }

enum { S_DIMS = 0, S_CELLS = 1, S_HUMAN = 2, S_START = 3, S_GOAL = 4, S_QUEUE = 5 };

// per-warp shared memory: free-cell flags (1 = free and inside dims), occupancy flags, BFS distances; with human_path = 1
// the A* search reuses dist as its g and fw / nf as its open / closed sets, and adds a level set and the parents
struct GenSmem {
    uint8_t *freec;     // [H*Wd]
    uint8_t *occ;       // [H*Wd]
    int16_t *dist;      // [H*Wd]
    uint32_t *fw, *nf;  // [ceil(H*Wd/32)] frontier bit sets of the current / next BFS level
    uint32_t *lvl, *par;
};
__host__ __device__ constexpr int gen_set_words(int cells) { return (astar4_words(cells) + 3) & ~3; }
__host__ __device__ constexpr int gen_par_words(int cells) { return ((cells + 15) / 16 + 3) & ~3; }

__global__ void __launch_bounds__(128) scenario_gen_kernel(const GenView g, const int per_warp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * (blockDim.x >> 5) + warp;
    if (w >= g.W) return;
    const int H = g.H, Wd = g.Wd, cells = H * Wd;
    unsigned char *base = smem_raw + (size_t)warp * per_warp;
    GenSmem s;
    s.freec = base;
    s.occ = base + ((cells + 15) & ~15);
    s.dist = reinterpret_cast<int16_t *>(base + 2 * ((cells + 15) & ~15));
    const int fwords = (cells + 31) / 32;
    s.fw = reinterpret_cast<uint32_t *>(base + 2 * ((cells + 15) & ~15) + ((cells * 2 + 15) & ~15));
    s.nf = s.fw + gen_set_words(cells);
    s.lvl = s.nf + gen_set_words(cells);          // only inside the per-warp block when human_path = 1
    s.par = s.lvl + gen_set_words(cells);
    const Astar4Smem as{s.dist, s.fw, s.nf, s.lvl, s.par};
    const uint32_t gw = (uint32_t)(w + g.world_offset);
    uint32_t err = 0;

    // ---- A. dimensions and obstacle map ---------------------------------------------------------------------------
    const U4 d0 = philox4(g.seed, gw, S_DIMS, 0);
    int rows, cols;
    float prob = 0.f;
    if (g.kind == 1) {                                   // generateWarehouse(num_block=(lo, hi))
        const int length = g.size_lo + (int)(d0.x % (uint32_t)(g.size_hi - g.size_lo + 1));   // np.random.randint(lo, hi+1)
        rows = length;
        cols = (int)((double)length / (2.0 / 3.0));                                            // int(length/lbRatio)
    } else {
        if (g.size_lo > 0 && g.size_hi > g.size_lo) {    // np.random.choice([lo, (lo+hi)/2, hi], p=[.5,.25,.25])
            const float u = u01(d0.x);
            rows = u < 0.5f ? g.size_lo : (u < 0.75f ? (int)(g.size_lo * .5 + g.size_hi * .5) : g.size_hi);
        } else {
            rows = g.size_lo > 0 ? g.size_lo : H;
        }
        cols = (g.size_lo > 0) ? rows : Wd;
        const float a = g.dlo, b = g.dhi, u = u01(d0.y);
        if (g.density_mode == 1 && b > a) {              // np.random.triangular(a, .33a + .66b, b)
            const float c = .33f * a + .66f * b, fc = (c - a) / (b - a);
            prob = u < fc ? a + sqrtf(u * (b - a) * (c - a)) : b - sqrtf((1.f - u) * (b - a) * (b - c));
        } else {
            prob = a + u * (b - a);
        }
    }
    if (rows > H) rows = H;
    if (cols > Wd) cols = Wd;
    int shelves = 0, free_space = 0;
    if (g.kind == 1) {                                   // shelfSize = 5, freeSpaceRatio = 1/3
        shelves = (int)(((double)cols * (1.0 - 1.0 / 3.0)) / 6.0);
        free_space = (int)((double)(cols - shelves * 6) / 2.0);
    }
    for (int c4 = lane; c4 < (cells + 3) / 4; c4 += 32) {
        U4 r = U4{0, 0, 0, 0};
        if (g.kind == 0) r = philox4(g.seed, gw, S_CELLS, (uint32_t)c4);
        const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = c4 * 4 + k;
            if (c >= cells) break;
            const int y = c / Wd, x = c - y * Wd;
            bool ob;
            if (y >= rows || x >= cols) ob = true;       // outside this world's dims
            else if (g.kind == 1) {
                const int rel = x - free_space;
                ob = (y & 1) && y < rows - 1 && rel >= 0 && rel < shelves * 6 && (rel % 6) < 5;
            } else ob = u01(rr[k]) < prob;
            s.freec[c] = ob ? 0 : 1;
            s.occ[c] = ob ? 1 : 0;
            g.obst[(size_t)w * cells + c] = ob ? 1 : 0;
        }
    }
    __syncwarp();
    // number of free cells (needed to bound rejection sampling)
    int nfree = 0;
    for (int c = lane; c < cells; c += 32) nfree += s.freec[c];
    nfree = __reduce_add_sync(FULL, nfree);
    if (nfree < 2 * g.N + 2) err |= 1u;                  // too crowded to place everything (flagged, still defined)

    // uniform free, unoccupied cell by rejection sampling in (rows x cols); all lanes get the same answer
    auto draw_cell = [&](uint32_t stream, uint32_t idx0, bool need_unocc) -> int {
        for (uint32_t t = 0; t < 64; ++t) {
            const U4 r = philox4(g.seed, gw, stream, idx0 * 64 + t);
            const uint32_t rs[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int y = (int)(rs[2 * k] % (uint32_t)rows), x = (int)(rs[2 * k + 1] % (uint32_t)cols);
                const int c = y * Wd + x;
                if (s.freec[c] && !(need_unocc && s.occ[c])) return c;
            }
        }
        for (int c = 0; c < cells; ++c) if (s.freec[c] && !(need_unocc && s.occ[c])) return c;   // exhaustive fallback
        return -1;
    };

    // ---- B. human: entrance on row 0 / column 0, goal, shortest out-and-back walk ---------------------------------
    int hpos = -1;
    {
        int cand = 0;
        for (int x = 0; x < cols; ++x) cand += s.freec[x];
        for (int y = 1; y < rows; ++y) cand += s.freec[y * Wd];
        if (cand > 0) {
            int k = (int)(philox4(g.seed, gw, S_HUMAN, 0).x % (uint32_t)cand);
            for (int x = 0; x < cols && hpos < 0; ++x) if (s.freec[x] && k-- == 0) hpos = x;
            for (int y = 1; y < rows && hpos < 0; ++y) if (s.freec[y * Wd] && k-- == 0) hpos = y * Wd;
        } else {
            err |= 2u;                                   // the reference would spin forever in getEntrance
            hpos = draw_cell(S_HUMAN, 1, false);
        }
    }
    if (hpos < 0) hpos = 0;
    __syncwarp();
    if (lane == 0) s.occ[hpos] = 1;                      // tempMap[human.position] = 1 (mapf_gym.py:177)
    __syncwarp();
    int16_t *tr = g.htrace + (size_t)w * g.L * 4;
    int tick = 0;
    int cur = hpos;
    for (int loop = 0; loop < g.human_loops && tick < g.L; ++loop) {
        int goal = -1, d = -1;
        for (int attempt = 0; attempt < 4 && d < 0; ++attempt) {
            goal = draw_cell(S_HUMAN, 2 + (uint32_t)loop * 8 + attempt, false);
            if (goal < 0 || goal == cur) { goal = -1; continue; }
            if (g.human_path == 1) {
                // astar_path(map, cur, goal): a shortest path, so d is the BFS distance and every draw stays the same
                d = astar4_search(as, H, Wd, cur, goal, [&](int c) { return s.freec[c] != 0; });
                if (d >= 0 && tick + 2 * d + 1 > g.L && loop == 0 && attempt < 3) d = -1;
                continue;
            }
            // BFS distance field from the goal: level-synchronous, the frontier kept as a bit set so that a level
            // costs work proportional to the frontier, not to the grid
            for (int c = lane; c < cells; c += 32) s.dist[c] = -1;
            for (int k = lane; k < fwords; k += 32) { s.fw[k] = 0; s.nf[k] = 0; }
            __syncwarp();
            if (lane == 0) { s.dist[goal] = 0; s.fw[goal >> 5] = 1u << (goal & 31); }
            __syncwarp();
            for (int level = 0; level < cells; ++level) {
                bool grew = false;
                for (int k = lane; k < fwords; k += 32) {
                    uint32_t b = s.fw[k];
                    while (b) {
                        const int c = 32 * k + __ffs(b) - 1; b &= b - 1;
                        const int y = c / Wd, x = c - y * Wd;
                        // several frontier cells may claim the same neighbour: they all write the same level
                        if (x + 1 < cols && s.freec[c + 1] && s.dist[c + 1] < 0) { s.dist[c + 1] = (int16_t)(level + 1); atomicOr(&s.nf[(c + 1) >> 5], 1u << ((c + 1) & 31)); grew = true; }
                        if (y + 1 < rows && s.freec[c + Wd] && s.dist[c + Wd] < 0) { s.dist[c + Wd] = (int16_t)(level + 1); atomicOr(&s.nf[(c + Wd) >> 5], 1u << ((c + Wd) & 31)); grew = true; }
                        if (x > 0 && s.freec[c - 1] && s.dist[c - 1] < 0) { s.dist[c - 1] = (int16_t)(level + 1); atomicOr(&s.nf[(c - 1) >> 5], 1u << ((c - 1) & 31)); grew = true; }
                        if (y > 0 && s.freec[c - Wd] && s.dist[c - Wd] < 0) { s.dist[c - Wd] = (int16_t)(level + 1); atomicOr(&s.nf[(c - Wd) >> 5], 1u << ((c - Wd) & 31)); grew = true; }
                    }
                }
                __syncwarp();
                if (!__any_sync(FULL, grew) || s.dist[cur] >= 0) break;
                for (int k = lane; k < fwords; k += 32) { s.fw[k] = s.nf[k]; s.nf[k] = 0; }
                __syncwarp();
            }
            __syncwarp();
            d = s.dist[cur];
            if (d >= 0 && tick + 2 * d + 1 > g.L && loop == 0 && attempt < 3) d = -1;   // walk would not fit: try another goal
        }
        if (d < 0) {                                     // no reachable goal: the human stands still
            if (loop == 0) {
                if (lane == 0) { tr[0] = tr[2] = (int16_t)(cur / Wd); tr[1] = tr[3] = (int16_t)(cur % Wd); }
                tick = 1;
                err |= 4u;
            }
            break;
        }
        if (tick + 2 * d + 1 > g.L) break;               // a further loop that does not fit: wrap the trace here
        // out: astar_4's path, or decreasing distance (neighbour order E, S, W, N); back: the same cells reversed
        if (lane == 0 && g.human_path == 1) {
            for (int c = goal;; c = astar4_parent(as, Wd, c)) {    // cell c is the k-th of the path, k = its g
                const int k = as.g[c];
                tr[(tick + k) * 4 + 0] = tr[(tick + 2 * d - k) * 4 + 0] = (int16_t)(c / Wd);
                tr[(tick + k) * 4 + 1] = tr[(tick + 2 * d - k) * 4 + 1] = (int16_t)(c % Wd);
                if (k == 0) break;
            }
        } else if (lane == 0) {
            int c = cur;
            for (int k = 0; k <= d; ++k) {
                tr[(tick + k) * 4 + 0] = (int16_t)(c / Wd); tr[(tick + k) * 4 + 1] = (int16_t)(c % Wd);
                tr[(tick + 2 * d - k) * 4 + 0] = (int16_t)(c / Wd); tr[(tick + 2 * d - k) * 4 + 1] = (int16_t)(c % Wd);
                if (k == d) break;
                const int y = c / Wd, x = c - y * Wd, want = s.dist[c] - 1;
                if (x + 1 < cols && s.dist[c + 1] == want) c = c + 1;
                else if (y + 1 < rows && s.dist[c + Wd] == want) c = c + Wd;
                else if (x > 0 && s.dist[c - 1] == want) c = c - 1;
                else c = c - Wd;
            }
        }
        if (lane == 0) {
            // next = path[s+1], or path[-1] on the last tick of the loop (getNextPos, mapf_gym.py:46-50)
            for (int k = 0; k < 2 * d + 1; ++k) {
                const int nk = k + 1 < 2 * d + 1 ? k + 1 : k;
                tr[(tick + k) * 4 + 2] = tr[(tick + nk) * 4 + 0];
                tr[(tick + k) * 4 + 3] = tr[(tick + nk) * 4 + 1];
            }
            if (loop == 0 && g.hp5) {                    // human.path[1:6] (mapf_gym.py:293-297)
                int16_t *p5 = g.hp5 + (size_t)w * 10;
                for (int k = 0; k < 5; ++k) {
                    const bool ok = k + 1 < 2 * d + 1;
                    p5[2 * k] = ok ? tr[(tick + k + 1) * 4 + 0] : (int16_t)-1;
                    p5[2 * k + 1] = ok ? tr[(tick + k + 1) * 4 + 1] : (int16_t)-1;
                }
            }
        }
        tick += 2 * d + 1;                               // the walk ends where it started
        __syncwarp();
    }
    if (tick == 0) {
        if (lane == 0) { tr[0] = tr[2] = (int16_t)(cur / Wd); tr[1] = tr[3] = (int16_t)(cur % Wd); }
        tick = 1;
    }
    if (lane == 0) {
        g.hlen[w] = tick;
        for (int k = tick; k < g.L; ++k) { tr[k * 4] = tr[(tick - 1) * 4]; tr[k * 4 + 1] = tr[(tick - 1) * 4 + 1]; tr[k * 4 + 2] = tr[(tick - 1) * 4 + 2]; tr[k * 4 + 3] = tr[(tick - 1) * 4 + 3]; }
        if (g.hp5 && (err & 4u)) for (int k = 0; k < 10; ++k) g.hp5[(size_t)w * 10 + k] = -1;
        if (g.dims) { g.dims[2 * w] = (int16_t)rows; g.dims[2 * w + 1] = (int16_t)cols; }
    }
    __syncwarp();

    // ---- C. agent starts and first goals: distinct free cells, in agent order (populateMap) ------------------------
    // The reference alternates start_i, goal_i; drawing all starts and then all goals gives the same joint law
    // (a uniformly random injection of 2N labels into the unoccupied free cells).
    for (int phase = 0; phase < 2; ++phase) {
        for (int i = 0; i < g.N; ++i) {                  // sequential in agent order; every lane computes the same cell
            const int c = draw_cell(phase == 0 ? S_START : S_GOAL, (uint32_t)i, true);
            const int cc = c < 0 ? hpos : c;
            if (c < 0) err |= 8u;
            __syncwarp();
            if (lane == 0) {
                s.occ[cc] = 1;
                int16_t *dst = phase == 0 ? g.starts + ((size_t)w * g.N + i) * 2 : g.goal_queue + ((size_t)w * g.N + i) * g.Q * 2;
                dst[0] = (int16_t)(cc / Wd); dst[1] = (int16_t)(cc % Wd);
            }
            __syncwarp();
        }
    }
    // ---- D. later goals: free cells, consecutive goals differ (lane = agent, strided) -------------------------------
    for (int i = lane; i < g.N; i += 32) {
        int16_t *q = g.goal_queue + ((size_t)w * g.N + i) * g.Q * 2;
        int prev = q[0] * Wd + q[1];
        for (int k = 1; k < g.Q; ++k) {
            int c = prev;
            for (uint32_t t = 0; t < 64 && c == prev; ++t) {
                const U4 r = philox4(g.seed, gw, S_QUEUE, ((uint32_t)i * (uint32_t)g.Q + (uint32_t)k) * 64 + t);
                const int y0 = (int)(r.x % (uint32_t)rows), x0 = (int)(r.y % (uint32_t)cols);
                const int y1 = (int)(r.z % (uint32_t)rows), x1 = (int)(r.w % (uint32_t)cols);
                if (s.freec[y0 * Wd + x0] && y0 * Wd + x0 != prev) c = y0 * Wd + x0;
                else if (s.freec[y1 * Wd + x1] && y1 * Wd + x1 != prev) c = y1 * Wd + x1;
            }
            q[2 * k] = (int16_t)(c / Wd); q[2 * k + 1] = (int16_t)(c % Wd);
            prev = c;
        }
    }
    const uint32_t eb = __reduce_or_sync(FULL, err);
    if (lane == 0 && g.gen_err) g.gen_err[w] = eb;
}

}  // namespace

cudaError_t launch_scenario_gen(const MapfGenConfig &c, uint8_t *obst, int16_t *dims, int16_t *starts, int16_t *goal_queue,
                                int16_t *htrace, int32_t *hlen, int16_t *hp5, uint32_t *gen_err, cudaStream_t stream) {
    GenView g;
    g.W = c.num_worlds; g.H = c.height; g.Wd = c.width; g.N = c.num_agents; g.Q = c.queue_len; g.L = c.trace_len;
    g.kind = c.kind; g.density_mode = c.density_mode; g.size_lo = c.size_lo; g.size_hi = c.size_hi;
    g.human_loops = c.human_loops < 1 ? 1 : c.human_loops;
    g.human_path = c.human_path;
    g.dlo = c.density_lo; g.dhi = c.density_hi; g.seed = c.seed; g.world_offset = c.world_offset;
    g.obst = obst; g.dims = dims; g.starts = starts; g.goal_queue = goal_queue; g.htrace = htrace; g.hp5 = hp5;
    g.hlen = hlen; g.gen_err = gen_err;
    const int cells = c.height * c.width;
    const int per_warp = 2 * ((cells + 15) & ~15) + ((cells * 2 + 15) & ~15) + 2 * gen_set_words(cells) * 4 +
                         (c.human_path == 1 ? (gen_set_words(cells) + gen_par_words(cells)) * 4 : 0);
    int wpb = 4;
    while (wpb > 1 && per_warp * wpb > 160 * 1024) wpb >>= 1;
    const size_t smem = (size_t)per_warp * wpb;
    cudaError_t e = cudaFuncSetAttribute(scenario_gen_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int blocks = (c.num_worlds + wpb - 1) / wpb;
    scenario_gen_kernel<<<blocks, wpb * 32, smem, stream>>>(g, per_warp);
    return cudaGetLastError();
}

}  // namespace mapf
