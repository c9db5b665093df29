// astar4.cu — mapf_astar4_paths: astar_4 for many (map, start, goal) triples at once, one warp per triple (astar4.cuh).
// Used to plan every leg of a batch of evaluation fixtures in one call (episode_io.scenario_from_fixed_episode_infos).
#include "astar4.cuh"
#include "common.cuh"

namespace mapf {

namespace {

struct Astar4Layout {                 // per-warp shared memory, 16-byte aligned pieces
    int words, g_bytes, set_bytes, par_bytes, total;
    __host__ __device__ explicit Astar4Layout(int cells)
        : words(astar4_words(cells)), g_bytes((cells * 2 + 15) & ~15), set_bytes(((words + 3) & ~3) * 4),
          par_bytes((((cells + 15) / 16 + 3) & ~3) * 4), total(g_bytes + 4 * set_bytes + par_bytes) {}
};

__global__ void __launch_bounds__(128) astar4_paths_kernel(const uint8_t *__restrict__ obst, long long n, int H, int Wd,
                                                           const int16_t *__restrict__ start_goal, int max_len,
                                                           int16_t *__restrict__ paths, int32_t *__restrict__ lens) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cells = H * Wd;
    const Astar4Layout lay(cells);
    unsigned char *base = smem_raw + (size_t)warp * lay.total;
    Astar4Smem s;
    s.g = reinterpret_cast<int16_t *>(base);
    s.open = reinterpret_cast<uint32_t *>(base + lay.g_bytes);
    s.closed = s.open + lay.set_bytes / 4;
    s.lvl = s.closed + lay.set_bytes / 4;
    uint32_t *freeb = s.lvl + lay.set_bytes / 4;      // bit set of the map's free cells
    s.par = freeb + lay.set_bytes / 4;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long i = (long long)blockIdx.x * (blockDim.x >> 5) + warp; i < n; i += nwarps) {
        const int16_t *sg = start_goal + i * 4;
        const int sr = sg[0], sc = sg[1], tr = sg[2], tc = sg[3];
        int16_t *out = paths + i * (long long)max_len * 2;
        int len;
        if (sr < 0 || sr >= H || sc < 0 || sc >= Wd || tr < 0 || tr >= H || tc < 0 || tc >= Wd) len = -3;
        else if (sr == tr && sc == tc) len = 0;
        else {
            const uint8_t *m = obst + i * (long long)cells;
            for (int k = 0; k < lay.words; ++k) {
                const int c = 32 * k + lane;
                const unsigned b = __ballot_sync(FULL, c < cells && m[c] == 0);
                if (lane == 0) freeb[k] = b;
            }
            __syncwarp();
            const int goal = tr * Wd + tc;
            const int d = astar4_search(s, H, Wd, sr * Wd + sc, goal,
                                        [&](int c) { return (freeb[c >> 5] >> (c & 31)) & 1u; });
            len = d < 0 ? -1 : d + 1 > max_len ? -2 : d + 1;
            if (len > 0 && lane == 0)
                for (int c = goal;; c = astar4_parent(s, Wd, c)) {       // cell c is the k-th of the path, k = its g
                    const int k = s.g[c];
                    out[2 * k] = (int16_t)(c / Wd); out[2 * k + 1] = (int16_t)(c % Wd);
                    if (k == 0) break;
                }
        }
        for (int k = (len > 0 ? len : 0) * 2 + lane; k < max_len * 2; k += 32) out[k] = -1;
        if (lane == 0) lens[i] = len;
        __syncwarp();
    }
}

}  // namespace

cudaError_t launch_astar4_paths(const uint8_t *obst, long long n, int H, int Wd, const int16_t *start_goal, int max_len,
                                int16_t *paths, int32_t *lens, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const Astar4Layout lay(H * Wd);
    int wpb = 4;
    while (wpb > 1 && lay.total * wpb > 160 * 1024) wpb >>= 1;
    const size_t smem = (size_t)lay.total * wpb;
    cudaError_t e = cudaFuncSetAttribute(astar4_paths_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long blocks = (n + wpb - 1) / wpb;
    astar4_paths_kernel<<<(unsigned)(blocks < (1 << 20) ? blocks : (1 << 20)), wpb * 32, smem, stream>>>(
        obst, n, H, Wd, start_goal, max_len, paths, lens);
    return cudaGetLastError();
}

}  // namespace mapf
