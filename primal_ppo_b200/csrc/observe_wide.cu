// observe_wide.cu — observation builder for worlds whose block does not fit one warp pass (more than 32 agents, or a
// field of view so large that 32 agents' bit strings exceed the per-warp scratch): BASELINE.json configs[4], 80x80
// worlds, 128 agents, FOV up to 31x31.
//
// Same arithmetic as observe_kernel (observe_world.cuh: observe_chunk), different mapping: ONE CTA of 8 warps per world.
// The world is staged once per CTA (obstacle bit rows, agent-presence bit rows, agent-id grid, cells and goals of all N
// agents); the warps then take chunks of L.CH agents round-robin, each with its own bit-string scratch.  With the
// warp-per-world mapping every warp carries its own copy of the staging (17 KB for a padded 110x110 world plus 24 KB
// of scratch), which leaves 4 warps per SM; sharing it gives 16-32 warps per SM, and a world's 3 MB observation block
// is written by eight warps instead of one.
#include "common.cuh"
#include "observe_world.cuh"

namespace mapf {

namespace {

using namespace ow;

constexpr int WIDE_WARPS = 8;

template <int C_T, int F_T, bool VEC4, bool BITS>
__global__ void __launch_bounds__(WIDE_WARPS * 32)
observe_wide_kernel(const EnvView v, float *__restrict__ obs, float *__restrict__ vec, const ObsLayout L,
                    const int shared_bytes, const int per_warp, int *__restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint4 lut[16];
    __shared__ int s_world;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW, HP = v.HP, nob = v.HP * v.RW;
    // CTA-shared staging uses the ObsLayout offsets of the staging part; per-warp scratch (aw, wb) follows it
    ObsSmem m;
    m.obits = reinterpret_cast<uint32_t *>(smem_raw);
    m.abits = reinterpret_cast<uint32_t *>(smem_raw + L.off_abits);
    m.grid = smem_raw + L.off_grid;
    m.sgoal = reinterpret_cast<uint32_t *>(smem_raw + L.off_goal);
    m.spos = m.sgoal + N;
    unsigned char *mine = smem_raw + shared_bytes + (size_t)warp * per_warp;
    m.aw = reinterpret_cast<uint32_t *>(mine);
    m.wb = reinterpret_cast<uint32_t *>(mine + ((size_t)L.CH * L.AST * 4 + 15) / 16 * 16);
    fill_lut(lut, tid);
    for (int k = tid; k < nob; k += blockDim.x) m.abits[k] = 0;
    for (int k = tid; k < (HP * GS) / 16; k += blockDim.x) reinterpret_cast<uint4 *>(m.grid)[k] = make_uint4(0, 0, 0, 0);
    const int nchunks = (N + L.CH - 1) / L.CH;
    const uint64_t pol = policy_evict_last();
    const int dir = tid == 0 ? walk_dir(v) : 0;           // serpentine order (common.cuh world_of)
    for (;;) {
        __syncthreads();                                   // previous world fully written, scratch clean
        if (tid == 0) s_world = world_of(v, atomicAdd(work_counter, 1), dir);
        __syncthreads();
        const int w = s_world;
        if (w >= v.W) break;
        // ---- stage the world once for the CTA ---------------------------------------------------------------------
        expand_obstacle_rows<true>(m.obits, v.obst_pack + (size_t)w * v.PW, v, tid, blockDim.x, pol);
        const uint32_t *posw = reinterpret_cast<const uint32_t *>(v.pos) + (size_t)w * N;
        const uint32_t *goalw = reinterpret_cast<const uint32_t *>(v.goal) + (size_t)w * N;
        for (int i = tid; i < N; i += blockDim.x) {
            const uint32_t pw = ld_keep(posw + i, pol);
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            m.grid[(r + P) * GS + c + P] = (uint8_t)(i + 1);
            atomicOr(&m.abits[(r + P) * RW + ((c + P) >> 5)], 1u << ((c + P) & 31));
            m.sgoal[i] = ld_keep(goalw + i, pol);
            m.spos[i] = pw;
        }
        const int2 ht = ld_keep_v2(reinterpret_cast<const int2 *>(v.hcur) + w, pol);
        const int nr = (int16_t)(ht.y & 0xffff), nc = (int16_t)((uint32_t)ht.y >> 16);            // human.getNextPos()
        int rows = v.H, cols = v.Wd;
        if (v.use_da | v.use_hp) { if (v.dims) { rows = v.dims[2 * w]; cols = v.dims[2 * w + 1]; } }
        __syncthreads();
        // ---- chunks of agents, round-robin over the warps ---------------------------------------------------------------
        for (int k = warp; k < nchunks; k += WIDE_WARPS) {
            const int c0 = k * L.CH;
            observe_chunk<C_T, F_T, VEC4, 32, BITS>(v, L, m, lut, w, Grp<32>(lane), c0, min(L.CH, N - c0), nr, nc, rows, cols, obs, vec);
        }
        __syncthreads();
        // ---- un-scatter so that the next world starts from a clean grid ------------------------------------------------
        for (int i = tid; i < N; i += blockDim.x) {
            const uint32_t pw = m.spos[i];
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            m.grid[(r + P) * GS + c + P] = 0;
            m.abits[(r + P) * RW + ((c + P) >> 5)] = 0;
        }
    }
    __syncthreads();
    finish_work(work_counter, gridDim.x, tid, v.order);   // the last CTA to finish re-arms the counter, flips the direction
}

}  // namespace

// Returns cudaErrorNotSupported when the shape is better served (or only served) by the warp-per-world kernel.
cudaError_t launch_observe_wide(const EnvView &v, float *obs, float *vec, int *work_counter, cudaStream_t stream, int fmt) {
    const int PB = v.C * v.F * v.F;
    // chunk size: per-warp scratch (aw + wb) of at most ~12 KB, and at least one chunk per warp when N allows it
    int CH = 32;
    while (CH > 2 && (chunk_scratch(CH, PB) > 12 * 1024 || (v.N + CH - 1) / CH < WIDE_WARPS)) CH >>= 1;
    if (chunk_scratch(CH, PB) > 28 * 1024) return cudaErrorNotSupported;
    ObsLayout L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH);
    L.alias = 0;
    L.fmt = fmt;
    const int shared_bytes = (int)cta_shared_bytes(L, v.N), per_warp = (int)warp_scratch_bytes(CH, PB);
    const size_t smem = (size_t)shared_bytes + (size_t)per_warp * WIDE_WARPS;
    if (smem > 200 * 1024) return cudaErrorNotSupported;
    return dispatch_obs(fmt, v.C, v.F, obs_vec4(fmt, v.N, PB, CH, obs), [&](auto t) {
        using T = decltype(t);
        return launch_persistent(observe_wide_kernel<T::C_T, T::F_T, T::VEC4, T::BITS>, WIDE_WARPS * 32, smem, v.W, INT_MAX,
                                 stream, v, obs, vec, L, shared_bytes, per_warp, work_counter);
    });
}

}  // namespace mapf
