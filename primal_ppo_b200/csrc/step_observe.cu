// step_observe.cu — one launch for the rollout loop's whole per-step env work (runner.py:64-100): joint-step
// resolution (step_world.cuh) followed, for the same world and by the same warp, by the observation build of the
// post-step state (observe_world.cuh).
//
// Why fuse: step resolution is issue/latency-bound (~1000 warp instructions per world, almost no HBM traffic) while the
// observation store is HBM-write-bound with the SM issue slots ~26 % busy.  Run back to back as two kernels they add
// up (0.13 ms + 0.68 ms for 65 536 worlds); inside one persistent kernel the step work of some warps hides under the
// stores of the others, the post-step cells / goals / human tick go from the step phase to the observe phase in
// registers (no state re-read), and the obstacle bit rows are staged once.
// N <= 32 only (lane = agent).  Results are bit-identical to mapf_step followed by mapf_observe.
#include "common.cuh"
#include "observe_world.cuh"
#include "step_world.cuh"

namespace mapf {

namespace {

using namespace sw;
using namespace ow;

// G = lanes per world: 32 = one world per warp; 8 / 16 = four / two small worlds per warp, each owned by a lane group that
// claims, loads and processes its worlds independently of the other groups of the warp (Grp<G>, group lane masks).
// Why groups: with 8 agents per world (BASELINE configs[1]) a warp-per-world step keeps 8 of 32 lanes busy and a world still
// costs ~15 us of dependent work, so the step phase — not the 15 KB of stores per world — bounded the launch (0.62 of the
// HBM roofline at 65 536 x 20x20x8).
template <int C_T, int F_T, bool VEC4, int MINB, int G, bool BITS>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MINB)
step_observe_kernel(const EnvView v, const int8_t *__restrict__ actions, const MapfStepOut out, float *__restrict__ obs,
                    float *__restrict__ vec, const ObsLayout L, const int per_group, const int step_off,
                    int *__restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint4 lut[16];
    constexpr int MPW = 32 / G;                               // worlds (groups) per warp
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const Grp<G> g(lane);
    const int gl = g.gl, grp = G == 32 ? 0 : lane / G;
    const int HP = v.HP, GS = v.GS, nob = v.HP * v.RW, npw = v.PW;
    unsigned char *base = smem_raw + ((size_t)warp * MPW + grp) * per_group;
    const ObsSmem m = obs_carve(base, L, v.N);
    // the step phase shares the obstacle bit rows and the agent-id grid with the observe phase; its own scratch
    // (trainValid staging, conflict masks, fixActions queue) sits behind the observe layout
    WarpSmem s;
    s.obits = m.obits;
    s.grid = m.grid;
    carve_step_scratch(s, base + step_off, G);
    fill_lut(lut, threadIdx.x);
    __syncthreads();

    // claim-then-load (see observe.cu).  ONE claim per warp hands out 32 / G consecutive worlds, one per lane group: the
    // groups of a warp start every world together and stay converged through the common path, so an instruction issues
    // once for all of them (groups that drift apart would each issue their own copy with G lanes active); only the rare
    // data-dependent sections (sequential status replay, fixActions queue, goal draws) run per group, under group masks.
    // Worlds are claimed in claim space (wb) and mapped to worlds in the launch's direction (serpentine order, world_of).
    const int dir = walk_dir(v);
    int wb = claim_work(work_counter, MPW, lane);
    int w = world_of(v, wb + grp, dir);
    const uint64_t pol = policy_evict_last();
    StepRegs cur, nxt;
    load_step_world<MODE_FUSED, G>(v, actions, nullptr, w, gl, npw, pol, cur);
    const bool direct_ob = npw > SOBW * G;
    bool first = true;

    while (wb < v.W) {
        const int wb1 = claim_work(work_counter, MPW, lane);
        const int w1 = world_of(v, wb1 + grp, dir);
        load_step_world<MODE_FUSED, G>(v, actions, nullptr, w1, gl, npw, pol, nxt);   // in flight during this world
        // (the prefetch distance and batch are re-read from the kernel parameters: no registers held across the loop)
        if (lane == 0 && prefetch_ahead(v) >= 0 && (wb1 & (prefetch_batch(v) - 1)) == 0)
            prefetch_world_batch(v, actions, wb1 + prefetch_ahead(v), dir, pol);

        if (w < v.W) {
            // packed obstacle words: registers -> scratch (the agent-presence rows, zeroed right after) -> padded rows
            if (!direct_ob) {
#pragma unroll
                for (int k = 0; k < SOBW; ++k) if (k * G + gl < npw) m.abits[k * G + gl] = cur.ob[k];
                g.sync();
                expand_obstacle_rows(m.obits, m.abits, v, gl, G);
            } else {
                expand_obstacle_rows<true>(m.obits, v.obst_pack + (size_t)w * npw, v, gl, G, pol);
            }
            g.sync();
            for (int k = gl; k < nob; k += G) m.abits[k] = 0;
            if (L.alias || first) {          // the chunk bit string of the previous world overlays the id grid when L.alias
                uint4 *g4 = reinterpret_cast<uint4 *>(m.grid);
                for (int k = gl; k < (HP * GS) / 16; k += G) g4[k] = make_uint4(0, 0, 0, 0);
                first = false;
            }
            g.sync();
            uint32_t new_pw, new_gw;
            resolve_world<MODE_FUSED, false, G>(v, out, s, w, g, cur, pol, new_pw, new_gw);      // leaves the id grid clean
            g.sync();
            // the human has ticked: its getNextPos() is the `next` field of the following trace entry
            const int nr = (int16_t)(cur.ht2.y & 0xffff), nc = (int16_t)((uint32_t)cur.ht2.y >> 16);
            observe_world<C_T, F_T, VEC4, G, BITS>(v, L, m, lut, w, g, new_pw, new_gw, nr, nc, obs, vec);
        }
        wb = wb1;
        w = w1;
        cur = nxt;
    }
    finish_work(work_counter, gridDim.x * (blockDim.x >> 5), lane, v.order);
}

}  // namespace

// Lanes per world: the narrowest lane group that holds the agents (8 / 16 / 32), provided the worlds are small enough for
// a warp to stage 32 / G of them (shared memory for at least three CTAs per SM) and below the store-dominated regime;
// MAPF_DBG_FLAGS bit 28 keeps one world per warp (A/B runs).
static int group_width(const EnvView &v, int fmt) {
    const int CH = obs_chunk(v.N, v.C * v.F * v.F);
    if (v.N > 16 || (v.dbg_flags & (1 << 28)) || CH < v.N) return 32;
    const int G = v.N <= 8 ? 8 : 16;
    ObsLayout L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH, G);
    L.fmt = fmt;
    if (obs_world_bytes(L, v.N) >= 32768) return 32;
    const size_t per_cta = (L.total + sw::step_scratch_bytes(G)) * (32 / G) * WARPS_PER_BLOCK;
    if (per_cta > 72 * 1024) return 32;
    if (v.PW > sw::SOBW * G * 4) return 32;       // keep the register-prefetched obstacle words useful
    return G;
}

// The fused kernel covers lane = agent worlds whose observation is built in one chunk (every training configuration);
// anything else (N > 32, FOV 31 with 32 agents, ...) is served by the CTA-per-world fused kernel (step_observe_wide.cu).
bool step_observe_fusable(const EnvView &v) {
    const int CH = obs_chunk(v.N, v.C * v.F * v.F);
    if (v.N > 32 || CH < v.N) return false;
    const ObsLayout L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH);
    return (L.total + sw::step_scratch_bytes(32)) * WARPS_PER_BLOCK <= 200 * 1024;
}

cudaError_t launch_step_observe(const EnvView &v, const int8_t *actions, const MapfStepOut &out, float *obs, float *vec,
                                int *work_counter, cudaStream_t stream, int fmt) {
    const int PB = v.C * v.F * v.F, CH = obs_chunk(v.N, PB);
    const int G = group_width(v, fmt), wpg = WARPS_PER_BLOCK * (32 / G);     // worlds per CTA
    ObsLayout L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH, G);
    L.fmt = fmt;
    const int step_off = (int)L.total, per_group = step_off + (int)step_scratch_bytes(G);
    const size_t smem = (size_t)per_group * wpg;
    if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
    const int need = (v.W + wpg - 1) / wpg;
    // As in observe.cu fewer write streams help store-dominated worlds (>= 32 KB of observations each), but here the step
    // phase needs warps to hide behind: in-process A/B at 40x40x32: 2 / 3 / 4 CTAs per SM = 0.772 / 0.722 / 0.731 ms.  The
    // 3-CTA instantiation is also COMPILED for 3 CTAs (80 registers instead of 64, no spills): 0.706 vs 0.721 ms.
    const bool big = obs_world_bytes(L, v.N) >= 32768;
    return dispatch_obs(fmt, v.C, v.F, obs_vec4(fmt, v.N, PB, CH, obs), [&](auto t) {
        using T = decltype(t);
        auto launch = [&](auto kern, int minb) {
            return launch_persistent(kern, WARPS_PER_BLOCK * 32, smem, need, minb, stream, v, actions, out, obs, vec, L,
                                     per_group, step_off, work_counter);
        };
        if (G == 8) return launch(step_observe_kernel<T::C_T, T::F_T, T::VEC4, 4, 8, T::BITS>, 4);
        if (G == 16) return launch(step_observe_kernel<T::C_T, T::F_T, T::VEC4, 4, 16, T::BITS>, 4);
        if (big) return launch(step_observe_kernel<T::C_T, T::F_T, T::VEC4, 3, 32, T::BITS>, 3);
        return launch(step_observe_kernel<T::C_T, T::F_T, T::VEC4, 4, 32, T::BITS>, 4);
    });
}

}  // namespace mapf
