// observe.cu — observation builder: one warp per world, persistent CTAs with dynamic world scheduling.
//
// Replaces MapfGym.getAllObservations / observe / worldWithAgents (mapf_gym.py:192-198, 246-336) for W worlds:
//   obs f32 [W,N,C,F,F]  (0/1 valued)   and   vec f32 [W,N,4] = [dx/d, dy/d, d, 0]
// written straight into the policy's input tensors.  The store of obs is ~95 % of all bytes of a step, so the
// kernel is organised around keeping 16-byte stores in flight:
//   prefetch the NEXT world's inputs (agent cells, goals, obstacle bit rows, human tick) are loaded into registers
//            while the current world is being written, and the index of the world after that is claimed with one
//            atomicAdd per warp (dynamic scheduling: SMs that drain faster take more worlds, no tail).
//   phase 1  lane = agent: build the agent's C*F*F observation as a BIT string.  Channels 0/1 are F-bit windows cut
//            out of padded obstacle / agent-presence bit rows with one funnel shift per row (no per-cell work);
//            channels 2-5 are a handful of single bits (own goal, clamped goals of visible agents, human).
//   phase 1b compact the per-agent bit strings into one contiguous bit string of the chunk (N*C*F*F bits).
//   phase 2  all 32 lanes expand bits to floats: one nibble -> one 16-byte LUT read -> one 16-byte streaming store,
//            512 contiguous bytes per warp instruction (each world's block N*C*F*F*4 B is contiguous in HBM).
// Algorithmic HBM traffic per world: write N*(4*C*F*F + 16) B; read N*8 B state + HP*RW*4 B obstacle bits + 8 B human.
#include "common.cuh"
#include "observe_world.cuh"

namespace mapf {

namespace {

using namespace ow;

// C_T/F_T > 0: compile-time channels / FOV (the training configuration 6 x 9 x 9); 0: runtime values from EnvView.
template <int C_T, int F_T, bool VEC4, bool BITS>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, 4)
observe_kernel(const EnvView v, float *__restrict__ obs, float *__restrict__ vec, const ObsLayout L,
               int *__restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint4 lut[16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int GS = v.GS, HP = v.HP, nob = v.HP * v.RW, npw = v.PW;
    const ObsSmem m = obs_carve(smem_raw + (size_t)warp * L.total, L, v.N);
    uint32_t *const obits = m.obits, *const abits = m.abits;
    uint8_t *const grid = m.grid;

    fill_lut(lut, threadIdx.x);
    __syncthreads();

    // dynamic world scheduling: w (inputs in registers) is processed while w1, claimed at the top of the iteration, is
    // being loaded.  Claim and load are adjacent in time so that worlds are LOADED in (nearly) claim order, which is
    // what lets the batched L2 prefetch run a fixed distance ahead of the loads.
    const int dir = walk_dir(v);
    int w = world_of(v, claim_work(work_counter, 1, lane), dir);
    const uint64_t pol = policy_evict_last();
    WorldRegs cur, nxt;
    load_world(v, w, lane, npw, pol, cur);
    const bool direct_ob = npw > OBW * 32;
    bool first = true;

    while (w < v.W) {
        const int c1 = claim_work(work_counter, 1, lane), w1 = world_of(v, c1, dir);
        load_world(v, w1, lane, npw, pol, nxt);                  // in flight while this world is processed
        // (the prefetch distance and batch are re-read from the kernel parameters: no registers held across the loop)
        if (lane == 0 && prefetch_ahead(v) >= 0 && (c1 & (prefetch_batch(v) - 1)) == 0)
            prefetch_world_batch(v, nullptr, c1 + prefetch_ahead(v), dir, pol);

        // ---- stage: packed obstacle words (registers -> scratch in the agent-presence rows -> padded rows), then clean
        //      agent rows / id grid
        if (!direct_ob) {
#pragma unroll
            for (int k = 0; k < OBW; ++k) if (k * 32 + lane < npw) abits[k * 32 + lane] = cur.ob[k];
            __syncwarp();
            expand_obstacle_rows(obits, abits, v, lane, 32);
        } else {
            expand_obstacle_rows<true>(obits, v.obst_pack + (size_t)w * npw, v, lane, 32, pol);
        }
        __syncwarp();
        for (int k = lane; k < nob; k += 32) abits[k] = 0;
        if (L.alias || first) {
            uint4 *g4 = reinterpret_cast<uint4 *>(grid);
            for (int k = lane; k < (HP * GS) / 16; k += 32) g4[k] = make_uint4(0, 0, 0, 0);
            first = false;
        }
        __syncwarp();
        const int nr = (int16_t)(cur.ht.y & 0xffff), nc = (int16_t)((uint32_t)cur.ht.y >> 16);   // human.getNextPos()
        observe_world<C_T, F_T, VEC4, 32, BITS>(v, L, m, lut, w, Grp<32>(lane), cur.pw, cur.gw, nr, nc, obs, vec);
        w = w1;
        cur = nxt;
    }
    finish_work(work_counter, gridDim.x * (blockDim.x >> 5), lane, v.order);
}

}  // namespace

cudaError_t launch_observe(const EnvView &v, float *obs, float *vec, int *work_counter, cudaStream_t stream, int fmt) {
    const int PB = v.C * v.F * v.F, CH = obs_chunk(v.N, PB);
    // worlds whose block needs several warp passes: one CTA per world with shared staging (observe_wide.cu)
    if ((v.N > 32 || CH < v.N || (v.dbg_flags & 4)) && !(v.dbg_flags & 2)) {
        const cudaError_t e = launch_observe_wide(v, obs, vec, work_counter, stream, fmt);
        if (e != cudaErrorNotSupported) return e;
    }
    ObsLayout L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH);
    L.fmt = fmt;
    int wpb = WARPS_PER_BLOCK;
    while (wpb > 1 && L.total * wpb > 200 * 1024) wpb >>= 1;
    if (L.total * wpb > 227 * 1024) return cudaErrorInvalidConfiguration;
    // Store-dominated worlds (>= 32 KB of observations each) run best with FEWER resident warps: the HBM write path prefers
    // fewer, longer write streams (write-pattern benchmark: 16 warps/SM beat 32 by 2 %), and this kernel has no other
    // latency to hide.  In-process A/B at 40x40x32: 1 / 2 / 3 / 4 CTAs per SM = 0.613 / 0.608 / 0.612 / 0.622 ms.
    const int max_per_sm = obs_world_bytes(L, v.N) >= 32768 ? 2 : INT_MAX;
    return dispatch_obs(fmt, v.C, v.F, obs_vec4(fmt, v.N, PB, CH, obs), [&](auto t) {
        using T = decltype(t);
        return launch_persistent(observe_kernel<T::C_T, T::F_T, T::VEC4, T::BITS>, wpb * 32, L.total * wpb,
                                 (v.W + wpb - 1) / wpb, max_per_sm, stream, v, obs, vec, L, work_counter);
    });
}

}  // namespace mapf
