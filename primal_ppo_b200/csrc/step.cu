// step.cu — joint-step resolution: one warp per world, lane = agent (N <= 32).
//
// Replaces, for W worlds at once, the five calls the rollout loop makes per step (runner.py:64-91):
//   getActionStatus (mapf_gym.py:434-480), calculateActionReward (:483-511), calculateCostReward (:528-533),
//   getTrainValid (:535-550), jointStep (:614-637) incl. fixActions (:552-612), and the mask refresh
//   getUnconditionallyGoodActions (:404-430 -> getInvalidActions :339-360, getRestrictedActions :363-402).
//
// The reference keeps per-agent Python lists (invalid / restricted / good) that it rebuilds after every jointStep.
// Here they are never stored: they are a pure function of (positions, obstacle bits, human tick, repetition action)
// and are recomputed at the start of the step as 5-bit masks in registers.  The obstacle tile (bit rows) and an
// agent-id byte grid live in shared memory; an agent looks at the 12 cells of the radius-2 diamond around itself:
//   restricted[a]  <=>  another agent within Manhattan distance 1 of the target cell of a        (SURVEY A.3)
//   conflict(i,a;j,b) <=> T_i(a)==T_j(b)  or  (T_i(a)==pos_j and T_j(b)==pos_i)
// Order dependence of getActionStatus (an agent that was already marked -3 is skipped and therefore does not mark
// its fellows) only matters when a human-collision agent conflicts with a restricted-class agent; that case is
// detected with a warp vote and resolved by replaying the reference's sequential loop on lane 0 (rare path).
// fixActions: agents with an unconditionally good action commit in parallel (their choice can not conflict with
// anything); the remaining queue is processed in the reference's FIFO order, each iteration executed by the lane
// that owns the agent, with the committed actions in shared memory.
#include "common.cuh"
#include "step_common.cuh"
#include "step_world.cuh"

namespace mapf {

namespace {

using namespace sw;

// Persistent CTAs, one warp per world at a time; worlds are claimed with one atomicAdd per warp and the next world's
// inputs are loaded into registers while the current one is being resolved.
template <int MODE>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, 4)
step_kernel(const EnvView v, const int8_t *__restrict__ actions, const int8_t *__restrict__ status_in,
            const MapfStepOut out, const int per_warp, int *__restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int HP = v.HP, RW = v.RW, GS = v.GS, npw = v.PW;
    WarpSmem s = carve(smem_raw + (size_t)warp * per_warp, HP, RW, GS);
    {
        uint4 *g4 = reinterpret_cast<uint4 *>(s.grid);
        for (int k = lane; k < (HP * GS) / 16; k += 32) g4[k] = make_uint4(0, 0, 0, 0);
    }
    const int dir = walk_dir(v);
    int w = world_of(v, claim_work(work_counter, 1, lane), dir);      // claim-then-load: see observe.cu
    const uint64_t pol = policy_evict_last();
    StepRegs cur, nxt;
    load_step_world<MODE>(v, actions, status_in, w, lane, npw, pol, cur);
    const bool direct_ob = npw > SOBW * 32;
    while (w < v.W) {
        const int c1 = claim_work(work_counter, 1, lane), w1 = world_of(v, c1, dir);
        load_step_world<MODE>(v, actions, status_in, w1, lane, npw, pol, nxt);
        // (the prefetch distance and batch are re-read from the kernel parameters: no registers held across the loop)
        if (lane == 0 && prefetch_ahead(v) >= 0 && (c1 & (prefetch_batch(v) - 1)) == 0)
            prefetch_world_batch(v, actions, c1 + prefetch_ahead(v), dir, pol);
        if (!direct_ob) {                       // the packed obstacle words are probed directly (resolve_world<.., true>)
#pragma unroll
            for (int k = 0; k < SOBW; ++k) if (k * 32 + lane < npw) s.obits[k * 32 + lane] = cur.ob[k];
        } else {
            const uint32_t *src = v.obst_pack + (size_t)w * npw;
            for (int k = lane; k < npw; k += 32) s.obits[k] = ld_keep(src + k, pol);
        }
        uint32_t new_pw, new_gw;
        resolve_world<MODE, true>(v, out, s, w, Grp<32>(lane), cur, pol, new_pw, new_gw);
        __syncwarp();
        w = w1;
        cur = nxt;
    }
    finish_work(work_counter, gridDim.x * (blockDim.x >> 5), lane, v.order);
}

}  // namespace

cudaError_t launch_step(const EnvView &v, const int8_t *actions, const int8_t *status_in, const MapfStepOut &out,
                        int mode, int *work_counter, cudaStream_t stream) {
    const int per_warp = (int)warp_smem_bytes(v.HP, v.RW, v.GS);
    const size_t smem = (size_t)per_warp * WARPS_PER_BLOCK;
    const int need = (v.W + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    auto launch = [&](auto kern) {
        return launch_persistent(kern, WARPS_PER_BLOCK * 32, smem, need, INT_MAX, stream, v, actions, status_in, out, per_warp,
                                 work_counter);
    };
    if (mode == MODE_EVALUATE) return launch(step_kernel<MODE_EVALUATE>);
    if (mode == MODE_JOINT) return launch(step_kernel<MODE_JOINT>);
    return launch(step_kernel<MODE_FUSED>);
}

}  // namespace mapf
