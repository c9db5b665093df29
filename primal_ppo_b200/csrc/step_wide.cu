// step_wide.cu — joint-step resolution for worlds with 32 < N <= 128 agents (BASELINE.json configs[4]: 80x80, 128 agents)
// as a stand-alone launch: one warp per world running step_wide_world (step_wide_world.cuh) with lane loops over agents.
// The rollout path for these shapes is the fused step_observe_wide_kernel (step_observe_wide.cu), where a whole CTA shares
// the same code; this kernel serves mapf_evaluate / mapf_joint_step / mapf_step.
#include "common.cuh"
#include "step_wide_world.cuh"

namespace mapf {

namespace {

using namespace sww;

constexpr int WIDE_WARPS = 4;

__host__ __device__ inline size_t wide_bytes(int HP, int RW, int GS) {
    return align16((size_t)HP * RW * 4) + align16((size_t)HP * GS) + scratch_bytes();
}

template <int MODE>
__global__ void __launch_bounds__(WIDE_WARPS * 32)
step_wide_kernel(const EnvView v, const int8_t *__restrict__ actions, const int8_t *__restrict__ status_in,
                 const MapfStepOut out, const int per_warp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * WIDE_WARPS + warp;
    if (w >= v.W) return;
    const int HP = v.HP, RW = v.RW, GS = v.GS;
    unsigned char *b = smem_raw + (size_t)warp * per_warp;
    WideSmem s;
    s.obits = reinterpret_cast<uint32_t *>(b); b += align16((size_t)HP * RW * 4);
    s.grid = b; b += align16((size_t)HP * GS);
    carve_scratch(s, b);
    expand_obstacle_rows<true>(s.obits, v.obst_pack + (size_t)w * v.PW, v, lane, 32, policy_evict_last());
    uint4 *g4 = reinterpret_cast<uint4 *>(s.grid);
    for (int k = lane; k < (HP * GS) / 16; k += 32) g4[k] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    int hnr, hnc;
    step_wide_world<MODE, false>(v, actions, status_in, out, s, w, lane, 32, hnr, hnc);
}

}  // namespace

cudaError_t launch_step_wide(const EnvView &v, const int8_t *actions, const int8_t *status_in, const MapfStepOut &out,
                             int mode, cudaStream_t stream) {
    if (v.N > NMAX) return cudaErrorInvalidValue;
    const int per_warp = (int)wide_bytes(v.HP, v.RW, v.GS);
    const size_t smem = (size_t)per_warp * WIDE_WARPS;
    const int blocks = (v.W + WIDE_WARPS - 1) / WIDE_WARPS;
    cudaError_t e = cudaSuccess;
#define LAUNCH(M)                                                                                                  \
    do {                                                                                                           \
        e = cudaFuncSetAttribute(step_wide_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);     \
        if (e == cudaSuccess) step_wide_kernel<M><<<blocks, WIDE_WARPS * 32, smem, stream>>>(v, actions, status_in, out, per_warp); \
    } while (0)
    if (mode == MODE_EVALUATE) LAUNCH(MODE_EVALUATE);
    else if (mode == MODE_JOINT) LAUNCH(MODE_JOINT);
    else LAUNCH(MODE_FUSED);
#undef LAUNCH
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

}  // namespace mapf
