// step_observe_wide.cu — one launch for the rollout loop's whole per-step env work (runner.py:64-100) for worlds that do
// not fit the warp-per-world fused kernel (step_observe.cu): more than 32 agents, or an observation block that needs
// several chunks (BASELINE.json configs[4]: 80x80 worlds, 128 agents, FOV 9..31).
//
// Mapping: ONE persistent CTA of 8 warps per world at a time (worlds are claimed dynamically).  The world is staged once
// for both phases — padded obstacle bit rows, agent-id grid — then
//   phase A: joint-step resolution by the whole CTA (step_wide_world.cuh: per-agent work spread over 256 threads, the
//            order-dependent parts on thread 0 / warp 0),
//   phase B: the post-step cells and goals go from shared memory straight into the observation build (no state re-read);
//            the eight warps take chunks of agents round-robin and stream the f32 block out (observe_world.cuh).
// With two or three CTAs resident per SM the latency-bound phase A of one world hides under the store-bound phase B of
// the others, which two back-to-back launches (step_wide_kernel, observe_wide_kernel) cannot do: at 80x80x128 / FOV 9 the
// two launches ran at 0.795 of the HBM roofline against 1.02 for the observation kernel alone.
// Results are bit-identical to mapf_step followed by mapf_observe.
#include "common.cuh"
#include "observe_world.cuh"
#include "step_wide_world.cuh"

namespace mapf {

namespace {

using namespace ow;
using namespace sww;

// WARPS per CTA / MINB resident CTAs per SM the kernel is compiled for.  The step phase of a world is latency-bound
// (~20 us: eight barrier-separated phases, global loads, thread-0 sections) and only hides under the stores of OTHER
// worlds, so what matters is the number of worlds in flight per SM = resident CTAs; small CTAs give more of them.
template <int C_T, int F_T, bool VEC4, bool BITS, int FW_WARPS, int MINB>
__global__ void __launch_bounds__(FW_WARPS * 32, MINB)
step_observe_wide_kernel(const EnvView v, const int8_t *__restrict__ actions, const MapfStepOut out, float *__restrict__ obs,
                         float *__restrict__ vec, const ObsLayout L, const int shared_bytes, const int scratch_off,
                         const int per_warp, int *__restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint4 lut[16];
    __shared__ int s_world;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW, HP = v.HP, nob = v.HP * v.RW;
    ObsSmem m;
    m.obits = reinterpret_cast<uint32_t *>(smem_raw);
    m.abits = reinterpret_cast<uint32_t *>(smem_raw + L.off_abits);
    m.grid = smem_raw + L.off_grid;
    m.sgoal = reinterpret_cast<uint32_t *>(smem_raw + L.off_goal);
    m.spos = m.sgoal + N;
    unsigned char *mine = smem_raw + shared_bytes + (size_t)warp * per_warp;
    m.aw = reinterpret_cast<uint32_t *>(mine);
    m.wb = reinterpret_cast<uint32_t *>(mine + ((size_t)L.CH * L.AST * 4 + 15) / 16 * 16);
    WideSmem s;
    s.obits = m.obits;
    s.grid = m.grid;
    carve_scratch(s, smem_raw + scratch_off);
    fill_lut(lut, tid);
    for (int k = tid; k < nob; k += blockDim.x) m.abits[k] = 0;
    for (int k = tid; k < (HP * GS) / 16; k += blockDim.x) reinterpret_cast<uint4 *>(m.grid)[k] = make_uint4(0, 0, 0, 0);
    const int nchunks = (N + L.CH - 1) / L.CH;
    const uint64_t pol = policy_evict_last();
    // prefetch distance: worlds here are 2..8 times larger than in the warp-per-world kernel, so fewer of them make a batch
    const int pf_batch = 64, pf_ahead = (v.dbg_flags & (1 << 29)) ? -1 : 128;
    const int dir = tid == 0 ? walk_dir(v) : 0;           // serpentine order (common.cuh world_of)
    for (;;) {
        __syncthreads();                                   // previous world fully written, grid / abits clean
        if (tid == 0) {
            const int c = atomicAdd(work_counter, 1);
            s_world = world_of(v, c, dir);
            // batched L2 prefetch of the state a few hundred claims ahead (common.cuh)
            if (pf_ahead >= 0 && (c & (pf_batch - 1)) == 0) prefetch_world_batch(v, actions, c + pf_ahead, dir, pol, pf_batch);
        }
        __syncthreads();
        const int w = s_world;
        if (w >= v.W) break;
        expand_obstacle_rows<true>(m.obits, v.obst_pack + (size_t)w * v.PW, v, tid, blockDim.x, pol);
        int rows = v.H, cols = v.Wd;
        if (v.use_da | v.use_hp) { if (v.dims) { rows = v.dims[2 * w]; cols = v.dims[2 * w + 1]; } }
        __syncthreads();
        // ---- phase A: the joint step, by the whole CTA ----------------------------------------------------------------------
        int nr, nc;                                        // human.getNextPos() after the tick
        step_wide_world<MODE_FUSED, true>(v, actions, nullptr, out, s, w, tid, blockDim.x, nr, nc);
        // ---- hand the post-step world to the observation build ---------------------------------------------------------------
        for (int i = tid; i < N; i += blockDim.x) {
            const uint32_t pw = s.npos[i];
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            m.grid[(r + P) * GS + c + P] = (uint8_t)(i + 1);
            atomicOr(&m.abits[(r + P) * RW + ((c + P) >> 5)], 1u << ((c + P) & 31));
            m.sgoal[i] = s.goal[i];
            m.spos[i] = pw;
        }
        __syncthreads();
        // ---- phase B: chunks of agents, round-robin over the warps -----------------------------------------------------------
        for (int k = warp; k < nchunks; k += FW_WARPS) {
            const int c0 = k * L.CH;
            observe_chunk<C_T, F_T, VEC4, 32, BITS>(v, L, m, lut, w, Grp<32>(lane), c0, min(L.CH, N - c0), nr, nc, rows, cols, obs, vec);
        }
        __syncthreads();
        for (int i = tid; i < N; i += blockDim.x) {        // un-scatter: the next world starts from a clean grid
            const uint32_t pw = m.spos[i];
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            m.grid[(r + P) * GS + c + P] = 0;
            m.abits[(r + P) * RW + ((c + P) >> 5)] = 0;
        }
    }
    __syncthreads();
    finish_work(work_counter, gridDim.x, tid, v.order);   // the last CTA to finish re-arms the counter, flips the direction
}

struct WidePlan {
    ObsLayout L;
    int shared_bytes, scratch_off, per_warp;
    size_t smem;
    bool ok;
};

WidePlan make_plan(const EnvView &v, int fmt, int FW_WARPS) {
    WidePlan p;
    p.ok = false;
    const int PB = v.C * v.F * v.F;
    // chunk size: at least one chunk per warp when N allows it; per-warp scratch (aw + wb) small enough for six resident
    // CTAs (~36 KB each) while the chunk keeps at least 8 agents (phase 1 runs one lane per agent), 12 KB at most
    const size_t staged = cta_shared_bytes(make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, 8), v.N);
    size_t budget = staged < 36 * 1024 ? (36 * 1024 - staged) / FW_WARPS : 0;
    if (budget > 12 * 1024) budget = 12 * 1024;
    // Balanced chunks: with `r` rounds every warp builds r chunks of CH = ceil(N / (warps * r)) agents, rounded up so that a
    // chunk's block stays 16-byte aligned (vector stores); the smallest r whose scratch fits the budget wins.  (Power-of-two
    // chunks left 33 agents as 5 chunks of 8 on 4 warps — one warp with twice the work — and 48 agents as 6.)
    const int need_al = fmt == OBS_BF16 ? 8 : 4;                   // (bits: records are word-aligned; f32 rule kept)
    int g = need_al;
    while (g > 1 && PB % g) g >>= 1;
    const int mult = need_al / g;                                   // CH must be a multiple of this
    int CH = 0;
    for (int r = 1; r <= 64 && CH == 0; ++r) {
        int ch = (v.N + FW_WARPS * r - 1) / (FW_WARPS * r);
        ch = (ch + mult - 1) / mult * mult;
        if (ch > 32) continue;
        if (chunk_scratch(ch, PB) <= 12 * 1024 && (ch <= 8 || chunk_scratch(ch, PB) <= budget)) CH = ch;
    }
    if (CH == 0) CH = mult <= 2 ? 2 : mult;
    if (chunk_scratch(CH, PB) > 28 * 1024) return p;
    p.L = make_layout(v.HP, v.RW, v.GS, v.N, v.C, v.F, CH);
    p.L.alias = 0;
    p.L.fmt = fmt;
    // [obits | abits | grid | goals + cells] shared by the CTA, then the per-warp observation scratch (aw, wb).  The step
    // phase's scratch is dead once the post-step cells / goals have been handed over, and the observation scratch is dead
    // during the step phase: they overlay each other (a __syncthreads separates the two uses).
    p.shared_bytes = (int)cta_shared_bytes(p.L, v.N);
    p.scratch_off = p.shared_bytes;
    p.per_warp = (int)warp_scratch_bytes(CH, PB);
    const size_t obs_scratch = (size_t)p.per_warp * FW_WARPS, step_scratch = align16(scratch_bytes());
    p.smem = (size_t)p.shared_bytes + (obs_scratch > step_scratch ? obs_scratch : step_scratch);
    p.ok = p.smem <= 200 * 1024;
    return p;
}

}  // namespace

// Shapes served by the CTA-per-world fused kernel: anything the joint step supports (N <= 128) whose staging fits.
bool step_observe_wide_fusable(const EnvView &v) {
    if (v.N > NMAX) return false;
    return make_plan(v, 0, 8).ok;
}

cudaError_t launch_step_observe_wide(const EnvView &v, const int8_t *actions, const MapfStepOut &out, float *obs, float *vec,
                                     int *work_counter, cudaStream_t stream, int fmt) {
    // Default: 4-warp CTAs when six of them fit an SM (measured on 80x80x128, ms per step for FOV 9 / 15 / 21 / 31:
    // two launches 0.861 / 0.971 / 0.950 / 1.032; 8 warps x 3: 1.033 / 1.018 / 0.887 / 1.027; 4 warps x 6: 0.701 / 0.898 /
    // 0.870 / 1.077 — at FOV 31 the per-warp observation scratch leaves three 4-warp CTAs, too few warps for the stores).
    int variant = (v.dbg_flags >> 24) & 7;                  // experiments: 1 = 8w x 3, 2 = 4w x 6, 3 = 4w x 8, 4 = 2w x 16
    if (variant == 0) {
        const WidePlan p4 = make_plan(v, fmt, 4);
        // ... and eight of them (compiled for 64 registers) when eight fit: mid-size worlds (33..100 agents) have a short
        // store phase per world, so they need even more worlds in flight (40x40x64: 0.771 vs 0.806 ms; 80x80x64: 0.384 vs 0.406)
        variant = !(p4.ok && p4.smem <= 40 * 1024) ? 1 : (p4.smem <= 28 * 1024 ? 3 : 2);
        // ... and up to 64 agents, 2-warp CTAs x 16: 33..64-agent worlds have the shortest store phase of all (64-124 KB) against
        // the same ~20 us step phase (40x40x33: 0.927 vs 1.139 ms; 40x40x48: 0.574 vs 0.680; 24x24x40: 0.609 vs 0.750)
        if (v.N <= 64) {
            const WidePlan p2 = make_plan(v, fmt, 2);
            if (p2.ok && p2.smem <= 24 * 1024) variant = 4;
        }
    }
    const int warps = variant == 1 ? 8 : (variant == 4 ? 2 : 4);
    WidePlan p = make_plan(v, fmt, warps);
    if (!p.ok && warps != 8) { variant = 1; p = make_plan(v, fmt, 8); }
    if (!p.ok) return cudaErrorNotSupported;
    return dispatch_obs(fmt, v.C, v.F, obs_vec4(fmt, v.N, p.L.PB, p.L.CH, obs), [&](auto t) {
        using T = decltype(t);
        auto launch = [&](auto kern, int cta_warps) {
            return launch_persistent(kern, cta_warps * 32, p.smem, v.W, INT_MAX, stream, v, actions, out, obs, vec, p.L,
                                     p.shared_bytes, p.scratch_off, p.per_warp, work_counter);
        };
        if (variant == 1) return launch(step_observe_wide_kernel<T::C_T, T::F_T, T::VEC4, T::BITS, 8, 3>, 8);
        if (variant == 2) return launch(step_observe_wide_kernel<T::C_T, T::F_T, T::VEC4, T::BITS, 4, 6>, 4);
        if (variant == 4) return launch(step_observe_wide_kernel<T::C_T, T::F_T, T::VEC4, T::BITS, 2, 16>, 2);
        return launch(step_observe_wide_kernel<T::C_T, T::F_T, T::VEC4, T::BITS, 4, 8>, 4);
    });
}

}  // namespace mapf
