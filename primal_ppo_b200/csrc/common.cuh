// common.cuh — shared device-side definitions of the B200 MAPF hot path (sm_100a).
//
// HBM layout (all env-owned buffers are SoA over worlds, allocated once in mapf_create):
//   obst_pack u32 [W, PW]      the obstacle map as a tightly packed bit matrix, bit r*Wd + c (1 = blocked, incl. cells
//                              outside a world's dims); PW words, a multiple of 4.  208 B per 40x40 world instead of
//                              1600 B.  Kernels expand it in shared memory into rows padded by P cells on every side
//                              (HP = H + 2P rows of RW words, row bit c + P is cell c): the expansion is ALU work, which
//                              is free next to the observation store, and every byte NOT read from HBM while 4 GB of
//                              stores drain is worth ~50 bytes of write bandwidth (DESIGN.md 4.8).
//   pos, goal i16 [W,N,2]      agent cell and current goal (row, col)
//   rep       i8  [W,N]        Agent.invalidActions[2]: the one repetition action, -1 when empty (mapf_gym.py:158-161)
//   qcur      i32 [W,N]        goals already handed out from goal_queue (Sequence.curIdx - 1, util.py:33-39)
//   htick     i32 [W]          human tick into htrace;  hcur i16 [W,4] = htrace[w, htick[w]] (saves a dependent load)
//   tape_cur  i32 [W], nstep i32 [W], err u32 [W], counters i64 [W,6]
// Everything else of the reference's Agent objects (invalid lists, restricted dict, good list) is a pure function of
// this state and is recomputed in registers at the start of every step (SURVEY.md Appendix A.1).
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

#include "../../include/mapf_b200.h"

namespace mapf {

constexpr int NA = 5;                 // EnvParameters.N_ACTIONS (alg_parameters.py:31)
constexpr int WARPS_PER_BLOCK = 8;    // one warp per world, 8 worlds per 256-thread CTA
constexpr unsigned FULL = 0xffffffffu;

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// status codes of getActionStatus (mapf_gym.py:440-444)
constexpr int ST_STATIC = -1, ST_HUMAN = -2, ST_AGENT = -3, ST_REPEAT = -4, ST_OK = 1;

// A lane group: G consecutive lanes of a warp that own one world (lane within the group = agent).  G = 32 is the whole warp
// (one world per warp); G = 8 / 16 pack four / two small worlds into a warp (BASELINE configs[1]: 8 agents per world).  All
// warp-level primitives take the group's lane mask, so the groups of a warp may diverge from one another freely.
template <int G>
struct Grp {
    int gl;          // lane within the group (= agent index)
    int base;        // first lane of the group
    unsigned mask;   // lanes of the group
    __device__ __forceinline__ explicit Grp(int lane)
        : gl(G == 32 ? lane : lane % G), base(G == 32 ? 0 : lane / G * G),
          mask(G == 32 ? FULL : (((1u << (G & 31)) - 1u) << (lane / G * G))) {}
    __device__ __forceinline__ unsigned ballot(bool p) const {                   // bit i = lane i OF THE GROUP
        const unsigned b = __ballot_sync(mask, p);
        return G == 32 ? b : ((b >> base) & ((1u << (G & 31)) - 1u));
    }
    __device__ __forceinline__ bool any(bool p) const { return __any_sync(mask, p) != 0; }
    __device__ __forceinline__ uint32_t shfl(uint32_t x, int k) const { return __shfl_sync(mask, x, base + k); }
    __device__ __forceinline__ int shfl(int x, int k) const { return __shfl_sync(mask, x, base + k); }
    __device__ __forceinline__ uint32_t reduce_or(uint32_t x) const { return __reduce_or_sync(mask, x); }
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
};

struct EnvView {
    int W, H, Wd, N, F, C, use_da, use_hp, Q, L, TL, hp5_per_tick;
    int P;        // padding of the shared-memory bit rows / the agent-id grid = max(2, F/2)
    int PW;       // u32 words of one world's packed obstacle bit matrix (multiple of 4)
    int HP;       // H + 2P
    int RW;       // u32 words per padded bit row (+1 spare word so a funnel read of word k+1 is always in range)
    int GS;       // byte stride of one row of the shared-memory agent-id grid (multiple of 16)
    int dbg_flags; // experiment switches (MAPF_DBG_FLAGS), 0 in production
    int world_offset; // global index of world 0 (sharded jobs): Philox counter = world_offset + w
    int goal_sampling; // 1: draw the next goal on device at arrival (MapfGym.getNextGoal) instead of popping goal_queue
    unsigned long long seed;
    // borrowed scenario
    const uint8_t *obst;
    const int16_t *starts, *goal_queue, *htrace, *hp5, *dims;
    const int32_t *hlen, *tape_len;
    const int8_t *tape;
    // owned state
    uint32_t *obst_pack;
    int16_t *pos, *goal;
    int8_t *rep;
    int32_t *qcur, *htick, *tape_cur, *nstep;
    int16_t *hcur;      // [W,4] the human's (pos, next) of the current tick = htrace[w, htick[w]] (kept by reset/step)
    int16_t *hnx;       // [W,4] the entry of the following tick (wrapped), so that a step has no dependent loads
    uint32_t *err;
    long long *counters;
    int *order;         // [1] walk direction of the next world-claiming launch (see world_of)
};

__device__ __forceinline__ int dr_of(int a) { return (a == 2) - (a == 4); }   // mapf_gym.py:97
__device__ __forceinline__ int dc_of(int a) { return (a == 1) - (a == 3); }
__device__ __forceinline__ int opp_of(int a) { return a == 0 ? 0 : ((a + 1) & 3) + 1; }  // {0:0,1:3,2:4,3:1,4:2} (:100)

// F <= 31 bits of a padded bit row starting at bit `off` (row has RW words, the last one spare).
__device__ __forceinline__ uint32_t row_window(const uint32_t *row, int off, int nbits) {
    const int k = off >> 5;
    const uint32_t v = __funnelshift_r(row[k], row[k + 1], off & 31);
    return v & ((1u << nbits) - 1u);
}
__device__ __forceinline__ uint32_t row_bit(const uint32_t *row, int off) { return (row[off >> 5] >> (off & 31)) & 1u; }

// L2 residency rule.  The env state (cells, goals, obstacle bit rows, human tick: ~55 MB for 65 536 worlds) is re-read
// every step while 4 GB of observations stream through the same L2.  DRAM reads interleaved with the write stream cost
// far more than their bytes (read/write bus turnarounds: measured -13 % write bandwidth for 1.6 % read bytes), so:
//   - env state that the next step reads is loaded AND stored with the evict_last policy (ld_keep* / st_keep*):
//     pos, goal, rep, obst_pack, htick, hcur, hnx, nstep, hlen, counters and the htrace lookahead entry;
//   - everything a step only produces is stored evict-first (st.global.cs, st_stream*): the observations, vec, the
//     MapfStepOut fields (incl. the trainValid rows and the packed host slab), so that it does not compete with the state.
// Rare-path accesses (err, qcur / goal_queue on arrival, tape, dims) stay plain.
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint32_t ld_keep(const void *p, uint64_t pol) {
    uint32_t v;
    asm volatile("ld.global.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int ld_keep_s8(const void *p, uint64_t pol) {
    int v;
    asm volatile("ld.global.L2::cache_hint.s8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int2 ld_keep_v2(const void *p, uint64_t pol) {
    int2 v;
    asm volatile("ld.global.L2::cache_hint.v2.b32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_keep(void *p, uint32_t v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.b32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_s8(void *p, int v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.b8 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_v2(void *p, int2 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v2.b32 [%0], {%1, %2}, %3;" ::"l"(p), "r"(v.x), "r"(v.y), "l"(pol) : "memory");
}
// *p += x for state only this thread touches (the per-world counters)
__device__ __forceinline__ void add_keep_s64(long long *p, long long x, uint64_t pol) {
    long long v;
    asm volatile("ld.global.L2::cache_hint.b64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    asm volatile("st.global.L2::cache_hint.b64 [%0], %1, %2;" ::"l"(p), "l"(v + x), "l"(pol) : "memory");
}
__device__ __forceinline__ void add_keep_s32(int32_t *p, int x, uint64_t pol) { st_keep(p, ld_keep(p, pol) + x, pol); }

// ---- packed obstacle bit matrix -> padded bit rows ---------------------------------------------------------------
// bits [off, off + n), n <= 32, of a packed bit array of `nwords` words; KEEP: `p` is the env's obst_pack in global
// memory, read with the evict_last policy `pol` (residency rule above), else shared memory
template <bool KEEP>
__device__ __forceinline__ uint32_t pack_extract(const uint32_t *p, int off, int n, int nwords, uint64_t pol) {
    const int k = off >> 5;
    const uint32_t lo = KEEP ? ld_keep(p + k, pol) : p[k];
    const uint32_t hi = (k + 1 < nwords) ? (KEEP ? ld_keep(p + k + 1, pol) : p[k + 1]) : 0u;
    const uint32_t x = __funnelshift_r(lo, hi, off & 31);
    return n >= 32 ? x : (x & ((1u << n) - 1u));
}
// word q of padded row pr: 1 = obstacle or out of bounds
template <bool KEEP>
__device__ __forceinline__ uint32_t padded_row_word(const uint32_t *packed, int H, int Wd, int P, int PW, int pr, int q,
                                                    uint64_t pol) {
    const int r = pr - P;
    if (r < 0 || r >= H) return 0xffffffffu;
    const int c0 = 32 * q - P;                                   // column held by bit 0 of this word
    const int lo = c0 > 0 ? c0 : 0, hi = c0 + 32 < Wd ? c0 + 32 : Wd;
    if (hi <= lo) return 0xffffffffu;
    const int n = hi - lo, sh = lo - c0;
    const uint32_t bits = pack_extract<KEEP>(packed, r * Wd + lo, n, PW, pol);
    const uint32_t mask = (n >= 32 ? 0xffffffffu : ((1u << n) - 1u)) << sh;
    return (bits << sh) | ~mask;
}
// all `nthreads` threads of a warp / CTA expand one world (packed lives in shared memory, or with KEEP in global memory)
template <bool KEEP = false>
__device__ __forceinline__ void expand_obstacle_rows(uint32_t *obits, const uint32_t *packed, const EnvView &v, int tid, int nthreads,
                                                     uint64_t pol = 0) {
    const int nob = v.HP * v.RW;
    for (int k = tid; k < nob; k += nthreads) {
        const int pr = k / v.RW;
        obits[k] = padded_row_word<KEEP>(packed, v.H, v.Wd, v.P, v.PW, pr, k - pr * v.RW, pol);
    }
}

// Philox4x32-10, counter = (world, step, draw, tag), key = seed: the stand-in for Python's `random.choice`
// (mapf_gym.py:588) when the caller supplies no tape.  Bit-identical to the oracle's philox_draw.
__device__ __forceinline__ uint32_t philox_draw(unsigned long long seed, uint32_t world, uint32_t step, uint32_t draw) {
    uint32_t c0 = world, c1 = step, c2 = draw, c3 = 0x4D415046u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

// All four words of the same generator with a caller-chosen tag in counter word 3: the free-cell draws of on-device
// goal sampling (tag "GOAL") use words 0 and 1 for (row, col).  Bit-identical to the oracle's philox4.
constexpr uint32_t PHILOX_TAG_GOAL = 0x474F414Cu;
__device__ __forceinline__ void philox4(unsigned long long seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                        uint32_t &o0, uint32_t &o1) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1;
}
// candidate cell of free-cell draw `d` (util.getFreeCell, util.py:72-74: two independent uniform integers), packed like pos
__device__ __forceinline__ uint32_t goal_candidate(unsigned long long seed, uint32_t world, uint32_t step, uint32_t d,
                                                   int rows, int cols) {
    uint32_t x0, x1;
    philox4(seed, world, step, d, PHILOX_TAG_GOAL, x0, x1);
    const uint32_t r = __umulhi(x0, (uint32_t)rows), c = __umulhi(x1, (uint32_t)cols);
    return r | (c << 16);
}
constexpr int GOAL_DRAW_CAP = 4096;   // draws per arrival before MAPF_ERR_NO_FREE_CELL (the reference would spin for ever)

// Bulk L2 prefetch of a contiguous range (TMA unit, no registers, no completion to wait for).
__device__ __forceinline__ void prefetch_l2_bulk(const void *p, size_t bytes, uint64_t pol) {
    bytes &= ~(size_t)15;
    if (bytes) asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(p), "r"((uint32_t)bytes), "l"(pol) : "memory");
}

// streaming stores: step outputs and observations are written once and consumed by another kernel much later
__device__ __forceinline__ void st_stream_v4(float *p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_stream(void *p, uint32_t v) {
    asm volatile("st.global.cs.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream(float *p, float v) { st_stream(static_cast<void *>(p), __float_as_uint(v)); }
__device__ __forceinline__ void st_stream_u16(void *p, uint32_t v) {
    asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void st_stream_u8(void *p, uint32_t v) {
    asm volatile("st.global.cs.b8 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Dynamic work distribution for the persistent kernels: counter[0] = next unit, counter[1] = warps that are done.
// The last warp to finish re-arms the counter, so no memset node is needed between launches.
__device__ __forceinline__ int claim_work(int *counter, int n, int lane) {
    int t = 0;
    if (lane == 0) t = atomicAdd(counter, n);
    return __shfl_sync(FULL, t, 0);
}
// `order`: the env's walk-direction word (world-claiming kernels), flipped by the last warp; every other warp has read it
// before its first claim, so the flip takes effect at the next launch.
__device__ __forceinline__ void finish_work(int *counter, int total_warps, int lane, int *order = nullptr) {
    if (lane == 0) {
        const int d = atomicAdd(counter + 1, 1);
        if (d == total_warps - 1) {
            counter[0] = 0; counter[1] = 0;
            if (order) *order ^= 1;
        }
    }
}

// World order of the world-claiming persistent kernels (step, observe, step_observe, observe_wide, step_observe_wide):
// serpentine.  Claims stay in claim space 0, 1, ...; a launch maps claim c to world c or W-1-c, and every launch reverses
// the direction of the one before.  Worlds are independent, so no result depends on the order, but the state a launch
// touched last is L2-resident and is what the next launch reads first (an ascending walk every time starts from the world
// touched longest ago, with ~4 GB of observation stores since).  The direction is a device word, so a captured or
// replayed launch sequence alternates too.  A claim c >= W stays c (no world).
constexpr int DBG_ASCENDING = 1 << 12;     // MAPF_DBG_FLAGS bit 12: ascending order every launch (A/B runs)
__device__ __forceinline__ int walk_dir(const EnvView &v) { return (v.dbg_flags & DBG_ASCENDING) ? 0 : *v.order; }
__device__ __forceinline__ int world_of(const EnvView &v, int c, int dir) { return (dir && c < v.W) ? v.W - 1 - c : c; }

// Launch of a persistent kernel: as many CTAs as are resident at once on the current device (at most max_per_sm per SM)
// and no more than need_blocks.  A failed runtime call is returned and nothing is launched.
template <typename... P, typename... A>
cudaError_t launch_persistent(void (*kern)(P...), int threads, size_t smem, long long need_blocks, int max_per_sm,
                              cudaStream_t stream, const A &...args) {
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (e != cudaSuccess) return e;
    per_sm = per_sm < 1 ? 1 : (per_sm > max_per_sm ? max_per_sm : per_sm);
    const long long cap = (long long)sms * per_sm;
    kern<<<(int)(need_blocks < cap ? need_blocks : cap), threads, smem, stream>>>(args...);
    return cudaGetLastError();
}

// Batched state prefetch.  A world's state is ~0.9 KB spread over a dozen SoA arrays; loaded world by world it reaches
// DRAM as ~430 000 isolated 128-byte reads per step, interleaved with 4 GB of observation stores — and every isolated
// read costs the HBM channel a write->read->write bus turnaround (measured: 1.6 % read bytes cost 13 % of the write
// bandwidth).  Claims are handed out in increasing order, so the warp that claims c1 with c1 % PFB == 0 asks the TMA unit
// to pull the state of the worlds of claims [c1 + ahead, c1 + ahead + PFB) (in the launch's direction `dir`, world_of)
// into L2 as a few large contiguous reads; the per-world register loads that follow a few microseconds later then hit L2.
constexpr int PFB = 256;
__device__ __forceinline__ int prefetch_batch(const EnvView &v) { return PFB << ((v.dbg_flags >> 8) & 7); }
__device__ __forceinline__ void prefetch_world_batch(const EnvView &v, const int8_t *actions, int c0, int dir, uint64_t pol,
                                                     int batch = 0) {
    if (c0 >= v.W) return;
    const int nb = min(batch > 0 ? batch : prefetch_batch(v), v.W - c0);
    const int w0 = dir ? v.W - c0 - nb : c0;             // lowest world of the batch
    const size_t n = (size_t)nb, wn = (size_t)w0 * v.N, nn = n * v.N;
    prefetch_l2_bulk(v.obst_pack + (size_t)w0 * v.PW, n * v.PW * 4, pol);
    prefetch_l2_bulk(reinterpret_cast<const uint32_t *>(v.pos) + wn, nn * 4, pol);
    prefetch_l2_bulk(reinterpret_cast<const uint32_t *>(v.goal) + wn, nn * 4, pol);
    prefetch_l2_bulk(reinterpret_cast<const int2 *>(v.hcur) + w0, n * 8, pol);
    if (actions) {
        prefetch_l2_bulk(v.rep + wn, nn, pol);
        if ((reinterpret_cast<uintptr_t>(actions + wn) & 15) == 0) prefetch_l2_bulk(actions + wn, nn, pol);
        prefetch_l2_bulk(reinterpret_cast<const int2 *>(v.hnx) + w0, n * 8, pol);
        prefetch_l2_bulk(v.htick + w0, n * 4, pol);
        prefetch_l2_bulk(v.hlen + w0, n * 4, pol);
        prefetch_l2_bulk(v.nstep + w0, n * 4, pol);
        prefetch_l2_bulk(v.counters + (size_t)w0 * 6, n * 48, pol);
    }
}
// distance (in worlds) between the world being loaded and the batch being prefetched; MAPF_DBG_FLAGS bits 4..7
// override it in units of PFB (0xF0 mask; value 15 = prefetch off)
__device__ __forceinline__ int prefetch_ahead(const EnvView &v) {
    const int k = (v.dbg_flags >> 4) & 15;
    return k == 15 ? -1 : (k ? k : 4) * prefetch_batch(v);
}

// Output format of the observation kernels: the reference's f32 layout, the same 0/1 values as bf16, or one bit per cell
// (u32 [W, N, AW], AW = MAPF_OBS_BITS_WORDS(C, F): each agent's C*F*F bits LSB first in its own word-aligned record).
enum ObsFormat { OBS_F32 = 0, OBS_BF16 = 1, OBS_BITS = 2 };

// launchers implemented in the .cu files
cudaError_t launch_reset(const EnvView &v, cudaStream_t s);
cudaError_t launch_step(const EnvView &v, const int8_t *actions, const int8_t *status_in, const MapfStepOut &out,
                        int mode, int *work_counter, cudaStream_t s);
cudaError_t launch_step_wide(const EnvView &v, const int8_t *actions, const int8_t *status_in, const MapfStepOut &out,
                             int mode, cudaStream_t s);
cudaError_t launch_observe(const EnvView &v, float *obs, float *vec, int *work_counter, cudaStream_t s, int fmt = OBS_F32);
bool step_observe_fusable(const EnvView &v);
cudaError_t launch_step_observe(const EnvView &v, const int8_t *actions, const MapfStepOut &out, float *obs, float *vec,
                                int *work_counter, cudaStream_t s, int fmt = OBS_F32);
bool step_observe_wide_fusable(const EnvView &v);
cudaError_t launch_step_observe_wide(const EnvView &v, const int8_t *actions, const MapfStepOut &out, float *obs, float *vec,
                                     int *work_counter, cudaStream_t s, int fmt = OBS_F32);
cudaError_t launch_observe_wide(const EnvView &v, float *obs, float *vec, int *work_counter, cudaStream_t s, int fmt = OBS_F32);
cudaError_t launch_bfs(const EnvView &v, const int32_t *agent_list, long long n, const int32_t *n_dev, int16_t *out,
                       int scatter, int *work_counter, cudaStream_t s);
cudaError_t launch_arrivals(const EnvView &v, const uint8_t *goals, int32_t *list, int32_t *n_dev, cudaStream_t s);
cudaError_t launch_gae(const float *r, const float *v, const float *last_v, const uint8_t *nonterminal, float g, float gl,
                       int T, long long cols, float *ret, float *adv, cudaStream_t s);

cudaError_t launch_gae2(const float *r, const float *v, const float *last_v, const float *cr, const float *cv,
                        const float *last_cv, const uint8_t *nonterminal, float g, float gl, int T, long long cols, float *ret,
                        float *cret, float *adv, float *cadv, cudaStream_t s);

cudaError_t launch_adv_moments(const float *ret, const float *cret, const float *old_v, const float *old_cv, long long n,
                               double *partials, cudaStream_t s);
cudaError_t launch_ppo_loss(const MapfPpoLossConfig &cfg, long long n, const float *policy, const float *value,
                            const float *cost_value, const float *sig, const float *ret, const float *cret, const float *old_v,
                            const float *old_cv, const int8_t *actions, const float *old_ps, const float *tv, float *g_policy,
                            float *g_value, float *g_cost_value, float *g_sig, double *partials, cudaStream_t s);

cudaError_t launch_sample_actions(const float *ps, long long rows, unsigned long long seed, uint32_t draw, int8_t *actions,
                                  float *chosen_p, cudaStream_t s);

cudaError_t launch_unpack_obs(const uint32_t *bits, long long src_rows, int N, int C, int F, const int64_t *rows,
                              long long n_rows, int out_bf16, void *out, cudaStream_t s);

cudaError_t launch_checksum_rows(const uint32_t *data, long long rows, long long words, unsigned long long *out, cudaStream_t s);

cudaError_t launch_scenario_gen(const MapfGenConfig &c, uint8_t *obst, int16_t *dims, int16_t *starts, int16_t *goal_queue,
                                int16_t *htrace, int32_t *hlen, int16_t *hp5, uint32_t *gen_err, cudaStream_t s);
cudaError_t launch_astar4_paths(const uint8_t *obst, long long n, int H, int Wd, const int16_t *start_goal, int max_len,
                                int16_t *paths, int32_t *lens, cudaStream_t s);

constexpr int MODE_EVALUATE = 0, MODE_JOINT = 1, MODE_FUSED = 2;

}  // namespace mapf
