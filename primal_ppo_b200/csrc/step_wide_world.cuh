// step_wide_world.cuh — joint-step resolution of ONE world with up to 128 agents by a GROUP of threads: a warp
// (step_wide_kernel, step_wide.cu) or a whole CTA (step_observe_wide_kernel, step_observe_wide.cu, where the eight warps
// that afterwards write the world's observations also share the step).
//
// Same semantics and reference lines as step_world.cuh (mapf_gym.py:339-637, runner.py:64-91).  Mapping: thread `tid` of
// `nthreads` loops over agents tid, tid + nthreads, ...; all per-agent masks live in shared memory so that the
// order-dependent parts (the sequential status replay, the fixActions queue) can be walked by thread 0 and the goal draws
// by the first warp.  Phases are separated by a group barrier (__syncwarp / __syncthreads).
#pragma once
#include "common.cuh"
#include "step_common.cuh"

namespace mapf {
namespace sww {

constexpr int NMAX = 128;

enum { K_SHADOW = 0, K_C1, K_C2, K_C3, K_ARR, K_VIOL, K_FIX, K_TRIG, K_ERR, K_COUNT = 12 };

struct WideSmem {
    uint32_t *obits;     // [HP*RW] padded obstacle bit rows (staged by the caller)
    uint8_t *grid;       // [HP*GS] agent id + 1, 0 = none (clean on entry and on exit)
    float *tv;           // [N*5]
    uint32_t *pos;       // [N] packed cell
    uint32_t *goal;      // [N]
    uint32_t *mm;        // [N] conflict partners of the chosen action, one id per byte
    uint32_t *npos;      // [N] packed cell after the move
    int *cnt;            // [K_COUNT] per-world counters / flags
    uint8_t *inv0, *inv1, *restr, *good, *confl;   // [N] 5-bit masks
    int8_t *act, *rep, *cls, *st, *commit;         // [N]
    uint8_t *queue;      // [256] ring of agent ids
};

// scratch of the step phase only (everything but obits / grid)
__host__ __device__ inline size_t scratch_bytes() { return NMAX * 5 * 4 + NMAX * 4 * 4 + K_COUNT * 4 + NMAX * 10 + 256; }

__device__ inline void carve_scratch(WideSmem &s, unsigned char *b) {
    s.tv = reinterpret_cast<float *>(b); b += NMAX * 5 * 4;
    s.pos = reinterpret_cast<uint32_t *>(b); b += NMAX * 4;
    s.goal = reinterpret_cast<uint32_t *>(b); b += NMAX * 4;
    s.mm = reinterpret_cast<uint32_t *>(b); b += NMAX * 4;
    s.npos = reinterpret_cast<uint32_t *>(b); b += NMAX * 4;
    s.cnt = reinterpret_cast<int *>(b); b += K_COUNT * 4;
    s.inv0 = b; b += NMAX; s.inv1 = b; b += NMAX; s.restr = b; b += NMAX; s.good = b; b += NMAX; s.confl = b; b += NMAX;
    s.act = reinterpret_cast<int8_t *>(b); b += NMAX; s.rep = reinterpret_cast<int8_t *>(b); b += NMAX;
    s.cls = reinterpret_cast<int8_t *>(b); b += NMAX; s.st = reinterpret_cast<int8_t *>(b); b += NMAX;
    s.commit = reinterpret_cast<int8_t *>(b); b += NMAX;
    s.queue = b;
}

template <bool CTA>
__device__ __forceinline__ void group_sync() {
    if (CTA) __syncthreads(); else __syncwarp();
}

// On entry: s.obits holds the world's padded obstacle rows, s.grid is all zero.  On exit: s.grid is all zero again,
// s.npos / s.goal hold the post-step cells and goals, the env state and `out` are written.  Returns false for
// MODE_EVALUATE (nothing moved).  (hnr, hnc) receive human.getNextPos() AFTER the tick (what the observation needs).
template <int MODE, bool CTA>
__device__ __forceinline__ void step_wide_world(const EnvView &v, const int8_t *__restrict__ actions,
                                                const int8_t *__restrict__ status_in, const MapfStepOut &out,
                                                const WideSmem &s, const int w, const int tid, const int nthreads,
                                                int &hnr, int &hnc) {
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW;
    const size_t base = (size_t)w * N;
    uint32_t errbits = 0;
    const uint64_t pol = policy_evict_last();         // residency rule (common.cuh)

    // ---- stage the agents ---------------------------------------------------------------------------------------------
    const int tick = (int)ld_keep(v.htick + w, pol);
    const int hlen = (int)ld_keep(v.hlen + w, pol);
    const int2 ht = ld_keep_v2(reinterpret_cast<const int2 *>(v.hcur) + w, pol);
    const int2 ht2 = ld_keep_v2(reinterpret_cast<const int2 *>(v.hnx) + w, pol);
    const int hr = (int16_t)(ht.x & 0xffff), hc = (int16_t)((uint32_t)ht.x >> 16);
    const int nr = (int16_t)(ht.y & 0xffff), nc = (int16_t)((uint32_t)ht.y >> 16);
    hnr = (int16_t)(ht2.y & 0xffff); hnc = (int16_t)((uint32_t)ht2.y >> 16);
    if (tid < K_COUNT) s.cnt[tid] = 0;
    for (int i = tid; i < N; i += nthreads) {
        const uint32_t pw = ld_keep(reinterpret_cast<const uint32_t *>(v.pos) + base + i, pol);
        s.pos[i] = pw;
        s.goal[i] = ld_keep(reinterpret_cast<const uint32_t *>(v.goal) + base + i, pol);
        int a = actions[base + i];
        if (a < 0 || a >= NA) { errbits |= MAPF_ERR_BAD_ACTION; a = 0; }
        s.act[i] = (int8_t)a;
        s.rep[i] = (int8_t)ld_keep_s8(v.rep + base + i, pol);
        const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
        s.grid[(r + P) * GS + c + P] = (uint8_t)(i + 1);
    }
    group_sync<CTA>();

    // ---- masks, class, fast status (getInvalidActions :339-360, getRestrictedActions :363-402, good :404-430) -----------
    for (int i = tid; i < N; i += nthreads) {
        const uint32_t pw = s.pos[i];
        const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
        const int a = s.act[i], rep = s.rep[i];
        uint32_t inv0 = 0, inv1 = 0;
#pragma unroll
        for (int k = 1; k < NA; ++k) {
            const int tr = r + ((k == 2) - (k == 4)), tc = c + ((k == 1) - (k == 3));
            if (row_bit(s.obits + (tr + P) * RW, tc + P)) inv0 |= 1u << k;
        }
#pragma unroll
        for (int k = 0; k < NA; ++k) {
            const int tr = r + ((k == 2) - (k == 4)), tc = c + ((k == 1) - (k == 3));
            const bool hv = (tr == nr && tc == nc) || (r == nr && c == nc && tr == hr && tc == hc);
            if (hv && !(inv0 >> k & 1)) inv1 |= 1u << k;
        }
        uint32_t restr, confl, mm;
        scan_diamond<true>(s.grid, GS, r + P, c + P, i + 1, s.act, a, restr, confl, mm);
        const uint32_t repbit = rep >= 0 ? (1u << rep) : 0u;
        const uint32_t good = ~(inv0 | inv1 | restr | repbit) & 31u;
        const uint32_t abit = 1u << a;
        const int cls = (inv0 & abit) ? C_INV0 : (inv1 & abit) ? C_INV1 : (good & abit) ? C_GOOD : C_E;
        const int st = cls == C_INV0 ? ST_STATIC : cls == C_INV1 ? ST_HUMAN : cls == C_GOOD ? ST_OK
                       : (confl & abit) ? ST_AGENT : (a == rep ? ST_REPEAT : ST_OK);
        s.inv0[i] = (uint8_t)inv0; s.inv1[i] = (uint8_t)inv1; s.restr[i] = (uint8_t)restr; s.good[i] = (uint8_t)good;
        s.confl[i] = (uint8_t)confl; s.mm[i] = mm; s.cls[i] = (int8_t)cls;
        s.st[i] = (int8_t)(MODE == MODE_JOINT ? status_in[base + i] : st);
    }
    group_sync<CTA>();
    if (MODE != MODE_JOINT) {                             // getActionStatus :434-480
        bool trig = false;
        for (int i = tid; i < N; i += nthreads) {
            if (s.cls[i] != C_E) continue;
            const uint32_t mm = s.mm[i];
#pragma unroll
            for (int k = 0; k < 4; ++k) { const int j = (mm >> (8 * k)) & 0xff; if (j != 0xff && s.cls[j] == C_INV1) trig = true; }
        }
        if (trig) s.cnt[K_TRIG] = 1;
        group_sync<CTA>();
        if (s.cnt[K_TRIG]) {                              // rare: replay the sequential loop (SURVEY A.5)
            if (tid == 0) {
                for (int i = 0; i < N; ++i) s.st[i] = 0;
                for (int i = 0; i < N; ++i) {
                    if (s.st[i] != 0) continue;
                    const int ci = s.cls[i];
                    if (ci == C_INV0) s.st[i] = ST_STATIC;
                    else if (ci == C_INV1) s.st[i] = ST_HUMAN;
                    else if (ci == C_GOOD) s.st[i] = ST_OK;
                    else {
                        const uint32_t mm = s.mm[i];
                        for (int k = 0; k < 4; ++k) { const int j = (mm >> (8 * k)) & 0xff; if (j != 0xff) { s.st[i] = ST_AGENT; s.st[j] = ST_AGENT; } }
                        if (s.st[i] == 0) s.st[i] = (s.act[i] == s.rep[i]) ? ST_REPEAT : ST_OK;
                    }
                }
            }
            group_sync<CTA>();
        }
    }

    // ---- reward / cost / trainValid / shadow goals (:483-550) ------------------------------------------------------------
    {
        int n_shadow = 0, n_c1 = 0, n_c2 = 0, n_c3 = 0;
        bool need_fix = false;
        for (int i = tid; i < N; i += nthreads) {
            const int st = s.st[i], a = s.act[i];
            const uint32_t pw = s.pos[i], gw = s.goal[i];
            const int tr = (int16_t)(pw & 0xffff) + dr_of(a), tc = (int16_t)(pw >> 16) + dc_of(a);
            if (st == ST_OK && tr == (int16_t)(gw & 0xffff) && tc == (int16_t)(gw >> 16)) n_shadow++;
            n_c1 += st == ST_STATIC; n_c2 += st == ST_HUMAN; n_c3 += st == ST_AGENT;
            need_fix |= (st == ST_STATIC || st == ST_HUMAN || st == ST_AGENT);
            if (MODE != MODE_JOINT) {
                if (out.status) st_stream_u8(out.status + base + i, (uint32_t)st);
                if (out.cost) {
                    const int d2 = (nr - tr) * (nr - tr) + (nc - tc) * (nc - tc);
                    st_stream(out.cost + base + i, d2 < 25 ? (float)((5.0 - sqrt((double)d2)) / 5.0) : 0.0f);
                }
                if (MODE == MODE_EVALUATE && out.reward) st_stream(out.reward + base + i, st == ST_REPEAT ? -0.35f : st == ST_OK ? -0.3f : -2.0f);
                if (MODE == MODE_EVALUATE && out.good_actions) st_stream_u8(out.good_actions + base + i, s.good[i]);
                if (out.train_valid) {
                    const uint32_t good = s.good[i], restr = s.restr[i], confl = s.confl[i];
#pragma unroll
                    for (int k = 0; k < NA; ++k) {
                        const uint32_t b = 1u << k;
                        s.tv[i * NA + k] = (good & b) ? 1.0f : (restr & b) ? ((confl & b) ? 0.0f : 1.0f) : 0.0f;
                    }
                }
            }
        }
        if (n_shadow) atomicAdd(&s.cnt[K_SHADOW], n_shadow);
        if (n_c1) atomicAdd(&s.cnt[K_C1], n_c1);
        if (n_c2) atomicAdd(&s.cnt[K_C2], n_c2);
        if (n_c3) atomicAdd(&s.cnt[K_C3], n_c3);
        if (need_fix) s.cnt[K_FIX] = 1;
    }
    group_sync<CTA>();
    if (MODE != MODE_JOINT) {
        if (tid == 0 && out.shadow_goals) st_stream(out.shadow_goals + w, (uint32_t)s.cnt[K_SHADOW]);
        if (out.train_valid) {
            float *dst = out.train_valid + base * NA;
            for (int k = tid; k < N * NA; k += nthreads) st_stream(dst + k, s.tv[k]);
        }
        if (MODE == MODE_EVALUATE) {
            if (errbits) atomicOr(reinterpret_cast<unsigned int *>(&s.cnt[K_ERR]), errbits);
            group_sync<CTA>();
            if (tid == 0 && s.cnt[K_ERR]) atomicOr(v.err + w, (uint32_t)s.cnt[K_ERR]);
            for (int i = tid; i < N; i += nthreads) {
                const uint32_t pw = s.pos[i];
                s.grid[((int16_t)(pw & 0xffff) + P) * GS + (int16_t)(pw >> 16) + P] = 0;
                s.npos[i] = pw;
            }
            group_sync<CTA>();
            return;
        }
    }

    // ---- fixActions (:552-612) --------------------------------------------------------------------------------------------
    if (s.cnt[K_FIX]) {
        for (int i = tid; i < N; i += nthreads) {
            const int st = s.st[i];
            int commit = (st == ST_OK) ? s.act[i] : -1;
            if (st < 0 && s.good[i]) commit = __ffs(s.good[i]) - 1;
            s.commit[i] = (int8_t)commit;
        }
        group_sync<CTA>();
        if (tid == 0) {
            int head = 0, tail = 0, iters = 0;
            uint32_t draw = 0;
            // problem agents that own a good action committed above; the reference's loop spends one iteration on each of
            // them before any re-queued agent, so they count towards the iteration cap (see step_world.cuh)
            for (int i = 0; i < N; ++i) {
                if (s.st[i] < 0 && !s.good[i]) s.queue[(tail++) & 255] = (uint8_t)i;
                else if (s.st[i] < 0) iters++;
            }
            while (head < tail) {
                if (++iters > FIX_CAP) { errbits |= MAPF_ERR_FIX_ITER_CAP; break; }
                const int k = s.queue[(head++) & 255];
                const uint32_t pw = s.pos[k];
                const int gr = (int16_t)(pw & 0xffff) + P, gc = (int16_t)(pw >> 16) + P;
                const uint32_t good = s.good[k], viable = ~((uint32_t)s.inv0[k] | s.inv1[k]) & 31u, restr = s.restr[k];
                int choice;
                uint32_t r2, c2, ev;
                scan_diamond<true>(s.grid, GS, gr, gc, k + 1, s.commit, -1, r2, c2, ev);
                const uint32_t ok = viable & ~(restr & c2);
                if (good) choice = __ffs(good) - 1;
                else if (ok) choice = __ffs(ok) - 1;
                else if (!viable) { errbits |= MAPF_ERR_NO_VIABLE; choice = 0; }
                else {
                    const int nv = __popc(viable);
                    if (v.TL > 0) {
                        const int8_t *tp = v.tape + (size_t)w * v.TL;
                        int cur = v.tape_cur[w];
                        const int tl = v.tape_len[w];
                        if (cur + 2 > tl) { errbits |= MAPF_ERR_TAPE; choice = __ffs(viable) - 1; cur = tl; }
                        else {
                            choice = tp[cur];
                            const int ne = tp[cur + 1];
                            if (choice < 0 || choice >= NA) { errbits |= MAPF_ERR_TAPE; choice = __ffs(viable) - 1; }
                            scan_diamond<true>(s.grid, GS, gr, gc, k + 1, s.commit, choice, r2, c2, ev);
                            int matched = 0, ncomp = 0;
                            for (int q = 0; q < 4; ++q) ncomp += ((ev >> (8 * q)) & 0xff) != 0xff;
                            for (int q = 0; q < ne && cur + 2 + q < tl; ++q) {
                                const int j = tp[cur + 2 + q];
                                bool in_ev = false;
                                for (int z = 0; z < 4; ++z) in_ev |= (int)((ev >> (8 * z)) & 0xff) == j;
                                if (j >= 0 && j < N && in_ev) { matched++; s.commit[j] = -1; s.queue[(tail++) & 255] = (uint8_t)j; }
                            }
                            if (matched != ncomp || ncomp != ne) errbits |= MAPF_ERR_TAPE;
                            cur += 2 + ne;
                        }
                        v.tape_cur[w] = cur;
                    } else {
                        int pick = (int)(philox_draw(v.seed, (uint32_t)(w + v.world_offset), (uint32_t)v.nstep[w], draw) % (uint32_t)nv);
                        uint32_t vm = viable;
                        while (pick--) vm &= vm - 1;
                        choice = __ffs(vm) - 1;
                        scan_diamond<true>(s.grid, GS, gr, gc, k + 1, s.commit, choice, r2, c2, ev);
                        // ascending eviction order: sort the (<= 4) packed ids
                        int ids[4], n = 0;
                        for (int z = 0; z < 4; ++z) { const int j = (ev >> (8 * z)) & 0xff; if (j != 0xff) ids[n++] = j; }
                        for (int x = 1; x < n; ++x) for (int y = x; y > 0 && ids[y - 1] > ids[y]; --y) { const int t = ids[y]; ids[y] = ids[y - 1]; ids[y - 1] = t; }
                        for (int z = 0; z < n; ++z) { s.commit[ids[z]] = -1; s.queue[(tail++) & 255] = (uint8_t)ids[z]; }
                    }
                    draw++;
                }
                s.commit[k] = (int8_t)choice;
            }
            // livelock cap / no viable action: every agent of the world stays in this step (see step_world.cuh)
            if (errbits & (MAPF_ERR_FIX_ITER_CAP | MAPF_ERR_NO_VIABLE)) for (int i = 0; i < N; ++i) s.commit[i] = 0;
        }
    } else {
        for (int i = tid; i < N; i += nthreads) s.commit[i] = s.act[i];
    }
    group_sync<CTA>();

    // ---- moves, goal arrival, human tick, violations (:620-633) ---------------------------------------------------------
    const int t2 = (tick + 1 >= hlen) ? 0 : tick + 1;
    const int h2r = (int16_t)(ht2.x & 0xffff), h2c = (int16_t)((uint32_t)ht2.x >> 16);
    {
        int n_arr = 0, n_viol = 0;
        for (int i = tid; i < N; i += nthreads) {
            int f = s.commit[i];
            if (f < 0) f = 0;
            const uint32_t pw = s.pos[i], gw = s.goal[i];
            const int nr_ = (int16_t)(pw & 0xffff) + dr_of(f), nc_ = (int16_t)(pw >> 16) + dc_of(f);
            const bool arrived = nr_ == (int16_t)(gw & 0xffff) && nc_ == (int16_t)(gw >> 16);
            const bool viol = (h2r - nr_) * (h2r - nr_) + (h2c - nc_) * (h2c - nc_) <= 24;
            const uint32_t npw = (uint32_t)(uint16_t)nr_ | ((uint32_t)(uint16_t)nc_ << 16);
            st_keep(reinterpret_cast<uint32_t *>(v.pos) + base + i, npw, pol);
            s.npos[i] = npw;
            s.cls[i] = (int8_t)arrived;                 // (the class array is free again: arrival flags for goal sampling)
            s.grid[((int16_t)(pw & 0xffff) + P) * GS + (int16_t)(pw >> 16) + P] = 0;       // leave the id grid clean
            st_keep_s8(v.rep + base + i, opp_of(f), pol);
            if (arrived && !v.goal_sampling) {                                     // Sequence.getNext util.py:33-39
                int k = v.qcur[base + i];
                if (k >= v.Q) k = v.Q - 1; else v.qcur[base + i] = k + 1;
                const uint32_t ngw = reinterpret_cast<const uint32_t *>(v.goal_queue)[(base + i) * v.Q + k];
                st_keep(reinterpret_cast<uint32_t *>(v.goal) + base + i, ngw, pol);
                s.goal[i] = ngw;
            }
            if (out.goals_reached) st_stream_u8(out.goals_reached + base + i, arrived);
            if (out.violated) st_stream_u8(out.violated + base + i, viol);
            if (out.fixed_actions) st_stream_u8(out.fixed_actions + base + i, (uint32_t)f);
            if (MODE == MODE_FUSED && out.reward) {
                const int st = s.st[i];
                const float reward = st == ST_REPEAT ? -0.35f : st == ST_OK ? -0.3f : -2.0f;
                st_stream(out.reward + base + i, arrived ? __fadd_rn(reward, 1.5f) : reward);    // runner.py:89-91
            }
            if (MODE == MODE_FUSED && out.packed) {                              // MAPF_PACKED_* (include/mapf_b200.h)
                const int st = s.st[i], a = s.act[i];
                const int tr = (int16_t)(pw & 0xffff) + dr_of(a), tc = (int16_t)(pw >> 16) + dc_of(a);
                const int d2 = (nr - tr) * (nr - tr) + (nc - tc) * (nc - tc);
                const uint32_t sc = st == ST_STATIC ? 0u : st == ST_HUMAN ? 1u : st == ST_AGENT ? 2u : st == ST_REPEAT ? 3u : 4u;
                st_stream_u16(out.packed + base + i, sc | ((uint32_t)arrived << 3) | ((uint32_t)viol << 4) | ((uint32_t)f << 5) |
                                                     ((uint32_t)min(d2, 25) << 8));
            }
            n_arr += arrived; n_viol += viol;
        }
        if (n_arr) atomicAdd(&s.cnt[K_ARR], n_arr);
        if (n_viol) atomicAdd(&s.cnt[K_VIOL], n_viol);
    }
    group_sync<CTA>();
    if (v.goal_sampling && s.cnt[K_ARR]) {
        // MapfGym.getNextGoal on arrival (mapf_gym.py:626, util.py:67-76); same draws as resolve_world (step_world.cuh):
        // the first warp tests 32 consecutive draws at a time and takes the first free one
        if (tid < 32) {
            const int lane = tid;
            int rows = v.H, cols = v.Wd;
            if (v.dims) { rows = v.dims[2 * w]; cols = v.dims[2 * w + 1]; }
            const uint32_t nstep_w = (uint32_t)v.nstep[w];
            uint32_t draw = 0;
            for (int i = 0; i < N; ++i) {
                if (!s.cls[i]) continue;                                 // warp-uniform (shared memory)
                uint32_t chosen = 0;
                bool found = false;
                for (int batch = 0; batch < GOAL_DRAW_CAP / 32 && !found; ++batch) {
                    const uint32_t cand = goal_candidate(v.seed, (uint32_t)(w + v.world_offset), nstep_w, draw + lane, rows, cols);
                    const int cr = (int)(cand & 0xffff), cc = (int)(cand >> 16);
                    bool free_ = !row_bit(s.obits + (cr + P) * RW, cc + P);
                    for (int j = 0; j < N && free_; ++j)
                        free_ = cand != (j <= i ? s.npos[j] : s.pos[j]) && cand != s.goal[j];
                    const uint32_t b = __ballot_sync(FULL, free_);
                    if (b) { const int k = __ffs(b) - 1; chosen = __shfl_sync(FULL, cand, k); draw += k + 1; found = true; }
                    else draw += 32;
                }
                if (!found) errbits |= MAPF_ERR_NO_FREE_CELL;
                else {
                    __syncwarp();
                    if (lane == 0) { s.goal[i] = chosen; st_keep(reinterpret_cast<uint32_t *>(v.goal) + base + i, chosen, pol); }
                    __syncwarp();
                }
            }
        }
    }
    if (errbits) atomicOr(reinterpret_cast<unsigned int *>(&s.cnt[K_ERR]), errbits);
    group_sync<CTA>();
    if (tid == 0) {
        st_keep(v.htick + w, (uint32_t)t2, pol);
        st_keep_v2(reinterpret_cast<int2 *>(v.hcur) + w, ht2, pol);
        const int t3 = (t2 + 1 >= hlen) ? 0 : t2 + 1;
        st_keep_v2(reinterpret_cast<int2 *>(v.hnx) + w, ld_keep_v2(v.htrace + ((size_t)w * v.L + t3) * 4, pol), pol);
        add_keep_s32(v.nstep + w, 1, pol);
        if (s.cnt[K_ERR]) atomicOr(v.err + w, (uint32_t)s.cnt[K_ERR]);
        long long *cn = v.counters + (size_t)w * 6;                              // util.py:56-65, runner.py:66-99
        add_keep_s64(cn + 0, s.cnt[K_ARR], pol); add_keep_s64(cn + 1, s.cnt[K_SHADOW], pol); add_keep_s64(cn + 2, s.cnt[K_C1], pol);
        add_keep_s64(cn + 3, s.cnt[K_C2], pol); add_keep_s64(cn + 4, s.cnt[K_C3], pol); add_keep_s64(cn + 5, s.cnt[K_VIOL], pol);
    }
}

}  // namespace sww
}  // namespace mapf
