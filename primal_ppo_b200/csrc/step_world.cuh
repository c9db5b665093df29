// step_world.cuh — joint-step resolution of ONE world by one lane group (lane of the group = agent; the whole warp for N <= 32,
// a quarter / half warp for N <= 8 / 16, see Grp in common.cuh): the device code shared by step_kernel (step.cu) and the fused
// step_observe_kernel (step_observe.cu).  See step.cu for the design notes and the reference lines (mapf_gym.py:339-637,
// runner.py:64-91).
#pragma once
#include "common.cuh"
#include "step_common.cuh"

namespace mapf {
namespace sw {

// problemAgents ring of 2 G entries: an agent is queued at most once at a time, so <= G live entries

struct WarpSmem {
    uint32_t *obits;   // [HP*RW]
    uint8_t *grid;     // [HP*GS] agent id + 1, 0 = none
    float *tv;         // [G*5]
    uint32_t *mmask;   // [G] agents in conflict with my chosen action
    int8_t *act;       // [G] sanitised joint action
    int8_t *cls;       // [G]
    int8_t *st;        // [G]
    int8_t *commit;    // [G] agentActionPairs[:,1]
    int8_t *rep;       // [G]
    int8_t *queue;     // [2G] problemAgents (ring buffer)
};

// scratch of the step phase for one group of G lanes (everything but obits / grid)
__host__ __device__ inline size_t step_scratch_bytes(int G) { return align16((size_t)G * 5 * 4 + G * 4 + 5 * G + 2 * G); }

__device__ inline void carve_step_scratch(WarpSmem &s, unsigned char *b, int G) {
    s.tv = reinterpret_cast<float *>(b); b += G * 5 * 4;
    s.mmask = reinterpret_cast<uint32_t *>(b); b += G * 4;
    s.act = reinterpret_cast<int8_t *>(b); b += G;
    s.cls = reinterpret_cast<int8_t *>(b); b += G;
    s.st = reinterpret_cast<int8_t *>(b); b += G;
    s.commit = reinterpret_cast<int8_t *>(b); b += G;
    s.rep = reinterpret_cast<int8_t *>(b); b += G;
    s.queue = reinterpret_cast<int8_t *>(b);
}

__host__ __device__ inline size_t warp_smem_bytes(int HP, int RW, int GS) {
    return align16((size_t)HP * RW * 4) + align16((size_t)HP * GS) + step_scratch_bytes(32);
}

__device__ inline WarpSmem carve(unsigned char *base, int HP, int RW, int GS) {
    WarpSmem s;
    s.obits = reinterpret_cast<uint32_t *>(base); base += align16((size_t)HP * RW * 4);
    s.grid = base; base += align16((size_t)HP * GS);
    carve_step_scratch(s, base, 32);
    return s;
}

constexpr int SOBW = 4;   // packed obstacle words prefetched per lane (PW <= 128: up to 64x64 cells; 40x40 needs 52)

// inputs of one world, prefetched one world ahead of the one being resolved
struct StepRegs {
    uint32_t pw, gw;          // cell, goal of agent `lane`
    int rep, act;             // repetition action, joint action
    int st_in;                // MODE_JOINT: status computed earlier by mapf_evaluate
    uint32_t ob[SOBW];        // packed obstacle words lane, lane+32, ...
    int2 ht, ht2;             // human (pos,next) at the current tick and after this step's tick
    int tick, hlen;
};

// `lane` is the lane within the group that owns world w, G the group width (32 = the whole warp)
template <int MODE, int G = 32>
__device__ __forceinline__ void load_step_world(const EnvView &v, const int8_t *__restrict__ actions,
                                                const int8_t *__restrict__ status_in, int w, int lane, int nob,
                                                uint64_t pol, StepRegs &r) {
    if (w < v.W) {
        const size_t idx = (size_t)w * v.N + (lane < v.N ? lane : 0);
        r.pw = ld_keep(reinterpret_cast<const uint32_t *>(v.pos) + idx, pol);
        r.gw = ld_keep(reinterpret_cast<const uint32_t *>(v.goal) + idx, pol);
        r.rep = ld_keep_s8(v.rep + idx, pol);
        r.act = __ldg(actions + idx);
        r.st_in = (MODE == MODE_JOINT) ? (int)__ldg(status_in + idx) : 0;
        const uint32_t *src = v.obst_pack + (size_t)w * v.PW;
#pragma unroll
        for (int k = 0; k < SOBW; ++k) r.ob[k] = (k * G + lane < nob) ? ld_keep(src + k * G + lane, pol) : 0u;
        r.ht = ld_keep_v2(reinterpret_cast<const int2 *>(v.hcur) + w, pol);
        r.ht2 = ld_keep_v2(reinterpret_cast<const int2 *>(v.hnx) + w, pol);
        r.tick = (int)ld_keep(v.htick + w, pol);
        r.hlen = (int)ld_keep(v.hlen + w, pol);
    }
}

// PACKED_OB: s.obits holds the world's PACKED obstacle bit matrix (step_kernel: the four wall probes per agent do not
// justify expanding padded rows); otherwise the padded bit rows (fused kernel, where the observation build needs them).
// `g` is the lane group that owns world w; `lane` = g.gl = the agent this thread stands for.
template <int MODE, bool PACKED_OB = false, int G = 32>
__device__ __forceinline__ void resolve_world(const EnvView &v, const MapfStepOut &out, const WarpSmem &s, const int w,
                                              const Grp<G> &g, const StepRegs &in, const uint64_t pol,
                                              uint32_t &new_pw, uint32_t &new_gw) {
    constexpr int QR = 2 * G;
    const int lane = g.gl;
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW;
    const bool active = lane < N;
    const size_t idx = (size_t)w * N + (active ? lane : 0);
    const uint32_t pw = in.pw, gw = in.gw;
    const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
    int goal_r = (int16_t)(gw & 0xffff), goal_c = (int16_t)(gw >> 16);
    const int rep = in.rep;
    int a = in.act;
    uint32_t errbits = 0;
    if (a < 0 || a >= NA) { if (active) errbits |= MAPF_ERR_BAD_ACTION; a = 0; }
    const int tick = in.tick;
    const int2 ht = in.ht;
    const int hr = (int16_t)(ht.x & 0xffff), hc = (int16_t)((uint32_t)ht.x >> 16);
    const int nr = (int16_t)(ht.y & 0xffff), nc = (int16_t)((uint32_t)ht.y >> 16);
    g.sync();
    const int gr = r + P, gc = c + P;
    if (active) {
        s.grid[gr * GS + gc] = (uint8_t)(lane + 1);
        s.act[lane] = (int8_t)a;
        s.rep[lane] = (int8_t)rep;
    }
    g.sync();

    // ---- masks (getInvalidActions :339-360, getRestrictedActions :363-402, good :404-430) -------------------
    uint32_t inv0 = 0, inv1 = 0;
#pragma unroll
    for (int k = 1; k < NA; ++k) {
        const int tr = r + ((k == 2) - (k == 4)), tc = c + ((k == 1) - (k == 3));
        bool blocked;
        if (PACKED_OB) {
            const int ci = tr * v.Wd + tc;
            blocked = (unsigned)tr >= (unsigned)v.H || (unsigned)tc >= (unsigned)v.Wd || ((s.obits[ci >> 5] >> (ci & 31)) & 1u);
        } else {
            blocked = row_bit(s.obits + (tr + P) * RW, tc + P);
        }
        if (blocked) inv0 |= 1u << k;                                                          // OOB or wall
    }
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const int tr = r + ((k == 2) - (k == 4)), tc = c + ((k == 1) - (k == 3));
        const bool hv = (tr == nr && tc == nc) || (r == nr && c == nc && tr == hr && tc == hc);
        if (hv && !(inv0 >> k & 1)) inv1 |= 1u << k;
    }
    uint32_t restr, confl, mmask;
    scan_diamond<false>(s.grid, GS, gr, gc, lane + 1, s.act, a, restr, confl, mmask);
    const uint32_t repbit = rep >= 0 ? (1u << rep) : 0u;
    const uint32_t good = ~(inv0 | inv1 | restr | repbit) & 31u;
    const uint32_t abit = 1u << a;
    const int tgt_r = r + dr_of(a), tgt_c = c + dc_of(a);

    // ---- status (getActionStatus :434-480) -----------------------------------------------------------------
    int st;
    if (MODE == MODE_JOINT) {
        st = in.st_in;
    } else {
        const int cls = (inv0 & abit) ? C_INV0 : (inv1 & abit) ? C_INV1 : (good & abit) ? C_GOOD : C_E;
        st = cls == C_INV0 ? ST_STATIC : cls == C_INV1 ? ST_HUMAN : cls == C_GOOD ? ST_OK
             : (confl & abit) ? ST_AGENT : (a == rep ? ST_REPEAT : ST_OK);
        if (active) s.cls[lane] = (int8_t)cls;
        g.sync();
        bool trig = false;
        if (active && cls == C_E) {
            uint32_t m = mmask;
            while (m) { const int j = __ffs(m) - 1; m &= m - 1; trig |= (s.cls[j] == C_INV1); }
        }
        if (g.any(trig)) {                       // rare: replay the sequential loop (SURVEY A.5)
            if (active) { s.mmask[lane] = mmask; s.st[lane] = 0; }
            g.sync();
            if (lane == 0) {
                for (int i = 0; i < N; ++i) {
                    if (s.st[i] != 0) continue;
                    const int ci = s.cls[i];
                    if (ci == C_INV0) s.st[i] = ST_STATIC;
                    else if (ci == C_INV1) s.st[i] = ST_HUMAN;
                    else if (ci == C_GOOD) s.st[i] = ST_OK;
                    else {
                        uint32_t m = s.mmask[i];
                        while (m) { const int j = __ffs(m) - 1; m &= m - 1; s.st[i] = ST_AGENT; s.st[j] = ST_AGENT; }
                        if (s.st[i] == 0) s.st[i] = (s.act[i] == s.rep[i]) ? ST_REPEAT : ST_OK;
                    }
                }
            }
            g.sync();
            if (active) st = s.st[lane];
        }
    }

    // ---- reward / cost / trainValid (:483-550) -------------------------------------------------------------
    float reward = st == ST_REPEAT ? -0.35f : st == ST_OK ? -0.3f : -2.0f;       // alg_parameters.py:36-43
    const bool sg = active && st == ST_OK && tgt_r == goal_r && tgt_c == goal_c;       // shadowGoal :501-504
    const uint32_t sgm = g.ballot(sg);
    const int d2 = (nr - tgt_r) * (nr - tgt_r) + (nc - tgt_c) * (nc - tgt_c);    // |human.getNextPos() - T(a)|^2 (:519)
    if (MODE != MODE_JOINT) {
        if (active) {
            if (out.status) st_stream_u8(out.status + idx, (uint32_t)st);
            if (out.cost) {
                // max(PENALTY_RADIUS - ||H' - T||, 0) / PENALTY_RADIUS in f64, then cast (:513-533)
                st_stream(out.cost + idx, d2 < 25 ? (float)((5.0 - sqrt((double)d2)) / 5.0) : 0.0f);
            }
            if (MODE == MODE_EVALUATE && out.reward) st_stream(out.reward + idx, reward);
            if (MODE == MODE_EVALUATE && out.good_actions) st_stream_u8(out.good_actions + idx, good);   // allGoodActions (:404-430)
        }
        if (lane == 0 && out.shadow_goals) st_stream(out.shadow_goals + w, (uint32_t)__popc(sgm));
        if (out.train_valid) {
            if (active) {
#pragma unroll
                for (int k = 0; k < NA; ++k) {
                    const uint32_t b = 1u << k;
                    s.tv[lane * NA + k] = (good & b) ? 1.0f : (restr & b) ? ((confl & b) ? 0.0f : 1.0f) : 0.0f;
                }
            }
            g.sync();
            float *dst = out.train_valid + (size_t)w * N * NA;
            for (int k = lane; k < N * NA; k += G) st_stream(dst + k, s.tv[k]);
        }
        if (MODE == MODE_EVALUATE) {
            const uint32_t eb = g.reduce_or(errbits);
            if (lane == 0 && eb) atomicOr(v.err + w, eb);
            g.sync();
            if (active) s.grid[gr * GS + gc] = 0;
            new_pw = pw; new_gw = gw;
            return;
        }
    }

    // ---- fixActions (:552-612), only if some status is -1/-2/-3 (:617) ------------------------------------
    int f = a;
    const bool bad = active && (st == ST_STATIC || st == ST_HUMAN || st == ST_AGENT);
    if (g.any(bad)) {
        int commit = (st == ST_OK) ? a : -1;
        const bool problem = active && st < 0;
        if (problem && good) commit = __ffs(good) - 1;                         // goodActions[0] (:568-571)
        if (active) s.commit[lane] = (int8_t)commit;
        const bool inq = problem && !good;
        const uint32_t qm = g.ballot(inq);
        if (qm) {
            if (inq) s.queue[__popc(qm & ((1u << lane) - 1u))] = (int8_t)lane;
            // The reference's loop pops EVERY problem agent, also those that own a good action (one iteration each, :568-571);
            // here they committed above without being queued.  They all precede the first re-queued agent, so counting them
            // up front makes the iteration cap fall on the same pop as in the oracle (a capped world then keeps evolving
            // identically on both sides; the cap itself cannot fall among the <= N initial entries).
            int head = 0, tail = __popc(qm), iters = __popc(g.ballot(problem && good != 0));
            uint32_t draw = 0;
            g.sync();
            // Every iteration is executed by the whole warp on warp-uniform values: the popped agent's masks arrive by
            // shuffle, lanes 0..11 each look at one cell of its radius-2 diamond, two `redux.or` collect the conflict
            // bits and the eviction set.  (One lane doing this alone made an iteration ~1.4 us of dependent
            // instructions; a world in the reference's livelock runs FIX_CAP of them and was the tail of the launch.)
            int tcur = (v.TL > 0) ? v.tape_cur[w] : 0;
            const int tcur0 = tcur;
            const uint32_t nstep_w = (uint32_t)v.nstep[w];
            uint32_t pd = 0;                       // Philox draws [32*(draw/32), +32), one per lane, made when first needed
            int pd_batch = -1;
            while (head < tail) {
                if (++iters > FIX_CAP) { errbits |= MAPF_ERR_FIX_ITER_CAP; break; }
                const int k = s.queue[(head++) & (QR - 1)];
                const uint32_t kgood = g.shfl(good, k);
                int choice;
                if (kgood) {
                    choice = __ffs(kgood) - 1;                                    // an evicted agent may own a good action (:568)
                } else {
                    const uint32_t viable = ~g.shfl(inv0 | inv1, k) & 31u;      // :575
                    const uint32_t krestr = g.shfl(restr, k);
                    const int kgr = g.shfl(gr, k), kgc = g.shfl(gc, k);
                    // the 12 cells of k's radius-2 diamond are shared out over the lanes of the group (one per lane for
                    // G >= 16, two for G = 8); myc[q] bit a: conflict(k, a; the agent on my q-th cell, its commit)
                    constexpr int CPL = (12 + G - 1) / G;
                    uint32_t myc[CPL], mycs = 0;
                    int myj[CPL];
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        myc[q] = 0; myj[q] = 0;
                        const int cell = lane + q * G;
                        if (cell < 12) {
                            const int dr = (int)((0x433322221110ull >> (4 * cell)) & 15) - 2;
                            const int dc = (int)((0x232143103212ull >> (4 * cell)) & 15) - 2;
                            const int code = s.grid[(kgr + dr) * GS + (kgc + dc)];
                            if (code != 0 && code != k + 1) {
                                myj[q] = code - 1;
                                const int b = s.commit[myj[q]];
                                const int tr = dr + (b >= 0 ? dr_of(b) : 0), tc = dc + (b >= 0 ? dc_of(b) : 0);   // T_j - pos_k
#pragma unroll
                                for (int a2 = 0; a2 < NA; ++a2) {
                                    const int ar = (a2 == 2) - (a2 == 4), ac = (a2 == 1) - (a2 == 3);
                                    bool cf = (b >= 0) && (tr == ar) && (tc == ac);                                      // vertex
                                    if (a2 != 0 && dr == ar && dc == ac) cf = cf || (b == (a2 == 1 ? 3 : a2 == 2 ? 4 : a2 == 3 ? 1 : 2));  // swap
                                    if (cf) myc[q] |= 1u << a2;
                                }
                            }
                        }
                        mycs |= myc[q];
                    }
                    auto evicted = [&](int choice_) {                             // agents whose commit conflicts with (k, choice_)
                        uint32_t e_ = 0;
#pragma unroll
                        for (int q = 0; q < CPL; ++q) if ((myc[q] >> choice_) & 1u) e_ |= 1u << myj[q];
                        return g.reduce_or(e_);
                    };
                    const uint32_t c2 = g.reduce_or(mycs);
                    const uint32_t ok = viable & ~(krestr & c2);                  // :577-584
                    if (ok) {
                        choice = __ffs(ok) - 1;
                    } else if (!viable) {
                        errbits |= MAPF_ERR_NO_VIABLE;                            // reference: IndexError (:588)
                        choice = 0;
                    } else {
                        const int nv = __popc(viable);
                        if (v.TL > 0) {                                           // recorded random.choice + eviction order
                            const int8_t *tp = v.tape + (size_t)w * v.TL;
                            const int tl = v.tape_len[w];
                            if (tcur + 2 > tl) { errbits |= MAPF_ERR_TAPE; choice = __ffs(viable) - 1; tcur = tl; }
                            else {
                                choice = tp[tcur];
                                const int ne = tp[tcur + 1];
                                if (choice < 0 || choice >= NA) { errbits |= MAPF_ERR_TAPE; choice = __ffs(viable) - 1; }
                                const uint32_t ev = evicted(choice);
                                uint32_t seen = 0;
                                for (int q = 0; q < ne && tcur + 2 + q < tl; ++q) {
                                    const int j = tp[tcur + 2 + q];
                                    if (j >= 0 && j < N && (ev >> j & 1)) {
                                        seen |= 1u << j;
                                        if (lane == 0) { s.commit[j] = -1; s.queue[tail & (QR - 1)] = (int8_t)j; }
                                        tail++;
                                    }
                                }
                                if (seen != ev || __popc(ev) != ne) errbits |= MAPF_ERR_TAPE;
                                tcur += 2 + ne;
                            }
                        } else {                                                  // Philox stand-in, ascending eviction
                            if ((int)(draw / G) != pd_batch) {                    // G draws cost the latency of one
                                pd_batch = (int)(draw / G);
                                pd = philox_draw(v.seed, (uint32_t)(w + v.world_offset), nstep_w, (draw & ~(uint32_t)(G - 1)) + lane);
                            }
                            const uint32_t x = g.shfl(pd, (int)(draw & (G - 1)));
                            // x % nv, nv in 1..5 (constant divisors: a multiply-high instead of a division loop)
                            int pick = nv == 1 ? 0 : nv == 2 ? (int)(x & 1u) : nv == 3 ? (int)(x % 3u) : nv == 4 ? (int)(x & 3u) : (int)(x % 5u);
                            uint32_t vm = viable;
                            while (pick--) vm &= vm - 1;
                            choice = __ffs(vm) - 1;
                            uint32_t ev = evicted(choice);
                            while (ev) {                                          // :593-596
                                const int j = __ffs(ev) - 1; ev &= ev - 1;
                                if (lane == 0) { s.commit[j] = -1; s.queue[tail & (QR - 1)] = (int8_t)j; }
                                tail++;
                            }
                        }
                        draw++;
                    }
                }
                if (lane == 0) s.commit[k] = (int8_t)choice;                      // :598
                g.sync();
            }
            if (v.TL > 0 && lane == 0 && tcur != tcur0) v.tape_cur[w] = tcur;
        }
        g.sync();
        if (active) { f = s.commit[lane]; if (f < 0) f = 0; }
        // The reference hangs (livelock) or raises (IndexError) here; whatever the loop had committed so far need not be
        // collision-free (an agent left at -1 stays where another may already be headed).  Every agent of such a world
        // stays in this step: nobody moves, so the world remains a valid state and keeps stepping identically in the oracle.
        if (errbits & (MAPF_ERR_FIX_ITER_CAP | MAPF_ERR_NO_VIABLE)) f = 0;
    }

    // ---- moves, goal arrival, human tick, constraint violations (:620-633) ----------------------------------
    const int nr_ = r + dr_of(f), nc_ = c + dc_of(f);
    const bool arrived = active && nr_ == goal_r && nc_ == goal_c;
    const int t2 = (tick + 1 >= in.hlen) ? 0 : tick + 1;
    const int2 ht2 = in.ht2;
    const int h2r = (int16_t)(ht2.x & 0xffff), h2c = (int16_t)((uint32_t)ht2.x >> 16);
    const bool viol = active && ((h2r - nr_) * (h2r - nr_) + (h2c - nc_) * (h2c - nc_) <= 24);   // cost_norm >= 0.01
    new_pw = (uint32_t)(uint16_t)nr_ | ((uint32_t)(uint16_t)nc_ << 16);
    new_gw = gw;
    const uint32_t am = g.ballot(arrived);
    if (v.goal_sampling && am) {
        // MapfGym.getNextGoal (mapf_gym.py:189-190, 626) = getFreeCell(worldWithAgentsAndGoals()) (util.py:67-76), for the
        // arrived agents in agent order: a cell is taken if it is an obstacle, the cell of an agent (agents <= i have
        // moved, the others have not: jointStep's loop is sequential, :620-627) or any agent's current goal.  The warp tests
        // 32 consecutive draws at a time and takes the first free one, which is what the sequential rejection loop does.
        int rows = v.H, cols = v.Wd;
        if (v.dims) { rows = v.dims[2 * w]; cols = v.dims[2 * w + 1]; }
        const uint32_t nstep_w = (uint32_t)v.nstep[w];
        uint32_t m = am, draw = 0;
        while (m) {
            const int i = __ffs(m) - 1; m &= m - 1;
            const uint32_t occ = (lane <= i) ? new_pw : pw;
            uint32_t chosen = 0;
            bool found = false;
            for (int batch = 0; batch < GOAL_DRAW_CAP / G && !found; ++batch) {
                const uint32_t cand = goal_candidate(v.seed, (uint32_t)(w + v.world_offset), nstep_w, draw + lane, rows, cols);
                const int cr = (int)(cand & 0xffff), cc = (int)(cand >> 16);
                bool free_;
                if (PACKED_OB) { const int ci = cr * v.Wd + cc; free_ = !((s.obits[ci >> 5] >> (ci & 31)) & 1u); }
                else free_ = !row_bit(s.obits + (cr + P) * RW, cc + P);
                for (int j = 0; j < N; ++j) {
                    const uint32_t pj = g.shfl(occ, j), gj = g.shfl(new_gw, j);
                    free_ = free_ && cand != pj && cand != gj;
                }
                const uint32_t b = g.ballot(free_);
                if (b) { const int k = __ffs(b) - 1; chosen = g.shfl(cand, k); draw += k + 1; found = true; }
                else draw += G;
            }
            if (!found) errbits |= MAPF_ERR_NO_FREE_CELL;          // goal unchanged (= the agent's own cell)
            else if (lane == i) new_gw = chosen;
        }
    }
    if (active) {
        st_keep(reinterpret_cast<uint32_t *>(v.pos) + idx, new_pw, pol);
        st_keep_s8(v.rep + idx, opp_of(f), pol);                                 // takeStep :158-161
        if (arrived) {
            if (!v.goal_sampling) {                                              // Sequence.getNext util.py:33-39
                int k = v.qcur[idx];
                if (k >= v.Q) k = v.Q - 1; else v.qcur[idx] = k + 1;
                new_gw = reinterpret_cast<const uint32_t *>(v.goal_queue)[idx * v.Q + k];
            }
            st_keep(reinterpret_cast<uint32_t *>(v.goal) + idx, new_gw, pol);
        }
        if (out.goals_reached) st_stream_u8(out.goals_reached + idx, arrived);
        if (out.violated) st_stream_u8(out.violated + idx, viol);
        if (out.fixed_actions) st_stream_u8(out.fixed_actions + idx, (uint32_t)f);
        if (MODE == MODE_FUSED && out.reward) st_stream(out.reward + idx, arrived ? __fadd_rn(reward, 1.5f) : reward);  // runner.py:89-91
        if (MODE == MODE_FUSED && out.packed) {                                  // MAPF_PACKED_* (include/mapf_b200.h)
            const uint32_t sc = st == ST_STATIC ? 0u : st == ST_HUMAN ? 1u : st == ST_AGENT ? 2u : st == ST_REPEAT ? 3u : 4u;
            st_stream_u16(out.packed + idx, sc | ((uint32_t)arrived << 3) | ((uint32_t)viol << 4) | ((uint32_t)f << 5) |
                                                ((uint32_t)min(d2, 25) << 8));
        }
    }
    const uint32_t vm_ = g.ballot(viol);
    const uint32_t c1 = g.ballot(active && st == ST_STATIC), c2b = g.ballot(active && st == ST_HUMAN),
                   c3 = g.ballot(active && st == ST_AGENT);
    const uint32_t eb = g.reduce_or(errbits);
    if (lane == 0) {
        st_keep(v.htick + w, (uint32_t)t2, pol);
        st_keep_v2(reinterpret_cast<int2 *>(v.hcur) + w, ht2, pol);
        const int t3 = (t2 + 1 >= in.hlen) ? 0 : t2 + 1;          // keep the entry after next resident too
        st_keep_v2(reinterpret_cast<int2 *>(v.hnx) + w, ld_keep_v2(v.htrace + ((size_t)w * v.L + t3) * 4, pol), pol);
        add_keep_s32(v.nstep + w, 1, pol);
        if (eb) atomicOr(v.err + w, eb);
        long long *cn = v.counters + (size_t)w * 6;                              // util.py:56-65, runner.py:66-99
        add_keep_s64(cn + 0, __popc(am), pol); add_keep_s64(cn + 1, __popc(sgm), pol); add_keep_s64(cn + 2, __popc(c1), pol);
        add_keep_s64(cn + 3, __popc(c2b), pol); add_keep_s64(cn + 4, __popc(c3), pol); add_keep_s64(cn + 5, __popc(vm_), pol);
    }
    g.sync();
    if (active) s.grid[gr * GS + gc] = 0;      // leave the id grid clean for the next world of this warp
}

}  // namespace sw
}  // namespace mapf
