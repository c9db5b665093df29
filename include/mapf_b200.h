/*
 * mapf_b200.h — C ABI of the B200-native batched MAPF environment hot path.
 *
 * The reference (Nielsencu/primal-ppo) has no FFI: its environment is a Python class,
 * `MapfGym` / `FixedMapfGym` (mapf_gym.py:163-669), driven by the rollout loop in runner.py:30-100
 * and followed by the GAE scan in runner.py:117-149.  This header is the boundary a maintainer binds
 * instead of those Python methods (INTEGRATION.md shows the ctypes stub): plain pointers and sizes, no
 * torch types.  Each entry point names the reference interface it replaces.
 *
 * Conventions
 *  - W worlds, N agents, H x Wd cells, C channels, F = FOV side.  Cells are (row, col).
 *  - Actions 0..4 = stay, (0,+1), (+1,0), (0,-1), (-1,0)                      (mapf_gym.py:97-98)
 *  - Unless a function name ends in `_host`, every data pointer is a DEVICE pointer on the env's device
 *    and the call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream).
 *    No allocation and no host synchronisation happens inside reset/evaluate/step/observe/bfs/gae (the staging of the
 *    *_host entry points is allocated by mapf_create).
 *  - Alignment: vec and the scenario's starts / goal_queue must be 4-byte aligned per (row, col) pair and vec 16-byte
 *    aligned; htrace 8-byte aligned; obs 4-byte (16-byte aligned buffers take the vector-store path).
 *  - A handle is single-stream: calls on one MapfEnv must be issued from one thread and are ordered on the streams
 *    passed; two calls of the same env must not run concurrently on different streams (every kernel family has its own
 *    work counter, re-armed by mapf_reset, but the env state itself is not versioned).
 *  - The caller owns every input/output buffer.  Scenario arrays passed to mapf_reset are BORROWED and
 *    must stay alive and unchanged until the next mapf_reset / mapf_destroy.
 *  - Return value: 0 on success, a negative MAPF_E_* code otherwise; mapf_last_error() gives the text.
 *    Data-dependent failures never abort a call: they set bits in err[w] (MAPF_ERR_*) for that world only.
 */
#ifndef MAPF_B200_H
#define MAPF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAPF_B200_ABI_VERSION 2

/* return codes */
#define MAPF_OK 0
#define MAPF_E_BAD_CONFIG (-1)
#define MAPF_E_NULL (-2)
#define MAPF_E_CUDA (-3)
#define MAPF_E_UNSUPPORTED (-4)
#define MAPF_E_STATE (-5)

/* per-world error bits (err[w]); the reference raises or hangs in these situations.  For NO_VIABLE and FIX_ITER_CAP every agent
 * of the world stays in that step (whatever fixActions had committed so far need not be collision-free), so a flagged world
 * remains a valid state and keeps stepping. */
#define MAPF_ERR_NO_VIABLE 1u    /* IndexError from random.choice([])        mapf_gym.py:588 */
#define MAPF_ERR_FIX_ITER_CAP 2u /* livelock of the fixActions while loop     mapf_gym.py:563 */
#define MAPF_ERR_BAD_ACTION 4u   /* action outside 0..4                       mapf_gym.py:452-456 */
#define MAPF_ERR_TAPE 8u         /* fixActions tape exhausted / inconsistent */
#define MAPF_ERR_NO_FREE_CELL 64u /* goal_sampling: no free cell found in 4096 draws (getFreeCell would spin for ever, util.py:72) */

typedef struct MapfEnv MapfEnv; /* opaque; one handle per (process, device); not thread-safe */

/* Replaces the constants read from alg_parameters.py (EnvParameters / NetParameters) and the ctor arguments of
 * FixedMapfGym (mapf_gym.py:649). */
typedef struct MapfConfig {
    int32_t num_worlds;   /* W */
    int32_t height;       /* H  (max rows over worlds) */
    int32_t width;        /* Wd (max cols over worlds) */
    int32_t num_agents;   /* N  = EnvParameters.N_AGENTS  (alg_parameters.py:30); 1..128 for step, up to 254 for observe/bfs */
    int32_t fov;          /* F  = EnvParameters.FOV_SIZE  (alg_parameters.py:33); odd, 3..31 */
    int32_t num_channel;  /* C  = NetParameters.NUM_CHANNEL (alg_parameters.py:104); 5 or 6 */
    int32_t use_da;       /* FixedMapfGym(useDA=)  danger-area disc in channel 4   (mapf_gym.py:289-290) */
    int32_t use_hp;       /* FixedMapfGym(useHP=)  human-path cells in channel 5   (mapf_gym.py:293-297) */
    int32_t queue_len;    /* Q: goals per agent in goal_queue */
    int32_t trace_len;    /* L: ticks per world in htrace */
    int32_t tape_stride;  /* TL: bytes per world in tape; 0 = no tape (Philox mode) */
    int32_t hp5_per_tick; /* 0: hp5 is [W,5,2]; 1: hp5 is [W,L,5,2] */
    uint64_t seed;        /* Philox key for the random branch of fixActions when no tape is given */
    int32_t device;       /* CUDA device ordinal */
    int32_t world_offset; /* global index of this env's world 0 (rank r of a sharded job: r*W): keys the Philox draws so
                             that world w behaves identically on whichever rank owns it */
    int32_t goal_sampling;/* 0: goals come from goal_queue (FixedMapfGym.getNextGoal, mapf_gym.py:668-669: Sequence.getNext);
                             1: on arrival the next goal is drawn ON DEVICE like MapfGym.getNextGoal (mapf_gym.py:189-190,
                                626) = util.getFreeCell (util.py:67-76) on worldWithAgentsAndGoals(): uniform rejection
                                sampling over cells free of obstacles, of every agent's cell (agents before the arriving one
                                already moved, the others not yet) and of every current goal.  Philox4x32-10 keyed by
                                (seed; world_offset + w, step, draw): the reference's distribution, not its MT19937 bits.
                                goal_queue[:, :, 0] still supplies the first goal. */
    int32_t reserved0;
} MapfConfig;

/* Exogenous inputs of a batch of worlds — what the reference draws from np.random / random at construction and on
 * goal arrival (mapf_gym.py:164-190, util.py:67-76) or receives through FixedMapfGym (mapf_gym.py:648-669). */
typedef struct MapfScenario {
    const uint8_t *obst;      /* [W,H,Wd]   1 = obstacle (reference -1), 0 = free */
    const int16_t *starts;    /* [W,N,2]    Sequence.items[0] */
    const int16_t *goal_queue;/* [W,N,Q,2]  Sequence.items[1:]; the last entry repeats when exhausted (util.py:33-36) */
    const int16_t *htrace;    /* [W,L,4]    human (pos_r,pos_c,next_r,next_c) per tick (mapf_gym.py:25-50) */
    const int32_t *hlen;      /* [W]        ticks before the trace wraps to 0 */
    const int16_t *hp5;       /* [W,5,2] or [W,L,5,2] human.path[1:6], -1 padded; may be NULL unless use_hp */
    const int8_t *tape;       /* [W,TL]     fixActions tape: [choice, n_evicted, ids...]*; NULL iff tape_stride==0 */
    const int32_t *tape_len;  /* [W] */
    const int16_t *dims;      /* [W,2] per-world (rows, cols) or NULL = (H, Wd) for all */
} MapfScenario;

/* Outputs of one step; any pointer may be NULL (that output is skipped). */
typedef struct MapfStepOut {
    int8_t *status;        /* [W,N]   getActionStatus        mapf_gym.py:434-480  (-1,-2,-3,-4,1) */
    float *reward;         /* [W,N]   calculateActionReward  mapf_gym.py:483-511  (+GOAL_REWARD in mapf_step, runner.py:89-91) */
    float *cost;           /* [W,N]   calculateCostReward    mapf_gym.py:528-533 */
    float *train_valid;    /* [W,N,5] getTrainValid          mapf_gym.py:535-550 */
    uint8_t *goals_reached;/* [W,N]   jointStep()[0]         mapf_gym.py:614-637 */
    uint8_t *violated;     /* [W,N]   jointStep()[1] */
    int32_t *shadow_goals; /* [W]     calculateActionReward()[1] */
    int8_t *fixed_actions; /* [W,N]   the actions actually executed (after fixActions, mapf_gym.py:552-612) */
    uint16_t *packed;      /* [W,N]   every per-agent result of the step in 16 bits (lossless; MAPF_PACKED_* below): what the
                              split-phase host call ships over PCIe in compact mode.  Written by mapf_step / mapf_step_observe. */
    uint8_t *good_actions; /* [W,N]   MapfGym.allGoodActions (mapf_gym.py:404-430, refreshed at :169/:635) as 5-bit masks, bit a =
                              action a is unconditionally good in the CURRENT state; written by mapf_evaluate only (the
                              masks do not depend on the actions passed) */
} MapfStepOut;

/* MapfStepOut.packed: bits 0-2 status code (0: -1 static, 1: -2 human, 2: -3 agent, 3: -4 repeat, 4: +1 ok), bit 3
 * goal reached, bit 4 constraint violated, bits 5-7 the executed action (after fixActions), bits 8-12 min(d2, 25) with d2 the
 * squared distance between human.getNextPos() and the agent's (unfixed) target cell.  The f32 outputs are functions of
 * these fields:  reward = {-2, -2, -2, -0.35, -0.3}[status code] (+ 1.5 when goal reached, runner.py:89-91);
 * cost = d2 < 25 ? (float)((5.0 - sqrt((double)d2)) / 5.0) : 0   (mapf_gym.py:513-533).  mapf_decode_results_host expands
 * a packed array into the reference's arrays on the host, bit for bit. */
#define MAPF_PACKED_STATUS(p) ((int)((p) & 7u))
#define MAPF_PACKED_GOAL(p) ((int)(((p) >> 3) & 1u))
#define MAPF_PACKED_VIOLATED(p) ((int)(((p) >> 4) & 1u))
#define MAPF_PACKED_ACTION(p) ((int)(((p) >> 5) & 7u))
#define MAPF_PACKED_D2(p) ((int)(((p) >> 8) & 31u))

int mapf_abi_version(void);
const char *mapf_last_error(void);

/* MapfGym.__init__ / FixedMapfGym.__init__ (mapf_gym.py:164-173, 648-663): allocate persistent state. */
int mapf_create(const MapfConfig *cfg, MapfEnv **out);
int mapf_destroy(MapfEnv *env);

/* populateMap (mapf_gym.py:175-184): starts, first goals, cleared repetition lists, human tick 0. */
int mapf_reset(MapfEnv *env, const MapfScenario *scenario, void *stream);

/* getActionStatus + calculateActionReward + calculateCostReward + getTrainValid (runner.py:64-82) without
 * mutating the env.  out->goals_reached / violated / fixed_actions are ignored. */
int mapf_evaluate(MapfEnv *env, const int8_t *actions, const MapfStepOut *out, void *stream);

/* jointStep(actions, actionStatus) (mapf_gym.py:614-637, runner.py:87): fixActions, moves, goal arrival, human tick,
 * constraint violations.  `status` is the array mapf_evaluate produced for the same actions. */
int mapf_joint_step(MapfEnv *env, const int8_t *actions, const int8_t *status, uint8_t *goals_reached,
                    uint8_t *violated, int8_t *fixed_actions, void *stream);

/* The five calls of runner.py:64-87 fused in one launch, plus `rewards[goalsReached==1] += GOAL_REWARD`
 * (runner.py:89-91). */
int mapf_step(MapfEnv *env, const int8_t *actions, const MapfStepOut *out, void *stream);

/* getAllObservations (mapf_gym.py:327-336): obs f32 [W,N,C,F,F], vec f32 [W,N,4], written in place.  vec must be
 * 16-byte aligned (one store per agent); obs may have any 4-byte alignment (16-byte aligned buffers take the fast path). */
int mapf_observe(MapfEnv *env, float *obs, float *vec, void *stream);

/* One env step of the rollout loop in ONE launch (runner.py:64-100): mapf_step followed by mapf_observe of the new
 * state, fused per world so that the step resolution hides under the observation stores.  Bit-identical to calling
 * the two entry points back to back (which is what happens for shapes the fused kernel does not cover: N > 32 or an
 * observation block that needs several chunks). */
int mapf_step_observe(MapfEnv *env, const int8_t *actions, const MapfStepOut *out, float *obs, float *vec, void *stream);

/* Optional output format (NOT the reference's layout): the same observations as bf16 [W,N,C,F,F] — every value is 0 or 1
 * and exact in bf16 — for GPU-resident training loops whose network runs under bf16 autocast anyway (the reference casts
 * the f32 observations to half precision at the first convolution, net.py:101).  Halves the bytes of the dominant store. */
int mapf_observe_bf16(MapfEnv *env, uint16_t *obs_bf16, float *vec, void *stream);
int mapf_step_observe_bf16(MapfEnv *env, const int8_t *actions, const MapfStepOut *out, uint16_t *obs_bf16, float *vec,
                           void *stream);

/* Optional bit-packed format (NOT the reference's layout): one bit per observation cell.  obs_bits is u32 [W,N,AW] with
 * AW = MAPF_OBS_BITS_WORDS(C, F): bit k of agent (w, i) is obs[w, i].flatten()[k] in the reference's [C,F,F] order, held in
 * word k / 32 at bit k % 32 (LSB first); the padding bits of an agent's last word are 0.  Every agent has its own
 * word-aligned record.  64 B per agent at 6 x 9 x 9 instead of 1944 B in f32: what lets a rollout buffer hold the
 * observations of a large batch (mapf_unpack_obs expands them for the network).  obs_bits must be 4-byte aligned (16-byte
 * aligned buffers with AW % 4 == 0 take 16-byte stores); vec is f32 [W,N,4] as in mapf_observe. */
#define MAPF_OBS_BITS_WORDS(C, F) (((C) * (F) * (F) + 31) / 32)
int mapf_observe_bits(MapfEnv *env, uint32_t *obs_bits, float *vec, void *stream);
int mapf_step_observe_bits(MapfEnv *env, const int8_t *actions, const MapfStepOut *out, uint32_t *obs_bits, float *vec,
                           void *stream);

/* Gather-and-expand of bit-packed observations (no env handle): obs_bits is [src_rows, agents, AW] (a row = one world of
 * one step); out[r] = the f32 (out_bf16 = 0) or bf16 (out_bf16 = 1) 0/1 values [agents, C, F, F] of source row rows[r]
 * (rows NULL: row r), for r < n_rows.  A row index outside [0, src_rows) gives an all-zero row.  obs_bits 4-byte aligned,
 * out aligned to its element size (16-byte aligned buffers take the fast path). */
int mapf_unpack_obs(const uint32_t *obs_bits, int64_t src_rows, int32_t agents, int32_t num_channel, int32_t fov,
                    const int64_t *rows /* NULL = rows 0..n_rows-1 */, int64_t n_rows, int32_t out_bf16, void *out,
                    void *stream);

/* makeBfsMap (mapf_gym.py:211-244) for the CURRENT goals.  agent_list: n flat ids (w*N+i), or NULL for all W*N
 * agents in order.  out: int16 [n,H,Wd]: -1 obstacle (and cells outside a world's dims), -2 unreached, >=0 distance. */
int mapf_bfs(MapfEnv *env, const int32_t *agent_list, int64_t n, int16_t *out, void *stream);

/* The in-loop refresh `makeBfsMap(agent)` on goal arrival (mapf_gym.py:627): recompute, in place, the maps of the
 * agents with goals_reached[w,i] == 1 inside bfs_maps int16 [W,N,H,Wd].  The arrival list is compacted on the device;
 * there is no host synchronisation. */
int mapf_bfs_refresh(MapfEnv *env, const uint8_t *goals_reached, int16_t *bfs_maps, void *stream);

/* GAE + returns of one stream (runner.py:120-149): r, v [T,cols]; last_v [cols]; nonterminal [T,cols] or NULL = all 1
 * (the reference uses the constant 1.0, runner.py:123); returns = adv + v; adv may be NULL.  gamma, lam are the Python
 * doubles; the kernel multiplies by float(gamma) and float(gamma*lam) without FMA contraction. */
int mapf_gae(const float *r, const float *v, const float *last_v, const uint8_t *nonterminal, double gamma,
             double lam, int32_t T, int64_t cols, float *returns, float *adv, void *stream);

/* Both streams of the rollout in ONE launch (runner.py:146-149 calls the scan twice: rewards / values and costRewards /
 * costValues): same arithmetic as two mapf_gae calls, bit for bit. */
int mapf_gae2(const float *r, const float *v, const float *last_v, const float *cost_r, const float *cost_v,
              const float *last_cost_v, const uint8_t *nonterminal, double gamma, double lam, int32_t T, int64_t cols,
              float *returns, float *cost_returns, float *adv, float *cost_adv, void *stream);

/* Joint-action sampling on device — replaces the per-agent host loop `np.random.choice(range(N_ACTIONS), p=ps[i])`
 * of Model.step / Model.evaluate (model.py:38-40, 58-59).  ps: f32 [rows,5] probabilities (rows = W*N); actions: int8
 * [rows]; chosen_p (optional): f32 [rows] probability of the drawn action.  Philox4x32-10 keyed by (seed; row, draw):
 * call with draw = 0, 1, 2, ... for successive steps.  Same distribution as the reference, not the same bits. */
int mapf_sample_actions(const float *ps, int64_t rows, uint64_t seed, uint32_t draw, int8_t *actions, float *chosen_p,
                        void *stream);

/* State read-back for checks and checkpoints (device pointers; any may be NULL):
 * pos/goal int16 [W,N,2], rep int8 [W,N] (the repetition action or -1, mapf_gym.py:161), err u32 [W]. */
int mapf_get_state(MapfEnv *env, int16_t *pos, int16_t *goal, int8_t *rep, uint32_t *err, void *stream);

/* The human walker of every world (Human.getPos / getNextPos / step, mapf_gym.py:25-50; device pointers, any may be
 * NULL): pos_next int16 [W,4] = (pos_r, pos_c, next_r, next_c) of the current tick, tick int32 [W]. */
int mapf_get_human(MapfEnv *env, int16_t *pos_next, int32_t *tick, void *stream);

/* Checkpoint / resume of everything reset and step mutate (cells, goals, repetition actions, queue cursors, human tick,
 * tape cursor, step count, error flags, episode counters) as one opaque device blob of mapf_state_bytes() bytes.  The
 * scenario arrays are not part of it (they are borrowed and immutable): a blob is valid for an env created with the same
 * MapfConfig and reset with the same scenario.  The reference has no counterpart (its envs are rebuilt every rollout,
 * runner.py:30). */
int64_t mapf_state_bytes(MapfEnv *env);
int mapf_save_state(MapfEnv *env, void *blob, void *stream);
int mapf_load_state(MapfEnv *env, const void *blob, void *stream);

/* Episode counters accumulated on device (util.py:56-65 OneEpPerformance, filled in runner.py:66-99):
 * int64 [W,6] = totalGoals, shadowGoals, staticCollide, humanCollide, agentCollide, constraintViolations. */
int mapf_get_counters(MapfEnv *env, int64_t *counters, void *stream);

/* ---- on-device scenario generation (throughput mode) ------------------------------------------------------------ */

/* Replaces, for W worlds at once, what MapfGym.__init__ draws on the host: the map (generateWarehouse,
 * map_generator.py:127-138, or the PRIMAL density map, map_generator.py:13-28), the human's entrance / goal / walk
 * (mapf_gym.py:9-50, astar_4.py) and the agents' starts and goals (populateMap mapf_gym.py:175-190, getFreeCell
 * util.py:67-76).  Philox4x32-10 keyed by (seed; world_offset + w, stream, draw): equal to the reference in distribution,
 * not in bits; the warehouse layout for a drawn length is bit-identical to generateWarehouse.  With human_path = 1 the
 * walk between the drawn cells is astar_4's path, bit for bit. */
typedef struct MapfGenConfig {
    int32_t num_worlds, height, width, num_agents; /* array shapes: every world is stored as height x width */
    int32_t kind;          /* 0 = density map, 1 = warehouse */
    int32_t density_mode;  /* kind 0: 0 = p ~ U[lo, hi], 1 = np.random.triangular(lo, .33 lo + .66 hi, hi) (map_generator.py:18) */
    float density_lo, density_hi;
    int32_t size_lo, size_hi; /* kind 1: length ~ U{lo..hi}, cols = int(length * 1.5); kind 0: side from {lo, (lo+hi)/2, hi}
                                 w.p. (.5, .25, .25) (map_generator.py:19), or fixed height x width when size_lo <= 0 */
    int32_t queue_len;     /* Q goals per agent */
    int32_t trace_len;     /* L ticks of human trace per world */
    int32_t human_loops;   /* 1 = LoopingHuman (one out-and-back walk, repeated); k > 1 = up to k walks with re-drawn goals
                              (Human.getNextGoal, mapf_gym.py:41-43) before the trace wraps */
    int32_t human_path;    /* the human's walk to each goal: 0 = descent of the BFS field with neighbour order E, S, W, N (a
                              shortest path, not astar_4's); 1 = astar_4 itself, bit-exact with its tie-breaking (the
                              reference's MapfGym).  The draws, maps and walk lengths are the same for both. */
    uint64_t seed;
    int32_t world_offset;  /* global index of world 0 (sharded jobs) */
    int32_t device;
} MapfGenConfig;

/* gen_err bits (per world, optional): 1 too few free cells, 2 no free cell on row 0 / column 0 (the reference would spin
 * forever in getEntrance), 4 no reachable goal within trace_len (human stands still), 8 an agent could not be placed. */
int mapf_generate_scenario(const MapfGenConfig *cfg, uint8_t *obst /*[W,H,Wd]*/, int16_t *dims /*[W,2]*/,
                           int16_t *starts /*[W,N,2]*/, int16_t *goal_queue /*[W,N,Q,2]*/, int16_t *htrace /*[W,L,4]*/,
                           int32_t *hlen /*[W]*/, int16_t *hp5 /*[W,5,2] or NULL*/, uint32_t *gen_err /*[W] or NULL*/,
                           void *stream);

/* astar_4 (astar_4.py:21-109) for n (map, start, goal) triples at once, bit-exact with its tie-breaking; one warp per
 * triple.  obst [n,H,Wd] (nonzero = wall; 1 <= H, Wd <= 128), start_goal [n,2,2] as (row, col) pairs.  lens[i] = k >= 1
 * for a path of k cells from start to goal inclusive, written to paths[i, :k]; 0 = start == goal; -1 = no path (the goal
 * is a wall or unreachable; a walled start is still expanded); -2 = the path has more than max_len cells; -3 = start or
 * goal outside the map.  Unused path cells are -1.  Asynchronous on stream; allocates nothing. */
int mapf_astar4_paths(const uint8_t *obst, int64_t n, int32_t H, int32_t Wd, const int16_t *start_goal, int32_t max_len,
                      int16_t *paths /*[n,max_len,2]*/, int32_t *lens /*[n]*/, void *stream);

/* ---- host-buffer entry points (what a CPU-side runner calls; copies are inside the call) ---------------- */

/* Host mirror of MapfStepOut: PINNED or pageable host memory; any pointer may be NULL.  For full PCIe speed carve the
 * action buffer and all of these out of ONE pinned allocation (measured: separately pinned 2 MB buffers copy up to 3x
 * slower than slices of a single slab). */
typedef struct MapfStepOutHost {
    int8_t *status; float *reward; float *cost; float *train_valid; uint8_t *goals_reached; uint8_t *violated;
    int32_t *shadow_goals; int8_t *fixed_actions; uint16_t *packed /* ignored */; uint8_t *good_actions /* ignored */;
} MapfStepOutHost;

/* SYNCHRONOUS form.  actions_host -> device, mapf_step, mapf_observe into obs_dev/vec_dev (device; the policy's input
 * tensors), step outputs -> host (copied on the env's copy stream while the observation kernel runs), stream
 * synchronised before return.  train_valid_dev (device, optional) receives trainValid [W,N,5] in HBM — like the
 * observations it is training data that the learner consumes on the GPU; out->train_valid (host) needs it.  If obs_host /
 * vec_host are non-NULL the observations are also copied to the host (what the reference's getAllObservations returns). */
int mapf_step_observe_host(MapfEnv *env, const int8_t *actions_host, const MapfStepOutHost *out, float *obs_dev,
                           float *vec_dev, float *train_valid_dev, float *obs_host, float *vec_host, void *stream);

/* SPLIT-PHASE form (what a rollout loop should use): nothing in runner.py:64-100 needs the rewards / status of step t
 * before step t+1 starts (they are appended to the rollout lists, runner.py:84-99), so the results of step t travel to the
 * host while step t+1 computes.
 *
 * All per-agent results of one step live in ONE contiguous "result slot" whose layout mapf_host_layout reports (same
 * layout on the device and on the host; every field 256-byte aligned).  Two wire formats, chosen by `flags`:
 *   full (default):        reward f32[W,N] | cost f32[W,N] | shadow_goals i32[W] | status i8[W,N] | goals_reached u8[W,N] |
 *                          violated u8[W,N] | fixed_actions i8[W,N]                       (12 B per agent)
 *   MAPF_HOST_COMPACT:     packed u16[W,N] (MapfStepOut.packed) | shadow_goals i32[W]     (2 B per agent, lossless;
 *                          mapf_decode_results_host expands it).  Eight GPUs of one box share the host's PCIe / memory
 *                          path: at 65 536 x 32 agents the full slab is 25 MB per step and GPU, the compact one 4.5 MB.
 *   | MAPF_HOST_TRAIN_VALID: train_valid f32[W,N,5] appended (needs train_valid_dev; the caller's tensor is the copy
 *                          source, so the next begin waits for this step's copy).
 *   | MAPF_HOST_OBS:        the step's observations and vec appended, for a runner whose policy reads them on the host
 *                          (the reference's getAllObservations, runner.py:31,100).  The observation block starts at
 *                          off_obs = slot_bytes of the same flags without MAPF_HOST_OBS and holds obs_dev as written:
 *                          W*N*C*F*F*4 (f32), W*N*C*F*F*2 (bf16) or W*N*MAPF_OBS_BITS_WORDS(C,F)*4 (bits) bytes, rounded up
 *                          to 256; vec f32[W,N,4] (W*N*16 bytes) follows it.  mapf_host_layout reports the total slot_bytes.
 *                          Both are copied from the caller's obs_dev / vec_dev, so a later begin whose outputs (obs_dev,
 *                          vec_dev, train_valid_dev) overlap them waits for this step's copy; one that writes into other
 *                          buffers (a rollout buffer's step t+1) does not.  Only later begins are ordered behind the
 *                          copy: any other writer to those buffers must first wait for that step (mapf_step_observe_host_wait).
 *                          A bit-packed slot is expanded on the host by
 *                          mapf_unpack_obs_host.
 * Observation format of obs_dev (orthogonal to the wire format; at most one of the two):
 *   default f32 [W,N,C,F,F] (mapf_step_observe); MAPF_HOST_OBS_BF16: bf16 [W,N,C,F,F] (mapf_step_observe_bf16);
 *   MAPF_HOST_OBS_BITS: u32 [W,N,MAPF_OBS_BITS_WORDS(C,F)] (mapf_step_observe_bits, obs_dev 4-byte aligned).  Setting both
 *   is MAPF_E_BAD_CONFIG.
 * mapf_step_observe_host_begin: actions_host -> device (own copy stream, double-buffered), ONE fused step+observe launch
 * on `stream` writing obs_dev / vec_dev (and train_valid_dev if given) and the env's device slot, then ONE device-to-host
 * copy of the slot into result_slot_host on the copy stream (plus the train_valid / observation copies the flags ask for).  Returns without any host synchronisation: work queued on
 * `stream` afterwards (the policy forward) sees obs_dev / vec_dev of this step.  The env keeps two device slots, so two
 * begins may be in flight; result_slot_host must stay untouched until the matching wait.
 * mapf_step_observe_host_wait(env, age): block the host until the results of the most recent begin (age 0) or of the one
 * before it (age 1) have landed in their result_slot_host, the MAPF_HOST_TRAIN_VALID / MAPF_HOST_OBS copies included. */
#define MAPF_HOST_TRAIN_VALID 1
#define MAPF_HOST_COMPACT 2
#define MAPF_HOST_OBS_BF16 4
#define MAPF_HOST_OBS_BITS 8
#define MAPF_HOST_OBS 16
typedef struct MapfHostLayout {
    int64_t slot_bytes; /* bytes of one result slot for the flags passed to mapf_host_layout */
    int64_t off_reward, off_cost, off_shadow_goals, off_status, off_goals_reached, off_violated, off_fixed_actions,
        off_train_valid, off_packed; /* -1 when absent */
} MapfHostLayout;
int mapf_host_layout(MapfEnv *env, int flags, MapfHostLayout *out);
int mapf_step_observe_host_begin(MapfEnv *env, const int8_t *actions_host, void *result_slot_host, int flags,
                                 void *obs_dev, float *vec_dev, float *train_valid_dev, void *stream);
int mapf_step_observe_host_wait(MapfEnv *env, int age);

/* HOST function (no GPU work): expand n packed results (MapfStepOut.packed / a compact slot's `packed` field) into the
 * reference's per-agent arrays; any pointer of `out` may be NULL; out->train_valid / shadow_goals / good_actions are not
 * touched.  Bit-identical to the arrays the full format carries. */
int mapf_decode_results_host(const uint16_t *packed, int64_t n, const MapfStepOutHost *out);

/* HOST function (no GPU work): mapf_unpack_obs on host memory, for a CPU-side consumer of bit-packed observations (the
 * observation block of a MAPF_HOST_OBS | MAPF_HOST_OBS_BITS slot).  Same arguments, checks, bit order and results: out[r]
 * = the f32 / bf16 0/1 values [agents, C, F, F] of source row rows[r] (rows NULL: row r); a row index outside
 * [0, src_rows) gives an all-zero row. */
int mapf_unpack_obs_host(const uint32_t *obs_bits, int64_t src_rows, int32_t agents, int32_t num_channel, int32_t fov,
                         const int64_t *rows /* NULL = rows 0..n_rows-1 */, int64_t n_rows, int32_t out_bf16, void *out);

/* ---- learner-side glue: the elementwise part of the PPO-Lagrangian minibatch loss (SURVEY 8 f3) ----------------------- */

/* Replaces the ~40 eager tensor ops of Model.train between the network outputs and `loss.backward()` (model.py:104-164):
 * advantage normalisation, probability ratio, clipped surrogate, clipped value / cost-value losses, entropy, valid-action
 * loss, cost term.  Two calls per minibatch:
 *   mapf_adv_moments: per-block partial sums [MAPF_PPO_LOSS_MAX_BLOCKS, 4] (double) of a, a^2, c, c^2 with
 *       a = returns - old_v, c = cost_returns - old_cv (model.py:106-108); the caller adds the rows (and all-reduces them
 *       over ranks so that every rank normalises with the GLOBAL minibatch statistics, SURVEY 8e) and forms
 *       mean / unbiased std;
 *   mapf_ppo_loss: with those statistics, one pass over the n = rows x agents elements computing the gradients of
 *       loss = -policy_loss - entropy_coef*entropy + value_coef*critic + valid_coef*valid + cost_value_coef*cost_critic
 *              + cost_coef*lagrangian*cost_loss                                            (model.py:153-164)
 *       with respect to the network outputs (g_policy [n,5], g_value [n], g_cost_value [n], g_sig [n,5]; any may be NULL)
 *       and per-block partial sums [MAPF_PPO_LOSS_MAX_BLOCKS, MAPF_PPO_LOSS_STATS] (double):
 *       0 surrogate, 1 entropy, 2 critic, 3 cost critic, 4 valid log-likelihood (all 5 actions), 5 ratio*cadv, 6 clipped
 *       count, 7 advantage, 8 cost advantage.  Every mean is sum / n_global (a rank's share of the global minibatch).
 * All pointers are device pointers; asynchronous on `stream`; the current device is used. */
#define MAPF_PPO_LOSS_MAX_BLOCKS 1024
#define MAPF_PPO_LOSS_STATS 10
typedef struct MapfPpoLossConfig {
    float clip_range, entropy_coef, value_coef, valid_coef, cost_value_coef, cost_coef; /* TrainingParameters, alg_parameters.py:53-91 */
    float lagrangian;             /* current multiplier (lagrange.py) */
    int32_t minus_adv_with_cadv;  /* model.py:111-113 */
    double n_global;              /* elements (rows x agents) of the GLOBAL minibatch */
    double adv_mean, adv_std, cadv_mean, cadv_std; /* statistics of the global minibatch (unbiased std) */
} MapfPpoLossConfig;
int mapf_adv_moments(const float *returns, const float *cost_returns, const float *old_v, const float *old_cv, int64_t n,
                     double *partials, void *stream);
int mapf_ppo_loss(const MapfPpoLossConfig *cfg, int64_t n, const float *policy, const float *value, const float *cost_value,
                  const float *policy_sig, const float *returns, const float *cost_returns, const float *old_v,
                  const float *old_cv, const int8_t *actions, const float *old_ps, const float *train_valid, float *g_policy,
                  float *g_value, float *g_cost_value, float *g_sig, double *partials, void *stream);

/* ---- integrity helper ------------------------------------------------------------------------------------------------- */

/* 64-bit checksum of every row of a [rows, row_bytes] device array (row_bytes a multiple of 4, data 4-byte aligned):
 *   out[r] = sum over 32-bit words i of mix64((uint64(x[r,i]) + 1) * 0x9E3779B97F4A7C15 + i * 0xC2B2AE3D27D4EB4F)   (mod 2^64),
 *   mix64(z) = (z ^ (z >> 29)) * 0xBF58476D1CE4E5B9, then z ^ (z >> 32).
 * Order-independent sum of position-keyed terms, so a 4 GB observation tensor is verified against another implementation
 * (the reference's arrays, hashed the same way on the host) without moving it: compare W 64-bit values.  The reference
 * has no counterpart. */
int mapf_checksum_rows(const void *data, int64_t rows, int64_t row_bytes, uint64_t *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MAPF_B200_H */
