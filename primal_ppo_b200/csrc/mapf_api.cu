// mapf_api.cu — the C ABI declared in include/mapf_b200.h (handle, reset, argument checking, host-buffer calls).
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"

using namespace mapf;

// work counters (2 ints each) of the persistent kernels: one per kernel family, so that a launch that aborted, or two
// families in flight on different streams, can never hand a stale counter to another kernel
enum { WC_STEP = 0, WC_OBSERVE = 1, WC_FUSED = 2, WC_BFS = 3, WC_FUSED_WIDE = 4, WC_COUNT = 8 };
// ... followed by the walk-direction word shared by all world-claiming families (EnvView::order, common.cuh world_of)
constexpr size_t WORK_BYTES = (WC_COUNT * 2 + 1) * sizeof(int);

struct MapfEnv {
    MapfConfig cfg;
    EnvView v;
    bool has_scenario;
    // arrivals compaction scratch for mapf_bfs_refresh
    int32_t *d_list, *d_count;
    int *d_work;   // [WC_COUNT][2] dynamic-scheduling counters, then the walk direction
    // ---- staging of the *_host entry points (allocated by mapf_create) --------------------------------------------------
    // two result slots (layout: MapfHostLayout without train_valid) and two action buffers, used alternately
    unsigned char *d_slot[2];
    int8_t *d_actions[2];
    MapfHostLayout lay;                      // layout of a full slot (no train_valid)
    MapfHostLayout lay_c;                    // layout of a compact slot (packed + shadow goals), carved from the same memory
    cudaStream_t copy_stream, h2d_stream;
    cudaEvent_t ev_step[2], ev_copied[2], ev_h2d[2];
    bool tv_copy_pending[2];                 // that begin also copied the caller's trainValid tensor
    // device ranges [begin, end) of the caller's obs_dev / vec_dev that a MAPF_HOST_OBS begin of slot k copies to the host
    // (empty when it copied none); a later begin whose outputs overlap one of them waits for that copy
    uintptr_t obs_src[2][2], vec_src[2][2];
    int next_slot;                          // slot the next begin uses; the most recent begin used next_slot ^ 1
    int begun;                               // number of begins so far (saturating at 2)
};

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
static int cuda_fail(cudaError_t e, const char *what) {
    return fail(MAPF_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
#define CU(call)                                              \
    do {                                                      \
        cudaError_t e_ = (call);                              \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);   \
    } while (0)

// every part of a host result slot starts on a 256-byte boundary
static int64_t round256(size_t x) { return (int64_t)((x + 255) & ~(size_t)255); }

namespace mapf {
namespace {

// populateMap (mapf_gym.py:175-184) + packing of the obstacle map into a bit matrix. One warp per world.
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) reset_kernel(const EnvView v) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * WARPS_PER_BLOCK + warp;
    if (w >= v.W) return;
    const int rows = v.dims ? v.dims[2 * w] : v.H, cols = v.dims ? v.dims[2 * w + 1] : v.Wd;
    const uint8_t *ob = v.obst + (size_t)w * v.H * v.Wd;
    uint32_t *dst = v.obst_pack + (size_t)w * v.PW;
    const int cells = v.H * v.Wd;
    for (int k = lane; k < v.PW; k += 32) {
        uint32_t bits = 0;
        for (int b = 0; b < 32; ++b) {
            const int idx = k * 32 + b;
            const int r = idx / v.Wd, c = idx - r * v.Wd;
            const bool blocked = idx >= cells || r >= rows || c >= cols || ob[idx] != 0;
            bits |= (blocked ? 1u : 0u) << b;
        }
        dst[k] = bits;
    }
    for (int i = lane; i < v.N; i += 32) {
        const size_t idx = (size_t)w * v.N + i;
        reinterpret_cast<uint32_t *>(v.pos)[idx] = reinterpret_cast<const uint32_t *>(v.starts)[idx];
        reinterpret_cast<uint32_t *>(v.goal)[idx] = reinterpret_cast<const uint32_t *>(v.goal_queue)[idx * v.Q];
        v.qcur[idx] = 1;                       // Sequence.getNext consumed the first goal (util.py:33-39)
        v.rep[idx] = -1;                       // setPos clears the repetition list (mapf_gym.py:134-139)
    }
    if (lane == 0) {
        v.htick[w] = 0; v.tape_cur[w] = 0; v.nstep[w] = 0; v.err[w] = 0;
        reinterpret_cast<int2 *>(v.hcur)[w] = *reinterpret_cast<const int2 *>(v.htrace + (size_t)w * v.L * 4);
        const int t1 = (1 >= v.hlen[w]) ? 0 : 1;
        reinterpret_cast<int2 *>(v.hnx)[w] = *reinterpret_cast<const int2 *>(v.htrace + ((size_t)w * v.L + t1) * 4);
    }
    if (lane < 6) v.counters[(size_t)w * 6 + lane] = 0;
}

}  // namespace

cudaError_t launch_reset(const EnvView &v, cudaStream_t s) {
    const int blocks = (v.W + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    reset_kernel<<<blocks, WARPS_PER_BLOCK * 32, 0, s>>>(v);
    return cudaGetLastError();
}
}  // namespace mapf

// Every entry point runs on the env's device whatever the caller's current device is, and leaves the caller's current
// device as it found it (a process that drives several GPUs from one thread keeps its own notion of "current").
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) { err = cudaSetDevice(dev); switched = err == cudaSuccess; }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
#define ON_DEVICE(dev)                \
    DeviceGuard dev_guard_(dev);      \
    if (dev_guard_.err != cudaSuccess) return cuda_fail(dev_guard_.err, "cudaSetDevice")

extern "C" {

int mapf_abi_version(void) { return MAPF_B200_ABI_VERSION; }
const char *mapf_last_error(void) { return g_err; }

int mapf_create(const MapfConfig *cfg, MapfEnv **out) {
    if (!cfg || !out) return fail(MAPF_E_NULL, "mapf_create: null argument");
    *out = nullptr;
    const MapfConfig &c = *cfg;
    if (c.num_worlds < 1 || c.height < 1 || c.width < 1 || c.num_agents < 1)
        return fail(MAPF_E_BAD_CONFIG, "mapf_create: W, H, Wd, N must be >= 1");
    if (c.height > 128 || c.width > 128) return fail(MAPF_E_UNSUPPORTED, "mapf_create: H, Wd <= 128 supported");
    if (c.num_agents > 254) return fail(MAPF_E_UNSUPPORTED, "mapf_create: N <= 254 supported");
    if (c.fov < 3 || c.fov > 31 || (c.fov & 1) == 0) return fail(MAPF_E_BAD_CONFIG, "mapf_create: fov must be odd in 3..31");
    if (c.num_channel != 5 && c.num_channel != 6) return fail(MAPF_E_BAD_CONFIG, "mapf_create: num_channel must be 5 or 6");
    if (c.queue_len < 1 || c.trace_len < 1 || c.tape_stride < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_create: bad Q / L / TL");
    ON_DEVICE(c.device);
    MapfEnv *e = new (std::nothrow) MapfEnv();
    if (!e) return fail(MAPF_E_CUDA, "mapf_create: out of host memory");
    memset(e, 0, sizeof(*e));
    e->cfg = c;
    EnvView &v = e->v;
    v.W = c.num_worlds; v.H = c.height; v.Wd = c.width; v.N = c.num_agents; v.F = c.fov; v.C = c.num_channel;
    v.use_da = c.use_da; v.use_hp = c.use_hp; v.Q = c.queue_len; v.L = c.trace_len; v.TL = c.tape_stride;
    v.hp5_per_tick = c.hp5_per_tick; v.seed = c.seed; v.world_offset = c.world_offset;
    v.goal_sampling = c.goal_sampling ? 1 : 0;
    v.P = c.fov / 2 > 2 ? c.fov / 2 : 2;
    v.HP = v.H + 2 * v.P;
    v.RW = (v.Wd + 2 * v.P + 31) / 32 + 1;
    v.GS = ((v.Wd + 2 * v.P + 15) / 16) * 16;
    v.PW = (((v.H * v.Wd + 31) / 32) + 3) & ~3;
    const size_t W = v.W, WN = (size_t)v.W * v.N;
    cudaError_t err = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) { if (err == cudaSuccess) err = cudaMalloc(p, bytes ? bytes : 1); };
    alloc((void **)&v.obst_pack, W * v.PW * 4);
    alloc((void **)&v.pos, WN * 4);
    alloc((void **)&v.goal, WN * 4);
    alloc((void **)&v.rep, WN);
    alloc((void **)&v.qcur, WN * 4);
    alloc((void **)&v.htick, W * 4);
    alloc((void **)&v.tape_cur, W * 4);
    alloc((void **)&v.nstep, W * 4);
    alloc((void **)&v.err, W * 4);
    alloc((void **)&v.counters, W * 6 * 8);
    alloc((void **)&v.hcur, W * 8);
    alloc((void **)&v.hnx, W * 8);
    alloc((void **)&e->d_work, WORK_BYTES);
    alloc((void **)&e->d_list, WN * 4);
    alloc((void **)&e->d_count, 4);
    // result-slot layout: f32 fields first, then the byte fields; every field 256-byte aligned
    {
        MapfHostLayout &L = e->lay;
        int64_t o = 0;
        L.off_reward = o; o += round256(WN * 4);
        L.off_cost = o; o += round256(WN * 4);
        L.off_shadow_goals = o; o += round256(W * 4);
        L.off_status = o; o += round256(WN);
        L.off_goals_reached = o; o += round256(WN);
        L.off_violated = o; o += round256(WN);
        L.off_fixed_actions = o; o += round256(WN);
        L.off_train_valid = -1;
        L.off_packed = -1;
        L.slot_bytes = o;
        MapfHostLayout &Lc = e->lay_c;
        Lc.off_reward = Lc.off_cost = Lc.off_status = Lc.off_goals_reached = Lc.off_violated = Lc.off_fixed_actions = -1;
        Lc.off_train_valid = -1;
        Lc.off_packed = 0;
        Lc.off_shadow_goals = round256(WN * 2);
        Lc.slot_bytes = Lc.off_shadow_goals + round256(W * 4);
    }
    for (int k = 0; k < 2; ++k) {
        alloc((void **)&e->d_slot[k], (size_t)e->lay.slot_bytes);
        alloc((void **)&e->d_actions[k], WN);
    }
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->h2d_stream, cudaStreamNonBlocking);
    for (int k = 0; k < 2 && err == cudaSuccess; ++k) {
        err = cudaEventCreateWithFlags(&e->ev_step[k], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_copied[k], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_h2d[k], cudaEventDisableTiming);
    }
    if (err != cudaSuccess) { mapf_destroy(e); return cuda_fail(err, "mapf_create: allocation"); }
    cudaMemset(e->d_work, 0, WORK_BYTES);
    v.order = e->d_work + WC_COUNT * 2;
    if (const char *f = getenv("MAPF_DBG_FLAGS")) v.dbg_flags = atoi(f);
    *out = e;
    return MAPF_OK;
}

int mapf_destroy(MapfEnv *e) {
    if (!e) return MAPF_OK;
    EnvView &v = e->v;
    cudaFree(v.obst_pack); cudaFree(v.pos); cudaFree(v.goal); cudaFree(v.rep); cudaFree(v.qcur); cudaFree(v.htick);
    cudaFree(v.tape_cur); cudaFree(v.nstep); cudaFree(v.err); cudaFree(v.counters); cudaFree(v.hcur); cudaFree(v.hnx);
    cudaFree(e->d_work); cudaFree(e->d_list); cudaFree(e->d_count);
    for (int k = 0; k < 2; ++k) {
        cudaFree(e->d_slot[k]); cudaFree(e->d_actions[k]);
        if (e->ev_step[k]) cudaEventDestroy(e->ev_step[k]);
        if (e->ev_copied[k]) cudaEventDestroy(e->ev_copied[k]);
        if (e->ev_h2d[k]) cudaEventDestroy(e->ev_h2d[k]);
    }
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->h2d_stream) cudaStreamDestroy(e->h2d_stream);
    delete e;
    return MAPF_OK;
}

int mapf_reset(MapfEnv *e, const MapfScenario *sc, void *stream) {
    if (!e || !sc) return fail(MAPF_E_NULL, "mapf_reset: null argument");
    if (!sc->obst || !sc->starts || !sc->goal_queue || !sc->htrace || !sc->hlen)
        return fail(MAPF_E_NULL, "mapf_reset: obst, starts, goal_queue, htrace, hlen are required");
    if (e->cfg.tape_stride > 0 && (!sc->tape || !sc->tape_len)) return fail(MAPF_E_NULL, "mapf_reset: tape_stride > 0 needs tape and tape_len");
    if (e->cfg.use_hp && e->cfg.num_channel == 6 && !sc->hp5) return fail(MAPF_E_NULL, "mapf_reset: use_hp needs hp5");
    EnvView &v = e->v;
    v.obst = sc->obst; v.starts = sc->starts; v.goal_queue = sc->goal_queue; v.htrace = sc->htrace; v.hlen = sc->hlen;
    v.hp5 = sc->hp5; v.tape = sc->tape; v.tape_len = sc->tape_len; v.dims = sc->dims;
    ON_DEVICE(e->cfg.device);
    // re-arm every work counter: a launch that faulted or was aborted must not leave later launches without work
    CU(cudaMemsetAsync(e->d_work, 0, WORK_BYTES, (cudaStream_t)stream));
    CU(launch_reset(v, (cudaStream_t)stream));
    e->has_scenario = true;
    return MAPF_OK;
}

static int check_env(const MapfEnv *e, const char *name) {
    if (!e) return fail(MAPF_E_NULL, "%s: null env", name);
    if (!e->has_scenario) return fail(MAPF_E_STATE, "%s: mapf_reset has not been called", name);
    return MAPF_OK;
}
#define NEED_ENV(name)                                  \
    if (int rc_ = check_env(e, name)) return rc_;       \
    ON_DEVICE(e->cfg.device)
#define WC(e, k) ((e)->d_work + 2 * (k))

// vec is written with one 16-byte store per agent
static int check_vec(const float *vec, const char *name) {
    if (reinterpret_cast<uintptr_t>(vec) & 15) return fail(MAPF_E_BAD_CONFIG, "%s: vec must be 16-byte aligned", name);
    return MAPF_OK;
}
static int check_step_n(const MapfEnv *e, const char *name) {
    if (e->v.N > 128) return fail(MAPF_E_UNSUPPORTED, "%s: joint-step resolution supports N <= 128 agents per world (got %d)", name, e->v.N);
    return MAPF_OK;
}
// N <= 32: lane = agent (step.cu); 32 < N <= 128: lane loops over agents (step_wide.cu)
static cudaError_t do_step(MapfEnv *e, const int8_t *actions, const int8_t *status, const MapfStepOut &o, int mode, cudaStream_t s) {
    if (e->v.N <= 32) return launch_step(e->v, actions, status, o, mode, WC(e, WC_STEP), s);
    return launch_step_wide(e->v, actions, status, o, mode, s);
}

// One env step of the rollout loop: the warp-per-world fused kernel (N <= 32, one observation chunk), else the
// CTA-per-world fused kernel (N <= 128), else the two launches back to back.  MAPF_DBG_FLAGS bit 0 forces the two launches.
static cudaError_t do_step_observe(MapfEnv *e, const int8_t *actions, const MapfStepOut &o, float *obs, float *vec,
                                   cudaStream_t s, int fmt) {
    const EnvView &v = e->v;
    if (!(v.dbg_flags & 1)) {
        if (step_observe_fusable(v)) return launch_step_observe(v, actions, o, obs, vec, WC(e, WC_FUSED), s, fmt);
        if (step_observe_wide_fusable(v)) return launch_step_observe_wide(v, actions, o, obs, vec, WC(e, WC_FUSED_WIDE), s, fmt);
    }
    cudaError_t err = do_step(e, actions, nullptr, o, MODE_FUSED, s);
    if (err != cudaSuccess) return err;
    return launch_observe(v, obs, vec, WC(e, WC_OBSERVE), s, fmt);
}

int mapf_evaluate(MapfEnv *e, const int8_t *actions, const MapfStepOut *out, void *stream) {
    NEED_ENV("mapf_evaluate");
    if (!actions || !out) return fail(MAPF_E_NULL, "mapf_evaluate: null argument");
    if (int rc = check_step_n(e, "mapf_evaluate")) return rc;
    CU(do_step(e, actions, nullptr, *out, MODE_EVALUATE, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_joint_step(MapfEnv *e, const int8_t *actions, const int8_t *status, uint8_t *goals_reached, uint8_t *violated,
                    int8_t *fixed_actions, void *stream) {
    NEED_ENV("mapf_joint_step");
    if (!actions || !status) return fail(MAPF_E_NULL, "mapf_joint_step: null argument");
    if (int rc = check_step_n(e, "mapf_joint_step")) return rc;
    MapfStepOut o;
    memset(&o, 0, sizeof(o));
    o.goals_reached = goals_reached; o.violated = violated; o.fixed_actions = fixed_actions;
    CU(do_step(e, actions, status, o, MODE_JOINT, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_step(MapfEnv *e, const int8_t *actions, const MapfStepOut *out, void *stream) {
    NEED_ENV("mapf_step");
    if (!actions || !out) return fail(MAPF_E_NULL, "mapf_step: null argument");
    if (int rc = check_step_n(e, "mapf_step")) return rc;
    CU(do_step(e, actions, nullptr, *out, MODE_FUSED, (cudaStream_t)stream));
    return MAPF_OK;
}

/* bit-packed output: one bit per observation cell, u32 [W,N,MAPF_OBS_BITS_WORDS(C,F)] */
static int check_bits(const uint32_t *obs_bits, const char *name) {
    if (reinterpret_cast<uintptr_t>(obs_bits) & 3) return fail(MAPF_E_BAD_CONFIG, "%s: obs_bits must be 4-byte aligned", name);
    return MAPF_OK;
}

// The observation entry points in format `fmt`: mapf_observe* (step = false; actions and out are not used) and
// mapf_step_observe*.
static int observe_call(const char *name, MapfEnv *e, bool step, const int8_t *actions, const MapfStepOut *out, void *obs,
                        float *vec, void *stream, int fmt) {
    NEED_ENV(name);
    if (!obs || !vec || (step && (!actions || !out))) return fail(MAPF_E_NULL, "%s: null argument", name);
    if (int rc = check_vec(vec, name)) return rc;
    if (fmt == OBS_BITS)
        if (int rc = check_bits(static_cast<const uint32_t *>(obs), name)) return rc;
    if (step) {
        if (int rc = check_step_n(e, name)) return rc;
        CU(do_step_observe(e, actions, *out, static_cast<float *>(obs), vec, (cudaStream_t)stream, fmt));
    } else {
        CU(launch_observe(e->v, static_cast<float *>(obs), vec, WC(e, WC_OBSERVE), (cudaStream_t)stream, fmt));
    }
    return MAPF_OK;
}

int mapf_observe(MapfEnv *e, float *obs, float *vec, void *stream) {
    return observe_call("mapf_observe", e, false, nullptr, nullptr, obs, vec, stream, OBS_F32);
}

int mapf_step_observe(MapfEnv *e, const int8_t *actions, const MapfStepOut *out, float *obs, float *vec, void *stream) {
    return observe_call("mapf_step_observe", e, true, actions, out, obs, vec, stream, OBS_F32);
}

/* bf16 variants: the same 0/1 observation values, half the bytes (optional format for GPU-resident training) */
int mapf_observe_bf16(MapfEnv *e, uint16_t *obs_bf16, float *vec, void *stream) {
    return observe_call("mapf_observe_bf16", e, false, nullptr, nullptr, obs_bf16, vec, stream, OBS_BF16);
}

int mapf_step_observe_bf16(MapfEnv *e, const int8_t *actions, const MapfStepOut *out, uint16_t *obs_bf16, float *vec, void *stream) {
    return observe_call("mapf_step_observe_bf16", e, true, actions, out, obs_bf16, vec, stream, OBS_BF16);
}

int mapf_observe_bits(MapfEnv *e, uint32_t *obs_bits, float *vec, void *stream) {
    return observe_call("mapf_observe_bits", e, false, nullptr, nullptr, obs_bits, vec, stream, OBS_BITS);
}

int mapf_step_observe_bits(MapfEnv *e, const int8_t *actions, const MapfStepOut *out, uint32_t *obs_bits, float *vec,
                           void *stream) {
    return observe_call("mapf_step_observe_bits", e, true, actions, out, obs_bits, vec, stream, OBS_BITS);
}

// argument checks shared by mapf_unpack_obs and mapf_unpack_obs_host
static int check_unpack(const char *name, const uint32_t *obs_bits, int64_t src_rows, int32_t agents, int32_t num_channel,
                        int32_t fov, int64_t n_rows, int32_t out_bf16, const void *out) {
    if (!obs_bits || !out) return fail(MAPF_E_NULL, "%s: null argument", name);
    if (src_rows < 0 || n_rows < 0) return fail(MAPF_E_BAD_CONFIG, "%s: negative row count", name);
    if (agents < 1 || agents > 254) return fail(MAPF_E_BAD_CONFIG, "%s: agents must be in 1..254", name);
    if (num_channel != 5 && num_channel != 6) return fail(MAPF_E_BAD_CONFIG, "%s: num_channel must be 5 or 6", name);
    if (fov < 3 || fov > 31 || (fov & 1) == 0) return fail(MAPF_E_BAD_CONFIG, "%s: fov must be odd in 3..31", name);
    if (out_bf16 != 0 && out_bf16 != 1) return fail(MAPF_E_BAD_CONFIG, "%s: out_bf16 must be 0 or 1", name);
    if (int rc = check_bits(obs_bits, name)) return rc;
    if (reinterpret_cast<uintptr_t>(out) & (out_bf16 ? 1 : 3))
        return fail(MAPF_E_BAD_CONFIG, "%s: out must be aligned to its element size", name);
    return MAPF_OK;
}

int mapf_unpack_obs(const uint32_t *obs_bits, int64_t src_rows, int32_t agents, int32_t num_channel, int32_t fov,
                    const int64_t *rows, int64_t n_rows, int32_t out_bf16, void *out, void *stream) {
    if (int rc = check_unpack("mapf_unpack_obs", obs_bits, src_rows, agents, num_channel, fov, n_rows, out_bf16, out)) return rc;
    if (n_rows == 0) return MAPF_OK;
    CU(launch_unpack_obs(obs_bits, src_rows, agents, num_channel, fov, rows, n_rows, out_bf16, out, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_bfs(MapfEnv *e, const int32_t *agent_list, int64_t n, int16_t *out, void *stream) {
    NEED_ENV("mapf_bfs");
    if (!out) return fail(MAPF_E_NULL, "mapf_bfs: null out");
    if (!agent_list) n = (int64_t)e->v.W * e->v.N;
    if (n < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_bfs: n < 0");
    if (n == 0) return MAPF_OK;
    CU(launch_bfs(e->v, agent_list, n, nullptr, out, 0, WC(e, WC_BFS), (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_bfs_refresh(MapfEnv *e, const uint8_t *goals_reached, int16_t *bfs_maps, void *stream) {
    NEED_ENV("mapf_bfs_refresh");
    if (!goals_reached || !bfs_maps) return fail(MAPF_E_NULL, "mapf_bfs_refresh: null argument");
    CU(launch_arrivals(e->v, goals_reached, e->d_list, e->d_count, (cudaStream_t)stream));
    CU(launch_bfs(e->v, e->d_list, (long long)e->v.W * e->v.N, e->d_count, bfs_maps, 1, WC(e, WC_BFS), (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_gae(const float *r, const float *v, const float *last_v, const uint8_t *nonterminal, double gamma, double lam,
             int32_t T, int64_t cols, float *returns, float *adv, void *stream) {
    if (!r || !v || !last_v || !returns) return fail(MAPF_E_NULL, "mapf_gae: null argument");
    if (T < 0 || cols < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_gae: negative size");
    // runner.py:138-143: GAMMA * next_nonterminal and GAMMA * LAM * next_nonterminal are Python doubles that NumPy
    // applies to f32 arrays as f32 scalars.
    const float g = (float)(gamma * 1.0), gl = (float)(gamma * lam * 1.0);
    CU(launch_gae(r, v, last_v, nonterminal, g, gl, T, cols, returns, adv, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_gae2(const float *r, const float *v, const float *last_v, const float *cr, const float *cv, const float *last_cv,
              const uint8_t *nonterminal, double gamma, double lam, int32_t T, int64_t cols, float *returns, float *cost_returns,
              float *adv, float *cost_adv, void *stream) {
    if (!r || !v || !last_v || !returns || !cr || !cv || !last_cv || !cost_returns) return fail(MAPF_E_NULL, "mapf_gae2: null argument");
    if (T < 0 || cols < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_gae2: negative size");
    const float g = (float)(gamma * 1.0), gl = (float)(gamma * lam * 1.0);
    CU(launch_gae2(r, v, last_v, cr, cv, last_cv, nonterminal, g, gl, T, cols, returns, cost_returns, adv, cost_adv, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_adv_moments(const float *returns, const float *cost_returns, const float *old_v, const float *old_cv, int64_t n,
                     double *partials, void *stream) {
    if (!returns || !cost_returns || !old_v || !old_cv || !partials) return fail(MAPF_E_NULL, "mapf_adv_moments: null argument");
    if (n < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_adv_moments: n < 0");
    CU(launch_adv_moments(returns, cost_returns, old_v, old_cv, n, partials, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_ppo_loss(const MapfPpoLossConfig *cfg, int64_t n, const float *policy, const float *value, const float *cost_value,
                  const float *policy_sig, const float *returns, const float *cost_returns, const float *old_v,
                  const float *old_cv, const int8_t *actions, const float *old_ps, const float *train_valid, float *g_policy,
                  float *g_value, float *g_cost_value, float *g_sig, double *partials, void *stream) {
    if (!cfg || !policy || !value || !cost_value || !policy_sig || !returns || !cost_returns || !old_v || !old_cv || !actions ||
        !old_ps || !train_valid || !partials)
        return fail(MAPF_E_NULL, "mapf_ppo_loss: null argument");
    if (n < 0 || !(cfg->n_global > 0)) return fail(MAPF_E_BAD_CONFIG, "mapf_ppo_loss: n >= 0 and n_global > 0 required");
    CU(launch_ppo_loss(*cfg, n, policy, value, cost_value, policy_sig, returns, cost_returns, old_v, old_cv, actions, old_ps,
                       train_valid, g_policy, g_value, g_cost_value, g_sig, partials, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_sample_actions(const float *ps, int64_t rows, uint64_t seed, uint32_t draw, int8_t *actions, float *chosen_p,
                        void *stream) {
    if (!ps || !actions) return fail(MAPF_E_NULL, "mapf_sample_actions: null argument");
    if (rows < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_sample_actions: rows < 0");
    CU(launch_sample_actions(ps, rows, seed, draw, actions, chosen_p, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_generate_scenario(const MapfGenConfig *c, uint8_t *obst, int16_t *dims, int16_t *starts, int16_t *goal_queue,
                           int16_t *htrace, int32_t *hlen, int16_t *hp5, uint32_t *gen_err, void *stream) {
    if (!c || !obst || !dims || !starts || !goal_queue || !htrace || !hlen)
        return fail(MAPF_E_NULL, "mapf_generate_scenario: null argument");
    if (c->num_worlds < 1 || c->height < 2 || c->width < 2 || c->num_agents < 1 || c->queue_len < 1 || c->trace_len < 1)
        return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: bad sizes");
    if (c->height > 128 || c->width > 128) return fail(MAPF_E_UNSUPPORTED, "mapf_generate_scenario: H, Wd <= 128 supported");
    if (c->kind == 1) {
        if (c->size_lo < 4 || c->size_hi < c->size_lo) return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: warehouse needs 4 <= size_lo <= size_hi");
        if (c->size_hi > c->height || (int)((double)c->size_hi / (2.0 / 3.0)) > c->width)
            return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: warehouse of length %d needs height >= %d and width >= %d",
                        c->size_hi, c->size_hi, (int)((double)c->size_hi / (2.0 / 3.0)));
    } else if (c->kind == 0) {
        if (c->density_lo < 0.f || c->density_hi < c->density_lo || c->density_hi >= 1.f)
            return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: need 0 <= density_lo <= density_hi < 1");
        if (c->size_lo > 0 && (c->size_hi < c->size_lo || c->size_hi > c->height || c->size_hi > c->width))
            return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: size range does not fit height x width");
    } else return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: kind must be 0 (density) or 1 (warehouse)");
    if (c->human_path != 0 && c->human_path != 1)
        return fail(MAPF_E_BAD_CONFIG, "mapf_generate_scenario: human_path must be 0 (BFS descent) or 1 (astar_4)");
    ON_DEVICE(c->device);
    CU(launch_scenario_gen(*c, obst, dims, starts, goal_queue, htrace, hlen, hp5, gen_err, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_astar4_paths(const uint8_t *obst, int64_t n, int32_t H, int32_t Wd, const int16_t *start_goal, int32_t max_len,
                      int16_t *paths, int32_t *lens, void *stream) {
    if (!obst || !start_goal || !paths || !lens) return fail(MAPF_E_NULL, "mapf_astar4_paths: null argument");
    if (n < 0 || H < 1 || H > 128 || Wd < 1 || Wd > 128 || max_len < 1)
        return fail(MAPF_E_BAD_CONFIG, "mapf_astar4_paths: need n >= 0, 1 <= H, Wd <= 128 and max_len >= 1");
    CU(launch_astar4_paths(obst, n, H, Wd, start_goal, max_len, paths, lens, (cudaStream_t)stream));
    return MAPF_OK;
}

int mapf_get_state(MapfEnv *e, int16_t *pos, int16_t *goal, int8_t *rep, uint32_t *err, void *stream) {
    if (!e) return fail(MAPF_E_NULL, "mapf_get_state: null env");
    ON_DEVICE(e->cfg.device);
    const size_t WN = (size_t)e->v.W * e->v.N;
    cudaStream_t s = (cudaStream_t)stream;
    if (pos) CU(cudaMemcpyAsync(pos, e->v.pos, WN * 4, cudaMemcpyDeviceToDevice, s));
    if (goal) CU(cudaMemcpyAsync(goal, e->v.goal, WN * 4, cudaMemcpyDeviceToDevice, s));
    if (rep) CU(cudaMemcpyAsync(rep, e->v.rep, WN, cudaMemcpyDeviceToDevice, s));
    if (err) CU(cudaMemcpyAsync(err, e->v.err, (size_t)e->v.W * 4, cudaMemcpyDeviceToDevice, s));
    return MAPF_OK;
}

int mapf_get_human(MapfEnv *e, int16_t *pos_next, int32_t *tick, void *stream) {
    NEED_ENV("mapf_get_human");
    cudaStream_t s = (cudaStream_t)stream;
    if (pos_next) CU(cudaMemcpyAsync(pos_next, e->v.hcur, (size_t)e->v.W * 8, cudaMemcpyDeviceToDevice, s));
    if (tick) CU(cudaMemcpyAsync(tick, e->v.htick, (size_t)e->v.W * 4, cudaMemcpyDeviceToDevice, s));
    return MAPF_OK;
}

// ---- checkpoint / resume of the env's mutable state ------------------------------------------------------------------
namespace {
struct StatePiece { void *p; size_t bytes; };
// every buffer step / reset mutate, in a fixed order; sizes are rounded up to 16 bytes inside the blob
int state_pieces(MapfEnv *e, StatePiece *out) {
    EnvView &v = e->v;
    const size_t W = v.W, WN = (size_t)v.W * v.N;
    int n = 0;
    out[n++] = {v.pos, WN * 4}; out[n++] = {v.goal, WN * 4}; out[n++] = {v.rep, WN}; out[n++] = {v.qcur, WN * 4};
    out[n++] = {v.htick, W * 4}; out[n++] = {v.tape_cur, W * 4}; out[n++] = {v.nstep, W * 4}; out[n++] = {v.err, W * 4};
    out[n++] = {v.counters, W * 48}; out[n++] = {v.hcur, W * 8}; out[n++] = {v.hnx, W * 8};
    return n;
}
}  // namespace

int64_t mapf_state_bytes(MapfEnv *e) {
    if (!e) return fail(MAPF_E_NULL, "mapf_state_bytes: null env");
    StatePiece pc[16];
    const int n = state_pieces(e, pc);
    size_t total = 0;
    for (int i = 0; i < n; ++i) total += (pc[i].bytes + 15) & ~(size_t)15;
    return (int64_t)total;
}

int mapf_save_state(MapfEnv *e, void *blob, void *stream) {
    NEED_ENV("mapf_save_state");
    if (!blob) return fail(MAPF_E_NULL, "mapf_save_state: null blob");
    StatePiece pc[16];
    const int n = state_pieces(e, pc);
    char *dst = static_cast<char *>(blob);
    for (int i = 0; i < n; ++i) {
        CU(cudaMemcpyAsync(dst, pc[i].p, pc[i].bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        dst += (pc[i].bytes + 15) & ~(size_t)15;
    }
    return MAPF_OK;
}

int mapf_load_state(MapfEnv *e, const void *blob, void *stream) {
    NEED_ENV("mapf_load_state");
    if (!blob) return fail(MAPF_E_NULL, "mapf_load_state: null blob");
    StatePiece pc[16];
    const int n = state_pieces(e, pc);
    const char *src = static_cast<const char *>(blob);
    for (int i = 0; i < n; ++i) {
        CU(cudaMemcpyAsync(pc[i].p, src, pc[i].bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        src += (pc[i].bytes + 15) & ~(size_t)15;
    }
    return MAPF_OK;
}

int mapf_get_counters(MapfEnv *e, int64_t *counters, void *stream) {
    if (!e || !counters) return fail(MAPF_E_NULL, "mapf_get_counters: null argument");
    ON_DEVICE(e->cfg.device);
    CU(cudaMemcpyAsync(counters, e->v.counters, (size_t)e->v.W * 6 * 8, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return MAPF_OK;
}

// ---- host-buffer entry points ---------------------------------------------------------------------------------------
namespace {

MapfStepOut slot_ptrs(const MapfEnv *e, int k) {
    unsigned char *b = e->d_slot[k];
    const MapfHostLayout &L = e->lay;
    MapfStepOut o;
    memset(&o, 0, sizeof(o));
    o.reward = reinterpret_cast<float *>(b + L.off_reward);
    o.cost = reinterpret_cast<float *>(b + L.off_cost);
    o.shadow_goals = reinterpret_cast<int32_t *>(b + L.off_shadow_goals);
    o.status = reinterpret_cast<int8_t *>(b + L.off_status);
    o.goals_reached = b + L.off_goals_reached;
    o.violated = b + L.off_violated;
    o.fixed_actions = reinterpret_cast<int8_t *>(b + L.off_fixed_actions);
    return o;
}

// Queue the joint action's host-to-device copy for slot k on the env's h2d stream and make `s` wait for it.  The buffer
// d_actions[k] was last read by the kernels of the begin two calls ago (ev_step[k]); the copy may therefore overlap the
// kernels of the previous begin.
int queue_actions(MapfEnv *e, int k, const int8_t *actions_host, cudaStream_t s) {
    const size_t WN = (size_t)e->v.W * e->v.N;
    if (e->begun >= 2) CU(cudaStreamWaitEvent(e->h2d_stream, e->ev_step[k], 0));
    else CU(cudaStreamWaitEvent(e->h2d_stream, e->ev_step[k ^ 1], 0));     // (first calls: order behind whatever ran last)
    CU(cudaMemcpyAsync(e->d_actions[k], actions_host, WN, cudaMemcpyHostToDevice, e->h2d_stream));
    CU(cudaEventRecord(e->ev_h2d[k], e->h2d_stream));
    CU(cudaStreamWaitEvent(s, e->ev_h2d[k], 0));
    // the device slot k is overwritten by this step: its previous contents must have left for the host
    if (e->begun >= 2) CU(cudaStreamWaitEvent(s, e->ev_copied[k], 0));
    // a trainValid copy of the previous begin reads the caller's tensor that this step may overwrite
    if (e->begun >= 1 && e->tv_copy_pending[k ^ 1]) CU(cudaStreamWaitEvent(s, e->ev_copied[k ^ 1], 0));
    return MAPF_OK;
}

// The observation format obs_dev is written in, from the flags of the split-phase call; -1 when both format flags are set.
int host_obs_format(int flags) {
    const bool bf16 = flags & MAPF_HOST_OBS_BF16, bits = flags & MAPF_HOST_OBS_BITS;
    if (bf16 && bits) return -1;
    return bits ? OBS_BITS : bf16 ? OBS_BF16 : OBS_F32;
}

size_t obs_bytes(const EnvView &v, int fmt) {
    const size_t WN = (size_t)v.W * v.N, PB = (size_t)v.C * v.F * v.F;
    return fmt == OBS_BITS ? WN * MAPF_OBS_BITS_WORDS(v.C, v.F) * 4 : WN * PB * (fmt == OBS_BF16 ? 2 : 4);
}

bool overlaps(uintptr_t lo, uintptr_t hi, const uintptr_t r[2]) { return lo < r[1] && r[0] < hi; }

// The host result slot of the split-phase call for `flags`: the device slot (full or compact), then trainValid
// (MAPF_HOST_TRAIN_VALID), then the observations in format `fmt` and vec (MAPF_HOST_OBS).  off_obs / off_vec are where
// the last two start.
struct HostSlot {
    MapfHostLayout lay;
    int64_t off_obs, off_vec;
};
HostSlot host_slot(const MapfEnv *e, int flags, int fmt) {
    const size_t WN = (size_t)e->v.W * e->v.N;
    HostSlot h;
    h.lay = (flags & MAPF_HOST_COMPACT) ? e->lay_c : e->lay;
    if (flags & MAPF_HOST_TRAIN_VALID) {
        h.lay.off_train_valid = h.lay.slot_bytes;
        h.lay.slot_bytes += round256(WN * NA * 4);
    }
    h.off_obs = h.lay.slot_bytes;
    h.off_vec = h.off_obs + round256(obs_bytes(e->v, fmt));
    if (flags & MAPF_HOST_OBS) h.lay.slot_bytes = h.off_vec + round256(WN * 16);
    return h;
}

}  // namespace

int mapf_host_layout(MapfEnv *e, int flags, MapfHostLayout *out) {
    if (!e || !out) return fail(MAPF_E_NULL, "mapf_host_layout: null argument");
    const int fmt = host_obs_format(flags);
    if (fmt < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_host_layout: MAPF_HOST_OBS_BF16 and MAPF_HOST_OBS_BITS are exclusive");
    *out = host_slot(e, flags, fmt).lay;
    return MAPF_OK;
}

int mapf_step_observe_host_begin(MapfEnv *e, const int8_t *actions_host, void *result_slot_host, int flags,
                                 void *obs_dev, float *vec_dev, float *train_valid_dev, void *stream) {
    NEED_ENV("mapf_step_observe_host_begin");
    if (int rc = check_vec(vec_dev, "mapf_step_observe_host_begin")) return rc;
    if (!actions_host || !result_slot_host || !obs_dev || !vec_dev) return fail(MAPF_E_NULL, "mapf_step_observe_host_begin: null argument");
    const bool with_tv = flags & MAPF_HOST_TRAIN_VALID, compact = flags & MAPF_HOST_COMPACT, with_obs = flags & MAPF_HOST_OBS;
    if (with_tv && !train_valid_dev) return fail(MAPF_E_NULL, "mapf_step_observe_host_begin: MAPF_HOST_TRAIN_VALID needs train_valid_dev");
    const int fmt = host_obs_format(flags);
    if (fmt < 0)
        return fail(MAPF_E_BAD_CONFIG, "mapf_step_observe_host_begin: MAPF_HOST_OBS_BF16 and MAPF_HOST_OBS_BITS are exclusive");
    if (fmt == OBS_BITS)
        if (int rc = check_bits(static_cast<const uint32_t *>(obs_dev), "mapf_step_observe_host_begin")) return rc;
    if (int rc = check_step_n(e, "mapf_step_observe_host_begin")) return rc;
    const EnvView &v = e->v;
    const size_t WN = (size_t)v.W * v.N, n_obs = obs_bytes(v, fmt);
    cudaStream_t s = (cudaStream_t)stream, cs = e->copy_stream;
    const int k = e->next_slot;
    if (int rc = queue_actions(e, k, actions_host, s)) return rc;
    // The observation copies of the previous begin read the caller's obs_dev / vec_dev while this step runs.  Only a step
    // that writes into one of those ranges waits for them (the copies of the begin before that were awaited by
    // queue_actions): a rollout that gives every step its own buffers keeps two steps overlapped.
    if (e->begun >= 1) {
        const uintptr_t ob = reinterpret_cast<uintptr_t>(obs_dev), vc = reinterpret_cast<uintptr_t>(vec_dev),
                        tv = reinterpret_cast<uintptr_t>(train_valid_dev);
        const uintptr_t *po = e->obs_src[k ^ 1], *pv = e->vec_src[k ^ 1];
        bool hit = overlaps(ob, ob + n_obs, po) || overlaps(ob, ob + n_obs, pv) || overlaps(vc, vc + WN * 16, po) ||
                   overlaps(vc, vc + WN * 16, pv);
        if (train_valid_dev) hit = hit || overlaps(tv, tv + WN * NA * 4, po) || overlaps(tv, tv + WN * NA * 4, pv);
        if (hit) CU(cudaStreamWaitEvent(s, e->ev_copied[k ^ 1], 0));
    }
    MapfStepOut o;
    size_t slot_bytes;
    if (compact) {
        memset(&o, 0, sizeof(o));
        o.packed = reinterpret_cast<uint16_t *>(e->d_slot[k] + e->lay_c.off_packed);
        o.shadow_goals = reinterpret_cast<int32_t *>(e->d_slot[k] + e->lay_c.off_shadow_goals);
        slot_bytes = (size_t)e->lay_c.slot_bytes;
    } else {
        o = slot_ptrs(e, k);
        slot_bytes = (size_t)e->lay.slot_bytes;
    }
    o.train_valid = train_valid_dev;
    CU(do_step_observe(e, e->d_actions[k], o, static_cast<float *>(obs_dev), vec_dev, s, fmt));
    CU(cudaEventRecord(e->ev_step[k], s));
    CU(cudaStreamWaitEvent(cs, e->ev_step[k], 0));
    char *const host = static_cast<char *>(result_slot_host);
    const HostSlot h = host_slot(e, flags, fmt);
    CU(cudaMemcpyAsync(host, e->d_slot[k], slot_bytes, cudaMemcpyDeviceToHost, cs));   // ONE copy
    if (with_tv) CU(cudaMemcpyAsync(host + h.lay.off_train_valid, train_valid_dev, WN * NA * 4, cudaMemcpyDeviceToHost, cs));
    const uintptr_t ob = reinterpret_cast<uintptr_t>(obs_dev), vc = reinterpret_cast<uintptr_t>(vec_dev);
    if (with_obs) {
        CU(cudaMemcpyAsync(host + h.off_obs, obs_dev, n_obs, cudaMemcpyDeviceToHost, cs));
        CU(cudaMemcpyAsync(host + h.off_vec, vec_dev, WN * 16, cudaMemcpyDeviceToHost, cs));
    }
    CU(cudaEventRecord(e->ev_copied[k], cs));
    e->tv_copy_pending[k] = with_tv;
    e->obs_src[k][0] = with_obs ? ob : 0; e->obs_src[k][1] = with_obs ? ob + n_obs : 0;
    e->vec_src[k][0] = with_obs ? vc : 0; e->vec_src[k][1] = with_obs ? vc + WN * 16 : 0;
    e->next_slot = k ^ 1;
    if (e->begun < 2) e->begun++;
    return MAPF_OK;
}

int mapf_decode_results_host(const uint16_t *packed, int64_t n, const MapfStepOutHost *out) {
    if (!packed || !out) return fail(MAPF_E_NULL, "mapf_decode_results_host: null argument");
    if (n < 0) return fail(MAPF_E_BAD_CONFIG, "mapf_decode_results_host: n < 0");
    static const int8_t status_of[8] = {-1, -2, -3, -4, 1, 1, 1, 1};
    static const float base_reward[8] = {-2.0f, -2.0f, -2.0f, -0.35f, -0.3f, -0.3f, -0.3f, -0.3f};   // alg_parameters.py:36-43
    float reward_lut[16], cost_lut[32];
    for (int k = 0; k < 16; ++k) reward_lut[k] = (k & 8) ? base_reward[k & 7] + 1.5f : base_reward[k & 7];   // runner.py:89-91
    for (int d2 = 0; d2 < 32; ++d2) cost_lut[d2] = d2 < 25 ? (float)((5.0 - sqrt((double)d2)) / 5.0) : 0.0f;  // mapf_gym.py:513-533
    for (int64_t i = 0; i < n; ++i) {
        const unsigned p = packed[i];
        if (out->status) out->status[i] = status_of[p & 7u];
        if (out->reward) out->reward[i] = reward_lut[p & 15u];
        if (out->cost) out->cost[i] = cost_lut[(p >> 8) & 31u];
        if (out->goals_reached) out->goals_reached[i] = (uint8_t)((p >> 3) & 1u);
        if (out->violated) out->violated[i] = (uint8_t)((p >> 4) & 1u);
        if (out->fixed_actions) out->fixed_actions[i] = (int8_t)((p >> 5) & 7u);
    }
    return MAPF_OK;
}

int mapf_unpack_obs_host(const uint32_t *obs_bits, int64_t src_rows, int32_t agents, int32_t num_channel, int32_t fov,
                         const int64_t *rows, int64_t n_rows, int32_t out_bf16, void *out) {
    if (int rc = check_unpack("mapf_unpack_obs_host", obs_bits, src_rows, agents, num_channel, fov, n_rows, out_bf16, out))
        return rc;
    // byte -> its eight 0/1 values, LSB first: one table lookup and copy per 8 cells
    static const struct Lut {
        float f[256][8];
        uint16_t h[256][8];
        Lut() {
            for (int b = 0; b < 256; ++b)
                for (int i = 0; i < 8; ++i) { f[b][i] = (b >> i) & 1 ? 1.0f : 0.0f; h[b][i] = (b >> i) & 1 ? 0x3f80 : 0; }
        }
    } lut;
    const int PB = num_channel * fov * fov, AW = MAPF_OBS_BITS_WORDS(num_channel, fov);
    const size_t esz = out_bf16 ? 2 : 4, row_out = (size_t)agents * PB * esz;
    for (int64_t r = 0; r < n_rows; ++r) {
        const int64_t s = rows ? rows[r] : r;
        char *dst = static_cast<char *>(out) + (size_t)r * row_out;
        if (s < 0 || s >= src_rows) { memset(dst, 0, row_out); continue; }
        const uint32_t *src = obs_bits + (size_t)s * agents * AW;
        for (int a = 0; a < agents; ++a, src += AW, dst += (size_t)PB * esz)
            for (int c = 0; c < PB; c += 8) {
                const unsigned byte = (src[c >> 5] >> (c & 31)) & 0xffu;
                const int n = PB - c < 8 ? PB - c : 8;
                memcpy(dst + c * esz, out_bf16 ? (const void *)lut.h[byte] : (const void *)lut.f[byte], n * esz);
            }
    }
    return MAPF_OK;
}

int mapf_step_observe_host_wait(MapfEnv *e, int age) {
    if (!e) return fail(MAPF_E_NULL, "mapf_step_observe_host_wait: null env");
    if (age < 0 || age > 1) return fail(MAPF_E_BAD_CONFIG, "mapf_step_observe_host_wait: age must be 0 or 1");
    if (e->begun <= age) return fail(MAPF_E_STATE, "mapf_step_observe_host_wait: no such begin in flight");
    const int k = (e->next_slot ^ 1) ^ age;
    CU(cudaEventSynchronize(e->ev_copied[k]));
    return MAPF_OK;
}

int mapf_step_observe_host(MapfEnv *e, const int8_t *actions_host, const MapfStepOutHost *out, float *obs_dev,
                           float *vec_dev, float *train_valid_dev, float *obs_host, float *vec_host, void *stream) {
    NEED_ENV("mapf_step_observe_host");
    if (int rc = check_vec(vec_dev, "mapf_step_observe_host")) return rc;
    if (!actions_host || !out || !obs_dev || !vec_dev) return fail(MAPF_E_NULL, "mapf_step_observe_host: null argument");
    if (out->train_valid && !train_valid_dev) return fail(MAPF_E_NULL, "mapf_step_observe_host: out->train_valid needs train_valid_dev");
    if (int rc = check_step_n(e, "mapf_step_observe_host")) return rc;
    const EnvView &v = e->v;
    const size_t W = v.W, WN = (size_t)v.W * v.N;
    cudaStream_t s = (cudaStream_t)stream, cs = e->copy_stream;
    const int k = e->next_slot;
    if (int rc = queue_actions(e, k, actions_host, s)) return rc;
    MapfStepOut o = slot_ptrs(e, k);                            // only compute what the caller asked for
    if (!out->status) o.status = nullptr;
    if (!out->reward) o.reward = nullptr;
    if (!out->cost) o.cost = nullptr;
    o.train_valid = train_valid_dev;
    if (!out->goals_reached) o.goals_reached = nullptr;
    if (!out->violated) o.violated = nullptr;
    if (!out->shadow_goals) o.shadow_goals = nullptr;
    if (!out->fixed_actions) o.fixed_actions = nullptr;
    // Synchronous form: the caller blocks until the results are on the host, so the copy has to hide inside this call.
    // The per-agent results are final once step_kernel has run: they travel on the copy stream while observe_kernel
    // writes the observations (measured at 65 536 x 32 agents: this split 0.97 ms per call; the fused kernel followed by
    // the copies 1.33 ms, the copy being exposed).  The split-phase form above uses the fused launch instead and hides the
    // copy behind the NEXT step.
    CU(do_step(e, e->d_actions[k], nullptr, o, MODE_FUSED, s));
    CU(cudaEventRecord(e->ev_step[k], s));
    CU(cudaStreamWaitEvent(cs, e->ev_step[k], 0));
    CU(launch_observe(v, obs_dev, vec_dev, WC(e, WC_OBSERVE), s));
    if (out->status) CU(cudaMemcpyAsync(out->status, o.status, WN, cudaMemcpyDeviceToHost, cs));
    if (out->reward) CU(cudaMemcpyAsync(out->reward, o.reward, WN * 4, cudaMemcpyDeviceToHost, cs));
    if (out->cost) CU(cudaMemcpyAsync(out->cost, o.cost, WN * 4, cudaMemcpyDeviceToHost, cs));
    if (out->train_valid) CU(cudaMemcpyAsync(out->train_valid, o.train_valid, WN * NA * 4, cudaMemcpyDeviceToHost, cs));
    if (out->goals_reached) CU(cudaMemcpyAsync(out->goals_reached, o.goals_reached, WN, cudaMemcpyDeviceToHost, cs));
    if (out->violated) CU(cudaMemcpyAsync(out->violated, o.violated, WN, cudaMemcpyDeviceToHost, cs));
    if (out->shadow_goals) CU(cudaMemcpyAsync(out->shadow_goals, o.shadow_goals, W * 4, cudaMemcpyDeviceToHost, cs));
    if (out->fixed_actions) CU(cudaMemcpyAsync(out->fixed_actions, o.fixed_actions, WN, cudaMemcpyDeviceToHost, cs));
    CU(cudaEventRecord(e->ev_copied[k], cs));
    e->tv_copy_pending[k] = false;
    e->obs_src[k][0] = e->obs_src[k][1] = e->vec_src[k][0] = e->vec_src[k][1] = 0;
    e->next_slot = k ^ 1;
    if (e->begun < 2) e->begun++;
    const size_t PB = (size_t)v.C * v.F * v.F;
    if (obs_host) CU(cudaMemcpyAsync(obs_host, obs_dev, WN * PB * 4, cudaMemcpyDeviceToHost, s));
    if (vec_host) CU(cudaMemcpyAsync(vec_host, vec_dev, WN * 16, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamWaitEvent(s, e->ev_copied[k], 0));
    CU(cudaStreamSynchronize(s));
    return MAPF_OK;
}

int mapf_checksum_rows(const void *data, int64_t rows, int64_t row_bytes, uint64_t *out, void *stream) {
    if (!data || !out) return fail(MAPF_E_NULL, "mapf_checksum_rows: null argument");
    if (rows < 0 || row_bytes < 0 || (row_bytes & 3) || (reinterpret_cast<uintptr_t>(data) & 3))
        return fail(MAPF_E_BAD_CONFIG, "mapf_checksum_rows: rows >= 0, row_bytes a multiple of 4, data 4-byte aligned");
    if (rows == 0) return MAPF_OK;
    CU(launch_checksum_rows(static_cast<const uint32_t *>(data), rows, row_bytes / 4, reinterpret_cast<unsigned long long *>(out), (cudaStream_t)stream));
    return MAPF_OK;
}

}  // extern "C"
