// observe_world.cuh — observation building of ONE world by one warp: the device code shared by observe_kernel
// (observe.cu) and the fused step_observe_kernel (step_observe.cu), and the per-chunk code the CTA-per-world kernels
// (observe_wide.cu, step_observe_wide.cu) and the unpack kernel (obs_bits.cu) share with them.  Also the host-side
// launch planning of all of them: chunk size, shared-memory layout, when 16-byte stores are allowed, and the mapping of
// the runtime format / shape onto a kernel instantiation.  See observe.cu for the design notes and the reference lines
// (mapf_gym.py:192-198, 246-336).
#pragma once
#include "common.cuh"

namespace mapf {
namespace ow {

constexpr int OBW = 4;   // packed obstacle words prefetched per lane (PW <= 128: up to 64x64 cells; 40x40 needs 52)

// u32 stride of one agent's bit string in shared memory: one spare word (phase 1b reads word k+1), odd so that lane-strided
// accesses are bank-conflict free
__host__ __device__ inline int agent_stride(int PB) {
    const int aw = (PB + 31) / 32 + 1;
    return (aw & 1) ? aw : aw + 1;
}

// u32 words of one agent's record in OBS_BITS output: MAPF_OBS_BITS_WORDS(C, F)
__host__ __device__ inline int bits_words(int PB) { return (PB + 31) / 32; }

struct ObsLayout {
    int PB;      // bits per agent = C*F*F
    int AST;     // u32 stride of one agent's padded bit string (odd -> conflict-free lane-strided access)
    int CH;      // agents per chunk (<= 32)
    int WB;      // u32 words of the chunk bit string
    int alias;   // 1: the chunk bit string overlays the staging area (single chunk per world)
    int fmt;     // ObsFormat: OBS_F32 (the reference's layout), OBS_BF16 (same 0/1 values, half the bytes) or OBS_BITS
    int step_n, step_e;   // (32 G) / PB, (32 G) % PB: how (agent, bit) advances when the word index advances by G (the group width)
    size_t off_abits, off_grid, off_goal, off_aw, off_wb, total;
};

// G = lanes that build one world (32 = a whole warp; 8 / 16 = lane groups, several small worlds per warp)
inline ObsLayout make_layout(int HP, int RW, int GS, int N, int C, int F, int CH, int G = 32) {
    ObsLayout L;
    L.PB = C * F * F;
    L.AST = agent_stride(L.PB);
    L.CH = CH;
    L.WB = (CH * L.PB + 31) / 32 + 2;
    L.alias = (CH >= N) ? 1 : 0;
    L.fmt = OBS_F32;
    L.step_n = (32 * G) / L.PB;
    L.step_e = (32 * G) % L.PB;
    size_t o = align16((size_t)HP * RW * 4);
    L.off_abits = o; o += align16((size_t)HP * RW * 4);
    L.off_grid = o; o += align16((size_t)HP * GS);
    const size_t staging = o;
    if (L.alias) {
        L.off_wb = 0;
        if (align16((size_t)L.WB * 4) > o) o = align16((size_t)L.WB * 4);
    }
    L.off_goal = o; o += align16((size_t)N * 8);      // goals [N] then cells [N]
    L.off_aw = o; o += align16((size_t)CH * L.AST * 4);
    if (!L.alias) { L.off_wb = o; o += align16((size_t)L.WB * 4); }
    (void)staging;
    L.total = o;
    return L;
}

// Observation bytes one world stores in L's format (the launch rules that prefer fewer write streams key on it)
inline size_t obs_world_bytes(const ObsLayout &L, int N) {
    if (L.fmt == OBS_BITS) return (size_t)N * bits_words(L.PB) * 4;
    return (size_t)N * L.PB * (L.fmt == OBS_BF16 ? 2 : 4);
}

// Bit-string scratch of one warp for a chunk of CH agents, as the chunk-size rules of the launchers estimate it: CH agent
// strings of (PB + 31) / 32 + 2 words, twice (per-agent strings aw, chunk string wb).
inline size_t chunk_scratch(int CH, int PB) { return (size_t)CH * ((PB + 31) / 32 + 2) * 4 * 2; }

// Agents per chunk of the warp-per-world kernels and of the unpack kernel: as many as fit ~24 KB of scratch per warp.
inline int obs_chunk(int N, int PB) {
    int CH = N < 32 ? N : 32;
    while (CH > 4 && chunk_scratch(CH, PB) > 24 * 1024) CH >>= 1;
    return CH;
}

// CTA-per-world kernels: the staging part of L ([obits | abits | grid | goals + cells]) is shared by the CTA, and each warp
// has its own scratch behind it (aw: CH agent strings at stride AST, then wb: the chunk bit string).
inline size_t cta_shared_bytes(const ObsLayout &L, int N) { return L.off_goal + align16((size_t)N * 8); }
inline size_t warp_scratch_bytes(int CH, int PB) {
    return align16((size_t)CH * agent_stride(PB) * 4) + align16((size_t)((CH * PB + 31) / 32 + 2) * 4);
}

// 16-byte stores (VEC4) need `obs` and the start of every chunk of CH agents 16-byte aligned.  Bits: every record is AW
// words.  f32 / bf16 (4 / 8 elements per store): N * PB, and CH * PB when a world takes several chunks.
inline bool obs_vec4(int fmt, int N, int PB, int CH, const void *obs) {
    if (reinterpret_cast<uintptr_t>(obs) & 15) return false;
    if (fmt == OBS_BITS) return bits_words(PB) % 4 == 0;
    const size_t al = fmt == OBS_BF16 ? 8 : 4;
    return ((size_t)N * PB) % al == 0 && (CH >= N || ((size_t)CH * PB) % al == 0);
}

// Compile-time parameters of an observation kernel: C_T / F_T = 6 / 9 (the training configuration) or 0 / 0 (runtime values
// from EnvView), VEC4 (16-byte stores), BITS (OBS_BITS output).
template <int C_, int F_, bool VEC4_, bool BITS_>
struct ObsVariant {
    static constexpr int C_T = C_, F_T = F_;
    static constexpr bool VEC4 = VEC4_, BITS = BITS_;
};

// Calls fn(ObsVariant<...>()) for the runtime format, channels x FOV and store width.
template <typename Fn>
cudaError_t dispatch_obs(int fmt, int C, int F, bool vec4, Fn &&fn) {
    const bool c69 = C == 6 && F == 9;
    if (fmt == OBS_BITS) {
        if (c69) return vec4 ? fn(ObsVariant<6, 9, true, true>()) : fn(ObsVariant<6, 9, false, true>());
        return vec4 ? fn(ObsVariant<0, 0, true, true>()) : fn(ObsVariant<0, 0, false, true>());
    }
    if (c69) return vec4 ? fn(ObsVariant<6, 9, true, false>()) : fn(ObsVariant<6, 9, false, false>());
    return vec4 ? fn(ObsVariant<0, 0, true, false>()) : fn(ObsVariant<0, 0, false, false>());
}

__device__ __forceinline__ void or_bits(uint32_t *words, int p, uint32_t val, int nbits) {
    const int k = p >> 5, s = p & 31;
    words[k] |= val << s;
    if (s + nbits > 32) words[k + 1] |= val >> (32 - s);
}
__device__ __forceinline__ void or_bit(uint32_t *words, int p) { words[p >> 5] |= 1u << (p & 31); }

// inputs of one world held in registers (prefetched one world ahead)
struct WorldRegs {
    uint32_t pw, gw;        // cell / goal of agent `lane` (agents >= 32 are loaded directly)
    uint32_t ob[OBW];       // packed obstacle words lane, lane+32, ...
    int2 ht;                // human (pos, next) of the current tick
};

template <int G = 32>
__device__ __forceinline__ void load_world(const EnvView &v, int w, int lane, int nob, uint64_t pol, WorldRegs &r) {
    if (w < v.W) {
        const size_t base = (size_t)w * v.N;
        const int i = lane < v.N ? lane : 0;
        r.pw = ld_keep(reinterpret_cast<const uint32_t *>(v.pos) + base + i, pol);
        r.gw = ld_keep(reinterpret_cast<const uint32_t *>(v.goal) + base + i, pol);
        const uint32_t *src = v.obst_pack + (size_t)w * v.PW;
#pragma unroll
        for (int k = 0; k < OBW; ++k) r.ob[k] = (k * G + lane < nob) ? ld_keep(src + k * G + lane, pol) : 0u;
        r.ht = ld_keep_v2(reinterpret_cast<const int2 *>(v.hcur) + w, pol);
    }
}

// Per-warp shared-memory views of one world (carved from ObsLayout offsets).
struct ObsSmem {
    uint32_t *obits, *abits, *sgoal, *spos, *aw, *wb;
    uint8_t *grid;
};
__device__ __forceinline__ ObsSmem obs_carve(unsigned char *base, const ObsLayout &L, int N) {
    ObsSmem m;
    m.obits = reinterpret_cast<uint32_t *>(base);
    m.abits = reinterpret_cast<uint32_t *>(base + L.off_abits);
    m.grid = base + L.off_grid;
    m.sgoal = reinterpret_cast<uint32_t *>(base + L.off_goal);
    m.spos = m.sgoal + N;
    m.aw = reinterpret_cast<uint32_t *>(base + L.off_aw);
    m.wb = reinterpret_cast<uint32_t *>(base + L.off_wb);
    return m;
}

// nibble -> four 0/1 floats for phase 2's 16-byte stores; filled by threads t < 16, the caller synchronises
__device__ __forceinline__ void fill_lut(uint4 *lut, const uint32_t t) {
    if (t < 16) {
        const uint32_t one = 0x3f800000u;
        lut[t] = make_uint4((t & 1u) ? one : 0u, (t & 2u) ? one : 0u, (t & 4u) ? one : 0u, (t & 8u) ? one : 0u);
    }
}


// Phases 1b and 2 of the observation build: `nch` per-agent bit strings of PB bits (stride AST words, in shared memory)
// are compacted into one contiguous bit string `wb` and expanded into f32 (fmt OBS_F32) or bf16 (OBS_BF16) 0/1 values at
// agent c0 of row `row` of `obs` ([rows, N, PB] f32 or bf16 elements) with streaming stores.  Shared by observe_chunk and unpack_obs_kernel (obs_bits.cu), which stages packed records.
template <bool VEC4, int G>
__device__ __forceinline__ void expand_records(const uint32_t *aw, const int AST, uint32_t *wb, const uint4 *lut,
                                               const Grp<G> &g, const int nch, const int PB, const int step_n,
                                               const int step_e, const int fmt, float *obs, const size_t row, const int N,
                                               const int c0) {
    const int lane = g.gl;
    // ---- phase 1b: compact to one contiguous bit string (word m <- 32 bits starting at agent n, bit e) ----------------
    const int TB = nch * PB;
    const int nwords = (TB + 31) >> 5;
    {
        int n = (lane << 5) / PB, e = (lane << 5) - n * PB;
        for (int m = lane; m < nwords; m += G) {
            const uint32_t *src = aw + n * AST;
            uint32_t x = __funnelshift_r(src[e >> 5], src[(e >> 5) + 1], e & 31);
            const int valid = PB - e;
            if (valid < 32) {
                x &= (1u << valid) - 1u;
                if (n + 1 < nch) x |= aw[(n + 1) * AST] << valid;
            }
            wb[m] = x;
            n += step_n; e += step_e;
            if (e >= PB) { e -= PB; n += 1; }
        }
    }
    g.sync();
    // ---- phase 2: bits -> floats, streaming stores ---------------------------------------------------------------------
    if (fmt == OBS_BF16) {
        // optional bf16 output: 8 bits -> 8 bf16 (1.0 = 0x3F80) -> one 16-byte store; the expansion is plain ALU
        uint16_t *dst16 = reinterpret_cast<uint16_t *>(obs) + (row * N + c0) * PB;
        if (VEC4) {
            const int n8 = TB >> 3;
            for (int q = lane; q < n8; q += G) {
                const uint32_t b = wb[q >> 2] >> ((q & 3) << 3);
                const uint32_t x0 = (b & 1u) * 0x3F80u | (b & 2u) * 0x1FC00000u;
                const uint32_t x1 = ((b >> 2) & 1u) * 0x3F80u | ((b >> 2) & 2u) * 0x1FC00000u;
                const uint32_t x2 = ((b >> 4) & 1u) * 0x3F80u | ((b >> 4) & 2u) * 0x1FC00000u;
                const uint32_t x3 = ((b >> 6) & 1u) * 0x3F80u | ((b >> 6) & 2u) * 0x1FC00000u;
                st_stream_v4(reinterpret_cast<float *>(dst16 + ((size_t)q << 3)), x0, x1, x2, x3);
            }
            for (int f = (n8 << 3) + lane; f < TB; f += G) dst16[f] = ((wb[f >> 5] >> (f & 31)) & 1u) ? 0x3F80 : 0;
        } else {
            for (int f = lane; f < TB; f += G) dst16[f] = ((wb[f >> 5] >> (f & 31)) & 1u) ? 0x3F80 : 0;
        }
        g.sync();
        return;
    }
    float *dst = obs + (row * N + c0) * PB;
    if (VEC4) {
        const int n4 = TB >> 2;
        const int sh = (lane & 7) << 2;
        const uint32_t *wp = wb + (lane >> 3);
        float *d4 = dst + (lane << 2);
#pragma unroll 4
        for (int q = lane; q < n4; q += G, wp += G / 8, d4 += 4 * G) {
            const uint4 val = lut[(*wp >> sh) & 15u];
            st_stream_v4(d4, val.x, val.y, val.z, val.w);
        }
    } else {
        for (int f = lane; f < TB; f += G) dst[f] = ((wb[f >> 5] >> (f & 31)) & 1u) ? 1.0f : 0.0f;
    }
    g.sync();
}

// One chunk of agents [c0, c0 + nch) of a staged world by one warp: phase 1 (per-agent bit strings), phase 1b
// (compaction), phase 2 (bits -> f32 / bf16, streaming stores) — or, in OBS_BITS, a direct store of the phase-1 strings.
// `aw` / `wb` are this warp's scratch; everything else of `m` is read-only here and may be shared by the warps of a CTA.
// BITS: the OBS_BITS instantiation (a separate one, so that the f32 / bf16 kernels compile exactly as without it).
template <int C_T, int F_T, bool VEC4, int G = 32, bool BITS = false>
__device__ __forceinline__ void observe_chunk(const EnvView &v, const ObsLayout &L, const ObsSmem &m, const uint4 *lut,
                                              const int w, const Grp<G> &g, const int c0, const int nch, const int nr,
                                              const int nc, const int rows, const int cols, float *__restrict__ obs,
                                              float *__restrict__ vec) {
    const int lane = g.gl;
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW;
    const int F = F_T > 0 ? F_T : v.F, C = C_T > 0 ? C_T : v.C, half = F >> 1;
    const int FF = F * F, PB = (C_T > 0 && F_T > 0) ? C_T * F_T * F_T : L.PB, AST = L.AST;
    const uint32_t *const obits = m.obits, *const abits = m.abits, *const sgoal = m.sgoal, *const spos = m.spos;
    uint32_t *const aw = m.aw, *const wb = m.wb;
    const uint8_t *const grid = m.grid;
    {
        const int i = c0 + lane;
        const bool act = lane < nch;
        // ---- phase 1: per-agent bit strings -------------------------------------------------------------------
        if (act) {
            uint32_t *my = aw + lane * AST;
            const uint32_t pw = spos[i], gw = sgoal[i];
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            const int gr = (int16_t)(gw & 0xffff), gc = (int16_t)(gw >> 16);
            const int top = r - half, left = c - half;                                    // :251
            const int off = left + P;
            if (F_T > 0) {
                // channels 0 and 1 accumulate in registers at compile-time bit positions
                constexpr int FT = F_T > 0 ? F_T : 1;
                constexpr int NACC = (2 * FT * FT + 31) / 32 + 1;
                uint32_t acc[NACC];
#pragma unroll
                for (int k = 0; k < NACC; ++k) acc[k] = 0;
#pragma unroll
                for (int y = 0; y < FT; ++y) {
                    const int prow = top + y + P;
                    uint32_t o = row_window(obits + prow * RW, off, FT);      // OOB or obstacle  (:270-276)
                    uint32_t g = row_window(abits + prow * RW, off, FT);      // agents           (:278-285)
                    if (y == FT / 2) { o |= 1u << (FT / 2); g &= ~(1u << (FT / 2)); }   // own cell -> channel 0 (:278-280)
                    constexpr int dummy = 0; (void)dummy;
                    const int p0 = y * FT, p1 = FT * FT + y * FT;
                    acc[p0 >> 5] |= o << (p0 & 31);
                    if ((p0 & 31) + FT > 32) acc[(p0 >> 5) + 1] |= o >> (32 - (p0 & 31));
                    acc[p1 >> 5] |= g << (p1 & 31);
                    if ((p1 & 31) + FT > 32) acc[(p1 >> 5) + 1] |= g >> (32 - (p1 & 31));
                }
#pragma unroll
                for (int k = 0; k < NACC; ++k) my[k] = acc[k];
                for (int k = NACC; k < AST; ++k) my[k] = 0;
            } else {
                for (int k = 0; k < AST; ++k) my[k] = 0;
                for (int y = 0; y < F; ++y) {
                    const int prow = top + y + P;
                    uint32_t o = row_window(obits + prow * RW, off, F);
                    uint32_t g = row_window(abits + prow * RW, off, F);
                    if (y == half) { o |= 1u << half; g &= ~(1u << half); }
                    or_bits(my, y * F, o, F);
                    or_bits(my, FF + y * F, g, F);
                }
            }
            // channel 3: goals of the agents visible in the window, clamped into it (:302-308)
            for (int y = 0; y < F; ++y) {
                const int prow = top + y + P;
                uint32_t g = row_window(abits + prow * RW, off, F);
                if (y == half) g &= ~(1u << half);
                while (g) {
                    const int x = __ffs(g) - 1; g &= g - 1;
                    const int j = grid[prow * GS + off + x] - 1;
                    const uint32_t jw = sgoal[j];
                    const int jr = (int16_t)(jw & 0xffff), jc = (int16_t)(jw >> 16);
                    const int mr = max(top, min(top + F - 1, jr)), mc = max(left, min(left + F - 1, jc));
                    or_bit(my, 3 * FF + (mr - top) * F + (mc - left));
                }
            }
            if (v.use_da) {                                              // danger disc |cell - H'| <= 5 (:289-290)
                for (int y = 0; y < F; ++y) {
                    const int rr = top + y, dy = rr > nr ? rr - nr : nr - rr;
                    if (rr >= 0 && rr < rows && dy <= 5) {
                        const int hw = dy == 0 ? 5 : dy <= 3 ? 4 : dy == 4 ? 3 : 0;
                        const int lo = max(max(nc - hw, 0), left), hi = min(min(nc + hw, cols - 1), left + F - 1);
                        if (lo <= hi) or_bits(my, 4 * FF + y * F + (lo - left), (1u << (hi - lo + 1)) - 1u, hi - lo + 1);
                    }
                }
            }
            if (gr >= top && gr < top + F && gc >= left && gc < left + F)                  // own goal (:298-300)
                or_bit(my, 2 * FF + (gr - top) * F + (gc - left));
            if (nr >= top && nr < top + F && nc >= left && nc < left + F)                  // human (:310-312)
                or_bit(my, 4 * FF + (nr - top) * F + (nc - left));
            if (v.use_hp && C == 6 && v.hp5) {                                             // (:293-297)
                const int tick = v.htick[w];
                const int16_t *p5 = v.hp5 + (v.hp5_per_tick ? ((size_t)w * v.L + tick) * 10 : (size_t)w * 10);
                for (int k = 0; k < 5; ++k) {
                    const int pr = p5[2 * k], pc = p5[2 * k + 1];
                    if (pr >= 0 && pr < rows && pc >= 0 && pc < cols && pr >= top && pr < top + F && pc >= left && pc < left + F)
                        or_bit(my, 5 * FF + (pr - top) * F + (pc - left));
                }
            }
            // vector (:316-323): f64 sqrt / divide, then cast
            const double dx = (double)(gr - r), dy_ = (double)(gc - c);
            const double d = sqrt(dx * dx + dy_ * dy_);
            float4 o4;
            o4.x = (float)(d != 0.0 ? dx / d : dx);
            o4.y = (float)(d != 0.0 ? dy_ / d : dy_);
            o4.z = (float)d;
            o4.w = 0.0f;
            st_stream_v4(vec + ((size_t)w * N + i) * 4, __float_as_uint(o4.x), __float_as_uint(o4.y), __float_as_uint(o4.z), __float_as_uint(o4.w));
        }
        g.sync();
        if (BITS) {
            // ---- bits output: the per-agent strings ARE the records (AW words each, padding bits 0); phases 1b and 2 are
            //      skipped.  The chunk's nch * AW words are contiguous in HBM: 16-byte streaming stores when AW % 4 == 0.
            const int AW = bits_words(PB);
            uint32_t *dstw = reinterpret_cast<uint32_t *>(obs) + ((size_t)w * N + c0) * AW;
            if (VEC4) {
                const int n4 = (nch * AW) >> 2;
                for (int q = lane; q < n4; q += G) {
                    const int a = (q << 2) / AW, k = (q << 2) - a * AW;
                    const uint32_t *src = aw + a * AST + k;
                    st_stream_v4(reinterpret_cast<float *>(dstw + ((size_t)q << 2)), src[0], src[1], src[2], src[3]);
                }
            } else {
                for (int m = lane; m < nch * AW; m += G) {
                    const int a = m / AW;
                    dstw[m] = aw[a * AST + (m - a * AW)];
                }
            }
            g.sync();
            return;
        }
        expand_records<VEC4, G>(aw, AST, wb, lut, g, nch, PB, L.step_n, L.step_e, L.fmt, obs, (size_t)w, N, c0);
    }
}

// One world's observations by one warp.  `pw_reg` / `gw_reg`: cell and goal of agent `lane` (agents >= 32 are read
// from HBM); (nr, nc) = human.getNextPos(); the obstacle bit rows are already staged in m.obits and m.abits / m.grid
// are clean on entry.  On exit they are clean again unless L.alias (then the caller re-zeroes them for the next world).
// C_T/F_T > 0: compile-time channels / FOV (the training configuration 6 x 9 x 9); 0: runtime values from EnvView.
template <int C_T, int F_T, bool VEC4, int G = 32, bool BITS = false>
__device__ __forceinline__ void observe_world(const EnvView &v, const ObsLayout &L, const ObsSmem &m, const uint4 *lut,
                                              const int w, const Grp<G> &g, const uint32_t pw_reg, const uint32_t gw_reg,
                                              const int nr, const int nc, float *__restrict__ obs,
                                              float *__restrict__ vec) {
    const int lane = g.gl;
    const int N = v.N, P = v.P, GS = v.GS, RW = v.RW, CH = L.CH;
    uint32_t *const abits = m.abits, *const sgoal = m.sgoal, *const spos = m.spos;
    uint8_t *const grid = m.grid;
    {
        const uint32_t *posw = reinterpret_cast<const uint32_t *>(v.pos) + (size_t)w * N;
        const uint32_t *goalw = reinterpret_cast<const uint32_t *>(v.goal) + (size_t)w * N;
        for (int i = lane; i < N; i += G) {
            const uint32_t pw = i < G ? pw_reg : __ldg(posw + i);
            const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
            grid[(r + P) * GS + c + P] = (uint8_t)(i + 1);
            atomicOr(&abits[(r + P) * RW + ((c + P) >> 5)], 1u << ((c + P) & 31));
            sgoal[i] = i < G ? gw_reg : __ldg(goalw + i);
            spos[i] = pw;
        }
        int rows = v.H, cols = v.Wd;
        if (v.use_da | v.use_hp) { if (v.dims) { rows = v.dims[2 * w]; cols = v.dims[2 * w + 1]; } }
        g.sync();

        for (int c0 = 0; c0 < N; c0 += CH)
            observe_chunk<C_T, F_T, VEC4, G, BITS>(v, L, m, lut, w, g, c0, min(CH, N - c0), nr, nc, rows, cols, obs, vec);
        if (!L.alias) {
            // un-scatter this world's agents so the next world starts from a clean grid
            for (int i = lane; i < N; i += G) {
                const uint32_t pw = spos[i];
                const int r = (int16_t)(pw & 0xffff), c = (int16_t)(pw >> 16);
                grid[(r + P) * GS + c + P] = 0;
                abits[(r + P) * RW + ((c + P) >> 5)] = 0;
            }
        }
        g.sync();
    }
}

}  // namespace ow
}  // namespace mapf
