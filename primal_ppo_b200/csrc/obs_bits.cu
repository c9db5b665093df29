// obs_bits.cu — gather-and-expand of bit-packed observations (mapf_unpack_obs): rows of u32 [N, AW] records (one bit per
// cell, the format of mapf_observe_bits / mapf_step_observe_bits) -> f32 or bf16 [n_rows, N, C, F, F] 0/1 values for the
// network, optionally through an int64 row index so that a minibatch gather and the expansion are one pass.
//
// One warp per output row (persistent grid, rows strided over the warps).  A chunk of the row's records is staged in
// shared memory at the phase-1 stride AST of the observation kernels, and from there the same device code as their
// phases 1b and 2 (observe_world.cuh: expand_records) compacts and expands it with streaming stores.  A row index outside
// [0, src_rows) stages zeros, so it yields an all-zero row.
// HBM traffic per row: read N*AW*4 B (+ 8 B of index), write N*C*F*F*4 B (f32) or *2 B (bf16).
#include "common.cuh"
#include "observe_world.cuh"

namespace mapf {

namespace {

using namespace ow;

constexpr int UNPACK_WARPS = 8;

template <bool VEC4>
__global__ void __launch_bounds__(UNPACK_WARPS * 32)
unpack_obs_kernel(const uint32_t *__restrict__ bits, const long long src_rows, const int N, const int PB, const int AW,
                  const int AST, const int CH, const int per_warp, const int step_n, const int step_e,
                  const int64_t *__restrict__ rows, const long long n_rows, const int fmt, void *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint4 lut[16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *const aw = reinterpret_cast<uint32_t *>(smem_raw + (size_t)warp * per_warp);
    uint32_t *const wb = reinterpret_cast<uint32_t *>(smem_raw + (size_t)warp * per_warp + align16((size_t)CH * AST * 4));
    fill_lut(lut, threadIdx.x);
    __syncthreads();
    const Grp<32> g(lane);
    const size_t row_words = (size_t)N * AW;
    const long long nwarps = (long long)gridDim.x * UNPACK_WARPS;
    for (long long r = (long long)blockIdx.x * UNPACK_WARPS + warp; r < n_rows; r += nwarps) {
        const long long s = rows ? rows[r] : r;
        const bool valid = s >= 0 && s < src_rows;
        const uint32_t *src = bits + (valid ? (size_t)s * row_words : 0);
        for (int c0 = 0; c0 < N; c0 += CH) {
            const int nch = min(CH, N - c0);
            for (int m = lane; m < nch * AW; m += 32) {          // coalesced read of the chunk's contiguous records
                const int a = m / AW;
                aw[a * AST + (m - a * AW)] = valid ? __ldcs(src + (size_t)c0 * AW + m) : 0u;
            }
            g.sync();
            expand_records<VEC4, 32>(aw, AST, wb, lut, g, nch, PB, step_n, step_e, fmt, static_cast<float *>(out), (size_t)r,
                                     N, c0);                                                // ends with g.sync()
        }
    }
}

}  // namespace

cudaError_t launch_unpack_obs(const uint32_t *bits, long long src_rows, int N, int C, int F, const int64_t *rows,
                              long long n_rows, int out_bf16, void *out, cudaStream_t stream) {
    const int PB = C * F * F, CH = obs_chunk(N, PB);
    const int per_warp = (int)warp_scratch_bytes(CH, PB);
    const int fmt = out_bf16 ? OBS_BF16 : OBS_F32;
    auto kern = obs_vec4(fmt, N, PB, CH, out) ? unpack_obs_kernel<true> : unpack_obs_kernel<false>;
    return launch_persistent(kern, UNPACK_WARPS * 32, (size_t)per_warp * UNPACK_WARPS, (n_rows + UNPACK_WARPS - 1) / UNPACK_WARPS,
                             INT_MAX, stream, bits, src_rows, N, PB, bits_words(PB), agent_stride(PB), CH, per_warp,
                             (32 * 32) / PB, (32 * 32) % PB, rows, n_rows, fmt, out);
}

}  // namespace mapf
