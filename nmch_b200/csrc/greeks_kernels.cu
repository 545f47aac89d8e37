// greeks_kernels.cu -- strike vector with pathwise delta AND pathwise vega (d price / d v_0) in one pass
// (SURVEY.md §8f rank 2 "a strike vector and pathwise delta/vega reuse the same paths at ~zero RNG cost"; the
// reference fixes K = S_0 and has no sensitivities, src/NMCH/methods/NMCH.cu:7).
//
// fe_tangent_kernel: the native FE step on the native Philox stream (the words, the instructions and therefore the
//   (S_T, V_T) of fe_philox_kernel, bit for bit) carrying the tangent (dV/dv_0, dS/dv_0) of every path in registers;
//   leaves S_T, V_T and dS_T/dv_0 in HBM (12 bytes per path) and reduces the K = S_0 payoff moments like every path kernel.
// strike_greeks_kernel: folds the two terminal arrays per strike: payoff moments, delta = 1{S_T > K} S_T / S_0,
//   vega = 1{S_T > K} dS_T/dv_0 and its square (for the standard error), through the deterministic ticket reduction.
//   A NaN path makes the strike's payoff, delta and vega sums NaN (DESIGN.md row A3); the in-the-money count stays a count.
#include "fe_step.cuh"
#include "kernels.cuh"

namespace nmchb {

constexpr int kTangentThreads = 256;
constexpr int kTangentPaths = 2;            // paths per thread: the tangent pair doubles the per-path state (52 registers, 32 warps per SM)
constexpr int kTangentTile = kTangentPaths * kTangentThreads;

// The loop of fe_philox_kernel (fe_kernels.cu) with the tangent step: one tile of kTangentTile paths per block, the
// Philox counter split where its low word would wrap so that the per-path invariants of rounds 1-2 are hoisted and the
// path-independent multiplies sit on the uniform datapath; a pass may start on the second half of a block (an odd
// number of steps before it) and end on a first half.
template <int FLOOR>
__global__ void __launch_bounds__(kTangentThreads, 4)
fe_tangent_kernel(const __grid_constant__ FeLaunch L, ReduceBuffers rb, float *__restrict__ S_out,
                  float *__restrict__ V_out, float *__restrict__ B_out)
{
    constexpr int P = kTangentPaths;
    NMCHB_ASSERT(blockDim.x == kTangentThreads && (int)blockIdx.x < L.blocks_per_point && L.n_points == 1);
    NMCHB_ASSERT(L.first_path % kTangentTile == 0);
    const unsigned long long local0 = (unsigned long long)blockIdx.x * kTangentTile;
    const unsigned long long g0 = L.first_path + local0;         // multiple of the tile: no carry below
    uint32_t path_hi = (uint32_t)(g0 >> 32);
    asm volatile("" : "+r"(path_hi));
    const uint32_t path_lo0 = (uint32_t)g0 + threadIdx.x;
    NMCHB_ASSERT(((g0 + (unsigned long long)(kTangentTile - 1)) >> 32) == (g0 >> 32));
    const FePoint pc = L.pt0;

    float S[P], V[P], A[P], B[P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
        S[j] = L.S0;
        V[j] = L.v0;
        A[j] = 1.0f;
        B[j] = 0.0f;
    }
    const unsigned long long w0 = L.draw_offset;
    unsigned long long blk = w0 >> 2;
    int n = L.N;
    const bool resume = (w0 & 2ull) != 0ull && n > 0;            // start on the second word pair of a block
    if (resume) {
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const U4 w = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), path_lo0 + j * kTangentThreads, path_hi, L.keys);
            fe_step_native_tangent<FLOOR>(S[j], V[j], A[j], B[j], w.z, w.w, L.rdt, L.zr, L.zc, pc);
        }
    }
    blk += resume ? 1ull : 0ull;
    n -= resume ? 1 : 0;
    int pairs = n >> 1;
    while (pairs > 0) {
        const uint32_t blk_hi = (uint32_t)(blk >> 32);
        const uint32_t blk_lo = (uint32_t)blk;
        const unsigned long long room = 0x100000000ull - (unsigned long long)blk_lo;
        const int chunk = ((unsigned long long)pairs < room) ? pairs : (int)room;
        PhiloxPathInv inv[P];
#pragma unroll
        for (int j = 0; j < P; ++j) inv[j] = philox_path_invariants(blk_hi, path_lo0 + j * kTangentThreads, L.keys);
#pragma unroll 1
        for (int it = 0; it < chunk; ++it) {
            const PhiloxBlockUniform bu = philox_block_uniform(blk_lo + (uint32_t)it, path_hi, L.keys);
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const U4 w = philox4x32_10_hoisted(bu, inv[j], L.keys);
                fe_step_native_tangent<FLOOR>(S[j], V[j], A[j], B[j], w.x, w.y, L.rdt, L.zr, L.zc, pc);
                fe_step_native_tangent<FLOOR>(S[j], V[j], A[j], B[j], w.z, w.w, L.rdt, L.zr, L.zc, pc);
            }
        }
        blk += (unsigned long long)chunk;
        pairs -= chunk;
    }
    if (n & 1) {
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const U4 w = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), path_lo0 + j * kTangentThreads, path_hi, L.keys);
            fe_step_native_tangent<FLOOR>(S[j], V[j], A[j], B[j], w.x, w.y, L.rdt, L.zr, L.zc, pc);
        }
    }
    double pay = 0.0, pay2 = 0.0;
#pragma unroll
    for (int j = 0; j < P; ++j) {
        const unsigned long long idx = local0 + (unsigned long long)(j * kTangentThreads) + threadIdx.x;
        if (idx < L.n_local) {
            const double x = payoff_or_nan(S[j], L.K);
            pay += x;
            pay2 += x * x;
            S_out[idx] = S[j];
            V_out[idx] = V[j];
            B_out[idx] = B[j];
        }
    }
    block_reduce_and_finish(pay, pay2, rb.partials, rb.tickets, rb.out, 0, blockIdx.x, L.blocks_per_point);
}

constexpr int kGreekThreads = 256;
constexpr int kGreekBlocks = 296;           // 2 per SM, contiguous slices, 16-byte loads (as strike_moments_kernel)

__device__ __forceinline__ void greek_fold(float s, float b, float K, float inv_S0, double &pay, double &pay2,
                                           double &delta, double &itm, double &vega, double &vega2)
{
    const double p = payoff_or_nan(s, K);
    pay += p;
    pay2 += p * p;
    if (s > K) {
        delta += (double)(s * inv_S0);
        itm += 1.0;
        vega += (double)b;
        vega2 += (double)b * (double)b;
    } else if (s != s) {                                     // a NaN path: carried into delta and vega too
        delta += (double)s;
        vega += (double)s;
        vega2 += (double)s;
    }
}

__global__ void __launch_bounds__(kGreekThreads)
strike_greeks_kernel(const float *__restrict__ S, const float *__restrict__ B, unsigned long long n,
                     const float *__restrict__ strikes, float inv_S0, ReduceBuffers rb)
{
    const int j = blockIdx.y;
    const float K = strikes[j];
    double pay = 0.0, pay2 = 0.0, delta = 0.0, itm = 0.0, vega = 0.0, vega2 = 0.0;
    const unsigned long long n4 = n / 4ull;
    const float4 *S4 = reinterpret_cast<const float4 *>(S);
    const float4 *B4 = reinterpret_cast<const float4 *>(B);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const float4 s = __ldg(S4 + i), b = __ldg(B4 + i);
        greek_fold(s.x, b.x, K, inv_S0, pay, pay2, delta, itm, vega, vega2);
        greek_fold(s.y, b.y, K, inv_S0, pay, pay2, delta, itm, vega, vega2);
        greek_fold(s.z, b.z, K, inv_S0, pay, pay2, delta, itm, vega, vega2);
        greek_fold(s.w, b.w, K, inv_S0, pay, pay2, delta, itm, vega, vega2);
    }
    if (blockIdx.x == 0)                                     // ragged tail
        for (unsigned long long i = n4 * 4ull + threadIdx.x; i < n; i += blockDim.x)
            greek_fold(S[i], B[i], K, inv_S0, pay, pay2, delta, itm, vega, vega2);
    block_reduce_and_finish(pay, pay2, rb.partials, rb.tickets, rb.out, 3 * j, blockIdx.x, gridDim.x);
    block_reduce_and_finish(delta, itm, rb.partials, rb.tickets, rb.out, 3 * j + 1, blockIdx.x, gridDim.x);
    block_reduce_and_finish(vega, vega2, rb.partials, rb.tickets, rb.out, 3 * j + 2, blockIdx.x, gridDim.x);
}

cudaError_t launch_fe_tangent(const FeLaunch &L, int floor_kind, ReduceBuffers rb, float *S_out, float *V_out, float *B_out,
                              cudaStream_t stream, KernelInfo *info)
{
    dim3 grid((unsigned)L.blocks_per_point, 1, 1);
    if (floor_kind == kFloorAbs)
        fe_tangent_kernel<kFloorAbs><<<grid, kTangentThreads, 0, stream>>>(L, rb, S_out, V_out, B_out);
    else
        fe_tangent_kernel<kFloorPlus><<<grid, kTangentThreads, 0, stream>>>(L, rb, S_out, V_out, B_out);
    if (info) {
        info->grid_x = (int)grid.x;
        info->grid_y = 1;
        info->block_threads = kTangentThreads;
        info->paths_per_thread = kTangentPaths;
        cudaFuncAttributes fa{};
        const void *fn = floor_kind == kFloorAbs ? (const void *)fe_tangent_kernel<kFloorAbs> : (const void *)fe_tangent_kernel<kFloorPlus>;
        if (cudaFuncGetAttributes(&fa, fn) == cudaSuccess) info->regs_per_thread = fa.numRegs;
        info->param_bytes = (int)(sizeof(FeLaunch) + sizeof(ReduceBuffers) + 3 * sizeof(float *));
    }
    return cudaGetLastError();
}

cudaError_t launch_strike_greeks(const float *d_S, const float *d_B, unsigned long long n_local, const float *d_strikes,
                                 int n_strikes, float S0, ReduceBuffers rb, cudaStream_t stream)
{
    dim3 grid(kGreekBlocks, (unsigned)n_strikes, 1);
    strike_greeks_kernel<<<grid, kGreekThreads, 0, stream>>>(d_S, d_B, n_local, d_strikes, 1.0f / S0, rb);
    return cudaGetLastError();
}

int greek_blocks_per_slot() { return kGreekBlocks; }
int tangent_tile_paths() { return kTangentTile; }

}  // namespace nmchb
