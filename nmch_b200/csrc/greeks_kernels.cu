// greeks_kernels.cu -- the strike family: a strike vector with pathwise delta, and optionally pathwise sensitivities from
// the same pass: the vega d price / d v_0 (compute_greeks, ND = 1) or d price / d p for all five of v_0, kappa, theta,
// sigma, rho (compute_sensitivities, ND = 5) (SURVEY.md §8f rank 2 "a strike vector and pathwise delta/vega reuse the
// same paths at ~zero RNG cost"; the reference fixes K = S_0 and has no sensitivities, src/NMCH/methods/NMCH.cu:7).
//
// fe_tangent_kernel<FLOOR, ND>: the native FE step on the native Philox stream (the words, the instructions and therefore
//   the (S_T, V_T) of fe_philox_kernel, bit for bit) carrying the tangents (dV/dp, dS/dp) of every path in registers;
//   leaves S_T, V_T and dS_T/dp in HBM (8 + 4 ND bytes per path) and reduces the K = S_0 payoff moments like every path
//   kernel.
// strike_fold_kernel<ND>: folds the terminal arrays per strike: payoff moments, delta = 1{S_T > K} S_T / S_0, and per
//   direction 1{S_T > K} dS_T/dp and its square (for the standard error), through the deterministic ticket reduction.
//   ND = 0 (compute_strikes) folds S_T alone, as left by any path kernel.  A NaN path makes the strike's payoff, delta
//   and sensitivity sums NaN (DESIGN.md row A3); the in-the-money count stays a count.
#include "fe_step.cuh"
#include "kernels.cuh"

namespace nmchb {

constexpr int kTangentThreads = 256;
// Paths per thread, from -Xptxas -v (sm_100a, no spills in any of these):
//   ND = 1 (compute_greeks): two paths, 52 registers at 4 blocks of 256 (32 warps per SM);
//   ND = 5 (compute_sensitivities): eleven floats of state per path instead of four.  One path takes 48 registers
//   (5 blocks of 256, 40 warps per SM); two paths fit 4 blocks in 64 (32 warps).  On a B200 (1000 W) one path per thread
//   is faster: 56.5 against 61.7 ms at 2^24 paths x 1000 steps (profiles/r03_sensitivities_time.json, DESIGN.md §4.6c).
//   -DNMCHB_SENS_PATHS=2 builds the other choice for that comparison.
#ifndef NMCHB_SENS_PATHS
#define NMCHB_SENS_PATHS 1
#endif
template <int ND> struct TangentShape;
template <> struct TangentShape<1> { static constexpr int kPaths = 2, kMinBlocks = 4; };
template <> struct TangentShape<kNumDirs> { static constexpr int kPaths = NMCHB_SENS_PATHS, kMinBlocks = 4; };

// The loop of fe_philox_kernel (fe_kernels.cu) with the tangent step: one tile of P * kTangentThreads paths per block,
// the Philox counter split where its low word would wrap so that the per-path invariants of rounds 1-2 are hoisted and
// the path-independent multiplies sit on the uniform datapath; a pass may start on the second half of a block (an odd
// number of steps before it) and end on a first half.  Direction d of dS_T lands in B_out[d * n_local + path] (structure
// of arrays, direction d at B_out + d * tangent_stride(n_local)); tf is read only when ND > 1.
template <int FLOOR, int ND>
__global__ void __launch_bounds__(kTangentThreads, TangentShape<ND>::kMinBlocks)
fe_tangent_kernel(const __grid_constant__ FeLaunch L, ReduceBuffers rb, float *__restrict__ S_out,
                  float *__restrict__ V_out, float *__restrict__ B_out, const __grid_constant__ TangentFold tf)
{
    constexpr int P = TangentShape<ND>::kPaths;
    constexpr int kTile = P * kTangentThreads;
    NMCHB_ASSERT(blockDim.x == kTangentThreads && (int)blockIdx.x < L.blocks_per_point && L.n_points == 1);
    NMCHB_ASSERT(L.first_path % kTile == 0);
    const unsigned long long local0 = (unsigned long long)blockIdx.x * kTile;
    const unsigned long long g0 = L.first_path + local0;         // multiple of the tile: no carry below
    uint32_t path_hi = (uint32_t)(g0 >> 32);
    asm volatile("" : "+r"(path_hi));
    const uint32_t path_lo0 = (uint32_t)g0 + threadIdx.x;
    NMCHB_ASSERT(((g0 + (unsigned long long)(kTile - 1)) >> 32) == (g0 >> 32));
    const FePoint pc = L.pt0;

    float S[P], V[P], A[P][ND], B[P][ND];
#pragma unroll
    for (int j = 0; j < P; ++j) {
        S[j] = L.S0;
        V[j] = L.v0;
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            A[j][d] = (d == kDirV0) ? 1.0f : 0.0f;
            B[j][d] = 0.0f;
        }
    }
    const unsigned long long w0 = L.draw_offset;
    unsigned long long blk = w0 >> 2;
    int n = L.N;
    const bool resume = (w0 & 2ull) != 0ull && n > 0;            // start on the second word pair of a block
    if (resume) {
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const U4 w = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), path_lo0 + j * kTangentThreads, path_hi, L.keys);
            fe_step_native_tangent<FLOOR, ND>(S[j], V[j], A[j], B[j], w.z, w.w, L.rdt, L.zr, L.zc, pc, tf);
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
                fe_step_native_tangent<FLOOR, ND>(S[j], V[j], A[j], B[j], w.x, w.y, L.rdt, L.zr, L.zc, pc, tf);
                fe_step_native_tangent<FLOOR, ND>(S[j], V[j], A[j], B[j], w.z, w.w, L.rdt, L.zr, L.zc, pc, tf);
            }
        }
        blk += (unsigned long long)chunk;
        pairs -= chunk;
    }
    if (n & 1) {
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const U4 w = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), path_lo0 + j * kTangentThreads, path_hi, L.keys);
            fe_step_native_tangent<FLOOR, ND>(S[j], V[j], A[j], B[j], w.x, w.y, L.rdt, L.zr, L.zc, pc, tf);
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
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                const unsigned long long at = (unsigned long long)d * tangent_stride(L.n_local) + idx;
                NMCHB_ASSERT(at < (unsigned long long)ND * tangent_stride(L.n_local));
                B_out[at] = B[j][d];
            }
        }
    }
    block_reduce_and_finish(pay, pay2, rb.partials, rb.tickets, rb.out, 0, blockIdx.x, L.blocks_per_point);
}

constexpr int kFoldThreads = 256;
constexpr int kFoldBlocks = 296;            // 2 per SM: every block streams a contiguous slice with 16-byte loads
// per-direction arrays of the fold: ND = 0 keeps one unused element (C++ has no zero-length arrays)
template <int ND> constexpr int kDirSlots = ND > 0 ? ND : 1;

// One path into the sums of one strike: payoff moments, delta = 1{S_T > K} S_T / S_0, the in-the-money count and, per
// direction, 1{S_T > K} dS_T/dp and its square.  b[d] is dS_T/dp_d of the path.
template <int ND>
__device__ __forceinline__ void greek_fold(float s, const float (&b)[kDirSlots<ND>], float K, float inv_S0, double &pay,
                                           double &pay2, double &delta, double &itm, double (&sens)[kDirSlots<ND>],
                                           double (&sens2)[kDirSlots<ND>])
{
    const double p = payoff_or_nan(s, K);
    pay += p;
    pay2 += p * p;
    if (s > K) {
        delta += (double)(s * inv_S0);
        itm += 1.0;
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            sens[d] += (double)b[d];
            sens2[d] += (double)b[d] * (double)b[d];
        }
    } else if (s != s) {                                     // a NaN path: carried into delta and every sensitivity too
        delta += (double)s;
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            sens[d] += (double)s;
            sens2[d] += (double)s;
        }
    }
}

// Reduction slots of strike j (relative to rb.tickets): (2 + ND) j = (payoff, payoff^2), + 1 = (delta, itm),
// + 2 + d = (sum, sum of squares) of direction d.  B holds ND arrays of n paths, tangent_stride(n) floats apart (not read
// when ND = 0).
template <int ND>
__global__ void __launch_bounds__(kFoldThreads)
strike_fold_kernel(const float *__restrict__ S, const float *__restrict__ B, unsigned long long n,
                   const float *__restrict__ strikes, float inv_S0, ReduceBuffers rb)
{
    constexpr int kSlots = 2 + ND;
    const unsigned long long stride = tangent_stride(n);
    const int j = blockIdx.y;
    const float K = strikes[j];
    constexpr int NB = kDirSlots<ND>;
    double pay = 0.0, pay2 = 0.0, delta = 0.0, itm = 0.0, sens[NB], sens2[NB];
#pragma unroll
    for (int d = 0; d < ND; ++d) sens[d] = sens2[d] = 0.0;
    const unsigned long long n4 = n / 4ull;
    const float4 *S4 = reinterpret_cast<const float4 *>(S);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const float4 s = __ldg(S4 + i);
        if constexpr (ND == 0) {
            // the loop form of the former S_T-only fold: ptxas schedules it faster than four calls (761 against
            // 798 us for 64 strikes at 2^24 paths on a B200), with the same additions in the same order
            const float v[4] = {s.x, s.y, s.z, s.w};
            const float none[NB] = {};
#pragma unroll
            for (int q = 0; q < 4; ++q) greek_fold<ND>(v[q], none, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
        } else {
            float4 b[ND];
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                NMCHB_ASSERT(4ull * i + 3ull < stride);
                b[d] = __ldg(reinterpret_cast<const float4 *>(B + (unsigned long long)d * stride) + i);
            }
            float bx[ND], by[ND], bz[ND], bw[ND];
#pragma unroll
            for (int d = 0; d < ND; ++d) { bx[d] = b[d].x; by[d] = b[d].y; bz[d] = b[d].z; bw[d] = b[d].w; }
            greek_fold<ND>(s.x, bx, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
            greek_fold<ND>(s.y, by, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
            greek_fold<ND>(s.z, bz, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
            greek_fold<ND>(s.w, bw, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
        }
    }
    if (blockIdx.x == 0)                                     // ragged tail
        for (unsigned long long i = n4 * 4ull + threadIdx.x; i < n; i += blockDim.x) {
            float bi[NB];
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                NMCHB_ASSERT(i < n);
                bi[d] = B[(unsigned long long)d * stride + i];
            }
            greek_fold<ND>(S[i], bi, K, inv_S0, pay, pay2, delta, itm, sens, sens2);
        }
    NMCHB_ASSERT(j >= 0 && j < (int)gridDim.y);
    block_reduce_and_finish(pay, pay2, rb.partials, rb.tickets, rb.out, kSlots * j, blockIdx.x, gridDim.x);
    block_reduce_and_finish(delta, itm, rb.partials, rb.tickets, rb.out, kSlots * j + 1, blockIdx.x, gridDim.x);
#pragma unroll
    for (int d = 0; d < ND; ++d)
        block_reduce_and_finish(sens[d], sens2[d], rb.partials, rb.tickets, rb.out, kSlots * j + 2 + d, blockIdx.x, gridDim.x);
}

template <int ND>
static cudaError_t launch_fe_tangent_nd(const FeLaunch &L, int floor_kind, const TangentFold &tf, ReduceBuffers rb,
                                        float *S_out, float *V_out, float *B_out, cudaStream_t stream, KernelInfo *info)
{
    dim3 grid((unsigned)L.blocks_per_point, 1, 1);
    if (floor_kind == kFloorAbs)
        fe_tangent_kernel<kFloorAbs, ND><<<grid, kTangentThreads, 0, stream>>>(L, rb, S_out, V_out, B_out, tf);
    else
        fe_tangent_kernel<kFloorPlus, ND><<<grid, kTangentThreads, 0, stream>>>(L, rb, S_out, V_out, B_out, tf);
    if (info) {
        info->grid_x = (int)grid.x;
        info->grid_y = 1;
        info->block_threads = kTangentThreads;
        info->paths_per_thread = TangentShape<ND>::kPaths;
        cudaFuncAttributes fa{};
        const void *fn = floor_kind == kFloorAbs ? (const void *)fe_tangent_kernel<kFloorAbs, ND>
                                                 : (const void *)fe_tangent_kernel<kFloorPlus, ND>;
        if (cudaFuncGetAttributes(&fa, fn) == cudaSuccess) info->regs_per_thread = fa.numRegs;
        info->param_bytes = (int)(sizeof(FeLaunch) + sizeof(ReduceBuffers) + 3 * sizeof(float *) + sizeof(TangentFold));
    }
    return cudaGetLastError();
}

cudaError_t launch_fe_tangent(const FeLaunch &L, int floor_kind, int n_dirs, const TangentFold &tf, ReduceBuffers rb,
                              float *S_out, float *V_out, float *B_out, cudaStream_t stream, KernelInfo *info)
{
    if (n_dirs == 1) return launch_fe_tangent_nd<1>(L, floor_kind, tf, rb, S_out, V_out, B_out, stream, info);
    if (n_dirs == kNumDirs) return launch_fe_tangent_nd<kNumDirs>(L, floor_kind, tf, rb, S_out, V_out, B_out, stream, info);
    return cudaErrorInvalidValue;
}

cudaError_t launch_strike_fold(const float *d_S, const float *d_B, int n_dirs, unsigned long long n_local,
                               const float *d_strikes, int n_strikes, float S0, ReduceBuffers rb, cudaStream_t stream)
{
    dim3 grid(kFoldBlocks, (unsigned)n_strikes, 1);
    if (n_dirs == 0)
        strike_fold_kernel<0><<<grid, kFoldThreads, 0, stream>>>(d_S, d_B, n_local, d_strikes, 1.0f / S0, rb);
    else if (n_dirs == 1)
        strike_fold_kernel<1><<<grid, kFoldThreads, 0, stream>>>(d_S, d_B, n_local, d_strikes, 1.0f / S0, rb);
    else if (n_dirs == kNumDirs)
        strike_fold_kernel<kNumDirs><<<grid, kFoldThreads, 0, stream>>>(d_S, d_B, n_local, d_strikes, 1.0f / S0, rb);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

int strike_blocks_per_slot() { return kFoldBlocks; }
int tangent_tile_paths(int n_dirs)
{
    return (n_dirs == 1 ? TangentShape<1>::kPaths : TangentShape<kNumDirs>::kPaths) * kTangentThreads;
}

}  // namespace nmchb
