// strike_kernels.cu -- strike vector + pathwise delta from the terminal prices of one path pass.
//
// The path kernels leave S_T of every local path in HBM (4 bytes per path; 64 MB at 2^24 paths, which stays in
// the 126 MB L2 between the two kernels).  This kernel folds them per strike: block (x, j) reduces a slice of the
// paths for strike j and writes two moment pairs -- (payoff, payoff^2) as reduction slot 2j and (delta, in-the-money
// count) as slot 2j+1 -- through the same deterministic FP64 ticket reduction as the path kernels.  A NaN path makes the
// strike's payoff and delta sums NaN, as in the path kernels (payoff_or_nan, DESIGN.md row A3); the count stays a count.
#include "kernels.cuh"

namespace nmchb {

constexpr int kStrikeThreads = 256;
constexpr int kStrikeBlocks = 296;          // 2 per SM: every block streams a contiguous slice with 16-byte loads

__global__ void __launch_bounds__(kStrikeThreads)
strike_moments_kernel(const float *__restrict__ S, unsigned long long n, const float *__restrict__ strikes,
                      float inv_S0, ReduceBuffers rb)
{
    const int j = blockIdx.y;
    const float K = strikes[j];
    double pay = 0.0, pay2 = 0.0, delta = 0.0, itm = 0.0;
    const unsigned long long n4 = n / 4ull;
    const float4 *S4 = reinterpret_cast<const float4 *>(S);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const float4 s = __ldg(S4 + i);
        const float v[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double p = payoff_or_nan(v[q], K);
            pay += p;
            pay2 += p * p;
            if (v[q] > K) {
                delta += (double)(v[q] * inv_S0);
                itm += 1.0;
            } else if (v[q] != v[q]) {                       // a NaN path: carried into delta too
                delta += (double)v[q];
            }
        }
    }
    if (blockIdx.x == 0) {                                   // ragged tail
        for (unsigned long long i = n4 * 4ull + threadIdx.x; i < n; i += blockDim.x) {
            const float v = S[i];
            const double p = payoff_or_nan(v, K);
            pay += p;
            pay2 += p * p;
            if (v > K) {
                delta += (double)(v * inv_S0);
                itm += 1.0;
            } else if (v != v) {
                delta += (double)v;
            }
        }
    }
    block_reduce_and_finish(pay, pay2, rb.partials, rb.tickets, rb.out, 2 * j, blockIdx.x, gridDim.x);
    block_reduce_and_finish(delta, itm, rb.partials, rb.tickets, rb.out, 2 * j + 1, blockIdx.x, gridDim.x);
}

cudaError_t launch_strike_moments(const float *d_S, unsigned long long n_local, const float *d_strikes, int n_strikes,
                                  float S0, ReduceBuffers rb, cudaStream_t stream)
{
    dim3 grid(kStrikeBlocks, (unsigned)n_strikes, 1);
    strike_moments_kernel<<<grid, kStrikeThreads, 0, stream>>>(d_S, n_local, d_strikes, 1.0f / S0, rb);
    return cudaGetLastError();
}

int strike_blocks_per_slot() { return kStrikeBlocks; }

}  // namespace nmchb
