// em_kernels.cu -- "exact method" (EM) Heston path kernels for sm_100a.
//
// Reference scheme (src/NMCH/methods/NMCH_EM.cu:213-260): per time step the variance makes an EXACT CIR
// transition  V' = c * Gamma(d + Poisson(lc * V)),  c = sigma^2 (1-e^{-k dt}) / (2k),  d = 2 k theta / sigma^2,
// lc = 2k e^{-k dt} / (sigma^2 (1 - e^{-k dt}));  the integrated variance is the trapezoid sum; one conditional
// log-normal draw gives S_T.
//
// em_native_kernel -- the product path.  V'/c is a scaled noncentral chi-square, sampled exactly by
//   d > 1/2 :  Gamma(d + Poisson(l)) =d= (Z + sqrt(2 l))^2 / 2 + Gamma(d - 1/2)           (one normal, one gamma
//              of CONSTANT shape: Marsaglia-Tsang constants are per-point, no Poisson, no data-dependent regime)
//              A trial takes 64 bits (23-bit radius, 18-bit angle, 23-bit accept uniform): two trials per Philox block.
//              Shape d - 1/2 < 1 needs the boost Gamma(a) = Gamma(a+1) U^(1/a); its uniform costs no random bits:
//              the accept test  -lg2 u < t  leaves, on acceptance, the excess  -lg2 u - t  as a fresh exponential
//              (memorylessness), so U = 2^-(excess) is uniform and independent of the accepted proposal.
//   d <= 1/2:  Poisson (inversion below 10, Hoermann PTRS above) then Marsaglia-Tsang gamma of shape d + N
//   Rejections do not loop inside a step: every loop iteration is a group of trials on fresh Philox bits and a lane
//   commits its step only if the trial accepted, so a warp never waits on its slowest lane's retry.  One
//   instantiation per sampler for launches whose points are all of one kind; a grid holding several kinds is ONE
//   launch of the kEmAny instantiation, which picks the sampler per block from the point record (block-uniform).
// em_compat_kernel -- validation path: the reference's own draw sequence (cuRAND's curand_poisson /
//   curand_normal / curand_uniform on a cuRAND-layout state) and its FP32 expressions, so results can be
//   compared with the reference's CUDA build on identical seeds.
#include <curand_kernel.h>

#include <algorithm>
#include <vector>

#include "compat_math.cuh"
#include "engine_internal.cuh"

namespace nmchb {

// ------------------------------------------------------------------------------------------
// native kernel
// ------------------------------------------------------------------------------------------
struct EmPoint {
    float scale;        // c
    float lc;
    float d;            // 2 k theta / sigma^2
    float a;            // fast path: gamma shape d - 1/2 (boosted by +1 when < 1)
    float mt_d, mt_c;   // Marsaglia-Tsang constants of the fast path's gamma
    float inv_a;        // 1/a when boosting, else 0
    // fast path with every constant folded (normals are produced as n' = n / c0, c0 = sqrt(2 ln 2)):
    float f_c;          // mt_c * c0
    float f_h;          // 0.5 * c0^2 * log2(e)    log test, log2 domain
    float f_dl;         // mt_d * log2(e)
    float f_g2s;        // mt_d * c                gamma term of V' = (c/2) (t^2 + 2 Gamma(a))
    float f_t1;         // c0 * sqrt(c/2)          V' = (f_t1 z' + sqrt(f_ev V))^2 + f_g2s v [boost]
    float f_ev;         // lc * c = e^{-k dt}
    float f_scale;      // c / 2                   (Poisson-mixture path)
    float f_hs;         // f_h / f_c^2             log test on the SCALED proposal xs = f_c x'
    float f_lg2s;       // log2(f_g2s)             boosted gamma term assembled in the log2 domain
    float k, ktheta_T, inv_sigma;
    int   kind;         // kEmSplit (boosted gamma, 1/2 < d < 3/2), kEmSplitPacked (d >= 3/2) or kEmMixture (d <= 1/2)
    int   index;        // position of the point in the caller's list (stream id, result slot): launches group points by kind
};

struct EmLaunch {
    PhiloxKeys keys;
    unsigned long long first_path, n_local;
    unsigned int call0;              // stream id of point 0 (engine call counter)
    int   N, n_points, blocks_per_point;
    float v0, K, half_dt, rho, one_m_rho2, lnS0_rT;
    EmPoint pt0;
};

__device__ __forceinline__ float u01_open(uint32_t w)          // (0,1), 23 bits
{
    return bits_to_1_2(w) - 0.99999994f;
}

__device__ __forceinline__ void box_muller_fast(uint32_t wa, uint32_t wb, float &n1, float &n2)
{
    const float r = sqrt_approx(-1.38629436f * lg2_approx(u01_open(wa)));     // sqrt(-2 ln u)
    const float ang = bits_to_1_2(wb) * 6.2831855f;
    n1 = r * sin_approx(ang);
    n2 = r * cos_approx(ang);
}

// log2(k!) for k < 10; copied to shared memory by the kernels that sample Poisson counts (a per-lane index into
// constant memory would serialise)
__constant__ float kLg2Factorial[10] = {0.0f, 0.0f, 1.0f, 2.5849625f, 4.5849625f, 6.9068906f,
                                        9.4918531f, 12.2992080f, 15.2992080f, 18.4691330f};

// One Hoermann-PTRS trial for Poisson(mu), mu >= 10, from two uniforms.  Returns accept, result in k.
// Branch-free: the algorithm's quick-acceptance squeeze is dropped (it only short-cuts trials the exact test accepts),
// and the exact test   ln(v inv_alpha / (a / us^2 + b)) <= -mu + k ln mu - ln k!   is evaluated in the log2 domain with
// single-instruction transcendentals, arranged so that none of them amplifies its 2^-22 absolute error:
//   k >= 10:  ln k! by Stirling (three terms: 1e-8 at k = 10), so the right side is
//               k (ln(1 - delta) + delta) - ln(2 pi k)/2 - 1/(12k) + 1/(360k^3),     delta = (k - mu) / k
//             ln(1 - delta) + delta = -delta s - 2 s^3 (1/3 + s^2/5 + s^4/7 + s^6/9 + s^8/11),  s = delta / (2 - delta)
//             (the atanh series; no cancellation; used while |s| < 0.3, i.e. |delta| < 0.46 -- beyond that the plain
//             lg2(mu / k) is far from zero and accurate enough).  ln(2 pi k)/2 rides in the left side's logarithm.
//   k < 10:   -mu + k ln mu - ln k! directly (table), values of order 10.
__device__ __forceinline__ bool ptrs_trial(float mu, float u_raw, float v, const float *__restrict__ lg2fact, float &k)
{
    constexpr float kLn2 = 0.69314718f, kLog2e = 1.44269504f;
    const float smu = sqrt_approx(mu);
    const float b = fmaf(2.53f, smu, 0.931f);
    const float a = fmaf(0.02483f, b, -0.059f);
    // the hat's constants may be approximate (MUFU.RCP, 1e-7): they only shape the proposal and enter the exact test
    // below consistently
    const float inv_alpha = fmaf(1.1328f, rcp_approx(b - 3.4f), 1.1239f);
    const float u = u_raw - 0.5f;
    const float us = 0.5f - fabsf(u);
    const float inv_us = rcp_approx(us);
    k = floorf(fmaf(fmaf(2.0f * a, inv_us, b), u, mu + 0.43f));
    const bool big = k >= 10.0f;
    const float t = v * inv_alpha * rcp_approx(fmaf(a * inv_us, inv_us, b));
    // left side (log2): lg2(t), plus lg2(2 pi k)/2 when Stirling is used: one logarithm of t^2 * 2 pi k, halved
    const float lhs = 0.5f * lg2_approx(big ? (t * t) * (6.28318531f * k) : t * t);
    const float ik = rcp_approx(big ? k : 1.0f);
    const float delta = (k - mu) * ik;
    const float sv = delta * rcp_approx(2.0f - delta);
    const float s2 = sv * sv;
    float poly = fmaf(s2, 1.0f / 11.0f, 1.0f / 9.0f);
    poly = fmaf(poly, s2, 1.0f / 7.0f);
    poly = fmaf(poly, s2, 1.0f / 5.0f);
    poly = fmaf(poly, s2, 1.0f / 3.0f);
    const float f_series = -fmaf(2.0f * sv * s2, poly, delta * sv);           // ln(1 - delta) + delta
    const bool near = fabsf(sv) < 0.3f;
    // one more logarithm serves both remaining cases: lg2(mu / k) (k >= 10, far from mu) or lg2(mu) (k < 10)
    const float lgx = lg2_approx(big ? mu * ik : mu);
    const float f_log = fmaf(lgx, kLn2, delta);                               // ln(mu/k) + 1 - mu/k
    const float ik2 = ik * ik;
    const float stirling = ik * fmaf(ik2, 1.0f / 360.0f, -1.0f / 12.0f);      // -1/(12k) + 1/(360k^3)
    const float rhs_big = fmaf(k, near ? f_series : f_log, stirling) * kLog2e;
    const int ki = big ? 0 : max((int)k, 0);
    const float rhs_small = fmaf(k, lgx, -fmaf(mu, kLog2e, lg2fact[ki]));
    const float rhs = big ? rhs_big : rhs_small;
    return (k >= 0.0f) && !(us < 0.013f && v > us) && (lhs <= rhs);
}

// Poisson by inversion (mu < 10): exact, one uniform.
__device__ __forceinline__ float poisson_inversion(float mu, float u)
{
    float p = ex2_approx(-1.44269504f * mu), cdf = p, k = 0.0f;
    while (u > cdf && k < 80.0f) {
        k += 1.0f;
        p *= mu * rcp_approx(k);
        cdf += p;
    }
    return k;
}

// One trial of the chi-square split from TWO Philox words, every constant folded on the host, no data-dependent
// branch:   2 V'/c = (Z + sqrt(2 l))^2 + 2 Gamma(a),   Z = c0 z', X = c0 x' from one Box-Muller pair.
//   radius uniform = wa[31:9] (23 bits)    angle = wa[8:0] : wc[31:23] (18 bits; an equispaced grid of 2^18 angles keeps
//   every trigonometric moment below that order exact)    accept-test uniform = wc[22:0] (23 bits)
// Marsaglia-Tsang trial for Gamma(a [+1]) with x = c0 xp, v = (1 + c x)^3: accept iff v > 0 and
//   lg2 u < rhs = (x^2/2 + d (1 - v)) log2 e + d log2 v         (the exact test; no squeeze, hence no divergence;
//   evaluated on the scaled proposal xs = mt_c x with f_hs = log2 e / (2 mt_c^2), so that v = (1 + xs)^3)
// BOOST (shape a < 1): Gamma(a) = Gamma(a+1) U^(1/a) with U = 2^(lg2 u - rhs): given acceptance, rhs - lg2 u is an
// exponential (rate ln 2) independent of the proposal -- the accept uniform's unused excess, so no extra random field
// and one MUFU.EX2 instead of LG2 + EX2.  (Marsaglia-Tsang's acceptance ratio never exceeds one, i.e. rhs <= 0.)
// Returns accept; zp = Z / c0, g2 = c Gamma(a) (the gamma term already scaled to V').
template <bool BOOST>
__device__ __forceinline__ bool em_split_trial(uint32_t wa, uint32_t wc, const EmPoint &pc, float &zp, float &g2)
{
    const float rad = sqrt_approx(-lg2_approx(u01_open(wa)));
    // (wa << 14 | wc >> 18) masked to mantissa bits 22..5, exponent of [1, 2) -- one funnel shift, one LOP3
    const float ang = __uint_as_float(and_or(__funnelshift_r(wc, wa, 18), 0x7fffe0u, 0x3f800000u)) * 6.2831855f;
    zp = rad * sin_approx(ang);
    // Every FP32 instruction below has at most ONE operand that is not a per-thread register (a point constant in a
    // uniform register, or an immediate): an FFMA with two of them costs a register move per trial.
    const float xs = (rad * pc.f_c) * cos_approx(ang);        // mt_c x: the proposal already scaled
    const float v1 = xs + 1.0f;
    const float v = v1 * v1 * v1;
    const float lv = lg2_approx(v);                           // v1 <= 0: NaN (v < 0) or -inf (v = 0), so the comparison
    float rhs = (xs * xs) * pc.f_hs;                          // below is false: no separate v1 > 0 test
    rhs = fmaf(1.0f - v, pc.f_dl, rhs);
    rhs = fmaf(lv, pc.mt_d, rhs);
    const float lu = lg2_approx(__uint_as_float(and_or(wc, 0x7fffffu, 0x3f800000u)) - 0.99999994f);
    if constexpr (BOOST) g2 = ex2_approx(fmaf(lu - rhs, pc.inv_a, lv + pc.f_lg2s));   // f_g2s v U^(1/a), one EX2
    else g2 = pc.f_g2s * v;
    return lu < rhs;
}

// Block shape of the native kernel (tuning builds may override: -DNMCHB_EM_THREADS=.. -DNMCHB_EM_MINB=..)
#ifndef NMCHB_EM_THREADS
#define NMCHB_EM_THREADS 256
#endif
#ifndef NMCHB_EM_MINB
#define NMCHB_EM_MINB 6
#endif
constexpr int kEmThreads = NMCHB_EM_THREADS;

// KIND: kEmSplit = the chi-square split with the boosted gamma (1/2 < d < 3/2); kEmSplitPacked = the split for points
// that need no boost (d >= 3/2); kEmMixture = the Poisson mixture (d <= 1/2); kEmAny = the sampler is read from the
// point record per block (block-uniform switch) -- what a sweep over points of several kinds launches, ONCE.
constexpr int kEmSplit = 0, kEmMixture = 1, kEmSplitPacked = 2, kEmAny = 3;

// The variance path of one thread: N exact CIR transitions on Philox blocks 0, 1, ... of its stream.  Returns with
// V = V_N, acc = V_1 + ... + V_N and blk = the first unused block (the terminal draw takes it).
template <int KIND, typename NextBlock>
__device__ __forceinline__ void em_variance_path(const EmLaunch &L, const EmPoint &pc, bool valid, NextBlock next_block,
                                                 const float *__restrict__ lg2fact, float &V, float &acc, uint32_t &blk)
{
    int step = valid ? 0 : L.N;                              // lanes past the end of the shard take part in the votes only
    if constexpr (KIND == kEmSplit || KIND == kEmSplitPacked) {
        // chi-square split: two trials per Philox block, four per iteration (em_split_trial).  Only the last FFMA pair
        // of a trial depends on V, so the four trials of a group overlap.  The loop is warp-uniform (vote): the block
        // counter is the same in every lane, and with it the path-independent multiplies of a block.
        // While EVERY lane still has four steps to go, a group of four trials cannot overshoot N: no bound test per trial.
        while (__all_sync(0xffffffffu, step + 4 <= L.N)) {
            const U4 b0 = next_block(blk), b1 = next_block(blk + 1u);
            blk += 2u;
            const uint32_t w[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float zp, g2;
                const bool ok = em_split_trial<KIND == kEmSplit>(w[2 * j], w[2 * j + 1], pc, zp, g2);
                const float t = fmaf(pc.f_t1, zp, sqrt_approx(pc.f_ev * V));
                const float Vn = fmaf(t, t, g2);
                if (ok) {
                    acc = __fadd_rn(acc, Vn);
                    V = Vn;
                    ++step;
                }
            }
        }
        // the last few steps of the warp's slowest and fastest lanes: the same group, with the bound test
        while (__any_sync(0xffffffffu, step < L.N)) {
            const U4 b0 = next_block(blk), b1 = next_block(blk + 1u);
            blk += 2u;
            const uint32_t w[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float zp, g2;
                const bool ok = em_split_trial<KIND == kEmSplit>(w[2 * j], w[2 * j + 1], pc, zp, g2);
                const float t = fmaf(pc.f_t1, zp, sqrt_approx(pc.f_ev * V));
                const float Vn = fmaf(t, t, g2);             // = (c/2) ((Z + sqrt(2 l))^2 + 2 Gamma(a))
                if (ok && step < L.N) {
                    acc = __fadd_rn(acc, Vn);
                    V = Vn;
                    ++step;
                }
            }
        }
    } else {
        // Poisson mixture (d <= 1/2): per iteration ONE Philox block (x, y, z, w) feeds a Poisson trial -- uniforms from
        // x[31:9] and y[31:9] -- and, from disjoint bits, one Marsaglia-Tsang trial for Gamma(d + N): radius z[31:9],
        // angle z[8:0] : w[31:23], accept uniform w[22:0]; the shape < 1 boost (N = 0) is recycled from the accept test
        // like in the split sampler.  A lane that already holds N skips the Poisson part, so a gamma retry never re-draws
        // (and never biases) N.  The gamma trial itself is branch-free with a per-lane shape:
        //   accept iff lg2 u < md (log2e (4.5 xs^2 + 1 - v) + lg2 v),  xs = x / sqrt(9 md),  v = (1 + xs)^3,  md = shape - 1/3.
        // Acceptance rates are >= 0.85 per trial and the host validates every folded constant (finite, positive),
        // so the loop terminates; the cap is a belt against a hang: a path that exhausts it ends early with V = NaN,
        // which the payoff stage carries into the sums (a NaN result, not a silently dropped path).
        bool have_np = false;
        float np = 0.0f;
        const uint32_t max_blocks = 64u * (uint32_t)L.N + 4096u;
        const float inv_d = rcp_approx(pc.d);
        while (step < L.N) {
            if (blk > max_blocks) { V = __int_as_float(0x7fc00000); break; }
            const U4 w = next_block(blk++);
            if (!have_np) {
                const float mu = pc.lc * V;
                if (mu < 10.0f) {
                    np = poisson_inversion(mu, u01_open(w.x));
                    have_np = true;
                } else {
                    have_np = ptrs_trial(mu, u01_open(w.x), u01_open(w.y), lg2fact, np);
                }
            }
            {
                const float shape0 = pc.d + np;
                const bool small = shape0 < 1.0f;                      // only for N = 0: Gamma(d) = Gamma(d + 1) U^(1/d)
                const float md = (small ? shape0 + 1.0f : shape0) - (1.0f / 3.0f);
                const float rad = sqrt_approx(-lg2_approx(u01_open(w.z)));
                const float ang = __uint_as_float(and_or(__funnelshift_r(w.w, w.z, 18), 0x7fffe0u, 0x3f800000u)) * 6.2831855f;
                const float xs = (rad * (1.1774100f * rsqrt_approx(9.0f * md))) * cos_approx(ang);   // c0 rad cos / sqrt(9 md)
                const float v1 = xs + 1.0f;
                const float v = v1 * v1 * v1;
                const float lv = lg2_approx(v);                        // v1 <= 0: NaN or -inf, the test below fails
                const float rhs = md * fmaf(fmaf(4.5f * xs, xs, 1.0f - v), 1.44269504f, lv);
                const float lu = lg2_approx(__uint_as_float(and_or(w.w, 0x7fffffu, 0x3f800000u)) - 0.99999994f);
                const float boost = ex2_approx((lu - rhs) * inv_d);
                const float gam = md * v * (small ? boost : 1.0f);
                if (have_np && lu < rhs) {
                    const float Vn = __fmul_rn(pc.scale, gam);
                    acc = __fadd_rn(acc, Vn);
                    V = Vn;
                    ++step;
                    have_np = false;
                }
            }
        }
    }
}

template <int KIND>
__global__ void __launch_bounds__(kEmThreads, NMCHB_EM_MINB)
em_native_kernel(const __grid_constant__ EmLaunch L, const EmPoint *__restrict__ pts, ReduceBuffers rb,
                 float *__restrict__ S_out, float *__restrict__ V_out)
{
    const EmPoint pc = (pts != nullptr) ? pts[blockIdx.y] : L.pt0;
    const int point = pc.index;
    // Paths of this block.  Written with the literal block size for the boosted split sampler and with blockDim.x for
    // the others: with the literal, ptxas keeps the two path-independent Philox multiplies of every block on the uniform
    // datapath (32 instead of 34 vector IMAD.WIDE per four trials) at the price of a few register moves -- measured on one
    // box (scripts/r02_em_ab.py): boosted 9.86 -> 9.74 ms, but unboosted 8.97 -> 9.10 and mixture 36.6 -> 37.6, so each
    // instantiation takes the form that is faster for it.
    const unsigned long long block0 = (KIND == kEmSplit) ? (unsigned long long)blockIdx.x * kEmThreads
                                                         : (unsigned long long)blockIdx.x * blockDim.x;
    const unsigned long long idx = block0 + threadIdx.x;
    const bool valid = idx < L.n_local;
    NMCHB_ASSERT(point >= 0 && point < L.n_points && blockDim.x == kEmThreads);
    // first_path is a multiple of 4096 (checked at create): the high counter word is the same for the whole block
    const unsigned long long g0 = L.first_path + block0;
    const uint32_t path_lo = (uint32_t)g0 + threadIdx.x;
    uint32_t path_hi = (uint32_t)(g0 >> 32);
    asm volatile("" : "+r"(path_hi));                       // computed once, not re-derived from blockIdx in the loop
    const uint32_t stream = L.call0 + (uint32_t)point;      // ctr.y: one stream per compute() call / point

    __shared__ float s_lg2fact[10];                        // log2(k!) for the Poisson sampler's small counts
    if constexpr (KIND == kEmMixture || KIND == kEmAny) {
        if (threadIdx.x < 10) s_lg2fact[threadIdx.x] = kLg2Factorial[threadIdx.x];
        __syncthreads();
    }
    float V = L.v0, acc = 0.0f, S = 0.0f;                  // acc = V_1 + ... + V_n so far
    {
        // counter = (trial block, stream, path_lo, path_hi): everything but the first word is fixed for this path
        const PhiloxPathInv inv = philox_path_invariants(stream, path_lo, L.keys);
        auto next_block = [&](uint32_t b) {
            return philox4x32_10_hoisted(philox_block_uniform(b, path_hi, L.keys), inv, L.keys);
        };
        uint32_t blk = 0;
        if constexpr (KIND == kEmAny) {
            if (pc.kind == kEmSplitPacked) em_variance_path<kEmSplitPacked>(L, pc, valid, next_block, s_lg2fact, V, acc, blk);
            else if (pc.kind == kEmSplit) em_variance_path<kEmSplit>(L, pc, valid, next_block, s_lg2fact, V, acc, blk);
            else em_variance_path<kEmMixture>(L, pc, valid, next_block, s_lg2fact, V, acc, blk);
        } else {
            em_variance_path<KIND>(L, pc, valid, next_block, s_lg2fact, V, acc, blk);
        }
        // terminal draw (NMCH_EM.cu:247-260, generalised to S_0, r, T)
        const U4 w = next_block(blk);
        float z, unused;
        box_muller_fast(w.x, w.y, z, unused);
        // trapezoid sum of NMCH_EM.cu:243,  sum_i (V_i + V_{i+1}) = 2 (V_1 + ... + V_N) + V_0 - V_N,  times dt / 2
        const float vI = fmaf(2.0f, acc, L.v0 - V) * L.half_dt;
        float m = pc.inv_sigma * (V - L.v0 - pc.ktheta_T + pc.k * vI);
        m = fmaf(L.rho, m, fmaf(-0.5f, vI, L.lnS0_rT));
        S = __expf(fmaf(sqrt_approx(L.one_m_rho2 * vI), z, m));
    }
    double pay = 0.0;
    if (valid) {
        pay = payoff_or_nan(S, L.K);
        if (S_out != nullptr && point == L.n_points - 1) {
            S_out[idx] = S;
            V_out[idx] = V;
        }
    }
    block_reduce_and_finish(pay, pay * pay, rb.partials, rb.tickets, rb.out, point, blockIdx.x, L.blocks_per_point);
}

// ------------------------------------------------------------------------------------------
// compat kernel: the reference's draws (cuRAND device API on a cuRAND-layout state) and expressions
// ------------------------------------------------------------------------------------------
struct EmCompatLaunch {
    unsigned long long n_local;
    int   N, n_points, blocks_per_point;
    float S0, v0, K, rho, dt;
    RawPoint raw0;
};

// Marsaglia-Tsang exactly as the reference draws it (NMCH_EM.cu:11-55): boost uniform BEFORE the loop, one
// cached-pair normal and one uniform per trial.
template <typename State>
__device__ __forceinline__ float gamma_compat(State *st, float alpha)
{
    float boost = 1.0f;
    if (alpha < 1.0f) {
        boost = powf(curand_uniform(st), 1.0f / alpha);
        alpha += 1.0f;
    }
    const float d = alpha - 1.0f / 3.0f;
    const float c = 1.0f / sqrtf(9.0f * d);
    for (;;) {
        float x, v;
        do {
            x = curand_normal(st);
            v = 1.0f + c * x;
        } while (v <= 0.0f);
        v = v * v * v;
        const float u = curand_uniform(st);
        const float x2 = x * x;
        if (u < 1.0f - 0.0331f * x2 * x2 || logf(u) < 0.5f * x2 + d * (1.0f - v + logf(v))) return d * v * boost;
    }
}

template <typename State>
__device__ __forceinline__ float em_path_compat(State *st, const EmCompatLaunch &L, const RawPoint &rp, float &V_T)
{
    const float k = rp.k, theta = rp.theta, sigma = rp.sigma, rho = L.rho, dt = L.dt, v_0 = L.v0;
    const float exp_kdt = expf(-k * dt);
    const float d = 2.0f * k * theta / (sigma * sigma);
    const float lambda_const = (2 * k * exp_kdt) / (sigma * sigma * (1 - exp_kdt));
    float Vt = v_0, vI = 0.0f;
    for (int i = 0; i < L.N; ++i) {
        const float lambda = lambda_const * Vt;
        const int N_p = curand_poisson(st, lambda);
        const float gam = gamma_compat(st, d + N_p);
        const float Vt_next = (sigma * sigma * (1.0f - exp_kdt) / (2.0f * k)) * gam;
        vI += (Vt + Vt_next);
        Vt = Vt_next;
    }
    vI *= dt * 0.5;                                            // double multiply, NMCH_EM.cu:247
    float m = (1.0f / sigma) * (Vt - v_0 - k * theta + k * vI);
    m = -0.5f * vI + rho * m;
    const float sigma2 = (1.0f - rho * rho) * vI;
    V_T = Vt;
    return expf(m + sqrtf(sigma2) * curand_normal(st));
}

__global__ void __launch_bounds__(256)
em_compat_xorwow_kernel(const __grid_constant__ EmCompatLaunch L, const RawPoint *__restrict__ pts, XorwowState xs,
                        ReduceBuffers rb, float *__restrict__ S_out, float *__restrict__ V_out)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < L.n_local;
    curandStateXORWOW_t st;
    if (valid) {
        st.d = xs.d[idx];
        st.v[0] = xs.v0[idx]; st.v[1] = xs.v1[idx]; st.v[2] = xs.v2[idx]; st.v[3] = xs.v3[idx]; st.v[4] = xs.v4[idx];
        st.boxmuller_flag = xs.bm_flag[idx];
        st.boxmuller_extra = xs.bm_extra[idx];
        st.boxmuller_flag_double = xs.bm_flag_d[idx];
        st.boxmuller_extra_double = xs.bm_extra_d[idx];
    }
    for (int point = 0; point < L.n_points; ++point) {
        const RawPoint rp = (pts != nullptr) ? pts[point] : L.raw0;
        double pay = 0.0;
        if (valid) {
            float V_T;
            const float S = em_path_compat(&st, L, rp, V_T);
            pay = (double)fmaxf(0.0f, S - L.K);
            if (S_out != nullptr && point == L.n_points - 1) {
                S_out[idx] = S;
                V_out[idx] = V_T;
            }
        }
        block_reduce_and_finish(pay, pay * pay, rb.partials, rb.tickets, rb.out, point, blockIdx.x, L.blocks_per_point);
    }
    if (valid) {                                               // streams continue (NMCH_EM.cu:280)
        xs.d[idx] = st.d;
        xs.v0[idx] = st.v[0]; xs.v1[idx] = st.v[1]; xs.v2[idx] = st.v[2]; xs.v3[idx] = st.v[3]; xs.v4[idx] = st.v[4];
        xs.bm_flag[idx] = st.boxmuller_flag;
        xs.bm_extra[idx] = st.boxmuller_extra;
        xs.bm_flag_d[idx] = st.boxmuller_flag_double;
        xs.bm_extra_d[idx] = st.boxmuller_extra_double;
    }
}

// cuRAND-layout states kept as an array of structures (Philox: 64 B, MRG32k3a: 48 B per path)
template <typename State>
__global__ void __launch_bounds__(256)
em_compat_state_kernel(const __grid_constant__ EmCompatLaunch L, const RawPoint *__restrict__ pts,
                       State *__restrict__ states, ReduceBuffers rb,
                       float *__restrict__ S_out, float *__restrict__ V_out)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < L.n_local;
    State st;
    if (valid) st = states[idx];
    for (int point = 0; point < L.n_points; ++point) {
        const RawPoint rp = (pts != nullptr) ? pts[point] : L.raw0;
        double pay = 0.0;
        if (valid) {
            float V_T;
            const float S = em_path_compat(&st, L, rp, V_T);
            pay = (double)fmaxf(0.0f, S - L.K);
            if (S_out != nullptr && point == L.n_points - 1) {
                S_out[idx] = S;
                V_out[idx] = V_T;
            }
        }
        block_reduce_and_finish(pay, pay * pay, rb.partials, rb.tickets, rb.out, point, blockIdx.x, L.blocks_per_point);
    }
    if (valid) states[idx] = st;
}

// cuRAND state per path, subsequence = global path index (reference: src/NMCH/random/random.cu:6-10).
// Philox: counter = (0, 0, path, 0), key = seed (curand_kernel.h:1022-1037); MRG32k3a: seed scramble + 3x3
// matrix-power skip of 2^76 draws per subsequence (curand_kernel.h:1274-1300).
template <typename State>
__global__ void curand_state_init_kernel(State *states, unsigned long long seed,
                                         unsigned long long first_path, unsigned long long n_local)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n_local) curand_init(seed, first_path + idx, 0, &states[idx]);
}

// FE for the MRG32k3a tag (the XORWOW / Philox tags have their own stream code in fe_kernels.cu): cuRAND's
// curand_normal2 on the MRG state (curand_normal.h:89-108, 466-469) + the reference's pinned update.
template <int FLOOR>
__global__ void __launch_bounds__(256)
fe_compat_mrg_kernel(const __grid_constant__ FeLaunch L, const RawPoint *__restrict__ pts,
                     curandStateMRG32k3a_t *__restrict__ states, ReduceBuffers rb, float *__restrict__ S_out,
                     float *__restrict__ V_out)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < L.n_local;
    curandStateMRG32k3a_t st;
    if (valid) st = states[idx];
    for (int point = 0; point < L.n_points; ++point) {
        const RawPoint rp = (pts != nullptr) ? pts[point] : L.raw0;
        float S = L.S0, V = L.v0;
        if (valid) {
            for (int n = 0; n < L.N; ++n) {
                const float2 g = curand_normal2(&st);
                fe_step_compat<FLOOR>(S, V, g.x, g.y, L.r, rp.k, L.rho, rp.theta, rp.sigma, L.dt, L.sqrt_dt, L.sqrt_rho);
            }
        }
        double pay = 0.0;
        if (valid) {
            pay = (double)fmaxf(0.0f, S - L.K);
            if (S_out != nullptr && point == L.n_points - 1) {
                S_out[idx] = S;
                V_out[idx] = V;
            }
        }
        block_reduce_and_finish(pay, pay * pay, rb.partials, rb.tickets, rb.out, point, blockIdx.x, L.blocks_per_point);
    }
    if (valid) states[idx] = st;
}

cudaError_t launch_fe_compat_mrg(const FeLaunch &L, int floor_kind, const RawPoint *d_pts, void *states,
                                 ReduceBuffers rb, float *S_out, float *V_out, cudaStream_t stream, KernelInfo *info)
{
    auto *st = static_cast<curandStateMRG32k3a_t *>(states);
    cudaFuncAttributes attr{};
    if (floor_kind == kFloorAbs) {
        fe_compat_mrg_kernel<kFloorAbs><<<(unsigned)L.blocks_per_point, 256, 0, stream>>>(L, d_pts, st, rb, S_out, V_out);
        cudaFuncGetAttributes(&attr, fe_compat_mrg_kernel<kFloorAbs>);
    } else {
        fe_compat_mrg_kernel<kFloorPlus><<<(unsigned)L.blocks_per_point, 256, 0, stream>>>(L, d_pts, st, rb, S_out, V_out);
        cudaFuncGetAttributes(&attr, fe_compat_mrg_kernel<kFloorPlus>);
    }
    if (info) *info = KernelInfo{L.blocks_per_point, 1, 256, 1, attr.numRegs, (int)(sizeof(FeLaunch) + 56)};
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static EmPoint fold_em_point(const nmch_params_t &p, float kf, float thetaf, float sigmaf)
{
    const double k = kf, theta = thetaf, sigma = sigmaf, dt = (double)p.T / p.N;
    const double e = std::exp(-k * dt), om = -std::expm1(-k * dt);
    EmPoint pt{};
    pt.scale = (float)(sigma * sigma * om / (2.0 * k));
    pt.lc = (float)(2.0 * k * e / (sigma * sigma * om));
    pt.d = (float)(2.0 * k * theta / (sigma * sigma));
    double a = 2.0 * k * theta / (sigma * sigma) - 0.5;
    pt.a = (float)a;
    pt.inv_a = 0.0f;
    if (a > 0.0) {
        if (a < 1.0) {
            pt.inv_a = (float)(1.0 / a);
            a += 1.0;
        }
        const double md = a - 1.0 / 3.0;
        pt.mt_d = (float)md;
        pt.mt_c = (float)(1.0 / std::sqrt(9.0 * md));
    }
    const double c0 = 1.1774100225154747, log2e = 1.4426950408889634;
    pt.f_c = (float)(pt.mt_c * c0);
    pt.f_h = (float)(0.5 * c0 * c0 * log2e);
    pt.f_dl = (float)(pt.mt_d * log2e);
    const double cc = sigma * sigma * om / (2.0 * k);
    pt.f_g2s = (float)(pt.mt_d * cc);
    pt.f_t1 = (float)(c0 * std::sqrt(0.5 * cc));
    pt.f_ev = (float)e;
    pt.f_scale = 0.5f * pt.scale;
    pt.f_hs = (pt.mt_c > 0.0f) ? (float)(0.5 * log2e / ((double)pt.mt_c * (double)pt.mt_c)) : 0.0f;   // (c0^2/2) log2 e / (mt_c c0)^2
    pt.f_lg2s = (pt.mt_d > 0.0f) ? (float)std::log2((double)pt.mt_d * cc) : 0.0f;
    pt.k = kf;
    pt.ktheta_T = (float)(k * theta * (double)p.T);
    pt.inv_sigma = (float)(1.0 / sigma);
    // tiny or negative d - 1/2 goes through the Poisson mixture
    pt.kind = !(pt.a > 1e-3f) ? kEmMixture : (pt.inv_a != 0.0f ? kEmSplit : kEmSplitPacked);
    return pt;
}

static bool em_point_finite(const EmPoint &pt)
{
    const float v[] = {pt.scale, pt.lc, pt.d, pt.a, pt.mt_d, pt.mt_c, pt.inv_a, pt.f_c, pt.f_h, pt.f_dl,
                       pt.f_g2s, pt.f_t1, pt.f_ev, pt.f_scale, pt.f_hs, pt.f_lg2s, pt.k, pt.ktheta_T, pt.inv_sigma};
    for (float x : v)
        if (!std::isfinite(x)) return false;
    return pt.scale > 0.0f && pt.lc > 0.0f;
}


template <typename State>
static int curand_states_init(nmch_engine *e)
{
    const size_t n = (size_t)e->n_local;
    cudaError_t err = engine_dev_malloc(e, &e->curand_states, n * sizeof(State), "cuRAND-layout states");
    if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "cudaMalloc(cuRAND-layout states)", err);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    curand_state_init_kernel<State><<<blocks, 256, 0, e->stream>>>(static_cast<State *>(e->curand_states), e->seed,
                                                                   e->first_path, e->n_local);
    err = cudaGetLastError();
    if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "curand_state_init_kernel", err);
    e->launches += 1;
    return NMCH_OK;
}

int em_philox_compat_init(nmch_engine *e) { return curand_states_init<curandStatePhilox4_32_10_t>(e); }
int mrg_compat_init(nmch_engine *e) { return curand_states_init<curandStateMRG32k3a_t>(e); }

void em_release(nmch_engine *e)
{
    engine_dev_free(e, e->curand_states);
    e->curand_states = nullptr;
}

int em_launch_points(nmch_engine *e, cudaStream_t stream, const float *k, const float *theta, const float *sigma,
                     int n_points, double *d_out, float *S_out, float *V_out)
{
    const nmch_params_t &p = e->p;
    const bool own = (k == nullptr);
    unsigned long long bpp = (e->n_local + (unsigned long long)kEmThreads - 1ull) / (unsigned long long)kEmThreads;
    if (bpp == 0 || bpp > 0x7fffffffull) return engine_fail(NMCH_ERR_ARG, "launch grid out of range");
    cudaError_t err;
    if (p.rng == NMCH_RNG_PHILOX) {
        std::vector<EmPoint> pts(n_points);
        for (int i = 0; i < n_points; ++i) {
            pts[i] = own ? fold_em_point(p, p.k, p.theta, p.sigma) : fold_em_point(p, k[i], theta[i], sigma[i]);
            pts[i].index = i;
            if (!em_point_finite(pts[i]))
                return engine_fail(NMCH_ERR_ARG, "EM: parameters out of the representable range (k dt or sigma^2 too small / large)");
        }
        // group the points by sampler (each keeps its index), slowest sampler first so that the tail of the launch is
        // made of the cheapest blocks: Poisson mixture, split with boost, split without boost
        auto rank_of = [](const EmPoint &q) { return q.kind == kEmMixture ? 0 : (q.kind == kEmSplit ? 1 : 2); };
        std::stable_sort(pts.begin(), pts.end(), [&](const EmPoint &a, const EmPoint &b) { return rank_of(a) < rank_of(b); });
        const bool one_kind = pts.front().kind == pts.back().kind;
        int rc = engine_ensure_buffers(e, n_points, bpp);
        if (rc) return rc;
        const EmPoint *d_pts = nullptr;
        if (!own) {
            rc = upload_records(e, stream, pts.data(), pts.size() * sizeof(EmPoint));
            if (rc) return rc;
            d_pts = static_cast<const EmPoint *>(e->d_points);
        }
        EmLaunch L{};
        L.keys = philox_expand_keys(e->seed);
        L.first_path = e->first_path;
        L.n_local = e->n_local;
        L.call0 = (unsigned int)e->em_calls;
        L.N = p.N;
        L.n_points = n_points;
        L.blocks_per_point = (int)bpp;
        L.v0 = p.v_0;
        L.K = p.S_0;
        L.half_dt = 0.5f * (p.T / (float)p.N);
        L.rho = p.rho;
        L.one_m_rho2 = 1.0f - p.rho * p.rho;
        L.lnS0_rT = (float)(std::log((double)p.S_0) + (double)p.r * (double)p.T);
        L.pt0 = pts[0];
        ReduceBuffers rb{e->d_partials, e->d_tickets, d_out};
        cudaFuncAttributes attr{};
        // ONE launch: blockIdx.y = point.  All points of one kind: that sampler's own instantiation; otherwise kEmAny,
        // whose blocks pick the sampler from their point record.
        dim3 grid((unsigned)bpp, (unsigned)n_points, 1);
        const int kind = one_kind ? pts.front().kind : kEmAny;
        if (kind == kEmSplit) {
            em_native_kernel<kEmSplit><<<grid, kEmThreads, 0, stream>>>(L, d_pts, rb, S_out, V_out);
            cudaFuncGetAttributes(&attr, em_native_kernel<kEmSplit>);
        } else if (kind == kEmSplitPacked) {
            em_native_kernel<kEmSplitPacked><<<grid, kEmThreads, 0, stream>>>(L, d_pts, rb, S_out, V_out);
            cudaFuncGetAttributes(&attr, em_native_kernel<kEmSplitPacked>);
        } else if (kind == kEmMixture) {
            em_native_kernel<kEmMixture><<<grid, kEmThreads, 0, stream>>>(L, d_pts, rb, S_out, V_out);
            cudaFuncGetAttributes(&attr, em_native_kernel<kEmMixture>);
        } else {
            em_native_kernel<kEmAny><<<grid, kEmThreads, 0, stream>>>(L, d_pts, rb, S_out, V_out);
            cudaFuncGetAttributes(&attr, em_native_kernel<kEmAny>);
        }
        err = cudaGetLastError();
        if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "em_native_kernel", err);
        e->kinfo = KernelInfo{(int)grid.x, n_points, kEmThreads, 1, attr.numRegs,
                              (int)(sizeof(EmLaunch) + sizeof(const EmPoint *) + sizeof(ReduceBuffers) + 2 * sizeof(float *))};
        e->em_calls += (unsigned long long)n_points;
        return NMCH_OK;
    }
    // compat modes
    bpp = (e->n_local + 255ull) / 256ull;
    int rc = engine_ensure_buffers(e, n_points, bpp);
    if (rc) return rc;
    const RawPoint *d_pts = nullptr;
    if (!own) {
        std::vector<RawPoint> pts(n_points);
        for (int i = 0; i < n_points; ++i) pts[i] = RawPoint{k[i], theta[i], sigma[i], 0.0f};
        rc = upload_records(e, stream, pts.data(), pts.size() * sizeof(RawPoint));
        if (rc) return rc;
        d_pts = static_cast<const RawPoint *>(e->d_points);
    }
    EmCompatLaunch L{};
    L.n_local = e->n_local;
    L.N = p.N;
    L.n_points = n_points;
    L.blocks_per_point = (int)bpp;
    L.S0 = p.S_0;
    L.v0 = p.v_0;
    L.K = p.S_0;
    L.rho = p.rho;
    L.dt = p.T / (float)p.N;
    L.raw0 = RawPoint{p.k, p.theta, p.sigma, 0.0f};
    ReduceBuffers rb{e->d_partials, e->d_tickets, d_out};
    cudaFuncAttributes attr{};
    if (p.rng == NMCH_RNG_XORWOW_COMPAT) {
        em_compat_xorwow_kernel<<<(unsigned)bpp, 256, 0, stream>>>(L, d_pts, e->xs, rb, S_out, V_out);
        cudaFuncGetAttributes(&attr, em_compat_xorwow_kernel);
    } else if (p.rng == NMCH_RNG_PHILOX_COMPAT) {
        em_compat_state_kernel<curandStatePhilox4_32_10_t><<<(unsigned)bpp, 256, 0, stream>>>(
            L, d_pts, static_cast<curandStatePhilox4_32_10_t *>(e->curand_states), rb, S_out, V_out);
        cudaFuncGetAttributes(&attr, em_compat_state_kernel<curandStatePhilox4_32_10_t>);
    } else {
        em_compat_state_kernel<curandStateMRG32k3a_t><<<(unsigned)bpp, 256, 0, stream>>>(
            L, d_pts, static_cast<curandStateMRG32k3a_t *>(e->curand_states), rb, S_out, V_out);
        cudaFuncGetAttributes(&attr, em_compat_state_kernel<curandStateMRG32k3a_t>);
    }
    err = cudaGetLastError();
    if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "em_compat_kernel", err);
    e->kinfo = KernelInfo{(int)bpp, 1, 256, 1, attr.numRegs, (int)(sizeof(EmCompatLaunch) + 64)};
    return NMCH_OK;
}

}  // namespace nmchb
