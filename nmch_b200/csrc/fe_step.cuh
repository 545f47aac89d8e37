// fe_step.cuh -- the native FE step, shared by the path kernels (fe_kernels.cu) and the tangent kernel
// (greeks_kernels.cu), so that both advance (S, V) with the same instructions on the same Philox words.
#pragma once
#include "kernels.cuh"

namespace nmchb {

// PRECISE_V: V' = g(V - kdt*V + (vb + q sin * vs)) with the product rounded once, instead of the folded
// V*va + vb + ... -- one more FP32 operation.  The folded va = 1 - k*dt carries a rounding error of up to 3e-8, i.e. a
// relative error of up to 3e-8 / (k dt) in the mean-reversion speed; fold_fe_point compensates vb so that the
// long-run level stays theta, which is all the 3-standard-error modes need.  The XORWOW_FAST mode promises 1e-5
// against the reference on identical draws and takes the exact form.
template <int FLOOR, bool PRECISE_V = false>
__device__ __forceinline__ void fe_step_native(float &S, float &V, uint32_t wa, uint32_t wb, float rdt,
                                               float zr, float zc, const FePoint &pc)
{
    // uniforms as cuRAND forms them (curand_uniform.h:69-72, curand_normal.h:72-75): u = x 2^-32 + 2^-33 in (0, 1],
    // angle = y (2 pi 2^-32) -- an integer-to-float conversion (I2FP) and one FFMA / FMUL.  Against bit
    // splicing ((w >> 9) | 0x3f800000, then a subtraction) this costs the same instruction count, but I2FP issues beside
    // the FP32 work where LEA.HI does not (profiles/r02_pipe_rates2.txt: -1 % on the kernel), and the native mode now
    // feeds the same uniforms as the draw-compatible modes into its fast transforms.
    constexpr float k2Pow32Inv = 2.3283064e-10f, k2Pow32Inv2Pi = 2.3283064e-10f * 6.2831855f;
    const float u = fmaf(__uint2float_rn(wa), k2Pow32Inv, k2Pow32Inv * 0.5f);
    const float l2 = lg2_approx(u);                   // <= 0
    const float q = sqrt_approx(-(V * l2));           // sqrt(V) * sqrt(-lg2 u)
    const float ang = __uint2float_rn(wb) * k2Pow32Inv2Pi;   // cuRAND adds half a step (7e-10 rad, below the angle's ulp)
    const float gs = q * sin_approx(ang);
    const float gc = q * cos_approx(ang);
    float m = fmaf(gs, zr, rdt);                      // relative increment; S' = S + S*m keeps r*dt at full precision
    m = fmaf(gc, zc, m);                              // (a folded 1 + r*dt would round by up to 6e-8 every step, a
    S = fmaf(S, m, S);                                //  systematic drift of N * 6e-8 on S_T)
    float vn;
    if constexpr (PRECISE_V) {
        vn = fmaf(-pc.kdt, V, V) + fmaf(gs, pc.vs, pc.vb);
    } else {
        vn = fmaf(V, pc.va, pc.vb);
        vn = fmaf(gs, pc.vs, vn);
    }
    V = (FLOOR == kFloorAbs) ? fabsf(vn) : fmaxf(vn, 0.0f);
}

// The same step carrying the pathwise tangent in ND directions (ND = 1: v_0 only; ND = kNumDirs: v_0, kappa, theta,
// sigma, rho):  A[d] = dV/dp_d,  B[d] = dS/dp_d  (A[v_0] = 1 at the start, every other tangent 0).
// (S, V) take EXACTLY the instructions of fe_step_native (same expressions in the same order), so a tangent pass
// reproduces the path pass bit for bit; the v_0 direction takes the same instructions for every ND, so its sums do not
// depend on how many other directions ride along.  Differentiating the step:  q = sqrt(V) e  =>  dq = q/(2V) dV, hence
// with h = A / (2V):   d(gs) = gs h,  d(gc) = gc h,
//   dm  = (gs zr + gc zc) h + gs dzr + gc dzc,          B' = B (1 + m) + S dm,
//   A'' = A va + V dva + dvb + gs vs h + gs dvs,        A' = g'(vn) A''   (g' = sign for |.|, 1{vn > 0} for (.)+),
// with the folded-constant derivatives of TangentFold (zero where a constant does not depend on the direction).  V does
// not depend on rho (the variance noise is the first normal alone), so the rho direction carries no A and A[kDirRho]
// is never read.
// V = 0 (the (.)+ floor parks paths there) has q = 0 and an infinite dq/dV; every A is then 0 (the floor's derivative
// zeroed it in the step that parked the path), and the 0 * inf is taken as 0: h = 0.  That is NOT "a parked path keeps
// zero tangents": in the next step dvb re-seeds A[kappa] and A[theta] with kappa-/theta-dependent values (the
// mean reversion pushes the path off 0 at a rate k theta dt), which the A'' line above does through V dva + dvb.
template <int FLOOR, int ND>
__device__ __forceinline__ void fe_step_native_tangent(float &S, float &V, float (&A)[ND], float (&B)[ND], uint32_t wa,
                                                       uint32_t wb, float rdt, float zr, float zc, const FePoint &pc,
                                                       const TangentFold &tf)
{
    static_assert(ND == 1 || ND == kNumDirs, "v_0 alone or all five directions");
    constexpr float k2Pow32Inv = 2.3283064e-10f, k2Pow32Inv2Pi = 2.3283064e-10f * 6.2831855f;
    const float u = fmaf(__uint2float_rn(wa), k2Pow32Inv, k2Pow32Inv * 0.5f);
    const float l2 = lg2_approx(u);
    const float q = sqrt_approx(-(V * l2));
    const float ang = __uint2float_rn(wb) * k2Pow32Inv2Pi;
    const float gs = q * sin_approx(ang);
    const float gc = q * cos_approx(ang);
    float m = fmaf(gs, zr, rdt);
    m = fmaf(gc, zc, m);
    float h[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        if (d == kDirRho) continue;
        h[d] = (V > 0.0f) ? __fdividef(0.5f * A[d], V) : 0.0f;
    }
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        const float dm = (d == kDirRho) ? fmaf(gc, tf.dzc_r, gs * tf.dzr_r) : fmaf(gc, zc, gs * zr) * h[d];
        B[d] = fmaf(S, dm, fmaf(B[d], m, B[d]));      // uses S before its update
    }
    S = fmaf(S, m, S);
    float vn = fmaf(V, pc.va, pc.vb);
    vn = fmaf(gs, pc.vs, vn);
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        if (d == kDirRho) continue;
        float an;
        if (d == kDirV0) {
            an = fmaf(gs * pc.vs, h[d], A[d] * pc.va);
        } else {
            const float c = (d == kDirKappa) ? fmaf(V, tf.dva_k, tf.dvb_k)       // V before its update
                          : (d == kDirTheta) ? tf.dvb_t
                                             : gs * tf.dvs_s;                    // kDirSigma
            an = fmaf(gs * pc.vs, h[d], fmaf(A[d], pc.va, c));
        }
        if (FLOOR == kFloorAbs)
            A[d] = (vn < 0.0f) ? -an : an;
        else
            A[d] = (vn > 0.0f) ? an : 0.0f;
    }
    V = (FLOOR == kFloorAbs) ? fabsf(vn) : fmaxf(vn, 0.0f);
}

}  // namespace nmchb
