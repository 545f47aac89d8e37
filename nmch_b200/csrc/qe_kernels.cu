// qe_kernels.cu -- Andersen's Quadratic-Exponential scheme with martingale correction (QE-M) for Heston.
//
// SURVEY.md §8f "next" row 3: a large-step third method next to the reference's FE and EM.  The reference's "exact"
// scheme pays one CIR transition per small step (N = 1000); QE matches the first two conditional moments of the
// CIR transition with either a squared shifted normal (psi <= 1.5) or a point mass at zero plus an exponential tail
// (psi > 1.5), integrates the log-price with the central discretisation (gamma1 = gamma2 = 1/2) and fixes the drift so
// that E[S] is exact.  It reaches the accuracy of N = 1000 Euler steps with 50-100 steps.  There is no reference
// implementation to be draw-compatible with, so this kernel exists for the native Philox stream only; it is checked
// against the semi-analytic price and a host restatement of the same scheme on the same draws (tests/test_gpu_qe.py).
//
// One Philox block per (path, step): words (x, y) -> Box-Muller pair (Z_v, Z_s), word z -> the uniform of the
// exponential branch; counter = (step, call/point id, path_lo, path_hi) like the EM kernel.
#include <vector>

#include "engine_internal.cuh"

namespace nmchb {

struct QePoint {
    float e;            // exp(-k dt)
    float m0;           // theta (1 - e)
    float c1, c2;       // s^2 = V c1 + c2
    float K2, K3, K4;   // log-price coefficients (gamma1 = gamma2 = 1/2); K1 cancels against the martingale drift
    float A;            // K2 + K4 / 2
    float pad;
};

struct QeLaunch {
    PhiloxKeys keys;
    unsigned long long first_path, n_local;
    unsigned int call0;
    int   N, n_points, blocks_per_point;
    float v0, K, lnS0, r_dt;
    QePoint pt0;
};

__device__ __forceinline__ float u01_open23(uint32_t w) { return bits_to_1_2(w) - 0.99999994f; }

__global__ void __launch_bounds__(256)
qe_kernel(const __grid_constant__ QeLaunch L, const QePoint *__restrict__ pts, ReduceBuffers rb,
          float *__restrict__ S_out, float *__restrict__ V_out)
{
    const int point = blockIdx.y;
    NMCHB_ASSERT(point < L.n_points && (int)blockIdx.x < L.blocks_per_point);
    const QePoint pc = (pts != nullptr) ? pts[point] : L.pt0;
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < L.n_local;
    const unsigned long long g = L.first_path + idx;
    const uint32_t path_lo = (uint32_t)g, path_hi = (uint32_t)(g >> 32);
    const uint32_t stream = L.call0 + (uint32_t)point;
    float V = L.v0, lnS = L.lnS0;
    if (valid) {
        const PhiloxPathInv inv = philox_path_invariants(stream, path_lo, L.keys);
        for (int n = 0; n < L.N; ++n) {
            const unsigned long long s = (unsigned long long)kPhiloxM0 * (uint32_t)n;
            const U4 w = philox4x32_10_hoisted((uint32_t)(s >> 32), (uint32_t)s, path_hi, inv, L.keys);
            // two independent normals and one uniform
            const float rad = sqrt_approx(-1.38629436f * lg2_approx(u01_open23(w.x)));
            const float ang = bits_to_1_2(w.y) * 6.2831855f;
            const float zv = rad * sin_approx(ang), zs = rad * cos_approx(ang);
            const float u = u01_open23(w.z);
            // conditional mean and variance of V(t+dt) given V(t)
            const float m = fmaf(V, pc.e, pc.m0);
            const float s2 = fmaf(V, pc.c1, pc.c2);
            const float psi = s2 * rcp_approx(m * m);
            float Vn, lnM;
            if (psi <= 1.5f) {
                // V' = a (b + Z)^2
                const float t = 2.0f * rcp_approx(psi);
                const float b2 = t - 1.0f + sqrt_approx(t * (t - 1.0f));
                const float a = m * rcp_approx(1.0f + b2);
                const float q = sqrt_approx(b2) + zv;
                Vn = a * q * q;
                const float den = fmaxf(1.0f - 2.0f * pc.A * a, 1e-6f);         // > 0 for the usual rho < 0; clamped so that
                                                                                // a large positive rho cannot produce NaN
                lnM = pc.A * b2 * a * rcp_approx(den) - 0.5f * __logf(den);
            } else {
                // V' = 0 with probability p, else exponential with rate beta
                const float p = (psi - 1.0f) * rcp_approx(psi + 1.0f);
                const float beta = (1.0f - p) * rcp_approx(m);
                Vn = (u <= p) ? 0.0f : __logf((1.0f - p) * rcp_approx(1.0f - u)) * rcp_approx(beta);
                lnM = __logf(p + beta * (1.0f - p) * rcp_approx(fmaxf(beta - pc.A, 1e-6f)));
            }
            if (!(m > 0.0f)) {               // theta = 0 and V = 0: the variance is absorbed at zero (psi = 0 * inf above)
                Vn = 0.0f;
                lnM = 0.0f;
            }
            // ln S' = ln S + r dt - ln M - K3 V / 2 + K2 V' + sqrt(K3 V + K4 V') Z_s   (K0* with K1 V folded in)
            const float var = fmaf(pc.K3, V, pc.K4 * Vn);
            lnS += L.r_dt - lnM - 0.5f * pc.K3 * V + pc.K2 * Vn + sqrt_approx(var) * zs;
            V = Vn;
        }
    }
    double pay = 0.0;
    if (valid) {
        const float S = __expf(lnS);
        pay = payoff_or_nan(S, L.K);
        if (S_out != nullptr && point == L.n_points - 1) {
            S_out[idx] = S;
            V_out[idx] = V;
        }
    }
    block_reduce_and_finish(pay, pay * pay, rb.partials, rb.tickets, rb.out, point, blockIdx.x, L.blocks_per_point);
}

static QePoint fold_qe_point(const nmch_params_t &p, float kf, float thetaf, float sigmaf)
{
    const double k = kf, theta = thetaf, sigma = sigmaf, rho = p.rho, dt = (double)p.T / p.N;
    const double e = std::exp(-k * dt), om = -std::expm1(-k * dt);
    QePoint q{};
    q.e = (float)e;
    q.m0 = (float)(theta * om);
    q.c1 = (float)(sigma * sigma * e * om / k);
    q.c2 = (float)(theta * sigma * sigma * om * om / (2.0 * k));
    const double g1 = 0.5, g2 = 0.5;
    const double K2 = g2 * dt * (k * rho / sigma - 0.5) + rho / sigma;
    const double K3 = g1 * dt * (1.0 - rho * rho), K4 = g2 * dt * (1.0 - rho * rho);
    q.K2 = (float)K2;
    q.K3 = (float)K3;
    q.K4 = (float)K4;
    q.A = (float)(K2 + 0.5 * K4);
    // Andersen's K0 and K1 never appear: the martingale-corrected K0* = -ln M - (K1 + K3/2) V replaces K0, and its
    // K1 V cancels the scheme's own K1 V term, leaving  r dt - ln M - K3 V / 2 + K2 V' + sqrt(K3 V + K4 V') Z.
    return q;
}

int qe_launch_points(nmch_engine *e, cudaStream_t stream, const float *k, const float *theta, const float *sigma,
                     int n_points, double *d_out, float *S_out, float *V_out)
{
    const nmch_params_t &p = e->p;
    if (p.rng != NMCH_RNG_PHILOX)
        return engine_fail(NMCH_ERR_ARG, "the QE scheme has no reference counterpart to be draw-compatible with: use rng = PHILOX");
    const bool own = (k == nullptr);
    const unsigned long long bpp = (e->n_local + 255ull) / 256ull;
    if (bpp == 0 || bpp > 0x7fffffffull) return engine_fail(NMCH_ERR_ARG, "launch grid out of range");
    std::vector<QePoint> pts(n_points);
    for (int i = 0; i < n_points; ++i)
        pts[i] = own ? fold_qe_point(p, p.k, p.theta, p.sigma) : fold_qe_point(p, k[i], theta[i], sigma[i]);
    int rc = engine_ensure_buffers(e, n_points, bpp);
    if (rc) return rc;
    const QePoint *d_pts = nullptr;
    if (!own) {
        rc = upload_records(e, stream, pts.data(), pts.size() * sizeof(QePoint));
        if (rc) return rc;
        d_pts = static_cast<const QePoint *>(e->d_points);
    }
    QeLaunch L{};
    L.keys = philox_expand_keys(e->seed);
    L.first_path = e->first_path;
    L.n_local = e->n_local;
    L.call0 = (unsigned int)e->em_calls;
    L.N = p.N;
    L.n_points = n_points;
    L.blocks_per_point = (int)bpp;
    L.v0 = p.v_0;
    L.K = p.S_0;
    L.lnS0 = (float)std::log((double)p.S_0);
    L.r_dt = p.r * (p.T / (float)p.N);
    L.pt0 = pts[0];
    ReduceBuffers rb{e->d_partials, e->d_tickets, d_out};
    dim3 grid((unsigned)bpp, (unsigned)n_points, 1);
    qe_kernel<<<grid, 256, 0, stream>>>(L, d_pts, rb, S_out, V_out);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "qe_kernel", err);
    cudaFuncAttributes attr{};
    cudaFuncGetAttributes(&attr, qe_kernel);
    e->kinfo = KernelInfo{(int)grid.x, (int)grid.y, 256, 1, attr.numRegs,
                          (int)(sizeof(QeLaunch) + sizeof(const QePoint *) + sizeof(ReduceBuffers) + 2 * sizeof(float *))};
    e->em_calls += (unsigned long long)n_points;
    return NMCH_OK;
}

}  // namespace nmchb
