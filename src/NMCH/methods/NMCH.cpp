// NMCH.cpp -- base of the method API over the engine C ABI (reference: src/NMCH/methods/NMCH.cu).
#include "NMCH/methods/NMCH.hpp"

#include <cmath>
#include <vector>

#define testNMCH(status) (nmch::utils::cuda::checkCUDA((status), __FILE__, __LINE__))

namespace nmch::methods {

template <typename rnd_state>
NMCH<rnd_state>::NMCH(int NTPB, int NB, float T, float S_0, float v_0, float r, float k, float rho, float theta,
                      float sigma, int N)
    : NTPB(NTPB), NB(NB), T(T), S_0(S_0), v_0(v_0), K(S_0), r(r), k(k), rho(rho), theta(theta), sigma(sigma), N(N),
      strike_price(0.0f), price_squared(0.0f)
{
    dt = T / N;
}

template <typename rnd_state>
NMCH<rnd_state>::~NMCH()
{
    // the reference leaks when finalize() is skipped (its destructors free nothing); here the handle is released
    if (group) nmch_group_destroy(group);
}

template <typename rnd_state>
void NMCH<rnd_state>::print_stats()
{
    // same lines as the reference (NMCH.cu:12-28; rho is not printed there either)
    printf("Base parameters:\n");
    printf("NTPB    = %d\n", NTPB);
    printf("NB      = %d\n", NB);
    printf("T       = %f\n", T);
    printf("S_0,K   = %f\n", S_0);
    printf("v_0     = %f\n", v_0);
    printf("r       = %f\n", r);
    printf("k       = %f\n", k);
    printf("theta   = %f\n", theta);
    printf("sigma   = %f\n", sigma);
    printf("N       = %d\n", N);
    printf("dt      = %f\n", dt);
}

template <typename rnd_state>
double NMCH<rnd_state>::get_std_error() const
{
    const double n = (double)path_count();
    const double m = sum_payoff / n, m2 = sum_payoff_sq / n;
    const double var = m2 - m * m;
    return var > 0.0 ? std::sqrt(var / n) : 0.0;
}

template <typename rnd_state>
void NMCH<rnd_state>::engine_init(int method, unsigned long long seed, float *tim_init)
{
    using traits = nmch::random::tag_traits<rnd_state>;
    nmch_params_t p{};
    p.NTPB = NTPB; p.NB = NB;
    p.T = T; p.S_0 = S_0; p.v_0 = v_0; p.r = r; p.k = k; p.rho = rho; p.theta = theta; p.sigma = sigma;
    p.N = N;
    p.method = method;
    p.floor = floor_plus ? NMCH_FLOOR_PLUS : NMCH_FLOOR_ABS;
    switch (traits::mode) {
    case nmch::random::stream_mode::xorwow_compat:
        p.rng = (xorwow_fast && method == NMCH_METHOD_FE) ? NMCH_RNG_XORWOW_FAST : NMCH_RNG_XORWOW_COMPAT;
        break;
    case nmch::random::stream_mode::philox_compat: p.rng = NMCH_RNG_PHILOX_COMPAT; break;
    case nmch::random::stream_mode::mrg32k3a_compat: p.rng = NMCH_RNG_MRG32K3A_COMPAT; break;
    default:                                                 // the FE-only opt-in streams are ignored by the other methods
        p.rng = philox_compat ? NMCH_RNG_PHILOX_COMPAT
                              : ((philox_dense && method == NMCH_METHOD_FE) ? NMCH_RNG_PHILOX_DENSE : NMCH_RNG_PHILOX);
        break;
    }
    p.device = -1;
    p.paths_per_thread = paths_per_thread;
    if (group) { nmch_group_destroy(group); group = nullptr; }
    testNMCH(nmch_group_create(&p, gpus, &group));
    testNMCH(nmch_group_init(group, seed));
    *tim_init = nmch_group_init_ms(group);
}

template <typename rnd_state>
void NMCH<rnd_state>::engine_compute(float *tim_exec)
{
    if (!group) testNMCH(NMCH_ERR_STATE);
    testNMCH(nmch_group_set_params(group, k, theta, sigma));       // setters act at the next compute (NMCH.hpp:76-80)
    nmch_moments_t m{};
    testNMCH(nmch_group_compute(group, &m));
    sum_payoff = m.sum_payoff;
    sum_payoff_sq = m.sum_payoff_sq;
    strike_price = (float)(m.sum_payoff / (double)m.n_paths);
    price_squared = (float)(m.sum_payoff_sq / (double)m.n_paths);
    *tim_exec = m.exec_ms;
}

template <typename rnd_state>
float NMCH<rnd_state>::compute_grid(int n_points, const float *kk, const float *tt, const float *ss, float *strike_out,
                                    float *sq_out, float *err_out)
{
    if (!group) testNMCH(NMCH_ERR_STATE);
    std::vector<nmch_moments_t> m((size_t)n_points);
    testNMCH(nmch_group_explore(group, kk, tt, ss, n_points, m.data()));
    const int n = (int)path_count();
    for (int i = 0; i < n_points; ++i) {
        const float e1 = (float)(m[i].sum_payoff / (double)m[i].n_paths);
        const float e2 = (float)(m[i].sum_payoff_sq / (double)m[i].n_paths);
        if (strike_out) strike_out[i] = e1;
        if (sq_out) sq_out[i] = e2;
        if (err_out)   // the reference's get_err() formula (NMCH_FE.hpp:50-55)
            err_out[i] = 1.96 * sqrt((double)(1.0f / (n - 1)) * (n * e2 - (e1 * e1))) / sqrt((double)n);
    }
    if (n_points > 0) {
        k = kk[n_points - 1]; theta = tt[n_points - 1]; sigma = ss[n_points - 1];
        sum_payoff = m.back().sum_payoff;
        sum_payoff_sq = m.back().sum_payoff_sq;
        strike_price = (float)(sum_payoff / (double)m.back().n_paths);
        price_squared = (float)(sum_payoff_sq / (double)m.back().n_paths);
    }
    return n_points > 0 ? m[0].exec_ms : 0.0f;
}

template <typename rnd_state>
float NMCH<rnd_state>::compute_strikes(int n_strikes, const float *strikes, float *price_out, float *sq_out, float *delta_out)
{
    if (!group) testNMCH(NMCH_ERR_STATE);
    testNMCH(nmch_group_set_params(group, k, theta, sigma));
    std::vector<nmch_strike_moments_t> m((size_t)(n_strikes > 0 ? n_strikes : 0));
    testNMCH(nmch_group_compute_strikes(group, strikes, n_strikes, m.data()));
    for (int j = 0; j < n_strikes; ++j) {
        const double n = (double)m[j].n_paths;
        if (price_out) price_out[j] = (float)(m[j].sum_payoff / n);
        if (sq_out) sq_out[j] = (float)(m[j].sum_payoff_sq / n);
        if (delta_out) delta_out[j] = (float)(m[j].sum_delta / n);
    }
    return n_strikes > 0 ? m[0].exec_ms : 0.0f;
}

template <typename rnd_state>
float NMCH<rnd_state>::compute_greeks(int n_strikes, const float *strikes, float *price_out, float *sq_out, float *delta_out,
                                      float *vega_out, float *vega_err_out)
{
    if (!group) testNMCH(NMCH_ERR_STATE);
    testNMCH(nmch_group_set_params(group, k, theta, sigma));
    std::vector<nmch_greek_moments_t> m((size_t)(n_strikes > 0 ? n_strikes : 0));
    testNMCH(nmch_group_compute_greeks(group, strikes, n_strikes, m.data()));
    for (int j = 0; j < n_strikes; ++j) {
        const double n = (double)m[j].n_paths;
        const double vega = m[j].sum_vega / n;
        const double var = m[j].sum_vega_sq / n - vega * vega;
        if (price_out) price_out[j] = (float)(m[j].sum_payoff / n);
        if (sq_out) sq_out[j] = (float)(m[j].sum_payoff_sq / n);
        if (delta_out) delta_out[j] = (float)(m[j].sum_delta / n);
        if (vega_out) vega_out[j] = (float)vega;
        if (vega_err_out) vega_err_out[j] = (float)std::sqrt((var > 0.0 ? var : 0.0) / (n > 1.0 ? n - 1.0 : 1.0));
    }
    return n_strikes > 0 ? m[0].exec_ms : 0.0f;
}

template <typename rnd_state>
float NMCH<rnd_state>::compute_sensitivities(int n_strikes, const float *strikes, float *price_out, float *sq_out,
                                             float *delta_out, float *sens_out, float *sens_err_out)
{
    if (!group) testNMCH(NMCH_ERR_STATE);
    testNMCH(nmch_group_set_params(group, k, theta, sigma));
    std::vector<nmch_sensitivity_moments_t> m((size_t)(n_strikes > 0 ? n_strikes : 0));
    testNMCH(nmch_group_compute_sensitivities(group, strikes, n_strikes, m.data()));
    for (int j = 0; j < n_strikes; ++j) {
        const double n = (double)m[j].n_paths;
        if (price_out) price_out[j] = (float)(m[j].sum_payoff / n);
        if (sq_out) sq_out[j] = (float)(m[j].sum_payoff_sq / n);
        if (delta_out) delta_out[j] = (float)(m[j].sum_delta / n);
        for (int d = 0; d < NMCH_SENS_COUNT; ++d) {
            const double mean = m[j].sum_sens[d] / n;
            const double var = m[j].sum_sens_sq[d] / n - mean * mean;
            if (sens_out) sens_out[(size_t)j * NMCH_SENS_COUNT + d] = (float)mean;
            if (sens_err_out)
                sens_err_out[(size_t)j * NMCH_SENS_COUNT + d] = (float)std::sqrt((var > 0.0 ? var : 0.0) / (n > 1.0 ? n - 1.0 : 1.0));
        }
    }
    return n_strikes > 0 ? m[0].exec_ms : 0.0f;
}

template <typename rnd_state>
void NMCH<rnd_state>::apply_legacy_k1_moment()
{
    // reference FE_k1 / EM_k1: SR = payoff / n; VR = SR * SR / n; price_squared = sum VR = (sum payoff^2) / n^3
    if (!legacy_k1_moment) return;
    const double n = (double)path_count();
    price_squared = (float)(sum_payoff_sq / n / n / n);
}

template <typename rnd_state>
void NMCH<rnd_state>::engine_finalize()
{
    if (group) testNMCH(nmch_group_finalize(group));               // idempotent, unlike the reference's double free
}

template class NMCH<curandStateXORWOW_t>;
template class NMCH<curandStateMRG32k3a_t>;
template class NMCH<curandStatePhilox4_32_10_t>;

}  // namespace nmch::methods
