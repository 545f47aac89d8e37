// NMCH/methods/NMCH.hpp -- base type of the method API, source-compatible with the reference
// (/root/reference/include/NMCH/methods/NMCH.hpp:28-115): same namespace, template parameter, constructor
// arguments, virtual lifecycle, getters and setters.  Underneath, every method object drives the sm_100a
// engine through the C ABI (include/nmch_b200.h) instead of owning cuRAND states and launching kernels.
#ifndef NMCH_HPP
#define NMCH_HPP

#include <stdio.h>

#include "NMCH/random/random.hpp"
#include "NMCH/utils/utils.hpp"
#include "nmch_b200.h"

namespace nmch::methods {

template <typename rnd_state>
class NMCH {
public:
    /* NTPB*NB = number of paths (launch geometry is internal to the engine); T maturity; S_0 spot (= strike);
       v_0 initial variance; r rate; k mean reversion; rho correlation; theta long-run variance; sigma vol of
       variance; N time steps (reference NMCH.hpp:42). */
    NMCH(int NTPB, int NB, float T, float S_0, float v_0, float r, float k, float rho, float theta, float sigma, int N);

    virtual void compute() = 0;
    virtual void print_stats();
    virtual void init(unsigned long long seed) = 0;
    virtual void finalize() = 0;

    float get_strike_price() const { return strike_price; }
    float get_price_squared() const { return price_squared; }

    void set_k(float k) { this->k = k; }
    void set_theta(float theta) { this->theta = theta; }
    void set_sigma(float sigma) { this->sigma = sigma; }

    /* ---- additive knobs (defaults reproduce the reference's behaviour); call before init() ---- */
    void set_floor_plus(bool on) { floor_plus = on; }             // g = (.)+ instead of |.| (README.md:37-40)
    void set_gpus(int n) { gpus = n < 1 ? 1 : n; }                // shard paths over n devices + one NCCL allreduce
    void set_philox_compat(bool on) { philox_compat = on; }       // Philox tag: cuRAND-draw-compatible validation mode
    void set_philox_dense(bool on) { philox_dense = on; }         // Philox tag, FE only (ignored otherwise): 3 steps per Philox block (+15 %, own mapping)
    void set_xorwow_fast(bool on) { xorwow_fast = on; }           // XORWOW tag, FE only (ignored otherwise): cuRAND's integer draws, native fast-math step
    void set_paths_per_thread(int p) { paths_per_thread = p; }
    /* Exact legacy output of the reference's K1 kernels (FE_k1 / EM_k1, reference NMCH_FE.cu:56-58, NMCH_EM.cu:129-131):
       they reduce (payoff/n)^2/n, so get_price_squared() of the *_K1* classes (K1_MM, K1_PgM, K1_PiM; not K2 / K3)
       returns E[X^2]/n^2 there.  Off by default (every class stores E[X^2]); on, the K1 classes reproduce the quirk --
       and with it the reference's get_err() and print_stats() lines, which are computed from that field.
       No effect on the K2 / K3 classes.  May be called at any time; acts at the next compute(). */
    void set_legacy_k1_moment(bool on) { legacy_k1_moment = on; }
    /* raw FP64 sums behind strike_price / price_squared, and the plain standard error of the mean */
    double get_sum_payoff() const { return sum_payoff; }
    double get_sum_payoff_sq() const { return sum_payoff_sq; }
    double get_std_error() const;
    /* The exploration sweep (reference src/NMCH/test/exploration.cu:71-88) as ONE launch: point i uses
       (k[i], theta[i], sigma[i]) on the stream position it would have after i sequential compute() calls,
       so the outputs equal n_points x { set_k; set_theta; set_sigma; compute(); get_*() }.  Returns the launch
       time in ms; outputs may be null. */
    float compute_grid(int n_points, const float *k, const float *theta, const float *sigma, float *strike_price_out,
                       float *price_squared_out, float *err_out);

    /* One compute() pass priced at a strike vector, with the pathwise delta E[1{S_T>K} S_T/S_0] (the reference fixes
       K = S_0, NMCH.cu:7).  Outputs (each n_strikes long, may be null): E[(S_T-K)^+], E[((S_T-K)^+)^2], delta.
       Returns the launch time in ms. */
    float compute_strikes(int n_strikes, const float *strikes, float *price_out, float *price_squared_out, float *delta_out);
    /* The same with the pathwise vega d E[(S_T-K)^+] / d v_0 and its standard error (FE on the native Philox stream
       only: the tangent rides the native Euler step; any other method / stream fails like every engine error). */
    float compute_greeks(int n_strikes, const float *strikes, float *price_out, float *price_squared_out, float *delta_out,
                         float *vega_out, float *vega_err_out);
    /* The same pass with the pathwise sensitivities d E[(S_T-K)^+] / dp for p = v_0, kappa, theta, sigma, rho (in the
       NMCH_SENS_* order of nmch_b200.h) and their standard errors: sens_out and sens_err_out hold NMCH_SENS_COUNT
       values per strike, strike after strike (may be null).  FE on the native Philox stream with |rho| < 1 only; any
       other method / stream fails like every engine error. */
    float compute_sensitivities(int n_strikes, const float *strikes, float *price_out, float *price_squared_out,
                                float *delta_out, float *sens_out, float *sens_err_out);

    virtual ~NMCH();

protected:
    int NTPB;
    int NB;
    float T;
    float S_0;
    float v_0;
    float K;   /* at the money: K = S_0 (reference NMCH.cu:7) */
    float r;
    float k;
    float rho;
    float theta;
    float sigma;
    int N;
    float dt;
    float strike_price;
    float price_squared;

    /* engine plumbing shared by the FE and EM families */
    nmch_group_t *group = nullptr;
    double sum_payoff = 0.0, sum_payoff_sq = 0.0;
    bool floor_plus = false, philox_compat = false, philox_dense = false, xorwow_fast = false;
    bool legacy_k1_moment = false;
    int gpus = 1, paths_per_thread = 0;

    void engine_init(int method, unsigned long long seed, float *tim_init);
    void engine_compute(float *tim_exec);
    void engine_finalize();
    void apply_legacy_k1_moment();   /* called by the classes that stand for the reference's K1 kernels */
    unsigned long long path_count() const { return (unsigned long long)NTPB * (unsigned long long)NB; }
};

}  // namespace nmch::methods

#endif  // NMCH_HPP
