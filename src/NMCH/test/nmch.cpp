// nmch.cpp -- the `NMCH` command line tool: same flags, defaults, output text and exit codes as the reference
// (src/NMCH/test/nmch.cu:49-139), host C++ over the method API.  Additive flags (defaults = reference behaviour):
//   --g abs|plus        variance floor (README.md:37-40; the reference codes only abs)
//   --rng philox|xorwow|philox-compat|philox-dense|xorwow-fast   generator tag / stream mode (reference CLI: Philox, nmch.cu:119,130)
//   --gpus N            shard the paths over N GPUs, one NCCL allreduce of the moments
//   --paths-per-thread P, --json (one machine-readable line after the report)
//   --legacy-k1         run the K1 class of the method (the reference CLI runs K3) with its E[X^2]/n^2 moment quirk
//                       (reference NMCH_FE.cu:56-58, NMCH_EM.cu:129-131), for exact legacy output
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "NMCH/methods/NMCH_EM.hpp"
#include "NMCH/methods/NMCH_FE.hpp"
#include "NMCH/methods/NMCH_QE.hpp"

using namespace nmch::methods;

namespace {

struct Options {
    int NTPB = 512, NB = 512, N = 1000, gpus = 1, ppt = 0;
    float T = 1.0f, S_0 = 1.0f, v_0 = 0.1f, r = 0.0f, k = 0.5f, rho = -0.7, theta = 0.1f, sigma = 0.3f;
    unsigned long long seed = 1234;
    std::string method = "fe", g = "abs", rng = "philox", strikes;
    bool json = false, legacy_k1 = false, vega = false, sensitivities = false;
};

void usage(const char *argv0)
{
    // the reference's help text, stale defaults included (nmch.cu:94-111), then the additive flags
    printf("Usage: %s [options]\n", argv0);
    printf("Options:\n");
    printf("  --NTPB <int>       Number of threads per block (default: 1024)\n");
    printf("  --NB <int>         Number of blocks (default: 512)\n");
    printf("  --T <float>        Time period (default: 1.0)\n");
    printf("  --S_0 <float>      Initial stock price (default: 1.0)\n");
    printf("  --v_0 <float>      Initial volatility (default: 0.1)\n");
    printf("  --r <float>        Risk-free rate (default: 0.0)\n");
    printf("  --k <float>        Mean reversion rate (default: 0.5)\n");
    printf("  --rho <float>      Correlation (default: -0.7)\n");
    printf("  --theta <float>    Long-term volatility (default: 0.1)\n");
    printf("  --sigma <float>    Volatility of volatility (default: 0.3)\n");
    printf("  --N <int>          Number of time steps (default: 50)\n");
    printf("  --seed <ull>       Random seed (default: 1234)\n");
    printf("  --method <string>  Method to use: fe or em (default: fe)\n");
    printf("  --help             Display this help message\n");
    printf("B200 engine options (actual defaults: NTPB 512, NB 512, N 1000):\n");
    printf("  --method qe        Quadratic-exponential large-step scheme (use with --N 50..100)\n");
    printf("  --g <abs|plus>     Variance floor g(.) (default: abs)\n");
    printf("  --rng <philox|xorwow|philox-compat|philox-dense|xorwow-fast>  Stream mode (default: philox; philox-dense and\n");
    printf("                     xorwow-fast: fe only; xorwow-fast = the reference's XORWOW draws, native fast-math step)\n");
    printf("  --gpus <int>       GPUs to shard the paths over (default: 1)\n");
    printf("  --paths-per-thread <int>  1, 2, 4 or 8 (default: auto)\n");
    printf("  --strikes <k1,k2,..>  Also price these strikes (and pathwise deltas) on a second pass of the streams\n");
    printf("  --vega                With --strikes: add the pathwise vega d price / d v_0 (fe, --rng philox only)\n");
    printf("  --sensitivities       With --strikes: add the pathwise d price / d p and its std error for p = v_0, k, theta,\n");
    printf("                        sigma, rho, all from the same pass (fe, --rng philox only, |rho| < 1)\n");
    printf("  --legacy-k1        Run the method's K1 class with the reference's K1 moment quirk (E[X^2] field = E[X^2]/n^2)\n");
    printf("  --json             Also print one JSON line with the raw moments\n");
}

template <typename M>
int run(const Options &o)
{
    M m(o.NTPB, o.NB, o.T, o.S_0, o.v_0, o.r, o.k, o.rho, o.theta, o.sigma, o.N);
    m.set_floor_plus(o.g == "plus");
    m.set_gpus(o.gpus);
    m.set_philox_compat(o.rng == "philox-compat");
    m.set_philox_dense(o.rng == "philox-dense");
    m.set_xorwow_fast(o.rng == "xorwow-fast");
    m.set_paths_per_thread(o.ppt);
    m.set_legacy_k1_moment(o.legacy_k1);
    m.init(o.seed);
    m.compute();
    m.print_stats();
    if (o.json) {
        const double n = (double)o.NTPB * (double)o.NB;
        const double units = o.method == "em" ? n : n * o.N;
        // the reference's err formula is NaN when price_squared carries the K1 quirk (n E[X^2]/n^2 - E[X]^2 < 0): JSON has no NaN
        char err_txt[32];
        const float err = m.get_err();
        if (err == err) snprintf(err_txt, sizeof err_txt, "%.9g", err);
        else snprintf(err_txt, sizeof err_txt, "null");
        printf("{\"method\": \"%s\", \"rng\": \"%s\", \"floor\": \"%s\", \"gpus\": %d, \"n_paths\": %.0f, \"N\": %d, "
               "\"sum_payoff\": %.17g, \"sum_payoff_sq\": %.17g, \"E\": %.9g, \"E2\": %.9g, \"std_error\": %.6g, "
               "\"err\": %s, \"exec_ms\": %.6f, \"%s\": %.6g}\n",
               o.method.c_str(), o.rng.c_str(), o.g.c_str(), o.gpus, n, o.N, m.get_sum_payoff(), m.get_sum_payoff_sq(),
               m.get_strike_price(), m.get_price_squared(), m.get_std_error(), err_txt, m.get_execution_time(),
               o.method == "em" ? "paths_per_s" : "path_steps_per_s", units / (m.get_execution_time() * 1e-3));
    }
    if (!o.strikes.empty()) {
        std::vector<float> ks;
        for (size_t p = 0; p < o.strikes.size();) {
            size_t q = o.strikes.find(',', p);
            if (q == std::string::npos) q = o.strikes.size();
            ks.push_back((float)atof(o.strikes.substr(p, q - p).c_str()));
            p = q + 1;
        }
        std::vector<float> pr(ks.size()), sq(ks.size()), dl(ks.size());
        if (o.sensitivities) {
            std::vector<float> sv(ks.size() * NMCH_SENS_COUNT), se(ks.size() * NMCH_SENS_COUNT);
            const float ms = m.compute_sensitivities((int)ks.size(), ks.data(), pr.data(), sq.data(), dl.data(), sv.data(), se.data());
            printf("strike, price, price_squared, delta, d_v0, d_v0_std_error, d_k, d_k_std_error, d_theta, d_theta_std_error, "
                   "d_sigma, d_sigma_std_error, d_rho, d_rho_std_error   (one pass, %f ms)\n", ms);
            for (size_t j = 0; j < ks.size(); ++j) {
                printf("%f, %f, %f, %f", ks[j], pr[j], sq[j], dl[j]);
                for (int d = 0; d < NMCH_SENS_COUNT; ++d)
                    printf(", %f, %f", sv[j * NMCH_SENS_COUNT + d], se[j * NMCH_SENS_COUNT + d]);
                printf("\n");
            }
        } else if (o.vega) {
            std::vector<float> vg(ks.size()), ve(ks.size());
            const float ms = m.compute_greeks((int)ks.size(), ks.data(), pr.data(), sq.data(), dl.data(), vg.data(), ve.data());
            printf("strike, price, price_squared, delta, vega_v0, vega_v0_std_error   (one pass, %f ms)\n", ms);
            for (size_t j = 0; j < ks.size(); ++j) printf("%f, %f, %f, %f, %f, %f\n", ks[j], pr[j], sq[j], dl[j], vg[j], ve[j]);
        } else {
            const float ms = m.compute_strikes((int)ks.size(), ks.data(), pr.data(), sq.data(), dl.data());
            printf("strike, price, price_squared, delta   (one pass, %f ms)\n", ms);
            for (size_t j = 0; j < ks.size(); ++j) printf("%f, %f, %f, %f\n", ks[j], pr[j], sq[j], dl[j]);
        }
    }
    m.finalize();
    return 0;
}

}  // namespace

int main(int argc, char **argv)
{
    Options o;
    for (int i = 1; i < argc; ++i) {
        auto has = [&](const char *f) { return strcmp(argv[i], f) == 0 && i + 1 < argc; };
        if (has("--NTPB")) o.NTPB = atoi(argv[++i]);
        else if (has("--NB")) o.NB = atoi(argv[++i]);
        else if (has("--T")) o.T = atof(argv[++i]);
        else if (has("--S_0")) o.S_0 = atof(argv[++i]);
        else if (has("--v_0")) o.v_0 = atof(argv[++i]);
        else if (has("--r")) o.r = atof(argv[++i]);
        else if (has("--k")) o.k = atof(argv[++i]);
        else if (has("--rho")) o.rho = atof(argv[++i]);
        else if (has("--theta")) o.theta = atof(argv[++i]);
        else if (has("--sigma")) o.sigma = atof(argv[++i]);
        else if (has("--N")) o.N = atoi(argv[++i]);
        else if (has("--seed")) o.seed = strtoull(argv[++i], nullptr, 10);
        else if (has("--method")) o.method = argv[++i];
        else if (has("--g")) o.g = argv[++i];
        else if (has("--rng")) o.rng = argv[++i];
        else if (has("--gpus")) o.gpus = atoi(argv[++i]);
        else if (has("--paths-per-thread")) o.ppt = atoi(argv[++i]);
        else if (has("--strikes")) o.strikes = argv[++i];
        else if (strcmp(argv[i], "--json") == 0) o.json = true;
        else if (strcmp(argv[i], "--legacy-k1") == 0) o.legacy_k1 = true;
        else if (strcmp(argv[i], "--vega") == 0) o.vega = true;
        else if (strcmp(argv[i], "--sensitivities") == 0) o.sensitivities = true;
        else if (strcmp(argv[i], "--help") == 0) { usage(argv[0]); return 0; }
    }
    if (o.rng != "philox" && o.rng != "xorwow" && o.rng != "philox-compat" && o.rng != "philox-dense" &&
        o.rng != "xorwow-fast") {
        printf("Unknown rng: %s\n", o.rng.c_str());
        return 1;
    }
    if ((o.rng == "philox-dense" || o.rng == "xorwow-fast") && o.method != "fe") {
        printf("--rng %s is a forward-Euler stream mode (use --method fe)\n", o.rng.c_str());
        return 1;
    }
    const bool x = o.rng == "xorwow" || o.rng == "xorwow-fast";
    if (o.legacy_k1 && o.method == "fe")
        return x ? run<NMCH_FE_K1_MM<curandStateXORWOW_t>>(o) : run<NMCH_FE_K1_MM<curandStatePhilox4_32_10_t>>(o);
    if (o.legacy_k1 && o.method == "em")
        return x ? run<NMCH_EM_K1_MM<curandStateXORWOW_t>>(o) : run<NMCH_EM_K1_MM<curandStatePhilox4_32_10_t>>(o);
    if (o.method == "fe")
        return x ? run<NMCH_FE_K3_MM<curandStateXORWOW_t>>(o) : run<NMCH_FE_K3_MM<curandStatePhilox4_32_10_t>>(o);
    if (o.method == "em")
        return x ? run<NMCH_EM_K3_MM<curandStateXORWOW_t>>(o) : run<NMCH_EM_K3_MM<curandStatePhilox4_32_10_t>>(o);
    if (o.method == "qe") {                                // additive: large-step QE-M scheme (native Philox stream only)
        if (o.rng != "philox") { printf("Method qe needs --rng philox\n"); return 1; }
        return run<NMCH_QE_K1_MM<curandStatePhilox4_32_10_t>>(o);
    }
    printf("Unknown method: %s\n", o.method.c_str());      // reference nmch.cu:135-137
    return 1;
}
