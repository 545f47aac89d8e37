// engine_internal.cuh -- the engine object behind the opaque nmch_engine_t handle, shared by engine.cu
// (FE + lifecycle) and em_kernels.cu (EM launches).
#pragma once
#include <vector>

#include "../../include/nmch_b200.h"
#include "kernels.cuh"

// one device allocation of an engine in the checked build: [guard | user bytes | guard]
struct nmch_guarded_alloc {
    void *base;
    void *user;
    size_t bytes;
    const char *name;
};

struct nmch_engine {
    nmch_params_t p{};
    int device = 0;
    int sm_count = 0;
    bool inited = false;
    unsigned long long seed = 0;
    unsigned long long n_paths = 0, first_path = 0, n_local = 0;
    unsigned long long draw_offset = 0;      // FE Philox modes: u32 words consumed per path so far
    unsigned long long em_calls = 0;         // EM native mode: compute() calls so far (selects a fresh stream)
    float init_ms = 0.0f;
    int threads = 128;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // reduction buffers
    double2 *d_partials = nullptr;
    size_t partials_cap = 0;
    unsigned int *d_tickets = nullptr;
    size_t tickets_cap = 0;
    double *h_out = nullptr;                 // mapped pinned host memory, written by the kernel
    double *h_out_dev = nullptr;             // its device alias
    size_t out_cap = 0;
    void *d_points = nullptr;                // FePoint[] / RawPoint[] / EmPoint[]
    size_t points_cap = 0;
    float *d_S = nullptr, *d_V = nullptr;    // parity hook buffers
    size_t sv_cap = 0;
    float *d_T = nullptr;                    // dS_T/dp of every local path: v_0 (compute_greeks) or all five directions,
                                             // tangent_stride(n_local) floats apart (compute_sensitivities)
    size_t t_cap = 0;
    // XORWOW-compat state
    nmchb::XorwowSkipTables *xtab = nullptr;
    nmchb::XorwowState xs{};
    uint32_t *d_xskip = nullptr;             // XORWOW offset-skip tables of the current sweep shape (chunked sweeps)
    unsigned long long xskip_draws = 0;      //   ... for chunks of this many draws
    int xskip_digits = 0;                    //   ... and this many base-4 digits of the chunk index
    void *curand_states = nullptr;           // cuRAND-layout states (AoS): Philox-compat EM, MRG32k3a-compat FE/EM
    nmchb::KernelInfo kinfo{};
    unsigned long long launches = 0;
    std::vector<nmch_guarded_alloc> guarded;  // checked build (-DNMCHB_CHECKS) only: every device buffer, for the guard sweep
};

namespace nmchb {

int engine_fail(int status, const char *what, cudaError_t err = cudaSuccess);
// Device memory of an engine.  Normal build: cudaMalloc / cudaFree.  Checked build: each buffer sits between two guard
// bands filled with a pattern, and engine_check_guards() (run by every blocking entry point after its sync, and by
// nmch_engine_check) fails with NMCH_ERR_CUDA naming the buffer whose band a kernel overwrote.
cudaError_t engine_dev_malloc(nmch_engine *e, void **ptr, size_t bytes, const char *name);
void engine_dev_free(nmch_engine *e, void *ptr);
int engine_check_guards(nmch_engine *e);
int engine_ensure_buffers(nmch_engine *e, size_t n_points, size_t blocks_per_point);
// Copies `bytes` of host records (parameter points, strikes) to e->d_points, growing it as needed, and waits for the copy:
// the source may be a staging buffer on the caller's stack or caller memory of unknown lifetime.
int upload_records(nmch_engine *e, cudaStream_t stream, const void *host, size_t bytes);

// em_kernels.cu
int em_launch_points(nmch_engine *e, cudaStream_t stream, const float *k, const float *theta, const float *sigma,
                     int n_points, double *d_out, float *S_out, float *V_out);
// qe_kernels.cu
int qe_launch_points(nmch_engine *e, cudaStream_t stream, const float *k, const float *theta, const float *sigma,
                     int n_points, double *d_out, float *S_out, float *V_out);
int em_philox_compat_init(nmch_engine *e);
int mrg_compat_init(nmch_engine *e);
cudaError_t launch_fe_compat_mrg(const FeLaunch &L, int floor_kind, const RawPoint *d_pts, void *states,
                                 ReduceBuffers rb, float *S_out, float *V_out, cudaStream_t stream, KernelInfo *info);
void em_release(nmch_engine *e);

static_assert(NMCH_SENS_COUNT == kNumDirs && NMCH_SENS_V0 == kDirV0 && NMCH_SENS_KAPPA == kDirKappa &&
                  NMCH_SENS_THETA == kDirTheta && NMCH_SENS_SIGMA == kDirSigma && NMCH_SENS_RHO == kDirRho,
              "the header's direction order is the kernels' order");
// The strike family (compute_strikes, compute_greeks, compute_sensitivities) is one pass with the tangent in n_dirs = 0, 1
// or NMCH_SENS_COUNT directions.  Per strike it leaves strike_doubles(n_dirs) raw sums: payoff, payoff^2, delta,
// in-the-money count, then the sum and the sum of squares of 1{S_T > K} dS_T/dp for each direction.
constexpr int strike_doubles(int n_dirs) { return 4 + 2 * n_dirs; }
// The stream form of that pass (engine.cu), shared by the engine's and the group's entry points.
int engine_strike_async(nmch_engine *e, void *cuda_stream, const float *strikes, int n_strikes, int n_dirs, double *d_out);

// one strike's raw sums (strike_doubles(n_dirs) of them, n_dirs as the struct implies) into the public struct
inline void strike_unpack(const double *m, float strike, unsigned long long n_paths, float ms, nmch_strike_moments_t *out)
{
    *out = nmch_strike_moments_t{strike, m[0], m[1], m[2], m[3], n_paths, ms};
}

inline void strike_unpack(const double *m, float strike, unsigned long long n_paths, float ms, nmch_greek_moments_t *out)
{
    *out = nmch_greek_moments_t{strike, m[0], m[1], m[2], m[3], m[4], m[5], n_paths, ms};
}

inline void strike_unpack(const double *m, float strike, unsigned long long n_paths, float ms,
                          nmch_sensitivity_moments_t *out)
{
    out->strike = strike;
    out->sum_payoff = m[0];
    out->sum_payoff_sq = m[1];
    out->sum_delta = m[2];
    out->sum_itm = m[3];
    for (int d = 0; d < NMCH_SENS_COUNT; ++d) {
        out->sum_sens[d] = m[4 + 2 * d];
        out->sum_sens_sq[d] = m[5 + 2 * d];
    }
    out->n_paths = n_paths;
    out->exec_ms = ms;
}

}  // namespace nmchb
