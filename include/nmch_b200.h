/*
 * nmch_b200.h -- C ABI of the B200-native Heston Monte-Carlo engine.
 *
 * This is the drop-in boundary between the reference's C++ method API (layer L3:
 * nmch::methods::NMCH_FE_* / NMCH_EM_*, /root/reference/include/NMCH/methods/NMCH_{FE,EM}.hpp) and the
 * hand-written sm_100a kernels.  Plain pointers and sizes only; no C++/torch types.
 * Every entry point names the reference interface it replaces (paths relative to
 * /root/reference).  The reference-side binding is shown in INTEGRATION.md.
 *
 * Conventions: every function returns 0 (NMCH_OK) or a negative nmch_status; the caller
 * serialises calls on one handle; distinct handles are independent.  There is NO CPU
 * fallback: without a CUDA device every compute entry point returns NMCH_ERR_CUDA.
 */
#ifndef NMCH_B200_H
#define NMCH_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nmch_engine nmch_engine_t;

typedef enum {
    NMCH_OK = 0,
    NMCH_ERR_ARG = -1,        /* bad argument / unsupported combination */
    NMCH_ERR_CUDA = -2,       /* a CUDA runtime call or kernel failed (see nmch_last_error) */
    NMCH_ERR_STATE = -3,      /* lifecycle misuse: compute before init, use after finalize */
    NMCH_ERR_NCCL = -4
} nmch_status;

/* which scheme: FE = NMCH_FE_* (src/NMCH/methods/NMCH_FE.cu), EM = NMCH_EM_* (NMCH_EM.cu);
 * QE = Andersen's quadratic-exponential large-step scheme with martingale correction (no reference equivalent:
 * SURVEY.md §8f row 3), native Philox stream only */
typedef enum { NMCH_METHOD_FE = 0, NMCH_METHOD_EM = 1, NMCH_METHOD_QE = 2 } nmch_method;
/* variance floor g(.) of README.md:37-40; the reference codes only ABS (NMCH_FE.cu:162) */
typedef enum { NMCH_FLOOR_ABS = 0, NMCH_FLOOR_PLUS = 1 } nmch_floor;
/* stream mode, selected by the reference's rnd_state template tag:
 *   PHILOX         native counter-based Philox4x32-10 fused into the step loop, fast-math transforms
 *                  (cuRAND counter layout, so the u32 words per (path, step) equal the reference's
 *                  Philox instantiation; floats agree to ~2^-23 per draw)
 *   XORWOW_COMPAT  curandStateXORWOW_t-compatible: same integer stream, same IEEE transforms and FMA
 *                  contraction as the reference's CUDA build
 *   PHILOX_COMPAT  curandStatePhilox4_32_10_t-compatible (reference CLI default, nmch.cu:119,130)
 *   MRG32K3A_COMPAT curandStateMRG32k3a_t-compatible (the third tag the reference instantiates, NMCH.cu:31)
 *   PHILOX_DENSE   opt-in FE throughput mode: the same Philox4x32-10 blocks cut into THREE (23-bit radius, 19-bit
 *                  angle) draws instead of two word pairs, i.e. a third fewer generator multiplies per step.  Statistically
 *                  equivalent, NOT word-compatible with cuRAND's per-step layout (checked against a restatement of its
 *                  own mapping and against the semi-analytic price)
 *   XORWOW_FAST    opt-in FE mode on the reference's default stream: the SAME cuRAND-XORWOW integer draws per path
 *                  as XORWOW_COMPAT (same seed scramble, subsequence skip-ahead and continuation across compute()
 *                  calls), pushed through the native fast-math step (cuRAND's uniforms, MUFU transforms) instead of
 *                  cuRAND's IEEE transforms.  Prices agree with the reference's CUDA build on identical seeds to
 *                  ~1e-6 relative (the 1e-5 tolerance of the XORWOW-compatible mode) at 2.5x its speed; per-path
 *                  values agree to ~1e-4, not to the last bits -- use XORWOW_COMPAT for draw-for-draw validation */
typedef enum { NMCH_RNG_PHILOX = 0, NMCH_RNG_XORWOW_COMPAT = 1, NMCH_RNG_PHILOX_COMPAT = 2,
               NMCH_RNG_MRG32K3A_COMPAT = 3, NMCH_RNG_PHILOX_DENSE = 4, NMCH_RNG_XORWOW_FAST = 5 } nmch_rng;

/* Replaces the constructor arguments of nmch::methods::NMCH (include/NMCH/methods/NMCH.hpp:42,
 * src/NMCH/methods/NMCH.cu:6-10).  Zero in an "auto" field selects the default. */
typedef struct {
    int   NTPB, NB;                 /* logical paths n = NTPB*NB (NMCH_FE.cu:317); launch geometry is internal */
    float T, S_0, v_0, r, k, rho, theta, sigma;
    int   N;                        /* time steps; dt = T/N */
    int   method, floor, rng;       /* nmch_method, nmch_floor, nmch_rng */
    int   device;                   /* CUDA ordinal; -1 = current device */
    unsigned long long n_paths;     /* auto(0) = NTPB*NB; lets n exceed the reference's int limit */
    unsigned long long first_path;  /* shard: this engine simulates paths [first_path, first_path+n_local) */
    unsigned long long n_local;     /* auto(0) = n_paths - first_path */
    int   paths_per_thread;         /* auto(0): picked from n_local; 1, 2, 4 or 8 */
    int   block_threads;            /* auto(0) = 256; 128 or 256 */
} nmch_params_t;

/* Replaces the two managed floats `sum[2]` (NMCH_FE.cu:376, 544-545) with raw FP64 sums:
 * E[X] = sum_payoff / n_paths, E[X^2] = sum_payoff_sq / n_paths. */
typedef struct {
    double sum_payoff;
    double sum_payoff_sq;
    unsigned long long n_paths;     /* paths behind the sums (n_local for a shard) */
    float  exec_ms;                 /* kernel + sync, the span of the reference's Tim_exec (NMCH_FE.cu:523-540) */
} nmch_moments_t;

/* ctor of NMCH_FE_* / NMCH_EM_* (NMCH_FE.cu:313-318, NMCH_EM.cu:376-382) */
int nmch_engine_create(const nmch_params_t *params, nmch_engine_t **out);
/* init(seed) (NMCH_FE.cu:367-386): allocates device buffers, builds generator state.
 * Philox: nothing to build (counter = path index); XORWOW: skip-ahead init kernel (random.cu:6-10). */
int nmch_engine_init(nmch_engine_t *e, unsigned long long seed);
/* set_k / set_theta / set_sigma (NMCH.hpp:76-80): host fields only, effective at next compute */
int nmch_engine_set_params(nmch_engine_t *e, float k, float theta, float sigma);
/* Positions every path's stream as if `words` 32-bit draws had already been consumed (the `offset` argument of
 * curand_init, which the reference always passes as 0, random.cu:9).  FE in the Philox modes only (a counter-based
 * stream seeks for free); `words` must be even.  Other modes return NMCH_ERR_ARG. */
int nmch_engine_seek(nmch_engine_t *e, unsigned long long words);
/* compute() (NMCH_FE.cu:516-546): one pass over all local paths, streams continue across calls */
int nmch_engine_compute(nmch_engine_t *e, nmch_moments_t *out);
/* Same pass, asynchronous: enqueued on `cuda_stream` (a cudaStream_t; NULL = the CUDA default stream),
 * raw sums {sum, sumsq} written to the DEVICE buffer d_moments[2] (e.g. an NCCL send buffer), no host
 * sync, no exec_ms.  This is what the multi-GPU layer calls before its single allreduce. */
int nmch_engine_compute_async(nmch_engine_t *e, void *cuda_stream, double *d_moments);
/* The exploration sweep of src/NMCH/test/exploration.cu:71-88 as ONE launch: point i uses
 * (k[i], theta[i], sigma[i]) and the stream position it would have had after i sequential compute()
 * calls, so explore() uses the same draws as n_points x { set_params; compute } and returns the same sums up to
 * the order of the FP64 summation (bit for bit when the two launches have the same shape: paths per thread and
 * tiles per block are picked from n_local x n_points).  out has n_points entries.  EM sweeps whose points need
 * different variance samplers (d = 2 k theta / sigma^2 below 1/2, between 1/2 and 3/2, above) are still ONE launch. */
int nmch_engine_explore(nmch_engine_t *e, const float *k, const float *theta, const float *sigma,
                        int n_points, nmch_moments_t *out);
int nmch_engine_explore_async(nmch_engine_t *e, void *cuda_stream, const float *k, const float *theta,
                              const float *sigma, int n_points, double *d_moments /* [2*n_points] */);
/* Parity hook (no reference equivalent: its kernels only emit sums): runs one compute() pass and also
 * returns the terminal S and V of local paths [0, count) into HOST arrays. */
int nmch_engine_compute_paths(nmch_engine_t *e, float *S_out, float *V_out, unsigned long long count,
                              nmch_moments_t *out);
/* ---- strike vector + pathwise delta in the same pass (SURVEY.md §8f rank 2; no reference equivalent: it fixes
 * K = S_0, src/NMCH/methods/NMCH.cu:7).  The paths of ONE compute() pass price n_strikes calls: the path kernel
 * keeps the terminal prices on the device (4 bytes per path) and a second small kernel folds them per strike with
 * the same deterministic FP64 reduction.  Streams advance exactly as for compute(). */
#define NMCH_MAX_STRIKES 64
typedef struct {
    float  strike;
    double sum_payoff;        /* sum (S_T - K)^+                      */
    double sum_payoff_sq;     /* sum ((S_T - K)^+)^2                  */
    double sum_delta;         /* sum 1{S_T > K} S_T / S_0   (pathwise d payoff / d S_0) */
    double sum_itm;           /* sum 1{S_T > K}                       */
    unsigned long long n_paths;
    float  exec_ms;
} nmch_strike_moments_t;
int nmch_engine_compute_strikes(nmch_engine_t *e, const float *strikes, int n_strikes, nmch_strike_moments_t *out);
/* stream form: 4*n_strikes raw sums {payoff, payoff^2, delta, itm} per strike into DEVICE memory, no host sync */
int nmch_engine_compute_strikes_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                      double *d_moments);
/* ---- ... and the pathwise vega (the second half of SURVEY.md §8f rank 2, "pathwise delta/vega"; no reference
 * equivalent).  FE on the native Philox stream only: one pass of the native step (the same words and instructions, so
 * the same S_T, as compute()) carries every path's tangent dS_T/dv_0 in registers; the fold then adds, per strike,
 * vega = 1{S_T > K} dS_T/dv_0 -- the sensitivity of the undiscounted price E[(S_T - K)^+] to the initial variance v_0
 * (the reference reports undiscounted prices too, NMCH_FE.cu:171-175) -- and its square for the standard error.
 * Other methods / stream modes return NMCH_ERR_ARG.  Streams advance exactly as for compute(). */
typedef struct {
    float  strike;
    double sum_payoff;        /* sum (S_T - K)^+                      */
    double sum_payoff_sq;     /* sum ((S_T - K)^+)^2                  */
    double sum_delta;         /* sum 1{S_T > K} S_T / S_0             */
    double sum_itm;           /* sum 1{S_T > K}                       */
    double sum_vega;          /* sum 1{S_T > K} dS_T/dv_0   (pathwise d payoff / d v_0) */
    double sum_vega_sq;       /* sum (1{S_T > K} dS_T/dv_0)^2         */
    unsigned long long n_paths;
    float  exec_ms;
} nmch_greek_moments_t;
int nmch_engine_compute_greeks(nmch_engine_t *e, const float *strikes, int n_strikes, nmch_greek_moments_t *out);
/* stream form: 6*n_strikes raw sums {payoff, payoff^2, delta, itm, vega, vega^2} per strike into DEVICE memory */
int nmch_engine_compute_greeks_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                     double *d_moments);

/* ---- ... and the pathwise sensitivities to every Heston parameter (no reference equivalent): the same pass carries
 * the tangent of every path in five directions p = v_0, kappa, theta, sigma, rho at once, so one pass returns the full
 * gradient of the FE-discretised, undiscounted price E[(S_T - K)^+] (the convention of compute_greeks) per strike:
 *   sum_sens[p] = sum 1{S_T > K} dS_T/dp,   sum_sens_sq[p] = sum (1{S_T > K} dS_T/dp)^2   (for the standard error).
 * The derivative is that of the FE map in the mathematical parameters (the host folds dt, kappa theta dt, ... in
 * double; their derivatives are folded the same way), not of the float32 rounding of that folding.  sum_sens[NMCH_SENS_V0]
 * and the four strike sums equal compute_greeks' and compute_strikes' bit for bit.  FE on the native Philox stream only;
 * other methods / stream modes, n_strikes outside 1..NMCH_MAX_STRIKES and |rho| >= 1 (where d sqrt(1 - rho^2) / d rho is
 * infinite) return NMCH_ERR_ARG and leave the engine as it was.  Streams advance exactly as for compute(). */
#define NMCH_SENS_V0    0
#define NMCH_SENS_KAPPA 1     /* the mean-reversion speed k of nmch_params_t */
#define NMCH_SENS_THETA 2
#define NMCH_SENS_SIGMA 3
#define NMCH_SENS_RHO   4
#define NMCH_SENS_COUNT 5
typedef struct {
    float  strike;
    double sum_payoff;        /* sum (S_T - K)^+                      */
    double sum_payoff_sq;     /* sum ((S_T - K)^+)^2                  */
    double sum_delta;         /* sum 1{S_T > K} S_T / S_0             */
    double sum_itm;           /* sum 1{S_T > K}                       */
    double sum_sens[NMCH_SENS_COUNT];      /* sum 1{S_T > K} dS_T/dp, p in NMCH_SENS_* order */
    double sum_sens_sq[NMCH_SENS_COUNT];   /* sum (1{S_T > K} dS_T/dp)^2          */
    unsigned long long n_paths;
    float  exec_ms;
} nmch_sensitivity_moments_t;
int nmch_engine_compute_sensitivities(nmch_engine_t *e, const float *strikes, int n_strikes,
                                      nmch_sensitivity_moments_t *out);
/* stream form: 14*n_strikes raw sums per strike into DEVICE memory, in the order
 * {payoff, payoff^2, delta, itm, sens[v_0], sens_sq[v_0], sens[kappa], sens_sq[kappa], sens[theta], sens_sq[theta],
 *  sens[sigma], sens_sq[sigma], sens[rho], sens_sq[rho]} */
int nmch_engine_compute_sensitivities_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                            double *d_moments);

/* finalize() (NMCH_FE.cu:326-331); idempotent here (the reference double-frees) */
int nmch_engine_finalize(nmch_engine_t *e);
void nmch_engine_destroy(nmch_engine_t *e);

/* Memory-safety probe (no reference equivalent; its only check is one testCUDA, NMCH_FE.cu:685).  Synchronises the
 * device and, in the checked build of this library (libnmch_b200_checked.so: -DNMCHB_CHECKS, device-side asserts on
 * every index the kernels form + guard bands around every device buffer), sweeps the guard bands: NMCH_ERR_CUDA names
 * the buffer a kernel wrote outside of, or reports the failed device assert.  The blocking entry points run the same
 * sweep themselves; this call is for *_async users.  In the normal build it is a synchronise that returns NMCH_OK.
 * nmch_checked_build() tells which build is loaded. */
int nmch_engine_check(nmch_engine_t *e);
int nmch_checked_build(void);
/* checked build only: plants an overrun behind the ticket array and verifies that the sweep reports it (NMCH_OK = it did) */
int nmch_checked_selftest(nmch_engine_t *e);

/* Tim_init (NMCH_FE.cu:370-385) and launch facts for reports */
float nmch_engine_init_ms(const nmch_engine_t *e);
typedef struct {
    int grid_x, grid_y, block_threads, paths_per_thread, regs_per_thread, sm_count;
    int kernel_param_bytes;                 /* bytes of kernel parameters uploaded by the last launch (the only H2D traffic of compute()) */
    unsigned long long kernel_launches;     /* kernels launched by this handle so far */
} nmch_launch_info_t;
int nmch_engine_launch_info(const nmch_engine_t *e, nmch_launch_info_t *out);

/* ---- multi-GPU group (one process, G devices): the path axis is sharded, paths [g*n/G, (g+1)*n/G) on
 * device g with disjoint generator subsequences (global path index = subsequence, random.cu:8-9), and ONE
 * ncclAllReduce(ncclDouble, ncclSum) over NVLink of the 2*n_points partial moments per compute()/explore().
 * The reference has no multi-GPU path (SURVEY.md §2: "Distributed backend: none"); a group of 1 is a plain
 * engine and needs no NCCL.  The C++ method classes (include/NMCH/methods/ headers) sit on this API. */
typedef struct nmch_group nmch_group_t;
int nmch_group_create(const nmch_params_t *params, int n_gpus, nmch_group_t **out);
int nmch_group_init(nmch_group_t *g, unsigned long long seed);
int nmch_group_set_params(nmch_group_t *g, float k, float theta, float sigma);
int nmch_group_compute(nmch_group_t *g, nmch_moments_t *out);            /* out: GLOBAL sums, n_paths = n */
int nmch_group_explore(nmch_group_t *g, const float *k, const float *theta, const float *sigma, int n_points,
                       nmch_moments_t *out);
int nmch_group_finalize(nmch_group_t *g);
void nmch_group_destroy(nmch_group_t *g);
int nmch_group_compute_strikes(nmch_group_t *g, const float *strikes, int n_strikes, nmch_strike_moments_t *out);
int nmch_group_compute_greeks(nmch_group_t *g, const float *strikes, int n_strikes, nmch_greek_moments_t *out);
/* one allreduce of 14*n_strikes doubles */
int nmch_group_compute_sensitivities(nmch_group_t *g, const float *strikes, int n_strikes, nmch_sensitivity_moments_t *out);
float nmch_group_init_ms(const nmch_group_t *g);
int nmch_group_size(const nmch_group_t *g);

const char *nmch_status_string(int status);
const char *nmch_last_error(void);          /* thread-local detail of the last failure */
int nmch_device_count(void);
const char *nmch_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NMCH_B200_H */
