// kernels.cuh -- launch-parameter blocks and launcher prototypes shared by the engine and the kernels.
#pragma once
#include <cstdint>
#include <vector>
#include <cuda_runtime.h>

#include "device_common.cuh"

namespace nmchb {

constexpr int kFloorAbs = 0, kFloorPlus = 1;
constexpr int kRngPhilox = 0, kRngXorwowCompat = 1, kRngPhiloxCompat = 2, kRngMrgCompat = 3, kRngPhiloxDense = 4, kRngXorwowFast = 5;
constexpr int kMaxTilePaths = 4096;     // native mode: first_path % kMaxTilePaths == 0 (no carry inside a tile)

// Per-point constants of the native FE kernel, folded on the host (fold_fe_point):
//   V' = g( V*va + vb + (sqrt(V)*n1)*vs ),  va = 1-k*dt, vb = theta*(1-va) (= k*theta*dt up to the rounding of va, so
//   that the long-run level of the folded map is theta exactly), vs = sigma*sqrt(dt)*sqrt(2 ln 2), kdt = k*dt
struct FePoint {
    float va, vb, vs, kdt;
};

// Per-point raw parameters for the compat kernels (they evaluate the reference's expressions verbatim).
struct RawPoint {
    float k, theta, sigma, pad;
};
static_assert(sizeof(RawPoint) == sizeof(FePoint), "the engine uploads raw records as FePoint{k, theta, sigma, 0}");

struct FeLaunch {
    PhiloxKeys keys;                    // expanded from the seed
    unsigned long long first_path;      // global index of local path 0 (= Philox subsequence of path 0)
    unsigned long long n_local;         // paths simulated by this engine
    unsigned long long draw_offset;     // u32 words each path has already consumed (stream position of point 0)
    // dense mode: the same position in STEPS, pre-divided on the host so that the kernel needs no 64-bit division
    // (which would leave the uniform datapath):  draw_offset / 2 = 3 * dense_q0 + dense_r0,  N = 3 * dense_qN + dense_rN
    unsigned long long dense_q0;
    unsigned int dense_r0, dense_qN, dense_rN;
    int   N;                            // time steps
    int   n_points;
    int   blocks_per_point;
    int   tiles_per_block;
    // XORWOW sweeps walked in chunks (fe_compat_kernel / fe_xorwow_fast_kernel): blockIdx.y = chunk of chunk_points
    // consecutive points; chunk c starts c * chunk_points * 2N draws into every path's stream (skip tables)
    int   chunk_points, n_chunks;
    float S0, v0, K;
    float rdt;                          // r*dt
    float zr, zc;                       // rho*sqrt(dt)*c0, sqrt(1-rho^2)*sqrt(dt)*c0, c0 = sqrt(2 ln 2)
    // compat kernels: the reference's own scalars (NMCH_FE.cu:135-153)
    float r, rho, dt, sqrt_dt, sqrt_rho;
    FePoint  pt0;                       // used when n_points == 1 (no parameter upload)
    RawPoint raw0;
};

// Directions of the pathwise tangent, in the order of nmch_sensitivity_moments_t (NMCH_SENS_V0 .. NMCH_SENS_RHO).
constexpr int kDirV0 = 0, kDirKappa = 1, kDirTheta = 2, kDirSigma = 3, kDirRho = 4, kNumDirs = 5;

// Derivatives of the folded step constants in the directions kappa, theta, sigma and rho (fold_tangent: double on the
// host, rounded once).  They are taken of the mathematical FE map (va = 1 - k dt, vb = k theta dt, vs = sigma sqrt(dt) c0,
// zr = rho sqrt(dt) c0, zc = sqrt(1 - rho^2) sqrt(dt) c0), not of the float32 rounding of the folding.
struct TangentFold {
    float dva_k;                        // d va / d kappa = -dt
    float dvb_k;                        // d vb / d kappa = theta dt
    float dvb_t;                        // d vb / d theta = kappa dt
    float dvs_s;                        // d vs / d sigma = sqrt(dt) c0 (not vs / sigma: sigma = 0 is a valid point)
    float dzr_r;                        // d zr / d rho   = sqrt(dt) c0
    float dzc_r;                        // d zc / d rho   = -rho / sqrt(1 - rho^2) sqrt(dt) c0
};

struct ReduceBuffers {
    double2      *partials;             // [n_points][blocks_per_point]
    unsigned int *tickets;              // [n_points], zero between launches
    double       *out;                  // [2*n_points] raw sums (device memory or mapped pinned host memory)
};

struct XorwowState {                    // structure of arrays, one entry per local path
    uint32_t *d, *v0, *v1, *v2, *v3, *v4;
    // Box-Muller caches used only by EM (curand_normal.h:313-326, 581-596)
    int *bm_flag;
    float *bm_extra;
    int *bm_flag_d;
    double *bm_extra_d;
};

struct KernelInfo {
    int grid_x, grid_y, block_threads, paths_per_thread, regs_per_thread;
    int param_bytes = 0;
};

// fe_kernels.cu
// exact_math: cuRAND's IEEE transforms + the reference's pinned update on the same Philox words (Philox-compat
// mode); d_pts then holds raw (k, theta, sigma, 0) records instead of folded constants
cudaError_t launch_fe_philox(const FeLaunch &L, int floor_kind, int paths_per_thread, int block_threads,
                             bool exact_math, const FePoint *d_pts, ReduceBuffers rb, float *S_out, float *V_out,
                             cudaStream_t stream, KernelInfo *info);
// dense-draw variant: three steps per Philox block (NMCH_RNG_PHILOX_DENSE); block size 128, P in {1, 2, 4}
cudaError_t launch_fe_dense(const FeLaunch &L, int floor_kind, int paths_per_thread, const FePoint *d_pts, ReduceBuffers rb,
                            float *S_out, float *V_out, cudaStream_t stream, KernelInfo *info);
// skip: device tables A^(q 4^m) with A = T^(2N * chunk_points) (xorwow_offset_tables_host), or nullptr when n_chunks == 1
cudaError_t launch_fe_compat(const FeLaunch &L, int floor_kind, const RawPoint *d_pts, XorwowState xs, const uint32_t *skip,
                             ReduceBuffers rb, float *S_out, float *V_out, cudaStream_t stream, KernelInfo *info);
// XORWOW integer stream + the native fast-math step (NMCH_RNG_XORWOW_FAST); d_pts holds folded FePoint records
cudaError_t launch_fe_xorwow_fast(const FeLaunch &L, int floor_kind, const FePoint *d_pts, XorwowState xs, const uint32_t *skip,
                                  ReduceBuffers rb, float *S_out, float *V_out, cudaStream_t stream, KernelInfo *info);

// greeks_kernels.cu: the native FE pass carrying the pathwise tangent in n_dirs = 1 (v_0) or 5 (v_0, kappa, theta, sigma,
// rho; fe_step.cuh) directions (leaves S_T, V_T and dS_T/dp of every direction on the device), and the one per-strike
// fold of every strike-family pass: payoff / delta sums from S_T alone (n_dirs = 0, after any path kernel) or with the
// sensitivities from d_B as well: 2 + n_dirs reduction slots = 4 + 2 n_dirs doubles per strike
cudaError_t launch_fe_tangent(const FeLaunch &L, int floor_kind, int n_dirs, const TangentFold &tf, ReduceBuffers rb,
                              float *S_out, float *V_out, float *B_out, cudaStream_t stream, KernelInfo *info);
cudaError_t launch_strike_fold(const float *d_S, const float *d_B, int n_dirs, unsigned long long n_local,
                               const float *d_strikes, int n_strikes, float S0, ReduceBuffers rb, cudaStream_t stream);
int strike_blocks_per_slot();
int tangent_tile_paths(int n_dirs);       // paths per block of fe_tangent_kernel
// floats between the tangent arrays of two directions: n_local rounded up to 16 bytes, so that every array takes float4 loads
__host__ __device__ inline unsigned long long tangent_stride(unsigned long long n_local) { return (n_local + 3ull) & ~3ull; }

// xorwow.cu
struct XorwowSkipTables;                // device tables M_m^q, q = 1..3, m = 0..31
cudaError_t xorwow_tables_create(XorwowSkipTables **out);
void        xorwow_tables_destroy(XorwowSkipTables *t);
// host side of the offset skip: tables of T^(draws * q * 4^m), q = 1..3, m < n_digits (device layout)
std::vector<uint32_t> xorwow_offset_tables_host(unsigned long long draws, int n_digits);
cudaError_t launch_xorwow_init(const XorwowSkipTables *t, unsigned long long seed,
                               unsigned long long first_path, unsigned long long n_local, XorwowState xs,
                               cudaStream_t stream);

}  // namespace nmchb
