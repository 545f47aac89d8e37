// engine.cu -- the C ABI (include/nmch_b200.h) over the sm_100a kernels.
//
// Host-side mirror of the reference's L2 drivers (src/NMCH/methods/NMCH_FE.cu:312-546,
// NMCH_EM.cu:376-575): allocate, time with CUDA events, launch, read two numbers back.
// Differences by design: one fused kernel per compute()/explore(), FP64 raw sums instead of two
// float atomics, every CUDA call checked, finalize() idempotent, no managed memory (the result is
// written by the kernel's single writer straight into mapped pinned host memory or into the
// caller's device buffer).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/nmch_b200.h"
#include <nvtx3/nvToolsExt.h>

#include "engine_internal.cuh"

using namespace nmchb;

namespace {

thread_local std::string g_last_error;

}  // namespace
namespace nmchb {
int engine_fail(int status, const char *what, cudaError_t err)
{
    char buf[512];
    if (err != cudaSuccess) {
        std::snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(err), cudaGetErrorString(err));
        (void)cudaGetLastError();       // a failed call leaves its code behind; do not let a later launch inherit it
    } else
        std::snprintf(buf, sizeof buf, "%s", what);
    g_last_error = buf;
    return status;
}
}  // namespace nmchb
namespace nmchb {
#ifdef NMCHB_CHECKS
constexpr size_t kGuardBytes = 256;
constexpr int kGuardByte = 0xA5;

cudaError_t engine_dev_malloc(nmch_engine *e, void **ptr, size_t bytes, const char *name)
{
    *ptr = nullptr;
    unsigned char *base = nullptr;
    const size_t padded = (bytes + 255) / 256 * 256;         // keep the user pointer and the tail guard 256-byte aligned
    cudaError_t err = cudaMalloc(&base, padded + 2 * kGuardBytes);
    if (err != cudaSuccess) return err;
    err = cudaMemset(base, kGuardByte, padded + 2 * kGuardBytes);
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { cudaFree(base); return err; }
    *ptr = base + kGuardBytes;
    e->guarded.push_back(nmch_guarded_alloc{base, *ptr, bytes, name});
    return cudaSuccess;
}

void engine_dev_free(nmch_engine *e, void *ptr)
{
    if (!ptr) return;
    for (size_t i = 0; i < e->guarded.size(); ++i)
        if (e->guarded[i].user == ptr) {
            cudaFree(e->guarded[i].base);
            e->guarded.erase(e->guarded.begin() + (long)i);
            return;
        }
    cudaFree(ptr);
}

int engine_check_guards(nmch_engine *e)
{
    std::vector<unsigned char> host(2 * kGuardBytes + 256);
    for (const nmch_guarded_alloc &g : e->guarded) {
        const unsigned char *base = static_cast<const unsigned char *>(g.base);
        const size_t tail_off = kGuardBytes + g.bytes;                       // first byte past the user's bytes
        const size_t tail_len = (g.bytes + 255) / 256 * 256 - g.bytes + kGuardBytes;
        cudaError_t err = cudaMemcpy(host.data(), base, kGuardBytes, cudaMemcpyDeviceToHost);
        if (err == cudaSuccess) err = cudaMemcpy(host.data() + kGuardBytes, base + tail_off, tail_len, cudaMemcpyDeviceToHost);
        if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "guard sweep", err);
        for (size_t i = 0; i < kGuardBytes + tail_len; ++i)
            if (host[i] != (unsigned char)kGuardByte) {
                char buf[160];
                std::snprintf(buf, sizeof buf, "checked build: guard band of device buffer '%s' (%zu bytes) overwritten %s it",
                              g.name, g.bytes, i < kGuardBytes ? "before" : "after");
                return engine_fail(NMCH_ERR_CUDA, buf);
            }
    }
    return NMCH_OK;
}
#else
cudaError_t engine_dev_malloc(nmch_engine *, void **ptr, size_t bytes, const char *) { return cudaMalloc(ptr, bytes); }
void engine_dev_free(nmch_engine *, void *ptr) { if (ptr) cudaFree(ptr); }
int engine_check_guards(nmch_engine *) { return NMCH_OK; }
#endif
}  // namespace nmchb
namespace {
inline int fail(int status, const char *what, cudaError_t err = cudaSuccess) { return engine_fail(status, what, err); }

#define CU_TRY(call)                                                    \
    do {                                                                \
        cudaError_t err__ = (call);                                     \
        if (err__ != cudaSuccess) return fail(NMCH_ERR_CUDA, #call, err__); \
    } while (0)

// NVTX range for profilers (nsys / ncu --nvtx); header-only NVTX3, a no-op unless a tool is attached
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (dev == prev) || (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

}  // namespace


namespace {

bool is_multiple_of(unsigned long long v, unsigned long long m) { return (v % m) == 0ull; }

int pick_paths_per_thread(const nmch_engine *e, int n_points)
{
    if (e->p.paths_per_thread > 0) return e->p.paths_per_thread;
    // Enough warps first (>= 16 resident per SM), then ILP: each extra path per thread hides more of
    // the dependent MUFU/FMA chain without costing occupancy (47 regs at P = 4).  Work = paths x points.
    const unsigned long long per_sm = e->n_local * (unsigned long long)n_points /
                                      (unsigned long long)(e->sm_count > 0 ? e->sm_count : 148);
    if (per_sm >= 4096ull) return 4;
    if (per_sm >= 2048ull) return 2;
    return 1;
}

FePoint fold_fe_point(const nmch_params_t &p, float k, float theta, float sigma, bool exact_v = false)
{
    // dt as the reference forms it (float, NMCH.cu:9); everything derived from it in double, rounded once
    const double dt = (double)(p.T / (float)p.N);
    const double c0 = 1.1774100225154747;                    // sqrt(2 ln 2)
    FePoint pt;
    pt.va = (float)(1.0 - (double)k * dt);
    pt.kdt = (float)((double)k * dt);
    // folded map V*va + vb: keep its fixed point at theta although va is rounded; exact map V - kdt*V + vb: plain k theta dt
    pt.vb = exact_v ? (float)((double)k * (double)theta * dt) : (float)((double)theta * (1.0 - (double)pt.va));
    pt.vs = (float)((double)sigma * std::sqrt(dt) * c0);
    return pt;
}

void fill_fe_launch(const nmch_engine *e, FeLaunch &L, int n_points, int blocks_per_point, int tiles_per_block)
{
    const nmch_params_t &p = e->p;
    const float dt = p.T / (float)p.N;
    const double c0 = 1.1774100225154747;                    // sqrt(2 ln 2)
    L.keys = philox_expand_keys(e->seed);
    L.first_path = e->first_path;
    L.n_local = e->n_local;
    L.draw_offset = e->draw_offset;
    L.dense_q0 = (e->draw_offset >> 1) / 3ull;
    L.dense_r0 = (unsigned int)((e->draw_offset >> 1) % 3ull);
    L.dense_qN = (unsigned int)p.N / 3u;
    L.dense_rN = (unsigned int)p.N % 3u;
    L.N = p.N;
    L.n_points = n_points;
    L.blocks_per_point = blocks_per_point;
    L.tiles_per_block = tiles_per_block;
    L.chunk_points = n_points;
    L.n_chunks = 1;
    L.S0 = p.S_0;
    L.v0 = p.v_0;
    L.K = p.S_0;                                             // at the money, NMCH.cu:7
    L.rdt = p.r * dt;
    L.zr = (float)((double)p.rho * std::sqrt((double)dt) * c0);
    L.zc = (float)(std::sqrt(1.0 - (double)p.rho * (double)p.rho) * std::sqrt((double)dt) * c0);
    L.r = p.r;
    L.rho = p.rho;
    L.dt = dt;
    L.sqrt_dt = sqrtf(dt);                                   // NMCH_FE.cu:152
    L.sqrt_rho = sqrtf(1 - p.rho * p.rho);                   // NMCH_FE.cu:153
    L.pt0 = fold_fe_point(p, p.k, p.theta, p.sigma, p.rng == NMCH_RNG_XORWOW_FAST);
    L.raw0 = RawPoint{p.k, p.theta, p.sigma, 0.0f};
}

int ensure_buffers(nmch_engine *e, size_t n_points, size_t blocks_per_point)
{
    const size_t need_partials = n_points * blocks_per_point;
    if (need_partials > e->partials_cap) {
        engine_dev_free(e, e->d_partials);
        e->d_partials = nullptr;
        e->partials_cap = 0;
        CU_TRY(engine_dev_malloc(e, (void **)&e->d_partials, need_partials * sizeof(double2), "partials"));
        e->partials_cap = need_partials;
    }
    if (n_points > e->tickets_cap) {
        engine_dev_free(e, e->d_tickets);
        e->d_tickets = nullptr;
        e->tickets_cap = 0;
        CU_TRY(engine_dev_malloc(e, (void **)&e->d_tickets, n_points * sizeof(unsigned int), "tickets"));
        // The next launch may be on any stream (the engine's, a group stream, a caller's -- all non-blocking, i.e. not
        // ordered against the legacy default stream the memset runs on): wait for it on the host before anyone launches.
        CU_TRY(cudaMemsetAsync(e->d_tickets, 0, n_points * sizeof(unsigned int), 0));
        CU_TRY(cudaStreamSynchronize(0));
        e->tickets_cap = n_points;
    }
    if (2 * n_points > e->out_cap) {
        if (e->h_out) cudaFreeHost(e->h_out);
        e->h_out = nullptr;
        e->out_cap = 0;
        CU_TRY(cudaHostAlloc((void **)&e->h_out, 2 * n_points * sizeof(double), cudaHostAllocMapped));
        CU_TRY(cudaHostGetDevicePointer((void **)&e->h_out_dev, e->h_out, 0));
        e->out_cap = 2 * n_points;
    }
    return NMCH_OK;
}

int ensure_sv(nmch_engine *e, size_t count)
{
    if (count > e->sv_cap) {
        engine_dev_free(e, e->d_S);
        engine_dev_free(e, e->d_V);
        e->d_S = e->d_V = nullptr;
        e->sv_cap = 0;
        CU_TRY(engine_dev_malloc(e, (void **)&e->d_S, count * sizeof(float), "S_T"));
        CU_TRY(engine_dev_malloc(e, (void **)&e->d_V, count * sizeof(float), "V_T"));
        e->sv_cap = count;
    }
    return NMCH_OK;
}

// The rejection samplers of EM and the moment matching of QE need k, sigma > 0 and finite, non-negative levels.
static int validate_point(int method, float k, float theta, float sigma, float v0)
{
    if (method == NMCH_METHOD_FE) return NMCH_OK;                       // the Euler step is total: any floats go through
    const bool ok = std::isfinite(k) && std::isfinite(theta) && std::isfinite(sigma) && k > 0.0f && sigma > 0.0f &&
                    theta >= 0.0f && v0 >= 0.0f;
    return ok ? NMCH_OK : fail(NMCH_ERR_ARG, "EM / QE need k > 0, sigma > 0, theta >= 0, v_0 >= 0 (finite)");
}

// A sweep on a sequential XORWOW stream walks its points inside the thread.  When the paths alone cannot fill the GPU
// (the reference's own exploration: 5120 paths x 200 points, exploration.cu:24-25) the walk is cut into chunks of
// consecutive points, one grid.y slice each, started by skipping chunk * chunk_points * 2N draws ahead.
int plan_xorwow_chunks(nmch_engine *e, cudaStream_t stream, int n_points, FeLaunch &L, const uint32_t **skip)
{
    L.chunk_points = n_points;
    L.n_chunks = 1;
    *skip = nullptr;
    const unsigned long long sms = (unsigned long long)(e->sm_count > 0 ? e->sm_count : 148);
    if (n_points < 2 || e->n_local >= sms * 1536ull) return NMCH_OK;            // the paths alone fill the GPU
    // Points per chunk: the makespan is (blocks on the busiest SM) x (points a block walks), plus one skip-ahead per
    // chunk (about 4 % of a 1000-step point).  More, shorter chunks balance the SMs better; pick the minimum.
    const unsigned long long bpp = (unsigned long long)L.blocks_per_point;
    double best = 0.0;
    int best_cp = n_points;
    const int cp_max = n_points < 256 ? n_points : 256;
    for (int cp = 1; cp <= cp_max; ++cp) {
        const unsigned long long chunks = ((unsigned long long)n_points + cp - 1) / cp;
        if (chunks > 65535ull) continue;                                       // grid.y
        const unsigned long long per_sm = (bpp * chunks + sms - 1ull) / sms;
        // one path per thread, no ILP: an SM needs about 48 warps (6 blocks of 256) in flight to run at full rate
        const double fill = per_sm >= 6ull ? 1.0 : (double)per_sm / 6.0;
        const double cost = (double)per_sm * ((double)cp + 0.05) / fill;
        if (cp == 1 || cost < best) { best = cost; best_cp = cp; }
    }
    L.chunk_points = best_cp;
    L.n_chunks = (n_points + L.chunk_points - 1) / L.chunk_points;
    if (L.n_chunks < 2) return NMCH_OK;
    const unsigned long long draws = 2ull * (unsigned long long)e->p.N * (unsigned long long)L.chunk_points;
    int digits = 0;
    for (unsigned int c = (unsigned int)(L.n_chunks - 1); c != 0u; c >>= 2) ++digits;
    if (!e->d_xskip || e->xskip_draws != draws || e->xskip_digits < digits) {
        const std::vector<uint32_t> host = xorwow_offset_tables_host(draws, digits);
        engine_dev_free(e, e->d_xskip);
        e->d_xskip = nullptr;
        e->xskip_draws = 0;
        e->xskip_digits = 0;
        CU_TRY(engine_dev_malloc(e, (void **)&e->d_xskip, host.size() * sizeof(uint32_t), "xorwow offset-skip tables"));
        CU_TRY(cudaMemcpyAsync(e->d_xskip, host.data(), host.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        CU_TRY(cudaStreamSynchronize(stream));                 // `host` is a local
        e->xskip_draws = draws;
        e->xskip_digits = digits;
    }
    *skip = e->d_xskip;
    return NMCH_OK;
}

// One launch over n_points parameter points.  k/theta/sigma are HOST arrays (nullptr => the engine's own
// current parameters, n_points == 1).  Raw sums go to d_out (device-accessible, 2*n_points doubles).
int launch_points(nmch_engine *e, cudaStream_t stream, const float *k, const float *theta, const float *sigma,
                  int n_points, double *d_out, float *S_out, float *V_out)
{
    const nmch_params_t &p = e->p;
    const bool exact = (p.rng == NMCH_RNG_PHILOX_COMPAT);        // Philox words, the reference's IEEE arithmetic
    const bool dense = (p.rng == NMCH_RNG_PHILOX_DENSE);         // three steps per Philox block
    const bool native = (p.rng == NMCH_RNG_PHILOX) || exact || dense;
    const bool own = (k == nullptr);
    for (int i = 0; i < n_points; ++i) {
        const int rc = own ? validate_point(p.method, p.k, p.theta, p.sigma, p.v_0)
                           : validate_point(p.method, k[i], theta[i], sigma[i], p.v_0);
        if (rc) return rc;
    }
    if (p.method == NMCH_METHOD_FE) {
        const bool xorwow_fast = (p.rng == NMCH_RNG_XORWOW_FAST);
        int P = 1, threads = 256, tiles_per_block = 1;
        unsigned long long bpp = (e->n_local + 255ull) / 256ull;   // the XORWOW and MRG kernels: one path per thread
        if (native) {
            P = pick_paths_per_thread(e, n_points);
            if (exact && P > 2) P = 2;
            if (dense && P > 4) P = 4;
            threads = dense ? 128 : e->threads;
            const unsigned long long tile = (unsigned long long)P * threads;
            const unsigned long long tiles = (e->n_local + tile - 1) / tile;
            // keep the per-point partial list short when many points share the launch
            if (n_points > 1 && tiles > 256ull) tiles_per_block = (int)((tiles + 255ull) / 256ull);
            bpp = (tiles + tiles_per_block - 1) / tiles_per_block;
        }
        if (bpp == 0 || bpp > 0x7fffffffull) return fail(NMCH_ERR_ARG, "launch grid out of range");
        FeLaunch L;
        fill_fe_launch(e, L, n_points, (int)bpp, tiles_per_block);
        int rc = ensure_buffers(e, n_points, bpp);
        if (rc) return rc;
        // Per-point records: the folded constants for the native step (XORWOW_FAST with the exact map of V), the raw
        // (k, theta, sigma, 0) for the reference's IEEE arithmetic (Philox-compat) and the compat kernels' RawPoint, which
        // has the same layout.
        const void *d_pts = nullptr;
        if (!own) {
            const bool raw = exact || !(native || xorwow_fast);
            std::vector<FePoint> pts(n_points);
            for (int i = 0; i < n_points; ++i)
                pts[i] = raw ? FePoint{k[i], theta[i], sigma[i], 0.0f} : fold_fe_point(p, k[i], theta[i], sigma[i], xorwow_fast);
            rc = upload_records(e, stream, pts.data(), pts.size() * sizeof(FePoint));
            if (rc) return rc;
            d_pts = e->d_points;
        }
        const FePoint *fe_pts = static_cast<const FePoint *>(d_pts);
        const RawPoint *raw_pts = static_cast<const RawPoint *>(d_pts);
        ReduceBuffers rb{e->d_partials, e->d_tickets, d_out};
        if (dense) {
            CU_TRY(launch_fe_dense(L, p.floor, P, fe_pts, rb, S_out, V_out, stream, &e->kinfo));
        } else if (native) {
            CU_TRY(launch_fe_philox(L, p.floor, P, threads, exact, fe_pts, rb, S_out, V_out, stream, &e->kinfo));
        } else if (p.rng == NMCH_RNG_MRG32K3A_COMPAT) {
            CU_TRY(launch_fe_compat_mrg(L, p.floor, raw_pts, e->curand_states, rb, S_out, V_out, stream, &e->kinfo));
        } else {
            const uint32_t *skip = nullptr;
            rc = plan_xorwow_chunks(e, stream, n_points, L, &skip);
            if (rc) return rc;
            if (xorwow_fast)
                CU_TRY(launch_fe_xorwow_fast(L, p.floor, fe_pts, e->xs, skip, rb, S_out, V_out, stream, &e->kinfo));
            else
                CU_TRY(launch_fe_compat(L, p.floor, raw_pts, e->xs, skip, rb, S_out, V_out, stream, &e->kinfo));
        }
        e->draw_offset += 2ull * (unsigned long long)p.N * (unsigned long long)n_points;
    } else if (p.method == NMCH_METHOD_EM) {
        int rc = em_launch_points(e, stream, k, theta, sigma, n_points, d_out, S_out, V_out);
        if (rc) return rc;
    } else {
        int rc = qe_launch_points(e, stream, k, theta, sigma, n_points, d_out, S_out, V_out);
        if (rc) return rc;
    }
    e->launches += 1;
    return NMCH_OK;
}

int check_ready(const nmch_engine *e)
{
    if (!e) return fail(NMCH_ERR_ARG, "null engine");
    if (!e->inited) return fail(NMCH_ERR_STATE, "engine not initialised (call nmch_engine_init first, or it was finalized)");
    return NMCH_OK;
}

void fill_moments(const nmch_engine *e, const double *src, int n_points, float ms, nmch_moments_t *out)
{
    for (int i = 0; i < n_points; ++i) {
        out[i].sum_payoff = src[2 * i];
        out[i].sum_payoff_sq = src[2 * i + 1];
        out[i].n_paths = e->n_local;
        out[i].exec_ms = ms;
    }
}

// The blocking entry points: the engine's device current, a host-visible result buffer of n_slots reduction slots (2 doubles
// each), launch(stream, d_out) timed on the engine's stream between ev0 and ev1, then unpack(h_out, exec_ms) and the guard
// sweep of the checked build.
template <class Launch, class Unpack>
int blocking_call(nmch_engine *e, size_t n_slots, Launch launch, Unpack unpack)
{
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    int rc = ensure_buffers(e, n_slots, 1);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(e->ev0, e->stream));
    rc = launch(e->stream, e->h_out_dev);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(e->ev1, e->stream));
    CU_TRY(cudaEventSynchronize(e->ev1));
    float ms = 0.0f;
    CU_TRY(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
    unpack(static_cast<const double *>(e->h_out), ms);
    return engine_check_guards(e);
}

int check_strike_call(const nmch_engine *e, const float *strikes, int n_strikes, const void *out)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!strikes || !out || n_strikes <= 0 || n_strikes > NMCH_MAX_STRIKES) return fail(NMCH_ERR_ARG, "bad strike arguments");
    return NMCH_OK;
}

// The derivatives of the folded step constants in kappa, theta, sigma and rho (fe_step.cuh), in double, rounded once.
TangentFold fold_tangent(const nmch_params_t &p)
{
    const double dt = (double)(p.T / (float)p.N);                 // as fold_fe_point forms it
    const double sdc = std::sqrt(dt) * 1.1774100225154747;         // sqrt(dt) sqrt(2 ln 2)
    const double rho = (double)p.rho;
    TangentFold tf;
    tf.dva_k = (float)(-dt);
    tf.dvb_k = (float)((double)p.theta * dt);
    tf.dvb_t = (float)((double)p.k * dt);
    tf.dvs_s = (float)sdc;
    tf.dzr_r = (float)sdc;
    tf.dzc_r = (float)(-rho / std::sqrt(1.0 - rho * rho) * sdc);
    return tf;
}

// One pass of the strike family on `stream`, shared by the blocking and the stream forms.  A path pass leaves S_T (and,
// for n_dirs >= 1, dS_T/dp in n_dirs directions) on the device; strike_fold_kernel<n_dirs> then folds strike_doubles(n_dirs)
// raw sums per strike into d_out.  n_dirs = 0 (compute_strikes) takes every method and stream; the tangent (1:
// compute_greeks, 5: compute_sensitivities) is carried by the native FE step only.  Those refusals come first: a refused
// call leaves the engine as it was.
int strike_pass(nmch_engine *e, cudaStream_t stream, const float *strikes, int n_strikes, int n_dirs, double *d_out)
{
    const nmch_params_t &p = e->p;
    if (n_dirs > 0 && (p.method != NMCH_METHOD_FE || p.rng != NMCH_RNG_PHILOX)) {
        char buf[160];
        std::snprintf(buf, sizeof buf, "%s: the pathwise tangent is carried by the native FE step (method FE, rng PHILOX)",
                      n_dirs == 1 ? "compute_greeks" : "compute_sensitivities");
        return fail(NMCH_ERR_ARG, buf);
    }
    if (n_dirs > 1 && !(std::fabs(p.rho) < 1.0f))      // also refuses a NaN rho
        return fail(NMCH_ERR_ARG, "compute_sensitivities: needs |rho| < 1 (d sqrt(1 - rho^2) / d rho is infinite at |rho| = 1)");
    int rc = ensure_sv(e, (size_t)e->n_local);
    if (rc) return rc;
    // reduction slots: 0 = the path kernel's own K = S_0 moments, then 2 + n_dirs per strike (payoff, delta, one per
    // direction)
    const size_t slots = 1 + (size_t)strike_doubles(n_dirs) / 2 * (size_t)n_strikes;
    rc = ensure_buffers(e, slots, (size_t)strike_blocks_per_slot());
    if (rc) return rc;
    rc = upload_records(e, stream, strikes, (size_t)n_strikes * sizeof(float));
    if (rc) return rc;
    if (n_dirs == 0) {
        rc = launch_points(e, stream, nullptr, nullptr, nullptr, 1, e->h_out_dev, e->d_S, e->d_V);
        if (rc) return rc;
    } else {
        const size_t t_need = n_dirs == 1 ? (size_t)e->n_local : (size_t)n_dirs * (size_t)tangent_stride(e->n_local);
        if (t_need > e->t_cap) {
            engine_dev_free(e, e->d_T);
            e->d_T = nullptr;
            e->t_cap = 0;
            CU_TRY(engine_dev_malloc(e, (void **)&e->d_T, t_need * sizeof(float), "dS_T/dp"));
            e->t_cap = t_need;
        }
        const unsigned long long tile = (unsigned long long)tangent_tile_paths(n_dirs);
        const unsigned long long bpp = (e->n_local + tile - 1ull) / tile;
        if (bpp == 0 || bpp > 0x7fffffffull) return fail(NMCH_ERR_ARG, "launch grid out of range");
        rc = ensure_buffers(e, 1, (size_t)bpp);
        if (rc) return rc;
        FeLaunch L;
        fill_fe_launch(e, L, 1, (int)bpp, 1);
        ReduceBuffers rb0{e->d_partials, e->d_tickets, e->h_out_dev};
        CU_TRY(launch_fe_tangent(L, p.floor, n_dirs, fold_tangent(p), rb0, e->d_S, e->d_V, e->d_T, stream, &e->kinfo));
        e->draw_offset += 2ull * (unsigned long long)p.N;          // the stream advances like one compute()
        e->launches += 1;
    }
    // same stream: the path kernel (and its use of the partial buffer) is complete before the fold starts
    ReduceBuffers rb{e->d_partials, e->d_tickets + 1, d_out};
    CU_TRY(launch_strike_fold(e->d_S, e->d_T, n_dirs, e->n_local, static_cast<const float *>(e->d_points), n_strikes, p.S_0,
                              rb, stream));
    e->launches += 1;
    return NMCH_OK;
}

// The blocking form of the strike family: n_dirs = 0, 1 or NMCH_SENS_COUNT, as the struct T carries.
template <class T>
int strike_call(nmch_engine *e, const float *strikes, int n_strikes, int n_dirs, T *out)
{
    const int rc = check_strike_call(e, strikes, n_strikes, out);
    if (rc) return rc;
    const size_t per = (size_t)strike_doubles(n_dirs);
    return blocking_call(
        e, 1 + per / 2 * (size_t)n_strikes,                     // slot 0: the path kernel's own K = S_0 moments
        [&](cudaStream_t s, double *d_out) { return strike_pass(e, s, strikes, n_strikes, n_dirs, d_out + 2); },
        [&](const double *h, float ms) {
            for (int j = 0; j < n_strikes; ++j) strike_unpack(h + 2 + per * (size_t)j, strikes[j], e->n_local, ms, &out[j]);
        });
}

}  // namespace

// em_kernels.cu and qe_kernels.cu need these engine internals
namespace nmchb {
int engine_ensure_buffers(nmch_engine *e, size_t n_points, size_t blocks_per_point)
{
    return ensure_buffers(e, n_points, blocks_per_point);
}

int upload_records(nmch_engine *e, cudaStream_t stream, const void *host, size_t bytes)
{
    if (bytes > e->points_cap) {
        engine_dev_free(e, e->d_points);
        e->d_points = nullptr;
        e->points_cap = 0;
        CU_TRY(engine_dev_malloc(e, &e->d_points, bytes, "points"));
        e->points_cap = bytes;
    }
    CU_TRY(cudaMemcpyAsync(e->d_points, host, bytes, cudaMemcpyHostToDevice, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    return NMCH_OK;
}

int engine_strike_async(nmch_engine *e, void *cuda_stream, const float *strikes, int n_strikes, int n_dirs, double *d_out)
{
    const int rc = check_strike_call(e, strikes, n_strikes, d_out);
    if (rc) return rc;
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    return strike_pass(e, static_cast<cudaStream_t>(cuda_stream), strikes, n_strikes, n_dirs, d_out);
}
}  // namespace nmchb

extern "C" {

int nmch_engine_create(const nmch_params_t *params, nmch_engine_t **out)
{
    if (!params || !out) return fail(NMCH_ERR_ARG, "null argument");
    const nmch_params_t &p = *params;
    if (p.N <= 0) return fail(NMCH_ERR_ARG, "N must be positive");
    if (p.method != NMCH_METHOD_FE && p.method != NMCH_METHOD_EM && p.method != NMCH_METHOD_QE)
        return fail(NMCH_ERR_ARG, "unknown method");
    if (p.method == NMCH_METHOD_QE && p.rng != NMCH_RNG_PHILOX)
        return fail(NMCH_ERR_ARG, "the QE scheme has no reference counterpart to be draw-compatible with: use rng = PHILOX");
    if (p.floor != NMCH_FLOOR_ABS && p.floor != NMCH_FLOOR_PLUS) return fail(NMCH_ERR_ARG, "unknown floor");
    if (p.rng < NMCH_RNG_PHILOX || p.rng > NMCH_RNG_XORWOW_FAST) return fail(NMCH_ERR_ARG, "unknown rng mode");
    if (p.rng == NMCH_RNG_PHILOX_DENSE && p.method != NMCH_METHOD_FE)
        return fail(NMCH_ERR_ARG, "PHILOX_DENSE is an FE stream mode");
    if (p.rng == NMCH_RNG_XORWOW_FAST && p.method != NMCH_METHOD_FE)
        return fail(NMCH_ERR_ARG, "XORWOW_FAST is an FE stream mode (EM on the XORWOW tag: XORWOW_COMPAT)");
    unsigned long long n = p.n_paths;
    if (n == 0) {
        if (p.NTPB <= 0 || p.NB <= 0) return fail(NMCH_ERR_ARG, "NTPB and NB must be positive");
        n = (unsigned long long)p.NTPB * (unsigned long long)p.NB;
    }
    if (p.first_path > n) return fail(NMCH_ERR_ARG, "first_path beyond n_paths");
    unsigned long long n_local = p.n_local ? p.n_local : n - p.first_path;
    if (n_local == 0 || p.first_path + n_local > n) return fail(NMCH_ERR_ARG, "empty or out-of-range shard");
    if ((p.rng == NMCH_RNG_PHILOX || p.rng == NMCH_RNG_PHILOX_DENSE ||
         (p.rng == NMCH_RNG_PHILOX_COMPAT && p.method == NMCH_METHOD_FE)) &&
        !is_multiple_of(p.first_path, kMaxTilePaths))
        return fail(NMCH_ERR_ARG, "the native Philox modes (and Philox-compatible FE) need first_path to be a multiple of 4096");
    if (p.paths_per_thread != 0 && p.paths_per_thread != 1 && p.paths_per_thread != 2 && p.paths_per_thread != 4 &&
        p.paths_per_thread != 8)
        return fail(NMCH_ERR_ARG, "paths_per_thread must be 0 (auto), 1, 2, 4 or 8");
    if (p.block_threads != 0 && p.block_threads != 128 && p.block_threads != 256)
        return fail(NMCH_ERR_ARG, "block_threads must be 0 (auto), 128 or 256");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(NMCH_ERR_CUDA, "no CUDA device: this engine has no CPU fallback");
    int dev = p.device;
    if (dev < 0) CU_TRY(cudaGetDevice(&dev));
    if (dev >= ndev) return fail(NMCH_ERR_ARG, "device ordinal out of range");
    nmch_engine *e = new (std::nothrow) nmch_engine();
    if (!e) return fail(NMCH_ERR_ARG, "out of host memory");
    e->p = p;
    e->device = dev;
    e->n_paths = n;
    e->first_path = p.first_path;
    e->n_local = n_local;
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) e->sm_count = prop.multiProcessorCount;
    *out = e;
    return NMCH_OK;
}

static int engine_init_impl(nmch_engine_t *e, unsigned long long seed);

int nmch_engine_init(nmch_engine_t *e, unsigned long long seed)
{
    if (!e) return fail(NMCH_ERR_ARG, "null engine");
    if (e->inited) return fail(NMCH_ERR_STATE, "engine already initialised");
    const int rc = engine_init_impl(e, seed);
    if (rc != NMCH_OK) {
        const std::string why = nmch_last_error();      // keep the cause: the clean-up below may overwrite it
        nmch_engine_finalize(e);
        engine_fail(rc, why.c_str());
    }
    return rc;
}

static int engine_init_impl(nmch_engine_t *e, unsigned long long seed)
{
    NvtxRange range("nmch_engine_init");
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    CU_TRY(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreate(&e->ev0));
    CU_TRY(cudaEventCreate(&e->ev1));
    CU_TRY(cudaEventRecord(e->ev0, e->stream));
    e->seed = seed;
    e->draw_offset = 0;
    e->em_calls = 0;
    e->threads = e->p.block_threads ? e->p.block_threads : 256;     // 256: 24.61 vs 24.69 ms at configs[1] (profiles/r02_fe_ab.txt)
    if (e->p.rng == NMCH_RNG_XORWOW_COMPAT || e->p.rng == NMCH_RNG_XORWOW_FAST) {
        const size_t n = (size_t)e->n_local;
        CU_TRY(xorwow_tables_create(&e->xtab));
        uint32_t *base = nullptr;
        CU_TRY(engine_dev_malloc(e, (void **)&base, 6 * n * sizeof(uint32_t), "xorwow states"));
        e->xs.d = base; e->xs.v0 = base + n; e->xs.v1 = base + 2 * n;
        e->xs.v2 = base + 3 * n; e->xs.v3 = base + 4 * n; e->xs.v4 = base + 5 * n;
        if (e->p.method == NMCH_METHOD_EM) {
            CU_TRY(engine_dev_malloc(e, (void **)&e->xs.bm_flag, n * sizeof(int), "xorwow bm_flag"));
            CU_TRY(engine_dev_malloc(e, (void **)&e->xs.bm_extra, n * sizeof(float), "xorwow bm_extra"));
            CU_TRY(engine_dev_malloc(e, (void **)&e->xs.bm_flag_d, n * sizeof(int), "xorwow bm_flag_d"));
            CU_TRY(engine_dev_malloc(e, (void **)&e->xs.bm_extra_d, n * sizeof(double), "xorwow bm_extra_d"));
        }
        CU_TRY(launch_xorwow_init(e->xtab, seed, e->first_path, e->n_local, e->xs, e->stream));
        e->launches += 1;
    } else if (e->p.rng == NMCH_RNG_PHILOX_COMPAT && e->p.method == NMCH_METHOD_EM) {
        int rc = em_philox_compat_init(e);
        if (rc) return rc;
    } else if (e->p.rng == NMCH_RNG_MRG32K3A_COMPAT) {
        int rc = mrg_compat_init(e);
        if (rc) return rc;
    }
    int rc = ensure_buffers(e, 1, 1);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(e->ev1, e->stream));
    CU_TRY(cudaEventSynchronize(e->ev1));
    CU_TRY(cudaEventElapsedTime(&e->init_ms, e->ev0, e->ev1));
    e->inited = true;
    return engine_check_guards(e);
}

int nmch_engine_set_params(nmch_engine_t *e, float k, float theta, float sigma)
{
    if (!e) return fail(NMCH_ERR_ARG, "null engine");
    e->p.k = k;
    e->p.theta = theta;
    e->p.sigma = sigma;
    return NMCH_OK;
}

int nmch_engine_seek(nmch_engine_t *e, unsigned long long words)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (e->p.method != NMCH_METHOD_FE || (e->p.rng != NMCH_RNG_PHILOX && e->p.rng != NMCH_RNG_PHILOX_COMPAT &&
                                          e->p.rng != NMCH_RNG_PHILOX_DENSE))
        return fail(NMCH_ERR_ARG, "seek is available for FE in the Philox stream modes only");
    if (words & 1ull) return fail(NMCH_ERR_ARG, "seek position must be an even number of 32-bit draws");
    e->draw_offset = words;
    return NMCH_OK;
}

int nmch_engine_compute(nmch_engine_t *e, nmch_moments_t *out)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!out) return fail(NMCH_ERR_ARG, "null output");
    NvtxRange range("nmch_engine_compute");
    return blocking_call(
        e, 1,
        [&](cudaStream_t s, double *d_out) { return launch_points(e, s, nullptr, nullptr, nullptr, 1, d_out, nullptr, nullptr); },
        [&](const double *h, float ms) { fill_moments(e, h, 1, ms, out); });
}

int nmch_engine_compute_async(nmch_engine_t *e, void *cuda_stream, double *d_moments)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!d_moments) return fail(NMCH_ERR_ARG, "null device output");
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);     // NULL = the CUDA default stream, as in the runtime API
    return launch_points(e, s, nullptr, nullptr, nullptr, 1, d_moments, nullptr, nullptr);
}

int nmch_engine_explore(nmch_engine_t *e, const float *k, const float *theta, const float *sigma, int n_points,
                        nmch_moments_t *out)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!k || !theta || !sigma || !out || n_points <= 0) return fail(NMCH_ERR_ARG, "bad exploration arguments");
    if (n_points > 65535) return fail(NMCH_ERR_ARG, "at most 65535 points per launch");
    NvtxRange range("nmch_engine_explore");
    return blocking_call(
        e, (size_t)n_points,
        [&](cudaStream_t s, double *d_out) { return launch_points(e, s, k, theta, sigma, n_points, d_out, nullptr, nullptr); },
        [&](const double *h, float ms) { fill_moments(e, h, n_points, ms, out); });
}

int nmch_engine_explore_async(nmch_engine_t *e, void *cuda_stream, const float *k, const float *theta,
                              const float *sigma, int n_points, double *d_moments)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!k || !theta || !sigma || !d_moments || n_points <= 0) return fail(NMCH_ERR_ARG, "bad exploration arguments");
    if (n_points > 65535) return fail(NMCH_ERR_ARG, "at most 65535 points per launch");
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);     // NULL = the CUDA default stream, as in the runtime API
    return launch_points(e, s, k, theta, sigma, n_points, d_moments, nullptr, nullptr);
}

int nmch_engine_compute_paths(nmch_engine_t *e, float *S_out, float *V_out, unsigned long long count,
                              nmch_moments_t *out)
{
    int rc = check_ready(e);
    if (rc) return rc;
    if (!S_out || !V_out || !out) return fail(NMCH_ERR_ARG, "null output");
    if (count > e->n_local) return fail(NMCH_ERR_ARG, "count exceeds the local path count");
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    rc = ensure_sv(e, (size_t)e->n_local);
    if (rc) return rc;
    rc = ensure_buffers(e, 1, 1);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(e->ev0, e->stream));
    rc = launch_points(e, e->stream, nullptr, nullptr, nullptr, 1, e->h_out_dev, e->d_S, e->d_V);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(e->ev1, e->stream));
    CU_TRY(cudaMemcpyAsync(S_out, e->d_S, count * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaMemcpyAsync(V_out, e->d_V, count * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream));
    float ms = 0.0f;
    CU_TRY(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
    fill_moments(e, e->h_out, 1, ms, out);
    return engine_check_guards(e);
}

int nmch_engine_compute_strikes(nmch_engine_t *e, const float *strikes, int n_strikes, nmch_strike_moments_t *out)
{
    return strike_call(e, strikes, n_strikes, 0, out);
}

int nmch_engine_compute_strikes_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                      double *d_moments)
{
    return engine_strike_async(e, cuda_stream, strikes, n_strikes, 0, d_moments);
}

// ---- strike vector with pathwise delta and vega / sensitivities (FE, native Philox stream) ---------------------------
int nmch_engine_compute_greeks(nmch_engine_t *e, const float *strikes, int n_strikes, nmch_greek_moments_t *out)
{
    return strike_call(e, strikes, n_strikes, 1, out);
}

int nmch_engine_compute_greeks_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                     double *d_moments)
{
    return engine_strike_async(e, cuda_stream, strikes, n_strikes, 1, d_moments);
}

int nmch_engine_compute_sensitivities(nmch_engine_t *e, const float *strikes, int n_strikes,
                                      nmch_sensitivity_moments_t *out)
{
    return strike_call(e, strikes, n_strikes, NMCH_SENS_COUNT, out);
}

int nmch_engine_compute_sensitivities_async(nmch_engine_t *e, void *cuda_stream, const float *strikes, int n_strikes,
                                            double *d_moments)
{
    return engine_strike_async(e, cuda_stream, strikes, n_strikes, NMCH_SENS_COUNT, d_moments);
}

int nmch_engine_finalize(nmch_engine_t *e)
{
    if (!e) return fail(NMCH_ERR_ARG, "null engine");
    // Idempotent (the reference double-frees), and also the clean-up path of an init() that failed half way:
    // every resource is released if present, whatever the lifecycle flag says.
    DeviceGuard guard(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    engine_dev_free(e, e->d_partials);
    engine_dev_free(e, e->d_tickets);
    if (e->h_out) cudaFreeHost(e->h_out);
    engine_dev_free(e, e->d_points);
    engine_dev_free(e, e->d_S);
    engine_dev_free(e, e->d_V);
    engine_dev_free(e, e->d_T);
    engine_dev_free(e, e->xs.d);
    engine_dev_free(e, e->xs.bm_flag);
    engine_dev_free(e, e->xs.bm_extra);
    engine_dev_free(e, e->xs.bm_flag_d);
    engine_dev_free(e, e->xs.bm_extra_d);
    engine_dev_free(e, e->d_xskip);
    e->d_xskip = nullptr;
    e->xskip_draws = 0;
    e->xskip_digits = 0;
    em_release(e);
    xorwow_tables_destroy(e->xtab);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->stream) cudaStreamDestroy(e->stream);
    e->d_partials = nullptr; e->partials_cap = 0;
    e->d_tickets = nullptr; e->tickets_cap = 0;
    e->h_out = e->h_out_dev = nullptr; e->out_cap = 0;
    e->d_points = nullptr; e->points_cap = 0;
    e->d_S = e->d_V = nullptr; e->sv_cap = 0;
    e->d_T = nullptr; e->t_cap = 0;
    e->xs = XorwowState{};
    e->xtab = nullptr;
    e->ev0 = e->ev1 = nullptr;
    e->stream = nullptr;
    e->inited = false;
    return NMCH_OK;
}

void nmch_engine_destroy(nmch_engine_t *e)
{
    if (!e) return;
    nmch_engine_finalize(e);
    delete e;
}

int nmch_engine_check(nmch_engine_t *e)
{
    int rc = check_ready(e);
    if (rc) return rc;
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    CU_TRY(cudaDeviceSynchronize());               // *_async work may sit on caller streams: a device assert surfaces here
    return engine_check_guards(e);
}

int nmch_checked_selftest(nmch_engine_t *e)
{
#ifdef NMCHB_CHECKS
    // Proves the guard sweep sees an overrun: write one word past the ticket array (what an off-by-one point index
    // would do), expect the sweep to fail naming "tickets", then repair the band.
    int rc = check_ready(e);
    if (rc) return rc;
    DeviceGuard guard(e->device);
    if (!guard.ok) return fail(NMCH_ERR_CUDA, "cudaSetDevice failed");
    const unsigned int junk = 0xdeadbeefu;
    unsigned char *past = reinterpret_cast<unsigned char *>(e->d_tickets) + e->tickets_cap * sizeof(unsigned int);
    CU_TRY(cudaMemcpy(past, &junk, sizeof junk, cudaMemcpyHostToDevice));
    const int seen = engine_check_guards(e);
    CU_TRY(cudaMemset(past, kGuardByte, sizeof junk));
    if (seen == NMCH_OK) return fail(NMCH_ERR_STATE, "checked build: the guard sweep missed a deliberate overrun");
    return engine_check_guards(e);                 // clean again after the repair
#else
    (void)e;
    return fail(NMCH_ERR_STATE, "not a checked build (load libnmch_b200_checked.so)");
#endif
}

int nmch_checked_build(void)
{
#ifdef NMCHB_CHECKS
    return 1;
#else
    return 0;
#endif
}

float nmch_engine_init_ms(const nmch_engine_t *e) { return e ? e->init_ms : 0.0f; }

int nmch_engine_launch_info(const nmch_engine_t *e, nmch_launch_info_t *out)
{
    if (!e || !out) return fail(NMCH_ERR_ARG, "null argument");
    out->grid_x = e->kinfo.grid_x;
    out->grid_y = e->kinfo.grid_y;
    out->block_threads = e->kinfo.block_threads;
    out->paths_per_thread = e->kinfo.paths_per_thread;
    out->regs_per_thread = e->kinfo.regs_per_thread;
    out->sm_count = e->sm_count;
    out->kernel_param_bytes = e->kinfo.param_bytes;
    out->kernel_launches = e->launches;
    return NMCH_OK;
}

const char *nmch_status_string(int status)
{
    switch (status) {
    case NMCH_OK: return "ok";
    case NMCH_ERR_ARG: return "invalid argument";
    case NMCH_ERR_CUDA: return "CUDA error";
    case NMCH_ERR_STATE: return "invalid engine state";
    case NMCH_ERR_NCCL: return "NCCL error";
    default: return "unknown status";
    }
}

const char *nmch_last_error(void) { return g_last_error.c_str(); }

int nmch_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char *nmch_version(void) { return "nmch_b200 0.1 (sm_100a)"; }

}  // extern "C"
