// group.cu -- single-process multi-GPU group over the engine C ABI: shard paths, one NCCL allreduce.
//
// NCCL is bound at run time (dlopen "libnccl.so.2") so the library has no link-time NCCL dependency and, in a
// process that already carries an NCCL (PyTorch), shares that copy.  A group of one device never touches NCCL.
#include <dlfcn.h>
#include <nccl.h>

#include <cstdio>
#include <string>
#include <vector>

#include "engine_internal.cuh"

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load()
    {
        if (handle) return true;
        handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!handle) handle = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!handle) return false;
        CommInitAll = reinterpret_cast<decltype(CommInitAll)>(dlsym(handle, "ncclCommInitAll"));
        CommDestroy = reinterpret_cast<decltype(CommDestroy)>(dlsym(handle, "ncclCommDestroy"));
        AllReduce = reinterpret_cast<decltype(AllReduce)>(dlsym(handle, "ncclAllReduce"));
        GroupStart = reinterpret_cast<decltype(GroupStart)>(dlsym(handle, "ncclGroupStart"));
        GroupEnd = reinterpret_cast<decltype(GroupEnd)>(dlsym(handle, "ncclGroupEnd"));
        GetErrorString = reinterpret_cast<decltype(GetErrorString)>(dlsym(handle, "ncclGetErrorString"));
        return CommInitAll && CommDestroy && AllReduce && GroupStart && GroupEnd && GetErrorString;
    }
};

NcclApi g_nccl;

}  // namespace

struct nmch_group {
    int n = 0;
    unsigned long long n_paths = 0;
    std::vector<nmch_engine_t *> eng;
    std::vector<int> dev;
    std::vector<cudaStream_t> stream;
    std::vector<cudaEvent_t> ev0, ev1;
    std::vector<double *> d_mom;
    std::vector<ncclComm_t> comm;
    double *h_mom = nullptr;
    size_t mom_cap = 0;
    bool inited = false;
    float init_ms = 0.0f;
};

namespace {

using nmchb::engine_fail;

// restores the caller's current device on every exit path of a group call
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
    ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

#define GROUP_CU_TRY(call)                                                       \
    do {                                                                         \
        cudaError_t err__ = (call);                                              \
        if (err__ != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, #call, err__); \
    } while (0)

int nccl_fail(const char *what, ncclResult_t r)
{
    char buf[256];
    std::snprintf(buf, sizeof buf, "%s: %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "nccl error");
    return engine_fail(NMCH_ERR_NCCL, buf);
}

int ensure_moments(nmch_group *g, size_t n_doubles)
{
    if (n_doubles <= g->mom_cap) return NMCH_OK;
    g->mom_cap = 0;
    for (int i = 0; i < g->n; ++i) {
        GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
        if (g->d_mom[i]) cudaFree(g->d_mom[i]);
        g->d_mom[i] = nullptr;
        cudaError_t err = cudaMalloc(&g->d_mom[i], n_doubles * sizeof(double));
        if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "cudaMalloc(group moments)", err);
    }
    if (g->h_mom) cudaFreeHost(g->h_mom);
    g->h_mom = nullptr;
    cudaError_t err = cudaMallocHost(&g->h_mom, n_doubles * sizeof(double));
    if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "cudaMallocHost(group moments)", err);
    g->mom_cap = n_doubles;
    return NMCH_OK;
}

// launch_on_device(i) enqueues device i's pass, n_doubles raw sums into g->d_mom[i] on g->stream[i]; then one grouped
// allreduce, the result of device 0 read back into g->h_mom; *ms = the slowest device's time
template <class Launch>
int group_run(nmch_group *g, size_t n_doubles, Launch launch_on_device, float *ms)
{
    int rc = ensure_moments(g, n_doubles);
    if (rc) return rc;
    for (int i = 0; i < g->n; ++i) {
        GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
        GROUP_CU_TRY(cudaEventRecord(g->ev0[i], g->stream[i]));
        rc = launch_on_device(i);
        if (rc) return rc;
    }
    if (g->n > 1) {
        ncclResult_t r = g_nccl.GroupStart();
        if (r != ncclSuccess) return nccl_fail("ncclGroupStart", r);
        for (int i = 0; i < g->n; ++i) {
            r = g_nccl.AllReduce(g->d_mom[i], g->d_mom[i], n_doubles, ncclDouble, ncclSum, g->comm[i], g->stream[i]);
            if (r != ncclSuccess) return nccl_fail("ncclAllReduce", r);
        }
        r = g_nccl.GroupEnd();
        if (r != ncclSuccess) return nccl_fail("ncclGroupEnd", r);
    }
    *ms = 0.0f;
    for (int i = 0; i < g->n; ++i) {
        GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
        if (i == 0)
            GROUP_CU_TRY(cudaMemcpyAsync(g->h_mom, g->d_mom[0], n_doubles * sizeof(double), cudaMemcpyDeviceToHost, g->stream[0]));
        GROUP_CU_TRY(cudaEventRecord(g->ev1[i], g->stream[i]));
    }
    for (int i = 0; i < g->n; ++i) {
        GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
        cudaError_t err = cudaEventSynchronize(g->ev1[i]);
        if (err != cudaSuccess) return engine_fail(NMCH_ERR_CUDA, "group pass", err);
        float t = 0.0f;
        GROUP_CU_TRY(cudaEventElapsedTime(&t, g->ev0[i], g->ev1[i]));
        if (t > *ms) *ms = t;
    }
    return NMCH_OK;
}

// compute (k == nullptr) or explore over n_points on every device
int run_points(nmch_group *g, const float *k, const float *theta, const float *sigma, int n_points, nmch_moments_t *out)
{
    if (!g || !g->inited) return engine_fail(NMCH_ERR_STATE, "group not initialised");
    float ms = 0.0f;
    const int rc = group_run(g, 2 * (size_t)n_points, [&](int i) {
        return k ? nmch_engine_explore_async(g->eng[i], g->stream[i], k, theta, sigma, n_points, g->d_mom[i])
                 : nmch_engine_compute_async(g->eng[i], g->stream[i], g->d_mom[i]);
    }, &ms);
    if (rc) return rc;
    for (int p = 0; p < n_points; ++p) {
        out[p].sum_payoff = g->h_mom[2 * p];
        out[p].sum_payoff_sq = g->h_mom[2 * p + 1];
        out[p].n_paths = g->n_paths;
        out[p].exec_ms = ms;
    }
    return NMCH_OK;
}

// the strike family (n_dirs = 0, 1 or NMCH_SENS_COUNT, as the struct T carries) on every device
template <class T>
int group_strikes(nmch_group *g, const float *strikes, int n_strikes, int n_dirs, T *out)
{
    if (!out) return engine_fail(NMCH_ERR_ARG, "bad strike arguments");
    if (!g || !g->inited) return engine_fail(NMCH_ERR_STATE, "group not initialised");
    if (!strikes || n_strikes <= 0 || n_strikes > NMCH_MAX_STRIKES) return engine_fail(NMCH_ERR_ARG, "bad strike arguments");
    DeviceRestore restore;
    const size_t per = (size_t)nmchb::strike_doubles(n_dirs);
    float ms = 0.0f;
    const int rc = group_run(g, per * (size_t)n_strikes, [&](int i) {
        return nmchb::engine_strike_async(g->eng[i], g->stream[i], strikes, n_strikes, n_dirs, g->d_mom[i]);
    }, &ms);
    if (rc) return rc;
    for (int j = 0; j < n_strikes; ++j) nmchb::strike_unpack(g->h_mom + per * (size_t)j, strikes[j], g->n_paths, ms, &out[j]);
    return NMCH_OK;
}

}  // namespace

extern "C" {

int nmch_group_create(const nmch_params_t *params, int n_gpus, nmch_group_t **out)
{
    if (!params || !out || n_gpus < 1) return engine_fail(NMCH_ERR_ARG, "bad group arguments");
    if (nmch_device_count() == 0) return engine_fail(NMCH_ERR_CUDA, "no CUDA device: this engine has no CPU fallback");
    if (n_gpus > nmch_device_count()) return engine_fail(NMCH_ERR_ARG, "more GPUs requested than visible");
    unsigned long long n = params->n_paths ? params->n_paths : (unsigned long long)params->NTPB * (unsigned long long)params->NB;
    if (n == 0) return engine_fail(NMCH_ERR_ARG, "no paths");
    // shards are multiples of 4096 paths (native-mode tile alignment); the last device takes the remainder
    unsigned long long per = n / (unsigned long long)n_gpus;
    if (n_gpus > 1) per = (per / 4096ull) * 4096ull;
    if (n_gpus > 1 && per == 0) return engine_fail(NMCH_ERR_ARG, "too few paths to shard (need >= 4096 per GPU)");
    auto *g = new nmch_group();
    g->n = n_gpus;
    g->n_paths = n;
    for (int i = 0; i < n_gpus; ++i) {
        nmch_params_t p = *params;
        p.n_paths = n;
        p.device = i;
        p.first_path = per * (unsigned long long)i;
        p.n_local = (i == n_gpus - 1) ? n - p.first_path : per;
        nmch_engine_t *e = nullptr;
        int rc = nmch_engine_create(&p, &e);
        if (rc) {
            nmch_group_destroy(g);
            return rc;
        }
        g->eng.push_back(e);
        g->dev.push_back(i);
    }
    g->stream.assign(n_gpus, nullptr);
    g->ev0.assign(n_gpus, nullptr);
    g->ev1.assign(n_gpus, nullptr);
    g->d_mom.assign(n_gpus, nullptr);
    *out = g;
    return NMCH_OK;
}

static int group_init_impl(nmch_group_t *g, unsigned long long seed)
{
    float ms = 0.0f;
    for (int i = 0; i < g->n; ++i) {
        GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
        GROUP_CU_TRY(cudaStreamCreateWithFlags(&g->stream[i], cudaStreamNonBlocking));
        GROUP_CU_TRY(cudaEventCreate(&g->ev0[i]));
        GROUP_CU_TRY(cudaEventCreate(&g->ev1[i]));
        int rc = nmch_engine_init(g->eng[i], seed);
        if (rc) return rc;
        const float t = nmch_engine_init_ms(g->eng[i]);
        if (t > ms) ms = t;
    }
    if (g->n > 1) {
        if (!g_nccl.load()) return engine_fail(NMCH_ERR_NCCL, "libnccl.so.2 not found: multi-GPU groups need NCCL");
        g->comm.assign(g->n, nullptr);
        ncclResult_t r = g_nccl.CommInitAll(g->comm.data(), g->n, g->dev.data());
        if (r != ncclSuccess) return nccl_fail("ncclCommInitAll", r);
    }
    g->init_ms = ms;
    g->inited = true;
    int rc = ensure_moments(g, 2);
    if (rc == NMCH_OK && g->n > 1) {
        // first collective on a communicator sets up its channels (~100 ms): pay that here, not in compute()
        for (int i = 0; i < g->n; ++i) {
            GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
            GROUP_CU_TRY(cudaMemsetAsync(g->d_mom[i], 0, 2 * sizeof(double), g->stream[i]));
        }
        ncclResult_t r = g_nccl.GroupStart();
        for (int i = 0; i < g->n && r == ncclSuccess; ++i)
            r = g_nccl.AllReduce(g->d_mom[i], g->d_mom[i], 2, ncclDouble, ncclSum, g->comm[i], g->stream[i]);
        if (r == ncclSuccess) r = g_nccl.GroupEnd();
        if (r != ncclSuccess) return nccl_fail("NCCL warm-up allreduce", r);
        for (int i = 0; i < g->n; ++i) {
            GROUP_CU_TRY(cudaSetDevice(g->dev[i]));
            GROUP_CU_TRY(cudaStreamSynchronize(g->stream[i]));
        }
    }
    return rc;
}

int nmch_group_init(nmch_group_t *g, unsigned long long seed)
{
    if (!g) return engine_fail(NMCH_ERR_ARG, "null group");
    if (g->inited) return engine_fail(NMCH_ERR_STATE, "group already initialised");
    DeviceRestore restore;
    const int rc = group_init_impl(g, seed);
    if (rc != NMCH_OK) {
        const std::string why = nmch_last_error();      // keep the cause: the clean-up below may overwrite it
        nmch_group_finalize(g);                         // releases whatever the failed init had created
        engine_fail(rc, why.c_str());
    }
    return rc;
}

int nmch_group_set_params(nmch_group_t *g, float k, float theta, float sigma)
{
    if (!g) return engine_fail(NMCH_ERR_ARG, "null group");
    for (auto *e : g->eng) nmch_engine_set_params(e, k, theta, sigma);
    return NMCH_OK;
}

int nmch_group_compute(nmch_group_t *g, nmch_moments_t *out)
{
    if (!out) return engine_fail(NMCH_ERR_ARG, "null output");
    DeviceRestore restore;
    return run_points(g, nullptr, nullptr, nullptr, 1, out);
}

int nmch_group_explore(nmch_group_t *g, const float *k, const float *theta, const float *sigma, int n_points,
                       nmch_moments_t *out)
{
    if (!k || !theta || !sigma || !out || n_points <= 0) return engine_fail(NMCH_ERR_ARG, "bad exploration arguments");
    DeviceRestore restore;
    return run_points(g, k, theta, sigma, n_points, out);
}

int nmch_group_compute_strikes(nmch_group_t *g, const float *strikes, int n_strikes, nmch_strike_moments_t *out)
{
    return group_strikes(g, strikes, n_strikes, 0, out);
}

int nmch_group_compute_greeks(nmch_group_t *g, const float *strikes, int n_strikes, nmch_greek_moments_t *out)
{
    return group_strikes(g, strikes, n_strikes, 1, out);
}

int nmch_group_compute_sensitivities(nmch_group_t *g, const float *strikes, int n_strikes, nmch_sensitivity_moments_t *out)
{
    return group_strikes(g, strikes, n_strikes, NMCH_SENS_COUNT, out);
}

int nmch_group_finalize(nmch_group_t *g)
{
    if (!g) return engine_fail(NMCH_ERR_ARG, "null group");
    // Idempotent, and also the clean-up path of an init() that failed half way: every resource is released if
    // present, whatever the lifecycle flag says (as nmch_engine_finalize does).
    DeviceRestore restore;
    for (int i = 0; i < g->n; ++i) {
        if (i >= (int)g->dev.size()) break;
        cudaSetDevice(g->dev[i]);
        if (i < (int)g->stream.size() && g->stream[i]) cudaStreamSynchronize(g->stream[i]);
        if (i < (int)g->comm.size() && g->comm[i]) g_nccl.CommDestroy(g->comm[i]);
        if (i < (int)g->eng.size() && g->eng[i]) nmch_engine_finalize(g->eng[i]);
        if (i < (int)g->d_mom.size() && g->d_mom[i]) { cudaFree(g->d_mom[i]); g->d_mom[i] = nullptr; }
        if (i < (int)g->ev0.size() && g->ev0[i]) { cudaEventDestroy(g->ev0[i]); g->ev0[i] = nullptr; }
        if (i < (int)g->ev1.size() && g->ev1[i]) { cudaEventDestroy(g->ev1[i]); g->ev1[i] = nullptr; }
        if (i < (int)g->stream.size() && g->stream[i]) { cudaStreamDestroy(g->stream[i]); g->stream[i] = nullptr; }
    }
    g->comm.clear();
    if (g->h_mom) cudaFreeHost(g->h_mom);
    g->h_mom = nullptr;
    g->mom_cap = 0;
    g->inited = false;
    return NMCH_OK;
}

void nmch_group_destroy(nmch_group_t *g)
{
    if (!g) return;
    nmch_group_finalize(g);
    for (auto *e : g->eng) nmch_engine_destroy(e);
    delete g;
}

float nmch_group_init_ms(const nmch_group_t *g) { return g ? g->init_ms : 0.0f; }
int nmch_group_size(const nmch_group_t *g) { return g ? g->n : 0; }

}  // extern "C"
