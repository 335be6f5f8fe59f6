// Lifecycle half of the C ABI (include/nfsp_b200.h): handles, errors, device queries.
#include <cstring>

#include "common.cuh"

namespace nfsp {

static thread_local char g_err[512] = "";

int set_error(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace nfsp

using namespace nfsp;

extern "C" int nfsp_version(void) { return 100; }

extern "C" const char *nfsp_last_error(void) { return g_err; }

extern "C" int nfsp_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len) {
    cudaDeviceProp prop;
    NFSP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (name && name_len > 0) {
        strncpy(name, prop.name, (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    return NFSP_OK;
}

extern "C" int nfsp_env_create(int rules, int64_t n_games, uint64_t seed, uint64_t game0, int device,
                               nfsp_env_t *out) {
    NFSP_CHECK_ARG(out != nullptr, "null out handle");
    *out = nullptr;
    NFSP_CHECK_ARG(rules == NFSP_RULES_LEGACY || rules == NFSP_RULES_NFSP, "unknown rules %d", rules);
    NFSP_CHECK_ARG(n_games >= 1 && n_games <= (int64_t)1 << 31, "n_games out of range");
    // Philox counter word 0 holds the low half of the global game id: game 2^32 would replay game 0's deals
    NFSP_CHECK_ARG(game0 <= ((uint64_t)1 << 32) - (uint64_t)n_games, "game0 + n_games must not exceed 2^32");
    int count = 0;
    // no CPU fallback: without a CUDA device this fails loudly
    NFSP_CUDA(cudaGetDeviceCount(&count));
    NFSP_CHECK_ARG(device >= 0 && device < count, "device %d not present (%d visible)", device, count);
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", device);
    cudaDeviceProp prop;
    NFSP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return set_error(NFSP_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                         prop.major, prop.minor);
    nfsp_env_s *h = new nfsp_env_s();
    h->rules = rules;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->n = n_games;
    h->seed = seed;
    h->game0 = game0;
    h->step = 0;
    h->d_state = nullptr;
    h->d_fsm = nullptr;
    h->d_wpack = nullptr;
    h->d_work = nullptr;
    h->d_wtc_wide = nullptr;
    h->has_weights = false;
    cudaError_t e = cudaMalloc(&h->d_state, sizeof(uint64_t) * (size_t)n_games);
    if (e != cudaSuccess) {
        delete h;
        return set_error(NFSP_E_CUDA, "cudaMalloc of %lld game words failed: %s", (long long)n_games,
                         cudaGetErrorString(e));
    }
    e = cudaMemset(h->d_state, 0, sizeof(uint64_t) * (size_t)n_games);
    if (e != cudaSuccess) {
        cudaFree(h->d_state);
        delete h;
        return set_error(NFSP_E_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    }
    {
        const int rc = nfsp_fsm_upload(h);
        if (rc != NFSP_OK) {
            cudaFree(h->d_state);
            delete h;
            return rc;
        }
    }
    *out = h;
    return NFSP_OK;
}

extern "C" int nfsp_env_destroy(nfsp_env_t h) {
    if (!h) return NFSP_OK;
    DeviceGuard guard(h->device);
    if (h->d_state) cudaFree(h->d_state);
    if (h->d_fsm) cudaFree(h->d_fsm);
    if (h->d_wpack) cudaFree(h->d_wpack);
    if (h->d_work) cudaFree(h->d_work);
    if (h->d_wtc_wide) cudaFree(h->d_wtc_wide);
    nfsp_tq_release(h);
    delete h;
    return NFSP_OK;
}

extern "C" int64_t nfsp_env_num_games(nfsp_env_t h) { return h ? h->n : 0; }
extern "C" int nfsp_env_rules(nfsp_env_t h) { return h ? h->rules : NFSP_E_ARG; }
extern "C" uint64_t nfsp_env_step_counter(nfsp_env_t h) { return h ? h->step : 0; }
extern "C" int nfsp_env_set_step_counter(nfsp_env_t h, uint64_t step) {
    NFSP_CHECK_ARG(h != nullptr, "null handle");
    h->step = step;
    return NFSP_OK;
}
extern "C" void *nfsp_env_state_ptr(nfsp_env_t h) { return h ? h->d_state : nullptr; }

extern "C" int nfsp_env_kernel_error(nfsp_env_t h, uint32_t *out) {
    NFSP_CHECK_ARG(h != nullptr && out != nullptr, "null argument");
    *out = 0u;
    if (!h->d_err) return NFSP_OK;
    DeviceGuard guard(h->device);
    NFSP_CUDA(cudaMemcpy(out, h->d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return NFSP_OK;
}

extern "C" int nfsp_rollout_tune(nfsp_env_t h, int patience_avg, int patience_br) {
    NFSP_CHECK_ARG(h != nullptr && patience_avg >= 0 && patience_br >= 0, "bad arguments");
    h->tq_patience[0] = (uint32_t)patience_avg;
    h->tq_patience[1] = (uint32_t)patience_br;
    return NFSP_OK;
}

extern "C" int nfsp_env_save_state(nfsp_env_t h, uint64_t *d_out, void *stream) {
    NFSP_CHECK_ARG(h != nullptr && d_out != nullptr, "null argument");
    DeviceGuard guard(h->device);
    NFSP_CUDA(cudaMemcpyAsync(d_out, h->d_state, sizeof(uint64_t) * (size_t)h->n, cudaMemcpyDeviceToDevice,
                              (cudaStream_t)stream));
    return NFSP_OK;
}

extern "C" int nfsp_env_load_state(nfsp_env_t h, const uint64_t *d_in, void *stream) {
    NFSP_CHECK_ARG(h != nullptr && d_in != nullptr, "null argument");
    DeviceGuard guard(h->device);
    NFSP_CUDA(cudaMemcpyAsync(h->d_state, d_in, sizeof(uint64_t) * (size_t)h->n, cudaMemcpyDeviceToDevice,
                              (cudaStream_t)stream));
    return NFSP_OK;
}
