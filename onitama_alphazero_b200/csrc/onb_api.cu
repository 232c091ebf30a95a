// onb_api.cu -- the extern "C" boundary of libonb.so (include/onb.h): context lifecycle, host<->device
// staging and error mapping. No torch types, no C++ exceptions, no CPU fallback.
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <string>
#include <vector>

#include "onb_gumbel.cuh"
#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {

cudaError_t launch_env_playout(Ctx* c, uint32_t* d_plies, unsigned long long* d_trace, uint32_t step0, uint32_t max_plies, int mode);

static int32_t fail(Ctx* c, int32_t code, const char* fmt, ...) {
    if (c) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(c->err, sizeof(c->err), fmt, ap);
        va_end(ap);
    }
    return code;
}
static int32_t cuda_fail(Ctx* c, cudaError_t e, const char* what) {
    return fail(c, ONB_E_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}
#define ONB_CUDA(c, call)                                   \
    do {                                                    \
        cudaError_t e__ = (call);                           \
        if (e__ != cudaSuccess) return cuda_fail(c, e__, #call); \
    } while (0)
// every entry point binds the context's device for the duration of the call (and puts the caller's device back): one host thread
// may drive contexts on several GPUs, and a drop-in library must not change the caller's current device behind its back
struct DeviceGuard {
    int prev = -1, mine;
    explicit DeviceGuard(int dev) : mine(dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != mine) cudaSetDevice(mine);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != mine) cudaSetDevice(prev);
    }
};
#define ONB_CHECK_CTX(ctx)            \
    if (!(ctx)) return ONB_E_INVALID; \
    DeviceGuard onb_device_guard__(reinterpret_cast<const Ctx*>(ctx)->cfg.device)

template <class T>
static cudaError_t dalloc(T** p, size_t count) {
    *p = nullptr;
    if (count == 0) return cudaSuccess;
    return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
}

// message of the last failed onb_create (no context exists yet to hold it); onb_create is expected to be called from one
// thread at a time per process
static char g_create_err[512] = "";

}  // namespace onb

using namespace onb;

extern "C" {

int32_t onb_version(void) { return ONB_VERSION; }

const char* onb_last_error(const onb_ctx* ctx) { return ctx ? reinterpret_cast<const Ctx*>(ctx)->err : g_create_err; }

int32_t onb_create(const onb_config* cfg, onb_ctx** out) {
    if (!cfg || !out || cfg->n_games <= 0) {
        snprintf(g_create_err, sizeof(g_create_err), "onb_create: invalid config");
        return ONB_E_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0 || cfg->device < 0 || cfg->device >= ndev) {
        snprintf(g_create_err, sizeof(g_create_err), "onb_create: no usable CUDA device %d (%s); there is no CPU fallback", cfg->device,
                 e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
        return ONB_E_CUDA;
    }
    Ctx* c = new (std::nothrow) Ctx();
    if (!c) return ONB_E_NOMEM;
    memset(c, 0, sizeof(*c));
    c->fixed_cards = -1;
    c->cfg = *cfg;
    c->n = cfg->n_games;
#define ONB_CREATE_CUDA(call)                                                                       \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            snprintf(g_create_err, sizeof(g_create_err), "onb_create: %s: %s", #call, cudaGetErrorString(e__)); \
            onb_destroy(reinterpret_cast<onb_ctx*>(c));                                             \
            return e__ == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;                     \
        }                                                                                           \
    } while (0)
    DeviceGuard onb_device_guard__(cfg->device);
    ONB_CREATE_CUDA(cudaSetDevice(cfg->device));
    if (cfg->stream) {
        c->stream = reinterpret_cast<cudaStream_t>(cfg->stream);
        c->own_stream = false;
    } else {
        ONB_CREATE_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    const size_t n = (size_t)c->n;
    ONB_CREATE_CUDA(dalloc(&c->d_states, n));
    ONB_CREATE_CUDA(dalloc(&c->d_masks, 2 * n));
    ONB_CREATE_CUDA(dalloc(&c->d_actions, n));
    ONB_CREATE_CUDA(dalloc(&c->d_stats, (size_t)ONB_STAT_COUNT));
    ONB_CREATE_CUDA(cudaMemsetAsync(c->d_stats, 0, ONB_STAT_COUNT * sizeof(unsigned long long), c->stream));
    if (cfg->alloc_planes) ONB_CREATE_CUDA(dalloc(&c->d_planes, n * 525));
    if (cfg->mcts_max_sims) {
        c->node_cap = cfg->mcts_node_cap ? cfg->mcts_node_cap : 1u + 40u * cfg->mcts_max_sims;
        if (c->node_cap < 64) c->node_cap = 64;
        ONB_CREATE_CUDA(dalloc(&c->d_nodes, n * (size_t)c->node_cap));
        ONB_CREATE_CUDA(dalloc(&c->d_tree_size, n));
        ONB_CREATE_CUDA(dalloc(&c->d_tree_flags, n));
        ONB_CREATE_CUDA(dalloc(&c->d_roots, n));
        ONB_CREATE_CUDA(dalloc(&c->d_leaf_node, n));
        ONB_CREATE_CUDA(dalloc(&c->d_leaf_state, n));
        ONB_CREATE_CUDA(dalloc(&c->d_leaf_planes, n * 525));
        ONB_CREATE_CUDA(dalloc(&c->d_policy, n * 50));
        ONB_CREATE_CUDA(dalloc(&c->d_value, n));
        ONB_CREATE_CUDA(dalloc(&c->d_pi, n * 50));
        ONB_CREATE_CUDA(dalloc(&c->d_best, n));
        ONB_CREATE_CUDA(dalloc(&c->d_root_visits, n));
        ONB_CREATE_CUDA(dalloc(&c->d_root_q, n));
        ONB_CREATE_CUDA(dalloc(&c->d_child_visits, n * 40));
    }
    ONB_CREATE_CUDA(cudaStreamSynchronize(c->stream));
#undef ONB_CREATE_CUDA
    *out = reinterpret_cast<onb_ctx*>(c);
    return ONB_OK;
}

int32_t onb_destroy(onb_ctx* ctx) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    cudaSetDevice(c->cfg.device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    void* ptrs[] = {c->d_states, c->d_masks, c->d_planes, c->d_actions, c->d_stats, c->d_io_states, c->d_moves, c->d_counts, c->d_nodes,
                    c->d_tree_size, c->d_tree_flags, c->d_roots, c->d_leaf_node, c->d_leaf_state, c->d_leaf_planes, c->d_policy, c->d_value,
                    c->d_pi, c->d_best, c->d_root_visits, c->d_root_q, c->d_child_visits, c->net[0].w, c->net[0].bias, c->net[0].head, c->net[1].w,
                    c->net[1].bias, c->net[1].head, c->d_ln_table, c->d_net_scratch, c->d_ab_score, c->d_ab_nodes, c->d_gb,
                    c->d_gb_tab, c->d_gb_base, c->d_gb_p, c->d_gb_r0, c->d_tb_values};
    reuse_free(c);
    tb_free(c);
    for (void* p : c->sp_buf)
        if (p) cudaFree(p);
    for (void* p : ptrs)
        if (p) cudaFree(p);
    for (void* p : c->scratch)
        if (p) cudaFree(p);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return ONB_OK;
}

int32_t onb_sync(onb_ctx* ctx) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

int32_t onb_get_stream(onb_ctx* ctx, void** stream) {
    ONB_CHECK_CTX(ctx);
    if (!stream) return ONB_E_INVALID;
    *stream = reinterpret_cast<void*>(reinterpret_cast<Ctx*>(ctx)->stream);
    return ONB_OK;
}

int32_t onb_buffer(onb_ctx* ctx, int32_t which, void** dev_ptr, int64_t* bytes) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    void* p = nullptr;
    int64_t b = 0;
    const int64_t n = c->n;
    switch (which) {
        case ONB_BUF_STATES: p = c->d_states; b = n * 16; break;
        case ONB_BUF_MASKS: p = c->d_masks; b = n * 8; break;
        case ONB_BUF_PLANES: p = c->d_planes; b = n * 2100; break;
        case ONB_BUF_ACTIONS: p = c->d_actions; b = n * 2; break;
        case ONB_BUF_LEAF_PLANES: p = c->d_leaf_planes; b = n * 2100; break;
        case ONB_BUF_POLICY: p = c->d_policy; b = n * 200; break;
        case ONB_BUF_VALUE: p = c->d_value; b = n * 4; break;
        case ONB_BUF_PI: p = c->d_pi; b = n * 200; break;
        case ONB_BUF_BEST: p = c->d_best; b = n * 2; break;
        case ONB_BUF_STATS: p = c->d_stats; b = ONB_STAT_COUNT * 8; break;
        default: return fail(c, ONB_E_INVALID, "onb_buffer: unknown buffer %d", which);
    }
    if (!p) return fail(c, ONB_E_STATE, "onb_buffer: buffer %d was not allocated by onb_create (see onb_config)", which);
    if (dev_ptr) *dev_ptr = p;
    if (bytes) *bytes = b;
    return ONB_OK;
}

int32_t onb_read_buffer(onb_ctx* ctx, int32_t which, void* host, int64_t bytes) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    void* p = nullptr;
    int64_t cap = 0;
    int32_t r = onb_buffer(ctx, which, &p, &cap);
    if (r) return r;
    if (!host || bytes < 0 || bytes > cap) return fail(c, ONB_E_INVALID, "onb_read_buffer: bad size %lld (buffer has %lld bytes)", (long long)bytes, (long long)cap);
    ONB_CUDA(c, cudaMemcpyAsync(host, p, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}
int32_t onb_write_buffer(onb_ctx* ctx, int32_t which, const void* host, int64_t bytes) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    void* p = nullptr;
    int64_t cap = 0;
    int32_t r = onb_buffer(ctx, which, &p, &cap);
    if (r) return r;
    if (!host || bytes < 0 || bytes > cap) return fail(c, ONB_E_INVALID, "onb_write_buffer: bad size %lld (buffer has %lld bytes)", (long long)bytes, (long long)cap);
    ONB_CUDA(c, cudaMemcpyAsync(p, host, (size_t)bytes, cudaMemcpyHostToDevice, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

// ---------------------------------------------------------------------------------------------- host helpers
int32_t onb_start_states(const uint8_t* decks5, int64_t n, onb_state* out) {
    if (!decks5 || !out || n < 0) return ONB_E_INVALID;
    for (int64_t i = 0; i < n; ++i) {
        const uint8_t* d = decks5 + 5 * i;
        for (int k = 0; k < 5; ++k)
            if (d[k] > 15) return ONB_E_INVALID;
        onb_state& s = out[i];
        s.pawns[0] = 0x00000D80u; s.pawns[1] = 0xD8000000u;  // state.rs:24-45
        s.kings[0] = 0x00000200u; s.kings[1] = 0x20000000u;
        memcpy(s.cards, d, 5);
        s.side = (uint8_t)((kBlueStampMask >> d[4]) & 1u);
        s.result = 0;
        s.flags = 0;
    }
    return ONB_OK;
}
uint32_t onb_rand_u32(uint64_t seed, uint64_t game, uint32_t step, uint32_t draw) { return rand_from_key(game_key(seed, game), step, draw); }
int32_t onb_deal(uint64_t seed, uint64_t game, uint32_t epoch, uint8_t out5[5]) {
    if (!out5) return ONB_E_INVALID;
    const uint32_t cards = deal_cards(game_key(seed, game), epoch);
    for (int k = 0; k < 5; ++k) out5[k] = (uint8_t)card_at(cards, k);
    return ONB_OK;
}
int32_t onb_attack_maps(uint32_t out800[800]) {
    if (!out800) return ONB_E_INVALID;
    for (int i = 0; i < 800; ++i) {  // internal bit n -> reference bit 31-n
        uint32_t v = kAttackHost.t[i], r = 0;
        for (int b = 0; b < 25; ++b)
            if (v & (1u << b)) r |= 1u << (31 - b);
        out800[i] = r;
    }
    return ONB_OK;
}

// ---------------------------------------------------------------------------------------------- env
static int32_t ensure_io(Ctx* c) {
    if (!c->d_io_states) ONB_CUDA(c, dalloc(&c->d_io_states, (size_t)c->n));
    return ONB_OK;
}

int32_t onb_env_reset(onb_ctx* ctx, const uint8_t* decks5_host, int64_t n_decks, uint32_t epoch) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (n_decks != 0 && n_decks != 1 && n_decks != c->n) return fail(c, ONB_E_INVALID, "onb_env_reset: n_decks must be 0, 1 or n_games");
    if (n_decks && !decks5_host) return fail(c, ONB_E_INVALID, "onb_env_reset: decks pointer is NULL");
    for (int64_t i = 0; i < 5 * n_decks; ++i)
        if (decks5_host[i] > 15) return fail(c, ONB_E_INVALID, "onb_env_reset: card id %d out of range", (int)decks5_host[i]);
    uint8_t* d_decks = nullptr;
    if (n_decks) {
        ONB_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&d_decks), (size_t)n_decks * 5));
        ONB_CUDA(c, cudaMemcpyAsync(d_decks, decks5_host, (size_t)n_decks * 5, cudaMemcpyHostToDevice, c->stream));
    }
    cudaError_t e = launch_env_reset(c, d_decks, n_decks, epoch);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (d_decks) cudaFree(d_decks);
    if (e != cudaSuccess) return cuda_fail(c, e, "onb_env_reset");
    c->fixed_cards = -1;
    if (n_decks == 1) {
        const uint8_t* d = decks5_host;
        c->fixed_cards = (int32_t)((d[0]) | (d[1] << 4) | (d[2] << 8) | (d[3] << 12) | (d[4] << 16));
    }
    c->mcts_phase = 0;
    return ONB_OK;
}

int32_t onb_env_reset_games(onb_ctx* ctx, const uint8_t* mask_host, uint32_t epoch, int64_t* n_reset) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    uint8_t* d = nullptr;
    const size_t mask_bytes = ((size_t)c->n + 7) & ~(size_t)7;  // layout: [n mask bytes, padded to 8][8-byte counter]
    ONB_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&d), mask_bytes + 8));
    unsigned long long* d_count = reinterpret_cast<unsigned long long*>(d + mask_bytes);
    cudaError_t e = cudaMemsetAsync(d_count, 0, 8, c->stream);
    if (e == cudaSuccess && mask_host) e = cudaMemcpyAsync(d, mask_host, (size_t)c->n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = launch_env_reset_where(c, mask_host ? d : nullptr, epoch, d_count);
    unsigned long long h = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d_count, 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(c, e, "onb_env_reset_games");
    if (n_reset) *n_reset = (int64_t)h;
    return ONB_OK;
}

int32_t onb_env_set_states(onb_ctx* ctx, const onb_state* states_host, int64_t first, int64_t n) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!states_host || first < 0 || n < 0 || first + n > c->n) return fail(c, ONB_E_INVALID, "onb_env_set_states: bad range");
    if (n == 0) return ONB_OK;
    int32_t r = ensure_io(c);
    if (r) return r;
    ONB_CUDA(c, cudaMemcpyAsync(c->d_io_states, states_host, (size_t)n * sizeof(onb_state), cudaMemcpyHostToDevice, c->stream));
    ONB_CUDA(c, launch_states_import(c, c->d_io_states, first, n));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    c->mcts_phase = 0;
    return ONB_OK;
}

int32_t onb_env_get_states(onb_ctx* ctx, onb_state* states_host, int64_t first, int64_t n) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!states_host || first < 0 || n < 0 || first + n > c->n) return fail(c, ONB_E_INVALID, "onb_env_get_states: bad range");
    if (n == 0) return ONB_OK;
    int32_t r = ensure_io(c);
    if (r) return r;
    ONB_CUDA(c, launch_states_export(c, c->d_io_states, first, n));
    ONB_CUDA(c, cudaMemcpyAsync(states_host, c->d_io_states, (size_t)n * sizeof(onb_state), cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

int32_t onb_env_legal_moves(onb_ctx* ctx, onb_action* moves_host, uint8_t* counts_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_moves) {
        ONB_CUDA(c, dalloc(&c->d_moves, (size_t)c->n * 40));
        ONB_CUDA(c, dalloc(&c->d_counts, (size_t)c->n));
    }
    ONB_CUDA(c, launch_legal_moves(c));
    if (moves_host) ONB_CUDA(c, cudaMemcpyAsync(moves_host, c->d_moves, (size_t)c->n * 40 * sizeof(uint16_t), cudaMemcpyDeviceToHost, c->stream));
    if (counts_host) ONB_CUDA(c, cudaMemcpyAsync(counts_host, c->d_counts, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

int32_t onb_env_legal_masks(onb_ctx* ctx, uint32_t* masks_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    ONB_CUDA(c, launch_observe(c, ONB_OUT_MASKS));
    if (masks_host) {
        ONB_CUDA(c, cudaMemcpyAsync(masks_host, c->d_masks, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return ONB_OK;
}

int32_t onb_env_encode(onb_ctx* ctx, float* planes_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_planes) return fail(c, ONB_E_STATE, "onb_env_encode: plane buffer not allocated (onb_config.alloc_planes = 0)");
    ONB_CUDA(c, launch_observe(c, ONB_OUT_PLANES));
    if (planes_host) {
        ONB_CUDA(c, cudaMemcpyAsync(planes_host, c->d_planes, (size_t)c->n * 2100, cudaMemcpyDeviceToHost, c->stream));
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return ONB_OK;
}

int32_t onb_env_step(onb_ctx* ctx, const onb_action* actions_host, uint32_t step, int32_t auto_reset, uint32_t out_flags) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if ((out_flags & ONB_OUT_PLANES) && !c->d_planes) return fail(c, ONB_E_STATE, "onb_env_step: plane buffer not allocated");
    if (actions_host) ONB_CUDA(c, cudaMemcpyAsync(c->d_actions, actions_host, (size_t)c->n * sizeof(uint16_t), cudaMemcpyHostToDevice, c->stream));
    ONB_CUDA(c, launch_env_step(c, kModeActions, step, auto_reset, out_flags));
    c->mcts_phase = 0;
    return ONB_OK;
}

int32_t onb_env_step_random(onb_ctx* ctx, uint32_t step, int32_t policy, int32_t auto_reset, uint32_t out_flags) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (policy != ONB_POLICY_UNIFORM && policy != ONB_POLICY_AGENT) return fail(c, ONB_E_INVALID, "onb_env_step_random: unknown policy %d", policy);
    if ((out_flags & ONB_OUT_PLANES) && !c->d_planes) return fail(c, ONB_E_STATE, "onb_env_step_random: plane buffer not allocated");
    ONB_CUDA(c, launch_env_step(c, policy, step, auto_reset, out_flags));
    c->mcts_phase = 0;
    return ONB_OK;
}

int32_t onb_env_choose_random(onb_ctx* ctx, uint32_t step, int32_t policy) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (policy != ONB_POLICY_UNIFORM && policy != ONB_POLICY_AGENT) return fail(c, ONB_E_INVALID, "onb_env_choose_random: unknown policy %d", policy);
    ONB_CUDA(c, launch_env_step(c, 4 + policy, step, 0, 0));
    return ONB_OK;
}

int32_t onb_env_run_random(onb_ctx* ctx, uint32_t step0, uint32_t n_steps, int32_t policy, int32_t auto_reset, uint32_t out_flags) {
    for (uint32_t s = 0; s < n_steps; ++s) {
        int32_t r = onb_env_step_random(ctx, step0 + s, policy, auto_reset, out_flags);
        if (r) return r;
    }
    return ONB_OK;
}

int32_t onb_env_playout(onb_ctx* ctx, uint32_t step0, uint32_t max_plies, int32_t policy, uint32_t* plies_host, uint64_t* trace_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (policy != ONB_POLICY_UNIFORM && policy != ONB_POLICY_AGENT) return fail(c, ONB_E_INVALID, "onb_env_playout: unknown policy %d", policy);
    uint32_t* d_plies = nullptr;
    unsigned long long* d_trace = nullptr;
    if (plies_host) ONB_CUDA(c, dalloc(&d_plies, (size_t)c->n));
    if (trace_host) ONB_CUDA(c, dalloc(&d_trace, (size_t)c->n));
    cudaError_t e = launch_env_playout(c, d_plies, d_trace, step0, max_plies, policy);
    if (e == cudaSuccess && plies_host) e = cudaMemcpyAsync(plies_host, d_plies, (size_t)c->n * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && trace_host) e = cudaMemcpyAsync(trace_host, d_trace, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && (plies_host || trace_host)) e = cudaStreamSynchronize(c->stream);
    if (d_plies) cudaFree(d_plies);
    if (d_trace) cudaFree(d_trace);
    if (e != cudaSuccess) return cuda_fail(c, e, "onb_env_playout");
    c->mcts_phase = 0;
    return ONB_OK;
}

int32_t onb_env_stats(onb_ctx* ctx, uint64_t stats_host[ONB_STAT_COUNT], int32_t clear) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (stats_host) ONB_CUDA(c, cudaMemcpyAsync(stats_host, c->d_stats, ONB_STAT_COUNT * 8, cudaMemcpyDeviceToHost, c->stream));
    if (clear) ONB_CUDA(c, cudaMemsetAsync(c->d_stats, 0, ONB_STAT_COUNT * 8, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

// ---------------------------------------------------------------------------------------------- perft
int32_t onb_perft(onb_ctx* ctx, const onb_state* roots_host, int64_t n, int32_t depth, uint64_t* nodes_host, uint64_t* wins_host, uint64_t* zero_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!roots_host || n <= 0 || depth < 1 || depth > 12 || !nodes_host) return fail(c, ONB_E_INVALID, "onb_perft: bad arguments");
    return run_perft(c, roots_host, n, depth, nodes_host, wins_host, zero_host);
}

// ---------------------------------------------------------------------------------------------- mcts
}  // extern "C"
namespace onb {
static bool knob_set(const char* name, bool numeric) {
    const char* v = getenv(name);
    if (!v) return false;
    return numeric ? atoi(v) != 0 : v[0] == '1';
}
// the combinations a Gumbel search does not support (include/onb.h, onb_mcts_set_gumbel); reuse: this begin keeps remembered trees
// (onb_fight never does, whatever the context's reuse switch says). Every begin clears gb_search first, so a search begun after the
// switch went off, or a refused begin, never runs the Gumbel kernels.
static int32_t gumbel_refusals(Ctx* c, const char* what, bool reuse) {
    c->gb_search = 0;
    if (!c->gb_on) return ONB_OK;
    if (reuse) return fail(c, ONB_E_STATE, "%s: the Gumbel root search does not combine with tree reuse (onb_mcts_set_reuse)", what);
    if (c->noise_on) return fail(c, ONB_E_STATE, "%s: the Gumbel root search does not combine with train-mode noise (onb_mcts_set_noise)", what);
    if (knob_set("ONB_MCTS_WARP_PER_TREE", false) || knob_set("ONB_MCTS_STEP_FUSION", false) || knob_set("ONB_MCTS_ROOT_SMEM", true))
        return fail(c, ONB_E_STATE, "%s: the Gumbel root search does not run with the exploration knobs ONB_MCTS_WARP_PER_TREE / "
                                    "ONB_MCTS_STEP_FUSION / ONB_MCTS_ROOT_SMEM", what);
    return ONB_OK;
}
// after the trees are begun: the search's GumbelDev (step = the serial, which advances) and, when (m, sims) changed, the table
static int32_t gumbel_begin(Ctx* c, uint32_t sims) {
    c->gb_search = c->gb_on;
    if (!c->gb_on) return ONB_OK;
    const uint32_t m = c->gb_cfg.max_considered, nt = sims ? sims - 1u : 0u;
    if (nt && (c->gb_tab_m != m || c->gb_tab_n != nt)) {
        std::vector<uint32_t> tab((size_t)m * nt);
        for (uint32_t r = 1; r <= m; ++r) onb_gumbel::seq_halving(r, nt, tab.data() + (size_t)(r - 1u) * nt);
        // from pageable memory: the copy has taken the data when the call returns, so tab may go out of scope
        ONB_CUDA(c, cudaMemcpyAsync(c->d_gb_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, c->stream));
        c->gb_tab_m = m;
        c->gb_tab_n = nt;
    }
    GumbelDev h;
    memset(&h, 0, sizeof(h));
    h.c_visit = c->gb_cfg.c_visit;
    h.c_scale = c->gb_cfg.c_scale;
    h.scale = c->gb_cfg.gumbel_scale;
    h.seed = c->gb_cfg.seed;
    h.step = c->gb_serial++;
    h.m = m;
    h.n_tab = nt;
    h.tab = c->d_gb_tab;
    h.base = c->d_gb_base;
    h.p = c->d_gb_p;
    h.r0 = c->d_gb_r0;
    ONB_CUDA(c, cudaMemcpyAsync(c->d_gb, &h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
    return ONB_OK;
}
}  // namespace onb
extern "C" {
int32_t onb_mcts_begin(onb_ctx* ctx, double c_puct, uint32_t sims) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_nodes) return fail(c, ONB_E_STATE, "onb_mcts_begin: context created with mcts_max_sims = 0");
    if (sims > c->cfg.mcts_max_sims) return fail(c, ONB_E_INVALID, "onb_mcts_begin: sims %u > mcts_max_sims %u", sims, c->cfg.mcts_max_sims);
    c->c_puct = c_puct;
    c->sims_target = sims;
    c->sims_done = 0;
    c->n_act = 0;  // the public search covers every game of the context
    c->d_tree_game = nullptr;
    c->mcts_phase = 0;
    int32_t rc = gumbel_refusals(c, "onb_mcts_begin", c->reuse_on != 0);
    if (rc != ONB_OK) return rc;
    if (c->reuse_on) {  // every game, trees laid out by remaining budget; finish puts the outputs back into game order
        ONB_CUDA(c, launch_reuse_begin(c, nullptr, c->n, sims));
        c->ru_search = 1;
        c->ru_public = 1;
    } else {
        c->ru_live = c->ru_search = c->ru_public = 0;  // a search without reuse forgets the remembered trees
        ONB_CUDA(c, launch_mcts_begin(c));
    }
    if ((rc = gumbel_begin(c, sims)) != ONB_OK) return rc;
    c->mcts_phase = 1;
    return ONB_OK;
}
int32_t onb_mcts_set_gumbel(onb_ctx* ctx, const onb_gumbel_config* cfg) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!cfg || !cfg->enabled) {
        c->gb_on = 0;
        return ONB_OK;
    }
    if (cfg->max_considered < 1 || cfg->max_considered > 40 || !std::isfinite(cfg->c_visit) || !std::isfinite(cfg->c_scale) ||
        !std::isfinite(cfg->gumbel_scale) || !(cfg->c_visit >= 0.0) || !(cfg->c_scale >= 0.0) || !(cfg->gumbel_scale >= 0.0))
        return fail(c, ONB_E_INVALID, "onb_mcts_set_gumbel: need 1 <= max_considered <= 40 and finite c_visit, c_scale, gumbel_scale >= 0");
    if (!c->d_nodes) return fail(c, ONB_E_STATE, "onb_mcts_set_gumbel: context created with mcts_max_sims = 0");
    if (!c->d_gb) {
        const size_t n = (size_t)c->n;
        cudaError_t e = dalloc(&c->d_gb, 1);
        if (e == cudaSuccess) e = dalloc(&c->d_gb_tab, (size_t)40 * c->cfg.mcts_max_sims);
        if (e == cudaSuccess) e = dalloc(&c->d_gb_base, n * kGbStride);
        if (e == cudaSuccess) e = dalloc(&c->d_gb_p, n * kGbStride);
        if (e == cudaSuccess) e = dalloc(&c->d_gb_r0, n);
        if (e != cudaSuccess) {
            for (void* p : {(void*)c->d_gb, (void*)c->d_gb_tab, (void*)c->d_gb_base, (void*)c->d_gb_p, (void*)c->d_gb_r0})
                if (p) cudaFree(p);
            c->d_gb = nullptr; c->d_gb_tab = nullptr; c->d_gb_base = c->d_gb_p = c->d_gb_r0 = nullptr;
            return e == cudaErrorMemoryAllocation ? fail(c, ONB_E_NOMEM, "onb_mcts_set_gumbel: out of device memory") : cuda_fail(c, e, "onb_mcts_set_gumbel");
        }
        c->gb_tab_m = c->gb_tab_n = 0;
    }
    c->gb_cfg = *cfg;
    c->gb_serial = cfg->step0;
    c->gb_on = 1;
    return ONB_OK;
}
int32_t onb_mcts_set_reuse(onb_ctx* ctx, int32_t enabled) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (enabled) {
        if (!c->d_nodes) return fail(c, ONB_E_STATE, "onb_mcts_set_reuse: context created with mcts_max_sims = 0");
        const cudaError_t e = reuse_alloc(c);
        if (e == cudaErrorInvalidValue) return fail(c, ONB_E_INVALID, "onb_mcts_set_reuse: mcts_node_cap %u is too large for tree reuse", c->node_cap);
        if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(c, ONB_E_NOMEM, "onb_mcts_set_reuse: out of device memory for the second node pool")
                                                                    : cuda_fail(c, e, "onb_mcts_set_reuse");
        c->reuse_on = 1;
    } else {
        c->reuse_on = 0;
        c->ru_live = 0;  // switching off forgets the remembered trees
    }
    return ONB_OK;
}
int32_t onb_mcts_reuse_stats(onb_ctx* ctx, uint64_t out[4], int32_t clear) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (out) memcpy(out, c->ru_stats, sizeof(c->ru_stats));
    if (clear) memset(c->ru_stats, 0, sizeof(c->ru_stats));
    return ONB_OK;
}
static int32_t refuse_after_reuse(Ctx* c, const char* what) {
    return fail(c, ONB_E_STATE, "%s: the search was begun with tree reuse on (onb_mcts_set_reuse), which only onb_mcts_run can continue; "
                                "switch reuse off before onb_mcts_begin for a caller-driven search", what);
}
int32_t onb_mcts_set_noise(onb_ctx* ctx, int32_t enabled, double epsilon, double alpha, uint64_t seed) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (enabled && (!(epsilon >= 0.0 && epsilon <= 1.0) || !(alpha > 0.0))) return fail(c, ONB_E_INVALID, "onb_mcts_set_noise: need 0 <= epsilon <= 1 and alpha > 0");
    c->noise_on = enabled ? 1 : 0;
    c->noise_eps = epsilon;
    c->noise_alpha = alpha;
    c->noise_seed = seed;
    return ONB_OK;
}
int32_t onb_mcts_select(onb_ctx* ctx) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->mcts_phase != 1) return fail(c, ONB_E_STATE, "onb_mcts_select: call onb_mcts_begin / onb_mcts_expand_backup first");
    if (c->ru_search) return refuse_after_reuse(c, "onb_mcts_select");
    if (c->gb_search && c->sims_done >= c->sims_target)
        return fail(c, ONB_E_STATE, "onb_mcts_select: a Gumbel search runs at most the begin's %u simulations", c->sims_target);
    ONB_CUDA(c, launch_mcts_select(c));
    c->mcts_phase = 2;
    return ONB_OK;
}
int32_t onb_mcts_eval(onb_ctx* ctx, int32_t evaluator) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->ru_search) return refuse_after_reuse(c, "onb_mcts_eval");
    if (c->mcts_phase != 2) return fail(c, ONB_E_STATE, "onb_mcts_eval: no leaves selected");
    if (evaluator == ONB_EVAL_NET) {
        if (!c->net[c->net_cur].loaded) return fail(c, ONB_E_STATE, "onb_mcts_eval: no network loaded (onb_net_load)");
        ONB_CUDA(c, launch_net_forward(c, c->d_leaf_planes, c->d_policy, c->d_value, trees(c)));
        return ONB_OK;
    }
    if (evaluator != ONB_EVAL_UNIFORM && evaluator != ONB_EVAL_HASH) return fail(c, ONB_E_INVALID, "onb_mcts_eval: unknown evaluator %d", evaluator);
    ONB_CUDA(c, launch_mcts_eval(c, evaluator));
    return ONB_OK;
}
int32_t onb_mcts_expand_backup(onb_ctx* ctx) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->ru_search) return refuse_after_reuse(c, "onb_mcts_expand_backup");
    if (c->mcts_phase != 2) return fail(c, ONB_E_STATE, "onb_mcts_expand_backup: call onb_mcts_select first");
    ONB_CUDA(c, launch_mcts_expand_backup(c));
    c->mcts_phase = 1;
    c->sims_done += 1;
    return ONB_OK;
}
// onb_mcts_run after a reuse begin: slot t runs max(0, sims - N_root) simulations; the slots are ordered by that budget, so round r
// runs the prefix [0, h_ru_off[r]) -- the network evaluates a shrinking batch, the fused kernel is launched once per run of rounds
// with the same prefix. Splitting a tree's simulations over several launches gives the same tree: the kernels keep nothing else.
static int32_t reuse_run(Ctx* c, int32_t evaluator, uint32_t sims) {
    if (sims != c->sims_target || c->sims_done != 0)
        return fail(c, ONB_E_INVALID, "onb_mcts_run: after a reuse begin, run once with the begin's visit target (%u), got %u", c->sims_target, sims);
    if (evaluator == ONB_EVAL_NET && !c->net[c->net_cur].loaded) return fail(c, ONB_E_STATE, "onb_mcts_run: no network loaded (onb_net_load)");
    const uint32_t* off = c->h_ru_off;
    cudaError_t e = cudaSuccess;
    if (evaluator == ONB_EVAL_NET) {
        for (uint32_t r = 0; r < sims && off[r] > 0 && e == cudaSuccess; ++r) {
            c->n_act = (int64_t)off[r];
            e = launch_mcts_select(c);
            if (e == cudaSuccess) e = launch_net_forward(c, c->d_leaf_planes, c->d_policy, c->d_value, (int64_t)off[r]);
            if (e == cudaSuccess) e = launch_mcts_expand_backup(c);
        }
    } else {
        for (uint32_t r = 0; r < sims && off[r] > 0 && e == cudaSuccess;) {
            uint32_t r1 = r + 1;
            while (r1 < sims && off[r1] == off[r]) ++r1;
            c->n_act = (int64_t)off[r];
            e = launch_mcts_run(c, evaluator, r1 - r);
            r = r1;
        }
    }
    c->n_act = c->ru_m;
    if (e != cudaSuccess) return cuda_fail(c, e, "onb_mcts_run");
    c->sims_done += sims;
    return ONB_OK;
}
int32_t onb_mcts_run(onb_ctx* ctx, int32_t evaluator, uint32_t sims) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->mcts_phase != 1) return fail(c, ONB_E_STATE, "onb_mcts_run: call onb_mcts_begin first");
    if (evaluator != ONB_EVAL_UNIFORM && evaluator != ONB_EVAL_HASH && evaluator != ONB_EVAL_NET)
        return fail(c, ONB_E_INVALID, "onb_mcts_run: unknown evaluator %d", evaluator);
    if (c->sims_done + sims > c->cfg.mcts_max_sims) return fail(c, ONB_E_INVALID, "onb_mcts_run: more simulations than mcts_max_sims");
    if (c->ru_search) return reuse_run(c, evaluator, sims);
    if (c->gb_search && c->sims_done + sims > c->sims_target)
        return fail(c, ONB_E_STATE, "onb_mcts_run: a Gumbel search runs at most the begin's %u simulations", c->sims_target);
    if (evaluator == ONB_EVAL_NET) {
        // the network sits between select and expand: three launches per simulation round, all on the context's stream.
        // ONB_MCTS_STEP_FUSION=1 (exploration knob): expand_backup(s) and select(s + 1) as ONE launch (k_mcts_step_g) -- measured SLOWER
        // on B200 (config 5, f16 network: 304.8 vs 293.9 ms per ply): the fused kernel carries both halves' shared tables (36.6 KB, one
        // CTA fewer per SM) and a block barrier between them, which costs more than the saved launch boundary
        if (!c->net[c->net_cur].loaded) return fail(c, ONB_E_STATE, "onb_mcts_run: no network loaded (onb_net_load)");
        const char* fuse_env = getenv("ONB_MCTS_STEP_FUSION");
        const bool fuse = fuse_env && fuse_env[0] == '1';
        if (sims > 0) ONB_CUDA(c, launch_mcts_select(c));
        for (uint32_t s = 0; s < sims; ++s) {
            ONB_CUDA(c, launch_net_forward(c, c->d_leaf_planes, c->d_policy, c->d_value, trees(c)));
            if (s + 1 == sims) {
                ONB_CUDA(c, launch_mcts_expand_backup(c));
            } else if (fuse) {
                ONB_CUDA(c, launch_mcts_step(c));
            } else {
                ONB_CUDA(c, launch_mcts_expand_backup(c));
                ONB_CUDA(c, launch_mcts_select(c));
            }
        }
        c->sims_done += sims;
        return ONB_OK;
    }
    ONB_CUDA(c, launch_mcts_run(c, evaluator, sims));
    c->sims_done += sims;
    return ONB_OK;
}
// onb_mcts_begin for a SUBSET of the games: tree t searches game d_games[t] (device list, ascending), t < m. d_games == nullptr: all games.
static int32_t mcts_begin_subset(Ctx* c, double c_puct, uint32_t sims, const int32_t* d_games, int64_t m) {
    onb_ctx* x = reinterpret_cast<onb_ctx*>(c);
    if (!d_games) return onb_mcts_begin(x, c_puct, sims);
    if (!c->d_nodes) return fail(c, ONB_E_STATE, "search: context created with mcts_max_sims = 0");
    if (sims > c->cfg.mcts_max_sims) return fail(c, ONB_E_INVALID, "search: sims %u > mcts_max_sims %u", sims, c->cfg.mcts_max_sims);
    if (m <= 0 || m > c->n) return fail(c, ONB_E_INVALID, "search: bad subset size");
    c->c_puct = c_puct;
    c->sims_target = sims;
    c->sims_done = 0;
    c->n_act = m;
    c->d_tree_game = d_games;
    c->ru_live = c->ru_search = c->ru_public = 0;  // a search without reuse forgets the remembered trees
    int32_t rc = gumbel_refusals(c, "search", false);
    if (rc != ONB_OK) return rc;
    ONB_CUDA(c, launch_mcts_begin(c));
    if ((rc = gumbel_begin(c, sims)) != ONB_OK) return rc;
    c->mcts_phase = 1;
    return ONB_OK;
}
// onb_self_play's search with reuse: the m games d_games (nullptr: all) in budget order; the outputs stay in slot order, the driver
// scatters them through d_tree_game
static int32_t reuse_begin_subset(Ctx* c, double c_puct, uint32_t sims, const int32_t* d_games, int64_t m) {
    const int32_t rc = gumbel_refusals(c, "onb_self_play", true);
    if (rc != ONB_OK) return rc;
    c->c_puct = c_puct;
    c->sims_target = sims;
    c->sims_done = 0;
    c->mcts_phase = 0;
    ONB_CUDA(c, launch_reuse_begin(c, d_games, d_games ? m : c->n, sims));
    c->ru_search = 1;
    c->ru_public = 0;
    c->mcts_phase = 1;
    return ONB_OK;
}
static int32_t self_play_search(Ctx* c, const onb_selfplay_config* cfg, const int32_t* d_games, int64_t m) {
    onb_ctx* x = reinterpret_cast<onb_ctx*>(c);
    int32_t rc = c->reuse_on ? reuse_begin_subset(c, cfg->c_puct, cfg->sims, d_games, m) : mcts_begin_subset(c, cfg->c_puct, cfg->sims, d_games, m);
    if (rc == ONB_OK) rc = onb_mcts_run(x, cfg->evaluator, cfg->sims);
    if (rc == ONB_OK) rc = onb_mcts_finish(x, nullptr, nullptr, nullptr, nullptr, nullptr);
    return rc;
}
int32_t onb_self_play(onb_ctx* ctx, const onb_selfplay_config* cfg, onb_selfplay_result* out) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!cfg || !out) return fail(c, ONB_E_INVALID, "onb_self_play: null argument");
    if (!c->d_planes || !c->d_nodes) return fail(c, ONB_E_STATE, "onb_self_play: the context needs alloc_planes and mcts_max_sims > 0");
    if (cfg->sims == 0 || cfg->sims > c->cfg.mcts_max_sims) return fail(c, ONB_E_INVALID, "onb_self_play: sims %u not in 1..mcts_max_sims", cfg->sims);
    if (cfg->n_games <= 0) return fail(c, ONB_E_INVALID, "onb_self_play: n_games must be positive");
    if (cfg->train && c->gb_on) return fail(c, ONB_E_INVALID, "onb_self_play: train-mode noise does not combine with the Gumbel root search");
    if (c->reuse_on && c->gb_on) return fail(c, ONB_E_STATE, "onb_self_play: tree reuse does not combine with the Gumbel root search");
    memset(out, 0, sizeof(*out));
    c->ru_live = 0;  // self-play starts from fresh deals: nothing is kept from earlier searches
    int32_t rc = onb_mcts_set_noise(ctx, cfg->train ? 1 : 0, 0.25, 0.03, cfg->noise_seed);
    if (rc != ONB_OK) return rc;
    const uint32_t serial = c->gb_serial;
    c->gb_serial = 0;  // one search per ply: the Gumbel step of ply p is p
    char err[400];
    err[0] = 0;
    try {
        rc = run_self_play(c, cfg, out, self_play_search, err, sizeof(err));
    } catch (const std::exception& ex) {
        snprintf(err, sizeof(err), "onb_self_play: %s", ex.what());
        rc = ONB_E_NOMEM;
    }
    c->gb_serial = serial;
    onb_mcts_set_noise(ctx, 0, 0.25, 0.03, 0);
    if (rc != ONB_OK) return fail(c, rc, "%s", err);
    return ONB_OK;
}
// one agent chooses for the m games in which it is to move (d_games) and leaves the actions in d_out[game]
static int32_t fight_move(Ctx* c, const onb_agent* ag, uint32_t ply, const int32_t* d_games, int64_t m, uint16_t* d_out) {
    onb_ctx* x = reinterpret_cast<onb_ctx*>(c);
    if (ag->kind == ONB_AGENT_RANDOM) {  // elementwise and cheap: chosen for every undecided game, the merge keeps this agent's games
        const int32_t rc = onb_env_choose_random(x, ply, ONB_POLICY_AGENT);
        if (rc != ONB_OK) return rc;
        ONB_CUDA(c, cudaMemcpyAsync(d_out, c->d_actions, (size_t)c->n * 2, cudaMemcpyDeviceToDevice, c->stream));
        return ONB_OK;
    }
    if (ag->kind == ONB_AGENT_ALPHABETA) {  // no tree: the kernel writes the actions of the listed games straight into d_out
        ONB_CUDA(c, launch_alphabeta(c, (int)ag->sims, d_games, m, d_out, nullptr, nullptr));
        return ONB_OK;
    }
    if (ag->kind == ONB_AGENT_TABLEBASE) {
        ONB_CUDA(c, launch_tb_best(c, d_games, m, d_out));
        return ONB_OK;
    }
    c->gb_on = 0;  // PUCT and UCT agents search without the Gumbel root step
    if (ag->kind == ONB_AGENT_GUMBEL) {
        c->gb_on = 1;
        c->gb_cfg.max_considered = ag->min_node_visits ? ag->min_node_visits : 16u;
        c->gb_cfg.c_visit = 50.0;
        c->gb_cfg.c_scale = ag->c;
        c->gb_cfg.gumbel_scale = 1.0;
        c->gb_cfg.seed = c->cfg.seed;
        c->gb_serial = ply;
    }
    int32_t rc = mcts_begin_subset(c, ag->kind == ONB_AGENT_GUMBEL ? 2.0 : ag->c, ag->sims, d_games, m);
    if (rc != ONB_OK) return rc;
    if (ag->kind == ONB_AGENT_PUCT || ag->kind == ONB_AGENT_GUMBEL) {
        if (ag->evaluator == ONB_EVAL_NET && (rc = onb_net_select(x, ag->net_slot)) != ONB_OK) return rc;
        rc = onb_mcts_run(x, ag->evaluator, ag->sims);
    } else {
        rc = onb_uct_run(x, (float)ag->c, ag->min_node_visits, ag->sims);
    }
    if (rc == ONB_OK) rc = onb_mcts_finish(x, nullptr, nullptr, nullptr, nullptr, nullptr);
    if (rc != ONB_OK) return rc;
    // the chosen moves become the agent's actions (ONB_ACTION_NONE for decided roots)
    ONB_CUDA(c, launch_mcts_scatter_best(c, d_out));
    return ONB_OK;
}
int32_t onb_fight(onb_ctx* ctx, const onb_agent* a, const onb_agent* b, const uint8_t* a_is_red_host, uint32_t max_plies, onb_fight_result* out,
                  uint8_t* results_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!a || !b || !a_is_red_host || !out) return fail(c, ONB_E_INVALID, "onb_fight: null argument");
    for (const onb_agent* ag : {a, b}) {
        if (ag->kind != ONB_AGENT_RANDOM && ag->kind != ONB_AGENT_PUCT && ag->kind != ONB_AGENT_UCT && ag->kind != ONB_AGENT_ALPHABETA &&
            ag->kind != ONB_AGENT_GUMBEL && ag->kind != ONB_AGENT_TABLEBASE)
            return fail(c, ONB_E_INVALID, "onb_fight: unknown agent kind %d", ag->kind);
        if (ag->kind == ONB_AGENT_TABLEBASE) {
            if (!c->tb_live) return fail(c, ONB_E_STATE, "onb_fight: a tablebase agent needs a solved table (onb_tb_solve)");
            continue;
        }
        if (ag->kind == ONB_AGENT_GUMBEL && (ag->min_node_visits > 40 || !std::isfinite(ag->c) || !(ag->c >= 0.0)))
            return fail(c, ONB_E_INVALID, "onb_fight: a Gumbel agent needs min_node_visits (m) <= 40 and a finite c (c_scale) >= 0");
        if (ag->kind == ONB_AGENT_ALPHABETA) {
            if (ag->sims < 1 || ag->sims > ONB_ALPHABETA_MAX_DEPTH)
                return fail(c, ONB_E_INVALID, "onb_fight: an alpha-beta agent needs 1 <= depth (sims) <= %d", ONB_ALPHABETA_MAX_DEPTH);
            continue;
        }
        if (ag->kind != ONB_AGENT_RANDOM && (!c->d_nodes || ag->sims == 0 || ag->sims > c->cfg.mcts_max_sims))
            return fail(c, ONB_E_INVALID, "onb_fight: a searching agent needs 1 <= sims <= mcts_max_sims");
    }
    if (a->kind == ONB_AGENT_TABLEBASE || b->kind == ONB_AGENT_TABLEBASE) {  // games stay in the table once they start in it
        unsigned long long* d_missing = nullptr;
        unsigned long long missing = 0;
        ONB_CUDA(c, dalloc(&d_missing, 1));
        cudaError_t e = cudaMemsetAsync(d_missing, 0, 8, c->stream);
        if (e == cudaSuccess) e = launch_tb_probe(c, nullptr, d_missing);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&missing, d_missing, 8, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(d_missing);
        ONB_CUDA(c, e);
        if (missing)
            return fail(c, ONB_E_INVALID, "onb_fight: %llu undecided games are not positions of the tablebase (card set or material)", missing);
    }
    memset(out, 0, sizeof(*out));
    int32_t rc = onb_mcts_set_noise(ctx, 0, 0.25, 0.03, 0);  // arenas search in eval mode (AlphaZeroMcts, not TrainingAlphaZeroMcts)
    if (rc != ONB_OK) return rc;
    const int gb_on = c->gb_on;  // the agents set the Gumbel switch per move; the context's own setting comes back afterwards
    const onb_gumbel_config gb_cfg = c->gb_cfg;
    const uint32_t gb_serial = c->gb_serial;
    if (a->kind == ONB_AGENT_GUMBEL || b->kind == ONB_AGENT_GUMBEL) {
        onb_gumbel_config on;
        memset(&on, 0, sizeof(on));
        on.enabled = 1;
        on.max_considered = 16;
        if ((rc = onb_mcts_set_gumbel(ctx, &on)) != ONB_OK) return rc;  // allocates the Gumbel buffers; the context's setting is restored below
        c->gb_on = gb_on;
        c->gb_cfg = gb_cfg;
        c->gb_serial = gb_serial;
    }
    char err[400];
    err[0] = 0;
    rc = run_fight(c, a, b, a_is_red_host, max_plies, out, fight_move, err, sizeof(err));
    c->gb_on = gb_on;
    c->gb_cfg = gb_cfg;
    c->gb_serial = gb_serial;
    if (rc != ONB_OK) return fail(c, rc, "%s", err);
    if (results_host) {
        ONB_CUDA(c, cudaMemcpyAsync(results_host, out->results, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return ONB_OK;
}
int32_t onb_fight_stats(onb_ctx* ctx, double rating_a, double rating_b, onb_fight_statistics* out, double* history_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!out) return fail(c, ONB_E_INVALID, "onb_fight_stats: null output");
    memset(out, 0, sizeof(*out));
    char err[400];
    err[0] = 0;
    const int32_t rc = run_fight_statistics(c, rating_a, rating_b, out, history_host, err, sizeof(err));
    if (rc != ONB_OK) return fail(c, rc, "%s", err);
    return ONB_OK;
}
int32_t onb_copy_to_host(onb_ctx* ctx, void* host, const void* device, int64_t bytes) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!host || !device || bytes < 0) return fail(c, ONB_E_INVALID, "onb_copy_to_host: bad arguments");
    if (bytes == 0) return ONB_OK;
    ONB_CUDA(c, cudaMemcpyAsync(host, device, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}
int32_t onb_uct_run(onb_ctx* ctx, float exploration_c, uint32_t min_node_visits, uint32_t playouts) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->mcts_phase != 1) return fail(c, ONB_E_STATE, "onb_uct_run: call onb_mcts_begin first");
    if (c->ru_search) return refuse_after_reuse(c, "onb_uct_run");
    if (c->gb_search) return fail(c, ONB_E_STATE, "onb_uct_run: the search was begun with the Gumbel root search on (onb_mcts_set_gumbel)");
    if (c->sims_done + playouts > c->cfg.mcts_max_sims) return fail(c, ONB_E_INVALID, "onb_uct_run: more playouts than mcts_max_sims");
    const uint32_t need = c->sims_done + playouts + 2;
    if (c->ln_cap < need) {  // ln(parent visits) as the reference computes it: f32 logf on the host
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
        if (c->d_ln_table) cudaFree(c->d_ln_table);
        c->d_ln_table = nullptr;
        c->ln_cap = 0;
        const uint32_t cap = need < c->cfg.mcts_max_sims + 2 ? c->cfg.mcts_max_sims + 2 : need;
        float* host = static_cast<float*>(malloc((size_t)cap * 4));
        if (!host) return fail(c, ONB_E_NOMEM, "onb_uct_run: out of host memory");
        for (uint32_t i = 0; i < cap; ++i) host[i] = logf((float)i);
        cudaError_t e = cudaMalloc(&c->d_ln_table, (size_t)cap * 4);
        if (e == cudaSuccess) e = cudaMemcpy(c->d_ln_table, host, (size_t)cap * 4, cudaMemcpyHostToDevice);
        free(host);
        ONB_CUDA(c, e);
        c->ln_cap = cap;
    }
    ONB_CUDA(c, launch_uct_run(c, exploration_c, min_node_visits, playouts));
    c->sims_done += playouts;
    return ONB_OK;
}
int32_t onb_alphabeta_run(onb_ctx* ctx, int32_t depth, onb_action* best_host, int32_t* score_host, uint64_t* nodes_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (depth < 1 || depth > ONB_ALPHABETA_MAX_DEPTH) return fail(c, ONB_E_INVALID, "onb_alphabeta_run: depth %d not in 1..%d", depth, ONB_ALPHABETA_MAX_DEPTH);
    const size_t n = (size_t)c->n;
    if (score_host && !c->d_ab_score) ONB_CUDA(c, dalloc(&c->d_ab_score, n));
    if (nodes_host && !c->d_ab_nodes) ONB_CUDA(c, dalloc(&c->d_ab_nodes, n));
    ONB_CUDA(c, launch_alphabeta(c, depth, nullptr, c->n, c->d_actions, score_host ? c->d_ab_score : nullptr, nodes_host ? c->d_ab_nodes : nullptr));
    if (best_host) ONB_CUDA(c, cudaMemcpyAsync(best_host, c->d_actions, n * 2, cudaMemcpyDeviceToHost, c->stream));
    if (score_host) ONB_CUDA(c, cudaMemcpyAsync(score_host, c->d_ab_score, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (nodes_host) ONB_CUDA(c, cudaMemcpyAsync(nodes_host, c->d_ab_nodes, n * 8, cudaMemcpyDeviceToHost, c->stream));
    if (best_host || score_host || nodes_host) ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}
int32_t onb_tb_solve(onb_ctx* ctx, const uint8_t cards5[5], int32_t max_pawns, onb_tb_class out[25]) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    char err[400];
    err[0] = 0;
    const int32_t rc = tb_solve(c, cards5, max_pawns, out, err, sizeof(err));
    if (rc != ONB_OK) return fail(c, rc, "%s", err);
    return ONB_OK;
}
int32_t onb_tb_free(onb_ctx* ctx) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    tb_free(c);
    return ONB_OK;
}
int32_t onb_tb_table(onb_ctx* ctx, int32_t red_pawns, int32_t blue_pawns, int16_t** dev_ptr, int64_t* entries) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->tb_live) return fail(c, ONB_E_STATE, "onb_tb_table: no tablebase is resident (onb_tb_solve)");
    if (!dev_ptr || red_pawns < 0 || blue_pawns < 0 || red_pawns + blue_pawns > c->tb_max_pawns)
        return fail(c, ONB_E_INVALID, "onb_tb_table: class (%d,%d) is not in the table (max_pawns %d)", red_pawns, blue_pawns, c->tb_max_pawns);
    const int k = 5 * red_pawns + blue_pawns;
    *dev_ptr = c->d_tb + c->tb_off[k];
    if (entries) *entries = c->tb_len[k];
    return ONB_OK;
}
int32_t onb_tb_probe(onb_ctx* ctx, int16_t* values_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->tb_live) return fail(c, ONB_E_STATE, "onb_tb_probe: no tablebase is resident (onb_tb_solve)");
    if (!values_host) return fail(c, ONB_E_INVALID, "onb_tb_probe: null output");
    const size_t n = (size_t)c->n;
    if (!c->d_tb_values) ONB_CUDA(c, dalloc(&c->d_tb_values, n));
    ONB_CUDA(c, launch_tb_probe(c, c->d_tb_values, nullptr));
    ONB_CUDA(c, cudaMemcpyAsync(values_host, c->d_tb_values, n * 2, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}
int32_t onb_tb_best(onb_ctx* ctx, onb_action* best_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->tb_live) return fail(c, ONB_E_STATE, "onb_tb_best: no tablebase is resident (onb_tb_solve)");
    ONB_CUDA(c, launch_tb_best(c, nullptr, c->n, c->d_actions));
    if (best_host) {
        ONB_CUDA(c, cudaMemcpyAsync(best_host, c->d_actions, (size_t)c->n * 2, cudaMemcpyDeviceToHost, c->stream));
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return ONB_OK;
}
int32_t onb_mcts_finish(onb_ctx* ctx, onb_action* best_host, float* pi_host, uint32_t* root_visits_host, double* root_q_host, uint32_t* child_visits_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (c->mcts_phase != 1) return fail(c, ONB_E_STATE, "onb_mcts_finish: search not in a finished-simulation state");
    if (c->ru_search && c->ru_public) {  // finish in slot order into the scratch, then back into game order
        float* pi = c->d_pi; uint16_t* best = c->d_best; uint32_t* rv = c->d_root_visits; double* q = c->d_root_q; uint32_t* cv = c->d_child_visits;
        c->d_pi = c->d_ru_pi; c->d_best = c->d_ru_best; c->d_root_visits = c->d_ru_rv; c->d_root_q = c->d_ru_q; c->d_child_visits = c->d_ru_cv;
        const cudaError_t e = launch_mcts_finish(c);
        c->d_pi = pi; c->d_best = best; c->d_root_visits = rv; c->d_root_q = q; c->d_child_visits = cv;
        ONB_CUDA(c, e);
        ONB_CUDA(c, launch_reuse_unpermute(c));
    } else {
        ONB_CUDA(c, launch_mcts_finish(c));
    }
    const size_t n = (size_t)c->n;
    bool any = false;
    if (best_host) { ONB_CUDA(c, cudaMemcpyAsync(best_host, c->d_best, n * 2, cudaMemcpyDeviceToHost, c->stream)); any = true; }
    if (pi_host) { ONB_CUDA(c, cudaMemcpyAsync(pi_host, c->d_pi, n * 200, cudaMemcpyDeviceToHost, c->stream)); any = true; }
    if (root_visits_host) { ONB_CUDA(c, cudaMemcpyAsync(root_visits_host, c->d_root_visits, n * 4, cudaMemcpyDeviceToHost, c->stream)); any = true; }
    if (root_q_host) { ONB_CUDA(c, cudaMemcpyAsync(root_q_host, c->d_root_q, n * 8, cudaMemcpyDeviceToHost, c->stream)); any = true; }
    if (child_visits_host) { ONB_CUDA(c, cudaMemcpyAsync(child_visits_host, c->d_child_visits, n * 160, cudaMemcpyDeviceToHost, c->stream)); any = true; }
    if (any) ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}
int32_t onb_mcts_play_best(onb_ctx* ctx, uint32_t out_flags) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_best) return fail(c, ONB_E_STATE, "onb_mcts_play_best: no search buffers");
    if ((out_flags & ONB_OUT_PLANES) && !c->d_planes) return fail(c, ONB_E_STATE, "onb_mcts_play_best: plane buffer not allocated");
    ONB_CUDA(c, launch_mcts_play_best(c, out_flags));
    c->mcts_phase = 0;
    return ONB_OK;
}
int32_t onb_mcts_dump_tree(onb_ctx* ctx, int64_t tree, int64_t cap, onb_tree_dump* out, int64_t* n_nodes) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_nodes || tree < 0 || tree >= c->n || !out) return fail(c, ONB_E_INVALID, "onb_mcts_dump_tree: bad arguments");
    uint32_t size = 0;
    if (c->ru_live) {  // trees laid out by budget: `tree` is a game; a game without a remembered tree has none (0 nodes)
        int32_t slot = -1;
        ONB_CUDA(c, cudaMemcpyAsync(&slot, c->d_ru_slot + tree, 4, cudaMemcpyDeviceToHost, c->stream));
        ONB_CUDA(c, cudaStreamSynchronize(c->stream));
        if (slot < 0) {
            if (n_nodes) *n_nodes = 0;
            return ONB_OK;
        }
        tree = slot;
    }
    ONB_CUDA(c, cudaMemcpyAsync(&size, c->d_tree_size + tree, 4, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_nodes) *n_nodes = size;
    if ((int64_t)size > cap) return fail(c, ONB_E_OVERFLOW, "onb_mcts_dump_tree: tree has %u nodes, cap %lld", size, (long long)cap);
    Node* h = (Node*)malloc((size_t)size * sizeof(Node));
    if (!h) return fail(c, ONB_E_NOMEM, "onb_mcts_dump_tree: host allocation failed");
    cudaError_t e = cudaMemcpyAsync(h, c->d_nodes + (size_t)tree * c->node_cap, (size_t)size * sizeof(Node), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { free(h); return cuda_fail(c, e, "onb_mcts_dump_tree"); }
    for (uint32_t i = 0; i < size; ++i) {
        if (out->visits) out->visits[i] = h[i].n;
        if (out->reward) out->reward[i] = h[i].w;
        if (out->prior) out->prior[i] = h[i].p;
        if (out->action) out->action[i] = h[i].action;
        if (out->parent) out->parent[i] = (int32_t)h[i].parent;
        if (out->first_child) out->first_child[i] = h[i].first_child;
        if (out->n_child) out->n_child[i] = h[i].n_child;
        if (out->flags) out->flags[i] = h[i].flags;
    }
    free(h);
    return ONB_OK;
}
// onb_mcts_tree_info with the trees laid out by budget: gathered into game order on the host (0 nodes for a game without a tree)
static int32_t reuse_tree_info(Ctx* c, uint32_t* n_nodes_host, uint8_t* flags_host) {
    const size_t n = (size_t)c->n;
    uint32_t* size = static_cast<uint32_t*>(malloc(n * 4));
    uint8_t* flags = static_cast<uint8_t*>(malloc(n));
    int32_t* slot = static_cast<int32_t*>(malloc(n * 4));
    cudaError_t e = (size && flags && slot) ? cudaSuccess : cudaErrorMemoryAllocation;
    if (e == cudaSuccess) e = cudaMemcpyAsync(size, c->d_tree_size, n * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(flags, c->d_tree_flags, n, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(slot, c->d_ru_slot, n * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess)
        for (size_t g = 0; g < n; ++g) {
            if (n_nodes_host) n_nodes_host[g] = slot[g] >= 0 ? size[slot[g]] : 0u;
            if (flags_host) flags_host[g] = slot[g] >= 0 ? flags[slot[g]] : (uint8_t)0;
        }
    free(size);
    free(flags);
    free(slot);
    if (e != cudaSuccess) return cuda_fail(c, e, "onb_mcts_tree_info");
    return ONB_OK;
}
int32_t onb_mcts_tree_info(onb_ctx* ctx, uint32_t* n_nodes_host, uint8_t* flags_host) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->d_nodes) return fail(c, ONB_E_STATE, "onb_mcts_tree_info: no search buffers");
    if (c->ru_live) return reuse_tree_info(c, n_nodes_host, flags_host);
    if (n_nodes_host) ONB_CUDA(c, cudaMemcpyAsync(n_nodes_host, c->d_tree_size, (size_t)c->n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (flags_host) ONB_CUDA(c, cudaMemcpyAsync(flags_host, c->d_tree_flags, (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    ONB_CUDA(c, cudaStreamSynchronize(c->stream));
    return ONB_OK;
}

int32_t onb_net_precision(onb_ctx* ctx, int32_t mode) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (mode != ONB_NET_F16 && mode != ONB_NET_TF32 && mode != ONB_NET_F32) return fail(c, ONB_E_INVALID, "onb_net_precision: unknown mode %d", mode);
    c->net_tf32 = mode;
    return ONB_OK;
}
int32_t onb_net_select(onb_ctx* ctx, int32_t slot) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (slot != 0 && slot != 1) return fail(c, ONB_E_INVALID, "onb_net_select: slot %d (two networks can be resident: 0, 1)", slot);
    c->net_cur = slot;
    return ONB_OK;
}
int32_t onb_net_load(onb_ctx* ctx, int32_t n_tensors, const char* const* names, const float* const* data, const int64_t* numel) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (n_tensors <= 0 || !names || !data || !numel) return fail(c, ONB_E_INVALID, "onb_net_load: null argument");
    std::string err;
    int32_t rc = ONB_E_INVALID;
    try {
        rc = net_load(c, n_tensors, names, data, numel, err);
    } catch (const std::exception& ex) {  // nothing may cross the C boundary
        err = ex.what();
        rc = ONB_E_NOMEM;
    }
    if (rc != ONB_OK) return fail(c, rc, "onb_net_load: %s", err.c_str());
    return ONB_OK;
}
int32_t onb_net_forward(onb_ctx* ctx, int32_t planes_buffer) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (!c->net[c->net_cur].loaded) return fail(c, ONB_E_STATE, "onb_net_forward: no network loaded (onb_net_load)");
    const float* planes = planes_buffer == ONB_BUF_LEAF_PLANES ? c->d_leaf_planes : planes_buffer == ONB_BUF_PLANES ? c->d_planes : nullptr;
    if (planes_buffer != ONB_BUF_LEAF_PLANES && planes_buffer != ONB_BUF_PLANES) return fail(c, ONB_E_INVALID, "onb_net_forward: not a plane buffer");
    if (!planes || !c->d_policy) return fail(c, ONB_E_STATE, "onb_net_forward: plane or policy/value buffers were not allocated by onb_create");
    ONB_CUDA(c, launch_net_forward(c, planes, c->d_policy, c->d_value, c->n));
    return ONB_OK;
}

int32_t onb_selftest(onb_ctx* ctx, int32_t which, uint64_t* mismatches) {
    ONB_CHECK_CTX(ctx);
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    if (which != ONB_SELFTEST_DIV) return fail(c, ONB_E_INVALID, "onb_selftest: unknown test");
    if (!mismatches) return fail(c, ONB_E_INVALID, "onb_selftest: null output");
    unsigned long long* d = nullptr;
    ONB_CUDA(c, cudaMalloc(&d, 8));
    cudaError_t e = cudaMemsetAsync(d, 0, 8, c->stream);
    if (e == cudaSuccess) e = launch_selftest_div(c, d);
    unsigned long long h = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    ONB_CUDA(c, e);
    *mismatches = (uint64_t)h;
    return ONB_OK;
}

}  // extern "C"
