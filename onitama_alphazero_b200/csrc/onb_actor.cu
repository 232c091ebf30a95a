// onb_actor.cu -- host-acted lockstep stepping with the round trip pipelined inside the library (include/onb.h, onb_actor_*).
//
// A host-side actor (the self-play driver of train.rs:55-80 with its policy on the host) needs, per step, the actions
// going in and "what happened" coming out. Stepping the whole context as one batch serialises H2D -> kernel -> D2H ->
// host; here the context's games are cut into n_sub contiguous sub-batches, each with its own stream, pinned host
// staging and completion event, so that while the host consumes sub-batch j the other n_sub - 1 are copying or
// stepping. No torch, no Python and no stream-wide synchronisation sits on the step: the host blocks on ONE event.
//
// Bytes across PCIe per game and step: 2 (action) in; out 8 (ONB_HOST_MASKS) and/or 0.25 (ONB_HOST_DONE, two bits).
#include <cstring>
#include <new>

#include "onb_internal.h"

namespace onb {

struct ActorSub {
    int64_t first, count;
    cudaStream_t stream;
    cudaEvent_t done;       // recorded after the sub-batch's last D2H copy
    uint32_t* d_done;       // [count/32][2] device
    // one pinned allocation: [actions u16 x count][masks u32 x 2 count][done u32 x 2 (count/32)][stats u64 x ONB_STAT_COUNT]
    uint8_t* h_block;
    onb_action* h_actions;
    uint32_t* h_masks;
    uint32_t* h_done;
    uint64_t* h_stats;
    bool in_flight;
};

struct Actor {
    Ctx* c;
    int n_sub;
    uint32_t out_flags, host_flags;
    cudaEvent_t fork;       // orders the sub-batch streams after the work queued on the context's stream
    bool forked;
    ActorSub* sub;
};

static int32_t actor_fail(Ctx* c, int32_t code, const char* what, cudaError_t e) {
    if (e != cudaSuccess) snprintf(c->err, sizeof(c->err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    else snprintf(c->err, sizeof(c->err), "%s", what);
    return code;
}
#define ACT_CUDA(c, call)                                                      \
    do {                                                                       \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess) return actor_fail(c, ONB_E_CUDA, #call, e__);  \
    } while (0)

struct ActorDeviceGuard {
    int prev = -1, mine;
    explicit ActorDeviceGuard(int dev) : mine(dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != mine) cudaSetDevice(mine);
    }
    ~ActorDeviceGuard() {
        if (prev >= 0 && prev != mine) cudaSetDevice(prev);
    }
};

static void actor_free(Actor* a) {
    if (!a) return;
    if (a->sub) {
        for (int j = 0; j < a->n_sub; ++j) {
            ActorSub& s = a->sub[j];
            if (s.stream) { cudaStreamSynchronize(s.stream); cudaStreamDestroy(s.stream); }
            if (s.done) cudaEventDestroy(s.done);
            if (s.d_done) cudaFree(s.d_done);
            if (s.h_block) cudaFreeHost(s.h_block);
        }
        delete[] a->sub;
    }
    if (a->fork) cudaEventDestroy(a->fork);
    delete a;
}

// first use after creation / after onb_actor_join: the sub-batch streams start behind whatever the context's stream holds
static cudaError_t actor_fork(Actor* a) {
    if (a->forked) return cudaSuccess;
    cudaError_t e = cudaEventRecord(a->fork, a->c->stream);
    for (int j = 0; j < a->n_sub && e == cudaSuccess; ++j) e = cudaStreamWaitEvent(a->sub[j].stream, a->fork, 0);
    if (e == cudaSuccess) a->forked = true;
    return e;
}

}  // namespace onb

using namespace onb;

extern "C" {

int32_t onb_actor_create(onb_ctx* ctx, int32_t n_sub, uint32_t out_flags, uint32_t host_flags, onb_actor** out) {
    if (!ctx || !out) return ONB_E_INVALID;
    Ctx* c = reinterpret_cast<Ctx*>(ctx);
    *out = nullptr;
    ActorDeviceGuard guard(c->cfg.device);
    if (n_sub < 1 || n_sub > 64) return actor_fail(c, ONB_E_INVALID, "onb_actor_create: n_sub must be in 1..64", cudaSuccess);
    if (host_flags & ~(ONB_HOST_MASKS | ONB_HOST_DONE | ONB_HOST_STATS)) return actor_fail(c, ONB_E_INVALID, "onb_actor_create: unknown host_flags", cudaSuccess);
    if ((out_flags & ONB_OUT_PLANES) && !c->d_planes) return actor_fail(c, ONB_E_STATE, "onb_actor_create: plane buffer not allocated", cudaSuccess);
    if (host_flags & ONB_HOST_MASKS) out_flags |= ONB_OUT_MASKS;
    Actor* a = new (std::nothrow) Actor();
    if (!a) return ONB_E_NOMEM;
    memset(a, 0, sizeof(*a));
    a->c = c;
    a->n_sub = n_sub;
    a->out_flags = out_flags;
    a->host_flags = host_flags;
    a->sub = new (std::nothrow) ActorSub[n_sub];
    if (!a->sub) { delete a; return ONB_E_NOMEM; }
    memset(a->sub, 0, sizeof(ActorSub) * (size_t)n_sub);
    cudaError_t e = cudaEventCreateWithFlags(&a->fork, cudaEventDisableTiming);
    // sub-batch boundaries on multiples of 64 games: plane tiles stay 16-byte aligned, done words stay whole
    const int64_t n = c->n, chunks = (n + 63) / 64;
    for (int j = 0; j < n_sub && e == cudaSuccess; ++j) {
        ActorSub& s = a->sub[j];
        const int64_t lo = chunks * j / n_sub * 64, hi = chunks * (j + 1) / n_sub * 64;
        s.first = lo < n ? lo : n;
        s.count = (hi < n ? hi : n) - s.first;
        e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming);
        const size_t words = (size_t)((s.count + 31) / 32) * 2;
        const size_t b_act = ((size_t)s.count * 2 + 63) & ~(size_t)63, b_mask = (size_t)s.count * 8, b_done = (words * 4 + 63) & ~(size_t)63,
                     b_stats = ONB_STAT_COUNT * 8;
        if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&s.h_block), b_act + b_mask + b_done + b_stats + 64, cudaHostAllocPortable);
        if (e == cudaSuccess) {
            memset(s.h_block, 0, b_act + b_mask + b_done + b_stats + 64);
            s.h_actions = reinterpret_cast<onb_action*>(s.h_block);
            s.h_masks = reinterpret_cast<uint32_t*>(s.h_block + b_act);
            s.h_done = reinterpret_cast<uint32_t*>(s.h_block + b_act + b_mask);
            s.h_stats = reinterpret_cast<uint64_t*>(s.h_block + b_act + b_mask + b_done);
            if (words) e = cudaMalloc(reinterpret_cast<void**>(&s.d_done), words * 4);
        }
    }
    if (e != cudaSuccess) {
        actor_free(a);
        return actor_fail(c, e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA, "onb_actor_create", e);
    }
    *out = reinterpret_cast<onb_actor*>(a);
    return ONB_OK;
}

int32_t onb_actor_destroy(onb_actor* actor) {
    if (!actor) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    ActorDeviceGuard guard(a->c->cfg.device);
    actor_free(a);
    return ONB_OK;
}

int32_t onb_actor_get_view(onb_actor* actor, int32_t sub, onb_actor_view* view) {
    if (!actor || !view) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    if (sub < 0 || sub >= a->n_sub) return actor_fail(a->c, ONB_E_INVALID, "onb_actor_get_view: no such sub-batch", cudaSuccess);
    const ActorSub& s = a->sub[sub];
    view->first = s.first;
    view->count = s.count;
    view->actions = s.h_actions;
    view->masks = (a->host_flags & ONB_HOST_MASKS) ? s.h_masks : nullptr;
    view->done = (a->host_flags & ONB_HOST_DONE) ? s.h_done : nullptr;
    view->stats = (a->host_flags & ONB_HOST_STATS) ? s.h_stats : nullptr;
    return ONB_OK;
}

int32_t onb_actor_submit(onb_actor* actor, int32_t sub, const onb_action* actions_host, uint32_t step, int32_t auto_reset) {
    if (!actor) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    Ctx* c = a->c;
    if (sub < 0 || sub >= a->n_sub) return actor_fail(c, ONB_E_INVALID, "onb_actor_submit: no such sub-batch", cudaSuccess);
    ActorSub& s = a->sub[sub];
    if (s.in_flight) return actor_fail(c, ONB_E_STATE, "onb_actor_submit: the sub-batch is in flight (onb_actor_wait first)", cudaSuccess);
    ActorDeviceGuard guard(c->cfg.device);
    ACT_CUDA(c, actor_fork(a));
    if (s.count > 0) {
        const onb_action* src = actions_host ? actions_host : s.h_actions;
        ACT_CUDA(c, cudaMemcpyAsync(c->d_actions + s.first, src, (size_t)s.count * sizeof(onb_action), cudaMemcpyHostToDevice, s.stream));
        ACT_CUDA(c, launch_env_step_slice(c, kModeActions, step, auto_reset, a->out_flags, s.first, s.count, s.stream,
                                          (a->host_flags & ONB_HOST_DONE) ? s.d_done : nullptr));
        if (a->host_flags & ONB_HOST_MASKS)
            ACT_CUDA(c, cudaMemcpyAsync(s.h_masks, c->d_masks + 2 * s.first, (size_t)s.count * 8, cudaMemcpyDeviceToHost, s.stream));
        if (a->host_flags & ONB_HOST_DONE)
            ACT_CUDA(c, cudaMemcpyAsync(s.h_done, s.d_done, (size_t)((s.count + 31) / 32) * 8, cudaMemcpyDeviceToHost, s.stream));
    }
    if (a->host_flags & ONB_HOST_STATS) ACT_CUDA(c, cudaMemcpyAsync(s.h_stats, c->d_stats, ONB_STAT_COUNT * 8, cudaMemcpyDeviceToHost, s.stream));
    ACT_CUDA(c, cudaEventRecord(s.done, s.stream));
    s.in_flight = true;
    c->search.phase = 0;
    return ONB_OK;
}

int32_t onb_actor_wait(onb_actor* actor, int32_t sub) {
    if (!actor) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    Ctx* c = a->c;
    if (sub < 0 || sub >= a->n_sub) return actor_fail(c, ONB_E_INVALID, "onb_actor_wait: no such sub-batch", cudaSuccess);
    ActorSub& s = a->sub[sub];
    if (!s.in_flight) return ONB_OK;
    ACT_CUDA(c, cudaEventSynchronize(s.done));
    s.in_flight = false;
    return ONB_OK;
}

int32_t onb_actor_join(onb_actor* actor) {
    if (!actor) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    Ctx* c = a->c;
    ActorDeviceGuard guard(c->cfg.device);
    if (!a->forked) return ONB_OK;
    for (int j = 0; j < a->n_sub; ++j) {
        ActorSub& s = a->sub[j];
        if (!s.in_flight) ACT_CUDA(c, cudaEventRecord(s.done, s.stream));
        ACT_CUDA(c, cudaStreamWaitEvent(c->stream, s.done, 0));
    }
    a->forked = false;
    return ONB_OK;
}

// The whole loop without a host policy: n_steps steps, the action of game g at step t read from trace_host[t * stride + g].
// This is the ring a host actor drives with submit/wait, run by the library itself (replay of recorded games, and the
// measurement of what the pipeline sustains when the host adds no think time).
int32_t onb_actor_replay(onb_actor* actor, const onb_action* trace_host, int64_t stride, uint32_t step0, uint32_t n_steps, int32_t auto_reset) {
    if (!actor) return ONB_E_INVALID;
    Actor* a = reinterpret_cast<Actor*>(actor);
    if (!trace_host || stride < a->c->n) return actor_fail(a->c, ONB_E_INVALID, "onb_actor_replay: bad trace", cudaSuccess);
    for (uint32_t t = 0; t < n_steps; ++t)
        for (int j = 0; j < a->n_sub; ++j) {
            int32_t rc = onb_actor_wait(actor, j);  // the host "has" the outputs of step t-1 of this sub-batch
            if (rc == ONB_OK) rc = onb_actor_submit(actor, j, trace_host + (int64_t)t * stride + a->sub[j].first, step0 + t, auto_reset);
            if (rc != ONB_OK) return rc;
        }
    for (int j = 0; j < a->n_sub; ++j) {
        int32_t rc = onb_actor_wait(actor, j);
        if (rc != ONB_OK) return rc;
    }
    return ONB_OK;
}

}  // extern "C"
