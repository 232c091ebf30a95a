// onb_selfplay.cu -- self_play (alphazero-training/src/train.rs:35-98) for all games of a context, natively: search, sample
// recording, move, game-over bookkeeping and the restart of finished slots all stay on the device; the host only reads one counter
// per ply to know when the requested number of games is complete. A worker of the reference plays its games one after the other
// (train.rs:218-245); here every slot starts its next game the moment the previous one is over, so all slots stay busy.
//
// Sample i = tick * n + slot (ply-major, every slot records every ply): planes = create_tensor_from_state of the searched position
// (train.rs:58), pi = the search's visit distribution, colour = side to move, serial = slot + n * (games already finished in the
// slot). When a game ends, z = reward(final result, sample colour) (train.rs:83-85, alphazero_mcts/mod.rs:45-53; 0 for a game cut
// at the ply cap) is written to the game's samples (the last `plies` samples of the slot: i, i - n, i - 2n, ...) and they become
// valid; samples of games still running when the quota is reached stay invalid.
#include <cstring>
#include <vector>

#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {
namespace {

__global__ void __launch_bounds__(256) k_sp_record(const uint4* __restrict__ states, int64_t n, const int32_t* __restrict__ generation, int64_t base,
                                                   uint8_t* __restrict__ color, int64_t* __restrict__ serial, uint8_t* __restrict__ valid,
                                                   float* __restrict__ z) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const Game g = unpack(states[s]);
    color[base + s] = (uint8_t)g.side;
    serial[base + s] = s + n * (int64_t)generation[s];
    valid[base + s] = 0;
    z[base + s] = 0.f;
}

// ---- deterministic stream compaction: idx[0 .. m) = ascending indices i with flags[i] != 0, *total = m -----------------------------
// Three small launches (count per 256-item block, single-block exclusive scan of the block counts, scatter); ascending order makes
// every consumer (which trees search which games, which finished slots are re-dealt first) independent of atomics' timing.
__global__ void __launch_bounds__(256) k_compact_count(const uint8_t* __restrict__ flags, int64_t n, uint32_t* __restrict__ block_counts) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int c = __syncthreads_count(i < n && flags[i] != 0);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = (uint32_t)c;
}
__global__ void __launch_bounds__(1024) k_compact_scan(uint32_t* __restrict__ block_counts, int nb, unsigned long long* __restrict__ total) {
    __shared__ uint32_t s_part[1024];
    const int per = (nb + 1023) / 1024, lo = threadIdx.x * per, hi = min(lo + per, nb);
    uint32_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += block_counts[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan of the 1024 partial sums
        const uint32_t v = threadIdx.x >= (unsigned)o ? s_part[threadIdx.x - o] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = s_part[threadIdx.x] - sum;  // exclusive prefix of this thread's chunk
    for (int i = lo; i < hi; ++i) {
        const uint32_t c = block_counts[i];
        block_counts[i] = run;
        run += c;
    }
    if (threadIdx.x == 1023) *total = (unsigned long long)s_part[1023];
}
__global__ void __launch_bounds__(256) k_compact_scatter(const uint8_t* __restrict__ flags, int64_t n, const uint32_t* __restrict__ block_offs,
                                                         int32_t* __restrict__ idx) {
    __shared__ uint32_t s_warp[8];
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const bool f = i < n && flags[i] != 0;
    const unsigned b = __ballot_sync(0xFFFFFFFFu, f);
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    if (lane == 0) s_warp[w] = __popc(b);
    __syncthreads();
    uint32_t off = block_offs[blockIdx.x];
    for (unsigned k = 0; k < w; ++k) off += s_warp[k];
    if (f) idx[off + __popc(b & ((1u << lane) - 1u))] = (int32_t)i;
}
cudaError_t compact(Ctx* c, const uint8_t* flags, int64_t n, uint32_t* block_counts, int32_t* idx, unsigned long long* total) {
    const int nb = (int)((n + 255) / 256);
    k_compact_count<<<nb, 256, 0, c->stream>>>(flags, n, block_counts);
    k_compact_scan<<<1, 1024, 0, c->stream>>>(block_counts, nb, total);
    k_compact_scatter<<<nb, 256, 0, c->stream>>>(flags, n, block_counts, idx);
    return cudaGetLastError();
}

// pi rows of the searched trees -> the sample rows of their games
__global__ void __launch_bounds__(256) k_scatter_rows50(const float* __restrict__ src, const int32_t* __restrict__ gid, float* __restrict__ dst, int64_t m) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m * 50) return;
    const int64_t t = e / 50;
    dst[(int64_t)gid[t] * 50 + (e - t * 50)] = src[e];
}

// self-play, after the move: which live slots' games are over (a win, or the ply cap of train.rs:74-79: max_plies counts down from 150
// and is tested after the move, so a game has at most max_plies + 2 plies)
__global__ void __launch_bounds__(256) k_sp_over(const uint4* __restrict__ states, int64_t n, const uint8_t* __restrict__ idle, int32_t* __restrict__ plies,
                                                 uint32_t max_plies, uint8_t* __restrict__ over) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint8_t o = 0;
    if (!idle[s]) {
        const int32_t p = plies[s] + 1;
        plies[s] = p;
        o = (unpack(states[s]).result != 0 || (uint32_t)p >= max_plies + 2u) ? 1 : 0;
    }
    over[s] = o;
}
// close the finished games in slot order: z = reward(result, sample colour) (train.rs:83-85; 0 for a game cut at the cap) on the game's
// samples (this ply's and the plies - 1 before it in the same slot), mark them valid; the first (target - started) of them start their
// slot's next game at once, the others leave their slot idle: exactly `target` games are ever started and every one of them is played
// to its end (a worker of the reference plays self_play_game_amnt games to completion, train.rs:44-98)
__global__ void __launch_bounds__(256) k_sp_finish(uint4* __restrict__ states, int64_t n, const int32_t* __restrict__ over_list,
                                                   const unsigned long long* __restrict__ n_over, int32_t* __restrict__ generation,
                                                   int32_t* __restrict__ plies, uint8_t* __restrict__ idle, uint8_t* __restrict__ live, int64_t base,
                                                   const uint8_t* __restrict__ color, uint8_t* __restrict__ valid, float* __restrict__ z, int64_t started,
                                                   int64_t target, int32_t fixed_cards, uint64_t seed, uint64_t game0, uint32_t epoch) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (int64_t)*n_over) return;
    const int64_t s = over_list[j];
    const Game g = unpack(states[s]);
    const int32_t p = plies[s];
    for (int32_t k = 0; k < p; ++k) {
        const int64_t i = base + s - (int64_t)k * n;
        z[i] = g.result == 0 ? 0.f : ((g.result - 1u) == (uint32_t)color[i] ? 1.f : -1.f);
        valid[i] = 1;
    }
    plies[s] = 0;
    if (started + j < target) {
        states[s] = pack(start_game(fixed_cards >= 0 ? (uint32_t)fixed_cards : deal_cards(game_key(seed, game0 + (uint64_t)s), epoch)));
        generation[s] += 1;
    } else {
        idle[s] = 1;
        live[s] = 0;
    }
}

// arena: who moves where. fa[i] / fb[i] = game i is undecided and agent A / B is to move (A moves when the side to move is its colour)
__global__ void __launch_bounds__(256) k_fight_plan(const uint4* __restrict__ states, int64_t n, const uint8_t* __restrict__ a_is_red,
                                                    uint8_t* __restrict__ fa, uint8_t* __restrict__ fb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Game g = unpack(states[i]);
    const bool live = g.result == 0, a_to_move = (g.side == 0u) == (a_is_red[i] != 0);
    fa[i] = live && a_to_move;
    fb[i] = live && !a_to_move;
}
// the action of the agent whose turn it is (evaluator.rs:379: agents[state.curr_agent_idx].generate_move)
__global__ void __launch_bounds__(256) k_fight_merge(const uint8_t* __restrict__ fa, const uint8_t* __restrict__ fb, int64_t n,
                                                     const uint16_t* __restrict__ act_a, const uint16_t* __restrict__ act_b, uint16_t* __restrict__ actions) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    actions[i] = fa[i] ? act_a[i] : (fb[i] ? act_b[i] : (uint16_t)0xFFFFu);
}
__global__ void __launch_bounds__(256) k_fight_tally(const uint4* __restrict__ states, int64_t n, const uint8_t* __restrict__ a_is_red,
                                                     uint8_t* __restrict__ results, unsigned long long* __restrict__ tally) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = unpack(states[i]).result;
    results[i] = (uint8_t)r;
    if (r == 0) atomicAdd(&tally[2], 1ull);                                             // draw: the ply cap ended the game
    else atomicAdd(&tally[((r == 1u) == (a_is_red[i] != 0)) ? 0 : 1], 1ull);            // agent A wins when its colour won
}

// FightStatistics::update folded over the games IN GAME ORDER (evaluator.rs:58-110; EloRating::elo_change, elo_rating.rs:53-70, K = 32):
// the Elo update of game i starts from the ratings game i - 1 left, so this is a sequential fold by construction -- one thread
// walks the results (a few hundred cycles per game). out: [0..2] W/L/D of agent A, [3..5] as Red, [6..8] as Blue; ratings: final
// (rating_a, rating_b); history (optional): [n][4] = before_a, after_a, before_b, after_b.
__global__ void k_elo_fold(const uint8_t* __restrict__ results, const uint8_t* __restrict__ a_is_red, int64_t n, double ra, double rb,
                           unsigned long long* __restrict__ out, double* __restrict__ ratings, double* __restrict__ history) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    unsigned long long cnt[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t r = results[i], color = a_is_red[i] ? 0u : 1u;
        const double ba = ra, bb = rb;
        int kind = 2;  // draw
        if (r == 1u || r == 2u) {
            const bool a_win = (r - 1u) == color;
            const double ea = 1.0 / (1.0 + pow(10.0, 2.5e-3 * (rb - ra))), eb = 1.0 / (1.0 + pow(10.0, 2.5e-3 * (ra - rb)));
            const double sa = a_win ? 1.0 : 0.0, sb = 1.0 - sa;
            ra = ba + 32.0 * (sa - ea);
            rb = bb + 32.0 * (sb - eb);
            kind = a_win ? 0 : 1;
        }
        cnt[kind] += 1;
        cnt[3 + 3 * color + kind] += 1;
        if (history) { history[4 * i + 0] = ba; history[4 * i + 1] = ra; history[4 * i + 2] = bb; history[4 * i + 3] = rb; }
    }
    for (int k = 0; k < 9; ++k) out[k] = cnt[k];
    ratings[0] = ra;
    ratings[1] = rb;
}

cudaError_t grow(Ctx* c, int slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 16;
    if (c->sp_cap[slot] < bytes) {
        if (c->sp_buf[slot]) cudaFree(c->sp_buf[slot]);
        c->sp_buf[slot] = nullptr;
        c->sp_cap[slot] = 0;
        const cudaError_t e = cudaMalloc(&c->sp_buf[slot], bytes);
        if (e != cudaSuccess) return e;
        c->sp_cap[slot] = bytes;
    }
    *out = c->sp_buf[slot];
    return cudaSuccess;
}

}  // namespace

// scratch slots of Ctx::sp_buf (grow-only). The arena has its own slots: the pointers an onb_selfplay_result hands out stay valid
// until the next onb_self_play even if an onb_fight runs in between.
enum : int {
    kSpPlanes = 0, kSpPi, kSpZ, kSpColor, kSpValid, kSpSerial, kSpGeneration, kSpPlies, kSpCounters, kSpValidIdx, kSpIdle, kSpLive, kSpOver,
    kSpLiveList, kSpOverList, kSpBlocks,
    kFtMask = 16, kFtResults, kFtActA, kFtActB, kFtCounters, kFtFlagA, kFtFlagB, kFtListA, kFtListB, kFtBlocks, kFtElo, kFtHistory
};
static_assert(kFtHistory < 32, "Ctx::sp_buf has 32 slots");

// Returns ONB_OK, or an ONB_E_* code with `err` filled. `search` runs one search (begin / run / finish) over the m games listed in
// d_games (device, ascending; nullptr = all games of the context).
int32_t run_self_play(Ctx* c, const onb_selfplay_config* cfg, onb_selfplay_result* out,
                      int32_t (*search)(Ctx*, const onb_selfplay_config*, const int32_t*, int64_t), char* err, size_t err_len) {
    const int64_t n = c->n;
    const int64_t cap_ticks = cfg->sample_cap / n;
    if (cap_ticks < 1) {
        snprintf(err, err_len, "onb_self_play: sample_cap %lld is smaller than one ply of %lld games", (long long)cfg->sample_cap, (long long)n);
        return ONB_E_INVALID;
    }
    const size_t cap = (size_t)cap_ticks * (size_t)n;
    float *planes = nullptr, *pi = nullptr, *z = nullptr;
    uint8_t *color = nullptr, *valid = nullptr, *idle = nullptr, *live = nullptr, *over = nullptr;
    int64_t *serial = nullptr, *idx = nullptr;
    int32_t *generation = nullptr, *plies = nullptr, *live_list = nullptr, *over_list = nullptr;
    uint32_t* blocks = nullptr;
    unsigned long long* counters = nullptr;  // [0] games over in this ply, [1] live slots after it
    cudaError_t e;
#define SP(call)                                                                       \
    do {                                                                               \
        e = (call);                                                                    \
        if (e != cudaSuccess) {                                                        \
            snprintf(err, err_len, "onb_self_play: %s: %s", #call, cudaGetErrorString(e)); \
            c->n_act = 0;                                                              \
            c->d_tree_game = nullptr;                                                  \
            return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;          \
        }                                                                              \
    } while (0)
    SP(grow(c, kSpPlanes, cap * 2100, (void**)&planes));
    SP(grow(c, kSpPi, cap * 200, (void**)&pi));
    SP(grow(c, kSpZ, cap * 4, (void**)&z));
    SP(grow(c, kSpColor, cap, (void**)&color));
    SP(grow(c, kSpValid, cap, (void**)&valid));
    SP(grow(c, kSpSerial, cap * 8, (void**)&serial));
    SP(grow(c, kSpGeneration, (size_t)n * 4, (void**)&generation));
    SP(grow(c, kSpPlies, (size_t)n * 4, (void**)&plies));
    SP(grow(c, kSpCounters, 16, (void**)&counters));
    SP(grow(c, kSpIdle, (size_t)n, (void**)&idle));
    SP(grow(c, kSpLive, (size_t)n, (void**)&live));
    SP(grow(c, kSpOver, (size_t)n, (void**)&over));
    SP(grow(c, kSpLiveList, (size_t)n * 4, (void**)&live_list));
    SP(grow(c, kSpOverList, (size_t)n * 4, (void**)&over_list));
    SP(grow(c, kSpBlocks, (size_t)((n + 255) / 256 + 1) * 4, (void**)&blocks));
    SP(cudaMemsetAsync(generation, 0, (size_t)n * 4, c->stream));
    SP(cudaMemsetAsync(plies, 0, (size_t)n * 4, c->stream));
    SP(cudaMemsetAsync(idle, 0, (size_t)n, c->stream));
    SP(cudaMemsetAsync(live, 1, (size_t)n, c->stream));
    c->fixed_cards = -1;                      // like onb_env_reset without decks: every game is dealt from the counter RNG
    SP(launch_env_reset(c, nullptr, 0, 0));
    const unsigned grid = (unsigned)((n + 255) / 256);
    // Exactly `target` games are started (every slot starts one; a slot whose game ends starts the next one while games remain to be
    // started) and ALL of them are played to the end: stopping as soon as n_games are complete would drop the games still running,
    // i.e. preferentially the long ones, and bias z / pi towards short games (the reference's workers each play their
    // self_play_game_amnt games to completion, train.rs:44-98).
    const int64_t target = cfg->n_games > n ? cfg->n_games : n;
    int64_t started = n, finished = 0, n_live = n, tick = 0;
    int truncated = 0;
    while (n_live > 0) {
        if (tick >= cap_ticks) {
            truncated = 1;
            break;
        }
        const int64_t base = tick * n;
        const bool all = n_live == n;
        SP(launch_observe(c, ONB_OUT_PLANES));  // planes of the position the search starts from (idle slots: rows stay invalid)
        SP(cudaMemcpyAsync(planes + (size_t)base * 525, c->d_planes, (size_t)n * 2100, cudaMemcpyDeviceToDevice, c->stream));
        k_sp_record<<<grid, 256, 0, c->stream>>>(c->d_states, n, generation, base, color, serial, valid, z);
        SP(cudaGetLastError());
        const int32_t rc = search(c, cfg, all ? nullptr : live_list, all ? 0 : n_live);   // only the slots with a game in progress
        if (rc != ONB_OK) {
            snprintf(err, err_len, "%s", c->err);
            c->n_act = 0;
            c->d_tree_game = nullptr;
            return rc;
        }
        if (!c->d_tree_game) {  // tree t searched game t
            SP(cudaMemcpyAsync(pi + (size_t)base * 50, c->d_pi, (size_t)n * 200, cudaMemcpyDeviceToDevice, c->stream));
        } else {                // the searched list (live_list, or with tree reuse that list ordered by remaining budget)
            const int64_t nt = trees(c);
            k_scatter_rows50<<<(unsigned)((nt * 50 + 255) / 256), 256, 0, c->stream>>>(c->d_pi, c->d_tree_game, pi + (size_t)base * 50, nt);
            SP(cudaGetLastError());
        }
        SP(cudaMemsetAsync(c->d_actions, 0xFF, (size_t)n * 2, c->stream));   // ONB_ACTION_NONE: idle slots are not stepped
        SP(launch_mcts_scatter_best(c, c->d_actions));
        SP(launch_env_step(c, kModeActions, 0, 0, 0));
        k_sp_over<<<grid, 256, 0, c->stream>>>(c->d_states, n, idle, plies, cfg->max_plies, over);
        SP(cudaGetLastError());
        SP(compact(c, over, n, blocks, over_list, counters));
        k_sp_finish<<<grid, 256, 0, c->stream>>>(c->d_states, n, over_list, counters, generation, plies, idle, live, base, color, valid, z, started, target,
                                                 c->fixed_cards, c->cfg.seed, c->cfg.game_id_base, (uint32_t)(tick + 1));
        SP(cudaGetLastError());
        SP(compact(c, live, n, blocks, live_list, counters + 1));
        unsigned long long h[2] = {0, 0};
        SP(cudaMemcpyAsync(h, counters, 16, cudaMemcpyDeviceToHost, c->stream));
        SP(cudaStreamSynchronize(c->stream));
        finished += (int64_t)h[0];
        started += (int64_t)h[0] < target - started ? (int64_t)h[0] : target - started;
        n_live = (int64_t)h[1];
        ++tick;
    }
    c->n_act = 0;
    c->d_tree_game = nullptr;
    // index list of the valid samples (ascending): flags to the host, indices back
    const size_t total = (size_t)tick * (size_t)n;
    std::vector<uint8_t> flags(total);
    std::vector<int64_t> keep;
    if (total) SP(cudaMemcpy(flags.data(), valid, total, cudaMemcpyDeviceToHost));
    keep.reserve(total);
    for (size_t i = 0; i < total; ++i)
        if (flags[i]) keep.push_back((int64_t)i);
    SP(grow(c, kSpValidIdx, keep.size() * 8, (void**)&idx));
    if (!keep.empty()) SP(cudaMemcpy(idx, keep.data(), keep.size() * 8, cudaMemcpyHostToDevice));
#undef SP
    out->n_samples = (int64_t)total;
    out->n_valid = (int64_t)keep.size();
    out->n_games = finished;
    out->plies_run = tick;
    out->truncated = truncated;
    out->planes = planes;
    out->pi = pi;
    out->z = z;
    out->color = color;
    out->serial = serial;
    out->valid_idx = idx;
    c->mcts_phase = 0;
    return ONB_OK;
}

// fight (evaluator.rs:355-399) for all games of the context in lockstep. Per ply the undecided games are split by whose turn it is
// (evaluator.rs:379: ONE agent moves per ply and game); `move` makes an agent choose for ITS m games only (d_games: ascending device
// list) and leaves the actions in d_out[game]. The merge, the step and the end-of-game test stay on the device; the host reads the
// two list lengths per ply.
int32_t run_fight(Ctx* c, const onb_agent* a, const onb_agent* b, const uint8_t* a_is_red_host, uint32_t max_plies, onb_fight_result* out,
                  int32_t (*move)(Ctx*, const onb_agent*, uint32_t, const int32_t*, int64_t, uint16_t*), char* err, size_t err_len) {
    const int64_t n = c->n;
    uint8_t *mask = nullptr, *results = nullptr, *fa = nullptr, *fb = nullptr;
    uint16_t *act_a = nullptr, *act_b = nullptr;
    int32_t *list_a = nullptr, *list_b = nullptr;
    uint32_t* blocks = nullptr;
    unsigned long long* counters = nullptr;  // [0] games where A moves, [1] games where B moves, [2..4] tally
    cudaError_t e;
#define FT(call)                                                                    \
    do {                                                                            \
        e = (call);                                                                 \
        if (e != cudaSuccess) {                                                     \
            snprintf(err, err_len, "onb_fight: %s: %s", #call, cudaGetErrorString(e)); \
            c->n_act = 0;                                                           \
            c->d_tree_game = nullptr;                                               \
            return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;       \
        }                                                                           \
    } while (0)
    FT(grow(c, kFtMask, (size_t)n, (void**)&mask));
    FT(grow(c, kFtResults, (size_t)n, (void**)&results));
    FT(grow(c, kFtActA, (size_t)n * 2, (void**)&act_a));
    FT(grow(c, kFtActB, (size_t)n * 2, (void**)&act_b));
    FT(grow(c, kFtCounters, 64, (void**)&counters));
    FT(grow(c, kFtFlagA, (size_t)n, (void**)&fa));
    FT(grow(c, kFtFlagB, (size_t)n, (void**)&fb));
    FT(grow(c, kFtListA, (size_t)n * 4, (void**)&list_a));
    FT(grow(c, kFtListB, (size_t)n * 4, (void**)&list_b));
    FT(grow(c, kFtBlocks, (size_t)((n + 255) / 256 + 1) * 4, (void**)&blocks));
    FT(cudaMemcpyAsync(mask, a_is_red_host, (size_t)n, cudaMemcpyHostToDevice, c->stream));
    const unsigned grid = (unsigned)((n + 255) / 256);
    int64_t plies_left = (int64_t)max_plies, tick = 0, searched = 0;
    for (;;) {
        k_fight_plan<<<grid, 256, 0, c->stream>>>(c->d_states, n, mask, fa, fb);
        FT(cudaGetLastError());
        FT(compact(c, fa, n, blocks, list_a, counters));
        FT(compact(c, fb, n, blocks, list_b, counters + 1));
        unsigned long long m[2] = {0, 0};
        FT(cudaMemcpyAsync(m, counters, 16, cudaMemcpyDeviceToHost, c->stream));
        FT(cudaStreamSynchronize(c->stream));
        if (m[0] + m[1] == 0) break;                // evaluator.rs:366: every game is decided
        for (int who = 0; who < 2; ++who) {
            if (m[who] == 0) continue;
            const int32_t rc = move(c, who ? b : a, (uint32_t)tick, who ? list_b : list_a, (int64_t)m[who], who ? act_b : act_a);
            if (rc != ONB_OK) {
                snprintf(err, err_len, "%s", c->err);
                c->n_act = 0;
                c->d_tree_game = nullptr;
                return rc;
            }
        }
        searched += (int64_t)(m[0] + m[1]);
        k_fight_merge<<<grid, 256, 0, c->stream>>>(fa, fb, n, act_a, act_b, c->d_actions);
        FT(cudaGetLastError());
        FT(launch_env_step(c, kModeActions, 0, 0, 0));
        ++tick;
        if (plies_left < 0) break;                  // evaluator.rs:386-392: checked after the move, then decremented (max_plies + 2 plies)
        plies_left -= 1;
    }
    c->n_act = 0;
    c->d_tree_game = nullptr;
    FT(cudaMemsetAsync(counters + 2, 0, 24, c->stream));
    k_fight_tally<<<grid, 256, 0, c->stream>>>(c->d_states, n, mask, results, counters + 2);
    FT(cudaGetLastError());
    unsigned long long tally[3] = {0, 0, 0};
    FT(cudaMemcpyAsync(tally, counters + 2, 24, cudaMemcpyDeviceToHost, c->stream));
    FT(cudaStreamSynchronize(c->stream));
#undef FT
    out->a_wins = (int64_t)tally[0];
    out->b_wins = (int64_t)tally[1];
    out->draws = (int64_t)tally[2];
    out->plies_run = tick;
    out->results = results;
    out->moves_chosen = searched;
    c->fight_valid = 1;
    c->mcts_phase = 0;
    return ONB_OK;
}

// FightStatistics (evaluator.rs:38-110) of the last onb_fight, folded on the device in game order
int32_t run_fight_statistics(Ctx* c, double rating_a, double rating_b, onb_fight_statistics* out, double* history_host, char* err, size_t err_len) {
    if (!c->fight_valid || !c->sp_buf[kFtResults] || !c->sp_buf[kFtMask]) {
        snprintf(err, err_len, "onb_fight_statistics: no onb_fight has run on this context");
        return ONB_E_STATE;
    }
    const int64_t n = c->n;
    unsigned long long* elo = nullptr;  // [9] counts, then 2 doubles
    double* history = nullptr;
    cudaError_t e = grow(c, kFtElo, 9 * 8 + 16, (void**)&elo);
    if (e == cudaSuccess && history_host) e = grow(c, kFtHistory, (size_t)n * 32, (void**)&history);
    double* ratings = reinterpret_cast<double*>(elo + 9);
    if (e == cudaSuccess) {
        k_elo_fold<<<1, 32, 0, c->stream>>>((const uint8_t*)c->sp_buf[kFtResults], (const uint8_t*)c->sp_buf[kFtMask], n, rating_a, rating_b, elo, ratings,
                                            history);
        e = cudaGetLastError();
    }
    unsigned long long h[11];
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, elo, sizeof(h), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && history_host) e = cudaMemcpyAsync(history_host, history, (size_t)n * 32, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        snprintf(err, err_len, "onb_fight_statistics: %s", cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;
    }
    out->wins = (int64_t)h[0]; out->loses = (int64_t)h[1]; out->draws = (int64_t)h[2];
    for (int col = 0; col < 2; ++col) {
        out->color_wins[col] = (int64_t)h[3 + 3 * col]; out->color_loses[col] = (int64_t)h[4 + 3 * col]; out->color_draws[col] = (int64_t)h[5 + 3 * col];
        const int64_t t = out->color_wins[col] + out->color_loses[col] + out->color_draws[col];
        out->color_winrate[col] = (double)out->color_wins[col] / (double)t;  // NaN when agent A never played this colour, as in the reference
    }
    out->winrate = (double)out->wins / (double)(out->wins + out->loses + out->draws);
    memcpy(&out->rating_a, &h[9], 8);
    memcpy(&out->rating_b, &h[10], 8);
    out->n_games = n;
    return ONB_OK;
}

}  // namespace onb
