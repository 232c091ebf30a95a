// onb_reuse.cu -- search-tree reuse between moves (onb_mcts_set_reuse, include/onb.h).
//
// Before a reuse-enabled search, per searched game:
//   1. plan:  find the child of the game's remembered root whose position equals the game's current state (the move that was
//             played), and the simulations that remain to the visit target: budget = max(0, sims - N_child) (no match: sims);
//   2. order: a stable counting sort of the games by budget, descending (per-256-game-block counts, one scan, placement), so that
//             the trees still searching in round r are the prefix [0, off[r]) of the slots: the unchanged search kernels then run
//             round r (or a run of rounds with the same prefix) over trees(c) = off[r];
//   3. copy:  compact the kept subtree (the child and its descendants) into the new slot of the second pool, in arena order: a
//             parent's index is below its children's and the child has the lowest index of its subtree, so the subtree is a
//             stable filter of the old pool from the child on. One warp per tree, two sweeps over the old pool: membership bits
//             (a node is kept iff its parent is), then the copy with parent / first_child renumbered by rank;
//   4. swap the pools (and the root / tree-size arrays read by step 1).
#include <cstdlib>
#include <cstring>

#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {
namespace {

constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr unsigned kFullMask = 0xFFFFFFFFu;
constexpr int kPlanBlock = 256;
constexpr int kCopyWarpsMax = 4;

__device__ __forceinline__ bool same_position(const Game& a, const Game& b) {
    return a.pawn_r == b.pawn_r && a.pawn_b == b.pawn_b && a.king_r == b.king_r && a.king_b == b.king_b && a.cards == b.cards &&
           a.side == b.side;
}

// 1. + the per-block part of 2: plan[i] = (old slot, kept node, budget, rank among the block's games with the same budget);
// mat[(sims - budget) * nb + block] = number of the block's games with that budget (mat zeroed by the caller)
__global__ void __launch_bounds__(kPlanBlock) k_reuse_plan(const uint4* __restrict__ states, const int32_t* __restrict__ list, int64_t m, int live,
                                                           const int32_t* __restrict__ slot_of_game, const uint4* __restrict__ old_roots,
                                                           const Node* __restrict__ old_nodes, uint32_t cap, uint32_t sims, uint4* __restrict__ plan,
                                                           uint32_t* __restrict__ mat, int nb) {
    __shared__ uint32_t s_b[kPlanBlock];
    const int64_t i = (int64_t)blockIdx.x * kPlanBlock + threadIdx.x;
    uint32_t old = kNone, keep = kNone, budget = kNone;
    if (i < m) {
        const int64_t g = list ? (int64_t)list[i] : i;
        budget = sims;
        const int32_t s = live ? slot_of_game[g] : -1;
        const Game cur = unpack(states[g]);
        if (s >= 0 && cur.result == 0) {
            old = (uint32_t)s;
            const Node* pool = old_nodes + (size_t)s * cap;
            const Game root = unpack(old_roots[s]);
            const uint32_t k = pool[0].n_child, fc = pool[0].first_child;
            for (uint32_t j = 0; j < k; ++j) {
                Game x = root;
                apply_move(x, pool[fc + j].action);
                if (same_position(x, cur)) {
                    keep = fc + j;
                    const uint32_t nk = pool[keep].n;
                    budget = nk >= sims ? 0u : sims - nk;
                    break;
                }
            }
        }
    }
    s_b[threadIdx.x] = budget;
    __syncthreads();
    uint32_t rank = 0;
    bool last = true;
    for (int j = 0; j < kPlanBlock; ++j) {
        if (s_b[j] != budget) continue;
        if (j < (int)threadIdx.x) ++rank;
        else if (j > (int)threadIdx.x) last = false;
    }
    if (i < m) {
        plan[i] = make_uint4(old, keep, budget, rank);
        if (last) mat[(size_t)(sims - budget) * nb + blockIdx.x] = rank + 1u;
    }
}

// 2. exclusive scan of mat (budget descending, then block), one CTA; off[r] = games with budget > r = scanned mat[(sims - r) * nb]
__global__ void __launch_bounds__(1024) k_reuse_scan(uint32_t* __restrict__ mat, int64_t len, int nb, uint32_t sims, uint32_t* __restrict__ off) {
    __shared__ uint32_t s_part[1024];
    const int64_t per = (len + 1023) / 1024, lo = threadIdx.x * per, hi = lo + per < len ? lo + per : len;
    uint32_t sum = 0;
    for (int64_t i = lo; i < hi; ++i) sum += mat[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const uint32_t v = threadIdx.x >= (unsigned)o ? s_part[threadIdx.x - o] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = s_part[threadIdx.x] - sum;
    for (int64_t i = lo; i < hi; ++i) {
        const uint32_t c = mat[i];
        mat[i] = run;
        run += c;
    }
    __syncthreads();
    for (uint32_t r = threadIdx.x; r <= sims; r += blockDim.x) off[r] = mat[(size_t)(sims - r) * nb];
}

// 2. placement: slot = scanned count of the (budget, block) cell + rank in the block; both maps updated (slot_of_game was reset)
__global__ void __launch_bounds__(256) k_reuse_place(const int32_t* __restrict__ list, int64_t m, uint4* __restrict__ plan, const uint32_t* __restrict__ mat,
                                                     int nb, uint32_t sims, int32_t* __restrict__ game_of_slot, int32_t* __restrict__ slot_of_game) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    uint4 p = plan[i];
    const uint32_t slot = mat[(size_t)(sims - p.z) * nb + (uint32_t)(i / kPlanBlock)] + p.w;
    const int32_t g = list ? list[i] : (int32_t)i;
    p.w = slot;
    plan[i] = p;
    game_of_slot[slot] = g;
    slot_of_game[g] = (int32_t)slot;
}

__device__ __forceinline__ uint32_t rank_of(const uint32_t* bits, const uint32_t* pre, uint32_t x) {
    return pre[x >> 5] + __popc(bits[x >> 5] & ((1u << (x & 31u)) - 1u));
}

// 3. one warp per searched game; dynamic shared memory: per warp bits[words] (kept flags, one word per 32 nodes) + pre[words]
// (kept nodes before the word)
__global__ void __launch_bounds__(kCopyWarpsMax * 32) k_reuse_copy(const uint4* __restrict__ states, const int32_t* __restrict__ list, int64_t m,
                                                                   const uint4* __restrict__ plan, const Node* __restrict__ old_nodes,
                                                                   const uint32_t* __restrict__ old_size, Node* __restrict__ new_nodes,
                                                                   uint4* __restrict__ new_roots, uint32_t* __restrict__ new_size,
                                                                   uint8_t* __restrict__ new_flags, uint32_t cap, uint32_t words) {
    extern __shared__ uint32_t s_mem[];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (i >= m) return;
    uint32_t* bits = s_mem + (size_t)warp * 2u * words;
    uint32_t* pre = bits + words;
    const uint4 pl = plan[i];
    const uint32_t keep = pl.y, slot = pl.w;
    const int64_t g = list ? (int64_t)list[i] : i;
    uint4* dst = reinterpret_cast<uint4*>(new_nodes + (size_t)slot * cap);
    uint32_t total = 1;
    if (keep == kNone) {  // a fresh root, as k_mcts_begin writes it (MctsNode::new(None, 0, None, player_color, 1.), mcts_arena.rs:57)
        if (lane == 0) {
            const double one = 1.0;
            dst[0] = make_uint4(0u, 0u, (uint32_t)__double2loint(one), (uint32_t)__double2hiint(one));
            dst[1] = make_uint4(0u, 0u, kNone, 0xFFFFu);
        }
    } else {
        const Node* src = old_nodes + (size_t)pl.x * cap;
        const uint4* src4 = reinterpret_cast<const uint4*>(src);
        const uint32_t size = old_size[pl.x];
        const uint32_t w0 = keep >> 5, w1 = (size + 31u) >> 5;
        uint32_t run = 0;
        // sweep 1: kept flags. A node is kept iff it is the child or its parent is kept; a parent in an earlier word is looked up,
        // one in the same word is resolved through the word's lanes (parent index < child index: the chain ends)
        for (uint32_t w = w0; w < w1; ++w) {
            const uint32_t idx = (w << 5) + lane;
            const bool in_range = idx >= keep && idx < size;
            const uint32_t p = in_range ? src[idx].parent : kNone;
            bool mem = idx == keep, res = !in_range || idx == keep;
            if (!res && p < (w << 5)) {
                res = true;
                mem = p >= keep && ((bits[p >> 5] >> (p & 31u)) & 1u);
            }
            for (;;) {
                const unsigned rb = __ballot_sync(kFullMask, res), mb = __ballot_sync(kFullMask, res && mem);
                if (rb == kFullMask) break;
                if (!res && ((rb >> (p & 31u)) & 1u)) {
                    res = true;
                    mem = (mb >> (p & 31u)) & 1u;
                }
            }
            const unsigned b = __ballot_sync(kFullMask, mem);
            if (lane == 0) { bits[w] = b; pre[w] = run; }
            run += __popc(b);
            __syncwarp();
        }
        // sweep 2: the kept records at their ranks, links renumbered (a node without children keeps first_child = 0)
        for (uint32_t w = w0; w < w1; ++w) {
            const uint32_t b = bits[w];
            if (!((b >> lane) & 1u)) continue;
            const uint32_t idx = (w << 5) + lane;
            const uint32_t ni = pre[w] + __popc(b & ((1u << lane) - 1u));
            const uint4 a = src4[2 * (size_t)idx];
            uint4 h = src4[2 * (size_t)idx + 1];  // n, first_child, parent, meta
            h.z = idx == keep ? kNone : rank_of(bits, pre, h.z);
            if ((h.w >> 16) & 0xFFu) h.y = rank_of(bits, pre, h.y);
            dst[2 * (size_t)ni] = a;
            dst[2 * (size_t)ni + 1] = h;
        }
        total = run;
    }
    if (lane == 0) {
        new_size[slot] = total;
        new_flags[slot] = 0;
        new_roots[slot] = states[g];
    }
}

// finish outputs, slot order -> game order
__global__ void __launch_bounds__(256) k_reuse_unpermute(const int32_t* __restrict__ game_of_slot, int64_t m, const float* __restrict__ pi,
                                                         const uint16_t* __restrict__ best, const uint32_t* __restrict__ rv, const double* __restrict__ q,
                                                         const uint32_t* __restrict__ cv, float* __restrict__ pi_o, uint16_t* __restrict__ best_o,
                                                         uint32_t* __restrict__ rv_o, double* __restrict__ q_o, uint32_t* __restrict__ cv_o) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m * 90) return;
    const int64_t t = e / 90, k = e - t * 90, g = game_of_slot[t];
    if (k < 50) pi_o[g * 50 + k] = pi[t * 50 + k];
    else cv_o[g * 40 + (k - 50)] = cv[t * 40 + (k - 50)];
    if (k == 0) { best_o[g] = best[t]; rv_o[g] = rv[t]; q_o[g] = q[t]; }
}

template <class T>
cudaError_t ralloc(T** p, size_t count) {
    if (*p) return cudaSuccess;
    return cudaMalloc(reinterpret_cast<void**>(p), (count ? count : 1) * sizeof(T));
}

}  // namespace

cudaError_t reuse_alloc(Ctx* c) {
    const size_t n = (size_t)c->n, nb = (n + kPlanBlock - 1) / kPlanBlock, smax = (size_t)c->cfg.mcts_max_sims;
    cudaError_t e;
    if ((e = ralloc(&c->d_nodes_alt, n * (size_t)c->node_cap)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_roots_alt, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_tree_size_alt, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_game, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_slot, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_plan, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_mat, (smax + 1) * nb)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_off, smax + 1)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_pi, n * 50)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_best, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_rv, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_q, n)) != cudaSuccess) return e;
    if ((e = ralloc(&c->d_ru_cv, n * 40)) != cudaSuccess) return e;
    if (!c->h_ru_off) {
        c->h_ru_off = static_cast<uint32_t*>(malloc((smax + 1) * sizeof(uint32_t)));
        if (!c->h_ru_off) return cudaErrorMemoryAllocation;
    }
    const uint32_t words = (c->node_cap + 31u) / 32u;
    const size_t smem = (size_t)words * 8u;  // one warp
    if (smem > 48u * 1024u) {
        if (smem > 227u * 1024u) return cudaErrorInvalidValue;
        if ((e = cudaFuncSetAttribute(k_reuse_copy, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

void reuse_free(Ctx* c) {
    void* ptrs[] = {c->d_nodes_alt, c->d_roots_alt, c->d_tree_size_alt, c->d_ru_game, c->d_ru_slot, c->d_ru_plan, c->d_ru_mat, c->d_ru_off,
                    c->d_ru_pi, c->d_ru_best, c->d_ru_rv, c->d_ru_q, c->d_ru_cv};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    free(c->h_ru_off);
}

cudaError_t launch_reuse_begin(Ctx* c, const int32_t* d_games, int64_t m, uint32_t sims) {
    const int nb = (int)((m + kPlanBlock - 1) / kPlanBlock);
    const int64_t len = (int64_t)(sims + 1) * nb;
    cudaError_t e = cudaMemsetAsync(c->d_ru_mat, 0, (size_t)len * 4, c->stream);
    if (e != cudaSuccess) return e;
    k_reuse_plan<<<nb, kPlanBlock, 0, c->stream>>>(c->d_states, d_games, m, c->ru_live, c->d_ru_slot, c->d_roots, c->d_nodes, c->node_cap, sims,
                                                     c->d_ru_plan, c->d_ru_mat, nb);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    k_reuse_scan<<<1, 1024, 0, c->stream>>>(c->d_ru_mat, len, nb, sims, c->d_ru_off);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(c->d_ru_slot, 0xFF, (size_t)c->n * 4, c->stream)) != cudaSuccess) return e;
    k_reuse_place<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(d_games, m, c->d_ru_plan, c->d_ru_mat, nb, sims, c->d_ru_game, c->d_ru_slot);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const uint32_t words = (c->node_cap + 31u) / 32u;
    const size_t per_warp = (size_t)words * 8u;
    int wpb = (int)((48u * 1024u) / per_warp);
    wpb = wpb < 1 ? 1 : wpb > kCopyWarpsMax ? kCopyWarpsMax : wpb;
    k_reuse_copy<<<(unsigned)((m + wpb - 1) / wpb), wpb * 32, per_warp * wpb, c->stream>>>(c->d_states, d_games, m, c->d_ru_plan, c->d_nodes,
                                                                                             c->d_tree_size, c->d_nodes_alt, c->d_roots_alt,
                                                                                             c->d_tree_size_alt, c->d_tree_flags, c->node_cap, words);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    Node* tn = c->d_nodes; c->d_nodes = c->d_nodes_alt; c->d_nodes_alt = tn;
    uint4* tr = c->d_roots; c->d_roots = c->d_roots_alt; c->d_roots_alt = tr;
    uint32_t* ts = c->d_tree_size; c->d_tree_size = c->d_tree_size_alt; c->d_tree_size_alt = ts;
    if ((e = cudaMemcpyAsync(c->h_ru_off, c->d_ru_off, (size_t)(sims + 1) * 4, cudaMemcpyDeviceToHost, c->stream)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
    c->n_act = m;
    c->d_tree_game = c->d_ru_game;
    c->ru_live = 1;
    c->ru_m = m;
    // counters: sum over rounds of the active trees = simulations; kept = trees whose budget is below the target
    uint64_t run = 0;
    for (uint32_t r = 0; r < sims; ++r) run += c->h_ru_off[r];
    c->ru_stats[0] += (uint64_t)m;
    c->ru_stats[1] += sims ? (uint64_t)m - c->h_ru_off[sims - 1] : 0u;
    c->ru_stats[2] += (uint64_t)m * sims - run;
    c->ru_stats[3] += run;
    return cudaSuccess;
}

cudaError_t launch_reuse_unpermute(Ctx* c) {
    const int64_t m = c->ru_m;
    k_reuse_unpermute<<<(unsigned)((m * 90 + 255) / 256), 256, 0, c->stream>>>(c->d_ru_game, m, c->d_ru_pi, c->d_ru_best, c->d_ru_rv, c->d_ru_q, c->d_ru_cv,
                                                                                 c->d_pi, c->d_best, c->d_root_visits, c->d_root_q, c->d_child_visits);
    return cudaGetLastError();
}

}  // namespace onb
