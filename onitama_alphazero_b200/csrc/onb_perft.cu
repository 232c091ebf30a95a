// onb_perft.cu -- perft-style legal-move enumeration (BASELINE config 2).
//
// Two phases: (1) lockstep breadth-first frontier expansion in HBM (32 B per node: read parent, write child)
// until there are enough independent subtrees to fill the machine; (2) every frontier node is finished by one
// thread's depth-first search with bulk counting at the last ply (k_perft_flat: a flat state machine, stack in shared
// memory). Phase 2 moves ~0 bytes per node and is issue-bound; see DESIGN.md.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {

// ---- phase 1: one BFS level -------------------------------------------------------------------------------
// COUNT_ONLY pass sizes the next frontier exactly; the fill pass writes it (order is irrelevant for perft).
template <bool COUNT_ONLY>
__global__ void __launch_bounds__(128) k_perft_expand(const uint4* __restrict__ in_states, const uint32_t* __restrict__ in_root, int64_t n_in,
                                                      uint4* __restrict__ out_states, uint32_t* __restrict__ out_root,
                                                      unsigned long long* __restrict__ cursor, unsigned long long* __restrict__ nodes,
                                                      unsigned long long* __restrict__ wins, unsigned long long* __restrict__ zero, int depth_total,
                                                      int level) {
    __shared__ uint32_t s_att[800];
    load_attack_table_to_smem(s_att);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n_in;
    Game g{};
    uint32_t root = 0, total = 0, nwin = 0;
    uint32_t own = 0, own_p = 0, win_t = 0, temple = 0, side = 0;
    if (live) {
        g = unpack(in_states[i]);
        root = in_root[i];
        side = g.side;
        own_p = side ? g.pawn_b : g.pawn_r;
        const uint32_t own_k = side ? g.king_b : g.king_r;
        const uint32_t en_p = side ? g.pawn_r : g.pawn_b, en_k = side ? g.king_r : g.king_b;
        own = own_p | own_k;
        win_t = en_k & ~en_p;
        temple = 1u << (side ? kRedTemple : kBlueTemple);
        for (uint32_t s = 0; s < 2; ++s) {
            const uint32_t* Ts = s_att + (side * 16u + card_at(g.cards, side * 2u + s)) * 25u;
            uint32_t rem = own;
            while (rem) {
                const int f = __ffs(rem) - 1;
                rem &= rem - 1;
                const uint32_t a = Ts[f] & ~own;
                const uint32_t wm = a & (win_t | (((own_p >> f) & 1u) ? 0u : temple));
                total += __popc(a);
                nwin += __popc(wm);
            }
        }
    }
    const uint32_t n_children = total - nwin;  // wins end the line
    // warp-aggregated reservation of output slots
    uint32_t incl = n_children;
    const uint32_t lane = threadIdx.x & 31u;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t warp_total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    unsigned long long base = 0;
    if (lane == 31 && warp_total) base = atomicAdd(cursor, (unsigned long long)warp_total);
    base = __shfl_sync(0xFFFFFFFFu, base, 31);
    if (COUNT_ONLY) return;
    {   // counters: one set of atomics per warp when every lane works for the same root (siblings sit together in the frontier)
        const unsigned full = 0xFFFFFFFFu;
        const uint32_t r0 = __shfl_sync(full, live ? root : 0xFFFFFFFFu, 0);
        const bool same = __all_sync(full, (live ? root : 0xFFFFFFFFu) == r0);
        if (same) {
            const uint32_t T = __reduce_add_sync(full, total), W = __reduce_add_sync(full, nwin), Z = __reduce_add_sync(full, live && total == 0 ? 1u : 0u);
            if (lane == 0 && live) {
                if (T) atomicAdd(&nodes[(int64_t)root * depth_total + level], (unsigned long long)T);
                if (W) atomicAdd(&wins[(int64_t)root * depth_total + level], (unsigned long long)W);
                if (Z) atomicAdd(&zero[(int64_t)root * depth_total + level], (unsigned long long)Z);
            }
        } else if (live) {
            atomicAdd(&nodes[(int64_t)root * depth_total + level], (unsigned long long)total);
            if (nwin) atomicAdd(&wins[(int64_t)root * depth_total + level], (unsigned long long)nwin);
            if (total == 0) atomicAdd(&zero[(int64_t)root * depth_total + level], 1ull);
        }
    }
    if (!live) return;
    unsigned long long pos = base + (incl - n_children);
    for (uint32_t s = 0; s < 2; ++s) {
        const uint32_t idx = side * 2u + s;
        const uint32_t* Ts = s_att + (side * 16u + card_at(g.cards, idx)) * 25u;
        uint32_t rem = own;
        while (rem) {
            const int f = __ffs(rem) - 1;
            rem &= rem - 1;
            const uint32_t king = ((own_p >> f) & 1u) ^ 1u;
            uint32_t a = Ts[f] & ~own;
            a &= ~(win_t | (king ? temple : 0u));
            while (a) {
                const uint32_t to = __ffs(a) - 1;
                a &= a - 1;
                Game ch = g;
                apply_move(ch, make_action(idx, (uint32_t)f, to, king));
                if (out_root) {
                    out_states[pos] = pack(ch);
                    out_root[pos] = root;
                } else {
                    // leaf format (the level k_perft_leaf2 reads): one 16-byte entry with the root id inside; both kings are on the
                    // board (a king capture ends the line), so a square index replaces each one-hot king board
                    out_states[pos] = make_uint4(ch.pawn_r | ((uint32_t)(__ffs(ch.king_r) - 1) << 25),
                                                 ch.pawn_b | ((uint32_t)(__ffs(ch.king_b) - 1) << 25) | (ch.side << 30), ch.cards, root);
                }
                ++pos;
            }
        }
    }
}

// ---- phase 2: depth-first search, one move per loop iteration ---------------------------------------------------------------
// A nested-loop DFS keeps everything in registers but its lanes drift apart (each lane sits at a different nesting level with a
// different trip count): ~14 % SIMT efficiency (DESIGN.md). This kernel runs the search as a state machine whose
// iteration either advances the (slot, piece) iterator of the current node or plays ONE move; positions at the last interior
// level are bulk-counted immediately. The per-level stack lives in shared memory ([level][word][thread], conflict free), the
// current level in registers, so every lane executes the same short instruction stream in every iteration.
constexpr int kFlatThreads = 128;
constexpr int kFlatWords = 7;  // op, ok, ep, ek, cards|side<<20, iterator, current destination mask | from << 25

struct BulkCount { uint32_t total, wins; };
__device__ __forceinline__ BulkCount bulk_count(const uint32_t* T, const RelGame& g) {
    const uint32_t own = g.op | g.ok;
    const uint32_t win_t = g.ek & ~g.ep;
    const uint32_t temple = 1u << (g.side ? kRedTemple : kBlueTemple);
    const uint32_t* T0 = T + (g.side * 16u + card_at(g.cards, g.side * 2u)) * 25u;
    const uint32_t* T1 = T + (g.side * 16u + card_at(g.cards, g.side * 2u + 1u)) * 25u;
    BulkCount c{0, 0};
    uint32_t rem = own;
    while (rem) {
        const int f = __ffs(rem) - 1;
        rem &= rem - 1;
        const uint32_t wm = win_t | (((g.op >> f) & 1u) ? 0u : temple);
        const uint32_t a0 = T0[f] & ~own, a1 = T1[f] & ~own;
        c.total += __popc(a0) + __popc(a1);
        c.wins += __popc(a0 & wm) + __popc(a1 & wm);
    }
    return c;
}

#ifndef ONB_PERFT_MINB
#define ONB_PERFT_MINB 1
#endif
template <int REM>
__global__ void __launch_bounds__(kFlatThreads, ONB_PERFT_MINB) k_perft_flat(const uint4* __restrict__ states, const uint32_t* __restrict__ roots, int64_t n_items,
                                                             unsigned long long* __restrict__ nodes, unsigned long long* __restrict__ wins,
                                                             unsigned long long* __restrict__ zero, int depth_total) {
    __shared__ __align__(16) uint32_t s_att[800];
    __shared__ uint32_t s_stk[(REM > 2 ? REM - 2 : 1) * kFlatWords * kFlatThreads];  // levels 0 .. REM-3 can have a level below them
    load_attack_table_to_smem(s_att);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const int64_t row = (int64_t)roots[i] * depth_total;
    const int d0 = depth_total - REM;  // the counters of the frontier node's children live at index d0
    RelGame g = to_rel(unpack(states[i]));
    if constexpr (REM == 1) {
        const BulkCount c = bulk_count(s_att, g);
        if (c.total) atomicAdd(&nodes[row + d0], (unsigned long long)c.total);
        if (c.wins) atomicAdd(&wins[row + d0], (unsigned long long)c.wins);
        if (c.total == 0) atomicAdd(&zero[row + d0], 1ull);
    } else {
    unsigned long long cnt_n[REM], cnt_w[REM];  // index = level of the PARENT whose children are counted
    uint32_t cnt_z[REM];
#pragma unroll
    for (int k = 0; k < REM; ++k) { cnt_n[k] = 0; cnt_w[k] = 0; cnt_z[k] = 0; }
    auto add_counts = [&](int lv, uint32_t tot, uint32_t w, uint32_t z) {  // level-indexed without dynamic register indexing
#pragma unroll
        for (int k = 0; k < REM - 1; ++k)
            if (k == lv) { cnt_n[k] += tot; cnt_w[k] += w; cnt_z[k] += z; }
    };
    int level = 0;
    uint32_t it = g.op | g.ok;        // own pieces of the current hand slot that were not visited yet
    uint32_t cur = 0, cur_f = 0;      // unplayed, non-winning destinations of the current piece, and its square
    uint32_t cur_slot = 0, had = 0;   // hand slot being enumerated; whether this node had any move so far
    uint32_t n_total = 0, n_wins = 0; // running child counts of the current node
    bool done = false;
    for (;;) {
        // (1) find the next move: advance over pieces and hand slots, leave finished nodes. Light and rarely more than one round,
        //     so that step (2), which dominates, is executed by all lanes of the warp together.
        while (cur == 0) {
            if (it) {  // next piece of the current hand slot
                const uint32_t own = g.op | g.ok;
                const int f = __ffs(it) - 1;
                it &= it - 1;
                const uint32_t wm = (g.ek & ~g.ep) | (((g.op >> f) & 1u) ? 0u : (1u << (g.side ? kRedTemple : kBlueTemple)));
                const uint32_t a = s_att[(g.side * 16u + card_at(g.cards, g.side * 2u + cur_slot)) * 25u + f] & ~own;
                n_total += __popc(a);
                n_wins += __popc(a & wm);
                had |= a ? 1u : 0u;
                cur = a & ~wm;  // a winning move ends its line
                cur_f = (uint32_t)f;
            } else if (cur_slot == 0) {  // second hand slot
                cur_slot = 1;
                it = g.op | g.ok;
            } else {  // node finished
                add_counts(level, n_total, n_wins, had ? 0u : 1u);
                if (level == 0) { done = true; break; }
                --level;
                const uint32_t* p = s_stk + (level * kFlatWords) * kFlatThreads + threadIdx.x;
                g.op = p[0 * kFlatThreads]; g.ok = p[1 * kFlatThreads]; g.ep = p[2 * kFlatThreads]; g.ek = p[3 * kFlatThreads];
                const uint32_t cs = p[4 * kFlatThreads];
                g.cards = cs & 0xFFFFFu; g.side = cs >> 20;
                const uint32_t itw = p[5 * kFlatThreads];
                it = itw & kAll25; cur_slot = (itw >> 25) & 1u; had = (itw >> 26) & 1u;
                const uint32_t cw = p[6 * kFlatThreads];
                cur = cw & kAll25; cur_f = cw >> 25;
                n_total = 0; n_wins = 0;  // the part counted before the descent was flushed then
            }
        }
        if (done) break;
        // (2) play one move
        const uint32_t to = __ffs(cur) - 1;
        cur &= cur - 1;
        RelGame ch = g;
        apply_move_rel(ch, make_action(g.side * 2u + cur_slot, cur_f, to, ((g.op >> cur_f) & 1u) ^ 1u));
        if (level == REM - 2) {  // the child is on the last interior level: count its children in bulk, do not descend
            const BulkCount c = bulk_count(s_att, ch);
            cnt_n[REM - 1] += c.total; cnt_w[REM - 1] += c.wins; cnt_z[REM - 1] += c.total == 0 ? 1u : 0u;
        } else {
            add_counts(level, n_total, n_wins, 0);
            uint32_t* p = s_stk + (level * kFlatWords) * kFlatThreads + threadIdx.x;
            p[0 * kFlatThreads] = g.op; p[1 * kFlatThreads] = g.ok; p[2 * kFlatThreads] = g.ep; p[3 * kFlatThreads] = g.ek;
            p[4 * kFlatThreads] = g.cards | (g.side << 20);
            p[5 * kFlatThreads] = it | (cur_slot << 25) | (had << 26);
            p[6 * kFlatThreads] = cur | (cur_f << 25);
            ++level;
            g = ch;
            it = g.op | g.ok; cur = 0; cur_f = 0; cur_slot = 0; had = 0; n_total = 0; n_wins = 0;
        }
    }
#pragma unroll
    for (int k = 0; k < REM; ++k) {
        if (cnt_n[k]) atomicAdd(&nodes[row + d0 + k], cnt_n[k]);
        if (cnt_w[k]) atomicAdd(&wins[row + d0 + k], cnt_w[k]);
        if (cnt_z[k]) atomicAdd(&zero[row + d0 + k], (unsigned long long)cnt_z[k]);
    }
    }
}

template <int REM>
static cudaError_t launch_dfs(Ctx* c, const uint4* st, const uint32_t* rt, int64_t n_items, unsigned long long* nodes, unsigned long long* wins,
                              unsigned long long* zero, int depth) {
    k_perft_flat<REM><<<(unsigned)((n_items + kFlatThreads - 1) / kFlatThreads), kFlatThreads, 0, c->stream>>>(st, rt, n_items, nodes, wins, zero,
                                                                                                             depth);
    return cudaGetLastError();
}

// ---- phase 2b: the last two levels of one frontier node per thread -----------------------------------------------------------
// With the frontier two plies above the horizon a thread generates the node's children and bulk-counts each child's moves: the
// opponent's hand is the same for all children (the mover's card goes to the neutral slot), so both attack-table rows are hoisted
// and a child costs ~10 table reads and popcounts. Work per thread is small and similar across a warp (the flat DFS above runs
// 16 of 32 lanes on average), and the counters are added per warp when all lanes share a root (frontier order keeps siblings together).
__global__ void __launch_bounds__(256) k_perft_leaf2(const uint4* __restrict__ states, const uint32_t* __restrict__ roots, int64_t n_items,
                                                     unsigned long long* __restrict__ nodes, unsigned long long* __restrict__ wins,
                                                     unsigned long long* __restrict__ zero, int depth_total, int level) {
    // the attack table is read from its global-memory mirror (L1 resident): ~20 reads per thread do not pay for staging it in shared
    // memory per CTA; the rows of the children's mover are read once per node and kept in registers
    const uint32_t* T = g_attack.t;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n_items;
    uint32_t root = 0xFFFFFFFFu, t0 = 0, w0 = 0, z0 = 0, t1 = 0, w1 = 0, z1 = 0;
    if (live) {
        Game g;
        if (roots) {
            g = unpack(states[i]);
            root = roots[i];
        } else {  // leaf format written by k_perft_expand (see there)
            const uint4 e = states[i];
            g.pawn_r = e.x & 0x1FFFFFFu; g.king_r = 1u << ((e.x >> 25) & 31u);
            g.pawn_b = e.y & 0x1FFFFFFu; g.king_b = 1u << ((e.y >> 25) & 31u);
            g.side = (e.y >> 30) & 1u; g.cards = e.z; g.result = 0; g.passed = 0;
            root = e.w;
        }
        const uint32_t side = g.side;
        const uint32_t own_p = side ? g.pawn_b : g.pawn_r, own_k = side ? g.king_b : g.king_r;
        const uint32_t en_p = side ? g.pawn_r : g.pawn_b, en_k = side ? g.king_r : g.king_b;
        const uint32_t own = own_p | own_k;
        const uint32_t win_t = en_k & ~en_p;
        const uint32_t temple = 1u << (side ? kRedTemple : kBlueTemple);
        const uint32_t temple2 = 1u << (side ? kBlueTemple : kRedTemple);  // the children's side moves towards the other temple
        const uint32_t* U0 = T + ((side ^ 1u) * 16u + card_at(g.cards, (side ^ 1u) * 2u)) * 25u;
        const uint32_t* U1 = T + ((side ^ 1u) * 16u + card_at(g.cards, (side ^ 1u) * 2u + 1u)) * 25u;
        // the opponent's pieces (the children's movers): square bit, both cards' masks, temple bit if it is the king
        constexpr int MAXP = 5;
        uint32_t pb[MAXP], m0[MAXP], m1[MAXP], tk[MAXP];
        const uint32_t en = en_p | en_k;
        const bool small = __popc(en) <= MAXP;  // always true for positions reachable by play; fabricated ones take the generic loop
        {
            uint32_t r = en;
#pragma unroll
            for (int j = 0; j < MAXP; ++j) {
                pb[j] = 0; m0[j] = 0; m1[j] = 0; tk[j] = 0;
                if (r) {
                    const int f2 = __ffs(r) - 1;
                    r &= r - 1;
                    pb[j] = 1u << f2;
                    m0[j] = __ldg(U0 + f2);
                    m1[j] = __ldg(U1 + f2);
                    tk[j] = ((en_p >> f2) & 1u) ? 0u : temple2;
                }
            }
        }
        // replies of the opponent when none of its pieces is captured: masks, their number, and the winning ones if this side's king stays
        uint32_t f0[MAXP], f1[MAXP], base_ct = 0, base_cw = 0;
#pragma unroll
        for (int j = 0; j < MAXP; ++j) {
            f0[j] = m0[j] & ~en;
            f1[j] = m1[j] & ~en;
            base_ct += __popc(f0[j]) + __popc(f1[j]);
            base_cw += __popc(f0[j] & (own_k | tk[j])) + __popc(f1[j] & (own_k | tk[j]));
        }
#pragma unroll 1
        for (uint32_t s = 0; s < 2; ++s) {
            const uint32_t* Ts = T + (side * 16u + card_at(g.cards, side * 2u + s)) * 25u;
            uint32_t rem = own;
#pragma unroll 1
            while (rem) {
                const int f = __ffs(rem) - 1;
                rem &= rem - 1;
                const uint32_t king = ((own_p >> f) & 1u) ^ 1u;
                const uint32_t a = __ldg(Ts + f) & ~own;
                const uint32_t wm = a & (win_t | (king ? temple : 0u));
                t0 += __popc(a);
                w0 += __popc(wm);
                uint32_t b = a & ~wm;  // wins end the line
                if (small) {
                    // The reply count of a child depends only on the opponent's own pieces, its winning replies only on where this
                    // side's king stands: a quiet pawn move changes neither -> counted in bulk; a quiet king move changes the target
                    // square only; captures (the opponent loses a pawn) take the per-child loop below.
                    const uint32_t quiet = b & ~en_p;
                    if (!king) {
                        const uint32_t nq = __popc(quiet);
                        t1 += nq * base_ct;
                        w1 += nq * base_cw;
                        z1 += base_ct == 0 ? nq : 0u;
                        b &= en_p;
                    } else {
                        uint32_t q = quiet;
                        while (q) {
                            const uint32_t tb = q & (0u - q);
                            q &= q - 1;
                            uint32_t cw = 0;
#pragma unroll
                            for (int j = 0; j < MAXP; ++j) cw += __popc(f0[j] & (tb | tk[j])) + __popc(f1[j] & (tb | tk[j]));
                            t1 += base_ct;
                            w1 += cw;
                            z1 += base_ct == 0;
                        }
                        b &= en_p;
                    }
                }
#pragma unroll 1
                while (b) {
                    const uint32_t tb = b & (0u - b);
                    b &= b - 1;
                    // the child position from its mover's (the opponent's) point of view
                    const uint32_t c_own_p = en_p & ~tb, c_own = c_own_p | en_k;  // a pawn on `to` is captured
                    const uint32_t c_en_k = king ? tb : own_k;                     // win target: the king that just moved or stayed
                    uint32_t ct = 0, cw = 0;
                    if (small) {
#pragma unroll
                        for (int j = 0; j < MAXP; ++j) {
                            const uint32_t alive = (pb[j] & c_own) ? ~c_own : 0u;  // a captured pawn (or an empty slot) has no moves
                            const uint32_t a0 = m0[j] & alive, a1 = m1[j] & alive;
                            const uint32_t tw = c_en_k | tk[j];
                            ct += __popc(a0) + __popc(a1);
                            cw += __popc(a0 & tw) + __popc(a1 & tw);
                        }
                    } else {
                        uint32_t r2 = c_own;
                        while (r2) {
                            const int f2 = __ffs(r2) - 1;
                            r2 &= r2 - 1;
                            const uint32_t tw = c_en_k | (((c_own_p >> f2) & 1u) ? 0u : temple2);
                            const uint32_t a0 = __ldg(U0 + f2) & ~c_own, a1 = __ldg(U1 + f2) & ~c_own;
                            ct += __popc(a0) + __popc(a1);
                            cw += __popc(a0 & tw) + __popc(a1 & tw);
                        }
                    }
                    t1 += ct;
                    w1 += cw;
                    z1 += ct == 0;
                }
            }
        }
        z0 = t0 == 0;
    }
    // counters: one set of atomics per warp when every lane works for the same root
    const unsigned full = 0xFFFFFFFFu;
    const bool same = __all_sync(full, root == __shfl_sync(full, root, 0));
    const int64_t row = (int64_t)root * depth_total + level;
    if (same) {
        if (root == 0xFFFFFFFFu) return;  // a warp beyond the end
        const uint32_t T0 = __reduce_add_sync(full, t0), W0 = __reduce_add_sync(full, w0), Z0 = __reduce_add_sync(full, z0);
        const uint32_t T1 = __reduce_add_sync(full, t1), W1 = __reduce_add_sync(full, w1), Z1 = __reduce_add_sync(full, z1);
        if ((threadIdx.x & 31) == 0) {
            if (T0) atomicAdd(&nodes[row], (unsigned long long)T0);
            if (W0) atomicAdd(&wins[row], (unsigned long long)W0);
            if (Z0) atomicAdd(&zero[row], (unsigned long long)Z0);
            if (T1) atomicAdd(&nodes[row + 1], (unsigned long long)T1);
            if (W1) atomicAdd(&wins[row + 1], (unsigned long long)W1);
            if (Z1) atomicAdd(&zero[row + 1], (unsigned long long)Z1);
        }
    } else if (live) {
        if (t0) atomicAdd(&nodes[row], (unsigned long long)t0);
        if (w0) atomicAdd(&wins[row], (unsigned long long)w0);
        if (z0) atomicAdd(&zero[row], (unsigned long long)z0);
        if (t1) atomicAdd(&nodes[row + 1], (unsigned long long)t1);
        if (w1) atomicAdd(&wins[row + 1], (unsigned long long)w1);
        if (z1) atomicAdd(&zero[row + 1], (unsigned long long)z1);
    }
}

static int32_t perft_fail(Ctx* c, cudaError_t e, const char* what) {
    snprintf(c->err, sizeof(c->err), "onb_perft: %s: %s", what, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? ONB_E_NOMEM : ONB_E_CUDA;
}

constexpr int kMaxDfs = 6;

static cudaError_t scratch_get(Ctx* c, int slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 16;
    if (c->scratch_cap[slot] < bytes) {
        if (c->scratch[slot]) cudaFree(c->scratch[slot]);
        c->scratch[slot] = nullptr;
        c->scratch_cap[slot] = 0;
        const size_t want = bytes + bytes / 8;  // a little headroom so similar calls do not reallocate
        cudaError_t e = cudaMalloc(&c->scratch[slot], want);
        if (e != cudaSuccess) return e;
        c->scratch_cap[slot] = want;
    }
    *out = c->scratch[slot];
    return cudaSuccess;
}

// Frontier -> counters for the `rem` plies that remain, in bounded memory: while more than two plies remain the frontier is expanded
// chunk by chunk into a per-level scratch pair and each chunk is finished recursively; two plies above the horizon k_perft_leaf2
// takes over. `slot` = first scratch slot of this recursion level (two slots per level).
static cudaError_t perft_finish(Ctx* c, const uint4* st, const uint32_t* rt, int64_t n_items, unsigned long long* nodes, unsigned long long* wins,
                                unsigned long long* zero, unsigned long long* d_cursor, int depth, int level, int slot) {
    const int rem = depth - level;
    if (n_items <= 0 || rem <= 0) return cudaSuccess;
    if (rem == 1) return launch_dfs<1>(c, st, rt, n_items, nodes, wins, zero, depth);
    if (rem == 2) {
        k_perft_leaf2<<<(unsigned)((n_items + 255) / 256), 256, 0, c->stream>>>(st, rt, n_items, nodes, wins, zero, depth, level);
        return cudaGetLastError();
    }
    if (slot + 1 >= 16) return cudaErrorInvalidValue;
    const int64_t chunk = 8 << 20;  // parents per chunk: at most 40 children each -> the child frontier stays below 6.7 GB
    for (int64_t off = 0; off < n_items; off += chunk) {
        const int64_t m = n_items - off < chunk ? n_items - off : chunk;
        unsigned long long total = 0;
        cudaError_t e = cudaMemsetAsync(d_cursor, 0, 8, c->stream);
        if (e != cudaSuccess) return e;
        k_perft_expand<true><<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(st + off, rt + off, m, nullptr, nullptr, d_cursor, nodes, wins, zero, depth,
                                                                                level);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if ((e = cudaMemcpyAsync(&total, d_cursor, 8, cudaMemcpyDeviceToHost, c->stream)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
        uint4* ns = nullptr;
        uint32_t* nr = nullptr;
        const bool leaf_next = depth - (level + 1) == 2;  // the children go straight to k_perft_leaf2: 16-byte entries with the root inside
        if ((e = scratch_get(c, slot, (size_t)total * 16, (void**)&ns)) != cudaSuccess) return e;
        if (!leaf_next && (e = scratch_get(c, slot + 1, (size_t)total * 4, (void**)&nr)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(d_cursor, 0, 8, c->stream)) != cudaSuccess) return e;
        k_perft_expand<false><<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(st + off, rt + off, m, ns, nr, d_cursor, nodes, wins, zero, depth, level);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if ((e = perft_finish(c, ns, nr, (int64_t)total, nodes, wins, zero, d_cursor, depth, level + 1, slot + 2)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

int32_t run_perft(Ctx* c, const onb_state* roots_host, int64_t n, int depth, uint64_t* nodes_host, uint64_t* wins_host, uint64_t* zero_host) {
    cudaError_t e;
    const size_t cnt = (size_t)n * depth;
    unsigned long long *d_nodes = nullptr, *d_wins = nullptr, *d_zero = nullptr, *d_cursor = nullptr;
    uint4* cur_s = nullptr; uint32_t* cur_r = nullptr;
    uint4* nxt_s = nullptr; uint32_t* nxt_r = nullptr;
    int pair = 0;  // which scratch pair (4/5 or 6/7) holds the current frontier
    int32_t rc = ONB_OK;
#define PF(call, what) do { e = (call); if (e != cudaSuccess) { rc = perft_fail(c, e, what); goto done; } } while (0)
    PF(scratch_get(c, 0, cnt * 8, (void**)&d_nodes), "alloc counters");
    PF(scratch_get(c, 1, cnt * 8, (void**)&d_wins), "alloc counters");
    PF(scratch_get(c, 2, cnt * 8, (void**)&d_zero), "alloc counters");
    PF(scratch_get(c, 3, 8, (void**)&d_cursor), "alloc cursor");
    PF(cudaMemsetAsync(d_nodes, 0, cnt * 8, c->stream), "memset");
    PF(cudaMemsetAsync(d_wins, 0, cnt * 8, c->stream), "memset");
    PF(cudaMemsetAsync(d_zero, 0, cnt * 8, c->stream), "memset");
    {
        // roots -> internal states. Roots that are already decided (State::current_state is a win) expand to nothing.
        std::vector<uint4> hs;
        std::vector<uint32_t> hr;
        hs.reserve((size_t)n); hr.reserve((size_t)n);
        for (int64_t i = 0; i < n; ++i) {
            const onb_state& s = roots_host[i];
            Game g;
            auto rev = [](uint32_t v) { uint32_t r = 0; for (int b = 0; b < 25; ++b) if (v & (1u << (31 - b))) r |= 1u << b; return r; };
            g.pawn_r = rev(s.pawns[0]); g.pawn_b = rev(s.pawns[1]); g.king_r = rev(s.kings[0]); g.king_b = rev(s.kings[1]);
            g.cards = (s.cards[0] & 15u) | ((s.cards[1] & 15u) << 4) | ((s.cards[2] & 15u) << 8) | ((s.cards[3] & 15u) << 12) | ((s.cards[4] & 15u) << 16);
            g.side = s.side & 1u; g.result = 0; g.passed = 0;
            if (current_state(g) != 0) continue;
            hs.push_back(pack(g)); hr.push_back((uint32_t)i);
        }
        int64_t n_cur = (int64_t)hs.size();
        if (n_cur > 0) {
            PF(scratch_get(c, 4, (size_t)n_cur * 16, (void**)&cur_s), "alloc frontier");
            PF(scratch_get(c, 5, (size_t)n_cur * 4, (void**)&cur_r), "alloc frontier");
            PF(cudaMemcpyAsync(cur_s, hs.data(), (size_t)n_cur * 16, cudaMemcpyHostToDevice, c->stream), "copy roots");
            PF(cudaMemcpyAsync(cur_r, hr.data(), (size_t)n_cur * 4, cudaMemcpyHostToDevice, c->stream), "copy roots");
            PF(cudaStreamSynchronize(c->stream), "sync");
            int level = 0;
            // breadth-first while the frontier is too small to fill 148 SMs or the remaining depth exceeds the DFS template range
            const int64_t bfs_nodes = 1 << 21;
            while (n_cur > 0 && ((depth - level) > kMaxDfs || ((depth - level) > 1 && n_cur < bfs_nodes))) {
                unsigned long long total = 0;
                PF(cudaMemsetAsync(d_cursor, 0, 8, c->stream), "memset");
                k_perft_expand<true><<<(unsigned)((n_cur + 127) / 128), 128, 0, c->stream>>>(cur_s, cur_r, n_cur, nullptr, nullptr, d_cursor, d_nodes, d_wins,
                                                                                            d_zero, depth, level);
                PF(cudaGetLastError(), "expand(count)");
                PF(cudaMemcpyAsync(&total, d_cursor, 8, cudaMemcpyDeviceToHost, c->stream), "copy cursor");
                PF(cudaStreamSynchronize(c->stream), "sync");
                if (total > (1ull << 31)) { snprintf(c->err, sizeof(c->err), "onb_perft: frontier of %llu nodes is too large", total); rc = ONB_E_OVERFLOW; goto done; }
                const int other = pair ^ 1;
                PF(scratch_get(c, 4 + 2 * other, (size_t)total * 16, (void**)&nxt_s), "alloc frontier");
                PF(scratch_get(c, 5 + 2 * other, (size_t)total * 4, (void**)&nxt_r), "alloc frontier");
                PF(cudaMemsetAsync(d_cursor, 0, 8, c->stream), "memset");
                k_perft_expand<false><<<(unsigned)((n_cur + 127) / 128), 128, 0, c->stream>>>(cur_s, cur_r, n_cur, nxt_s, nxt_r, d_cursor, d_nodes, d_wins,
                                                                                             d_zero, depth, level);
                PF(cudaGetLastError(), "expand(fill)");
                PF(cudaStreamSynchronize(c->stream), "sync");
                cur_s = nxt_s; cur_r = nxt_r;
                pair = other;
                n_cur = (int64_t)total;
                ++level;
            }
            const int rem = depth - level;
            const char* dfs_env = getenv("ONB_PERFT_DFS");  // exploration knob: finish with the flat DFS instead of expand + two-ply kernel
            if (!(dfs_env && dfs_env[0] == '1')) {
                PF(perft_finish(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, d_cursor, depth, level, 8), "finish");
            } else if (n_cur > 0 && rem > 0) {
                switch (rem) {
                    case 1: PF(launch_dfs<1>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                    case 2: PF(launch_dfs<2>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                    case 3: PF(launch_dfs<3>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                    case 4: PF(launch_dfs<4>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                    case 5: PF(launch_dfs<5>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                    default: PF(launch_dfs<6>(c, cur_s, cur_r, n_cur, d_nodes, d_wins, d_zero, depth), "dfs"); break;
                }
            }
        }
    }
    PF(cudaMemcpyAsync(nodes_host, d_nodes, cnt * 8, cudaMemcpyDeviceToHost, c->stream), "copy out");
    if (wins_host) PF(cudaMemcpyAsync(wins_host, d_wins, cnt * 8, cudaMemcpyDeviceToHost, c->stream), "copy out");
    if (zero_host) PF(cudaMemcpyAsync(zero_host, d_zero, cnt * 8, cudaMemcpyDeviceToHost, c->stream), "copy out");
    PF(cudaStreamSynchronize(c->stream), "sync");
#undef PF
done:
    return rc;
}

}  // namespace onb
