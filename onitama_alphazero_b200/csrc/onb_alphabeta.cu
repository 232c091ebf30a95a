// onb_alphabeta.cu -- the alpha-beta arena opponent (ONB_AGENT_ALPHABETA, DESIGN.md §5d): a fixed-depth negamax with
// alpha-beta pruning (fail-hard), one game per thread.
//
// The search is the flat state machine of k_perft_flat (onb_perft.cu): the node being searched lives in registers, the
// nodes above it in a shared-memory stack ([level][word][thread], conflict free), and every loop iteration plays exactly ONE
// move, so the lanes of a warp run the same short instruction stream even though each searches its own tree.
#include "onb_internal.h"
#include "onb_rules.cuh"

namespace onb {

constexpr int kAbThreads = 128;
// op, ok, ep, ek, cards | side << 20 | slot << 21, piece iterator, destinations | from << 25, alpha, beta
constexpr int kAbWords = 9;
constexpr uint32_t kAbPassFrom = 31;  // `from` of the two pass children of a node without a legal move (destination bit = hand slot)

struct AbScan {
    uint32_t moves;  // union of all destinations (0: no legal move)
    uint32_t wins;   // union of the destinations of moves that win at once (capture the enemy king / own king on the enemy temple)
};
// the win mask is the one of bulk_count: the enemy king's square (unless a pawn shares it: the pawn would be captured), plus the
// enemy temple for the king's moves -- exactly the moves for which apply_move_rel returns non-zero
__device__ __forceinline__ AbScan ab_scan(const uint32_t* T, const RelGame& g) {
    const uint32_t own = g.op | g.ok;
    const uint32_t win_t = g.ek & ~g.ep;
    const uint32_t temple = 1u << (g.side ? kRedTemple : kBlueTemple);
    const uint32_t* T0 = T + (g.side * 16u + card_at(g.cards, g.side * 2u)) * 25u;
    const uint32_t* T1 = T + (g.side * 16u + card_at(g.cards, g.side * 2u + 1u)) * 25u;
    AbScan s{0, 0};
    uint32_t rem = own;
    while (rem) {
        const int f = __ffs(rem) - 1;
        rem &= rem - 1;
        const uint32_t a = (T0[f] | T1[f]) & ~own;
        s.moves |= a;
        s.wins |= a & (win_t | (((g.op >> f) & 1u) ? 0u : temple));
    }
    return s;
}
// the first winning move in generation order (hand slot, from, to ascending); only asked for at the root
__device__ __forceinline__ uint32_t ab_first_win(const uint32_t* T, const RelGame& g) {
    const uint32_t own = g.op | g.ok;
    const uint32_t win_t = g.ek & ~g.ep;
    const uint32_t temple = 1u << (g.side ? kRedTemple : kBlueTemple);
    for (uint32_t s = 0; s < 2; ++s) {
        const uint32_t* Ts = T + (g.side * 16u + card_at(g.cards, g.side * 2u + s)) * 25u;
        uint32_t rem = own;
        while (rem) {
            const int f = __ffs(rem) - 1;
            rem &= rem - 1;
            const uint32_t king = ((g.op >> f) & 1u) ^ 1u;
            const uint32_t w = Ts[f] & ~own & (win_t | (king ? temple : 0u));
            if (w) return make_action(g.side * 2u + s, (uint32_t)f, (uint32_t)(__ffs(w) - 1), king);
        }
    }
    return 0xFFFFu;  // unreachable when ab_scan found a win
}

// Searches games[i] (i < m; games == nullptr: game i) to `depth` plies. out[game] = best action (ONB_ACTION_NONE for a decided
// game); score_out / nodes_out (optional) [game] = the root's negamax score and the number of positions entered.
__global__ void __launch_bounds__(kAbThreads) k_alphabeta(const uint4* __restrict__ states, const int32_t* __restrict__ games, int64_t m, int depth,
                                                          uint16_t* __restrict__ out, int32_t* __restrict__ score_out,
                                                          unsigned long long* __restrict__ nodes_out) {
    __shared__ __align__(16) uint32_t s_att[800];
    __shared__ uint32_t s_stk[(ONB_ALPHABETA_MAX_DEPTH - 1) * kAbWords * kAbThreads];  // levels 0 .. depth-2 can have a level below them
    load_attack_table_to_smem(s_att);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int64_t game = games ? (int64_t)games[i] : i;
    const Game g0 = unpack(states[game]);
    if (g0.result != 0 || current_state(g0) != 0) {  // a decided game is not searched
        out[game] = 0xFFFFu;
        if (score_out) score_out[game] = 0;
        if (nodes_out) nodes_out[game] = 0;
        return;
    }
    RelGame g = to_rel(g0);
    unsigned long long nodes = 1;
    uint32_t best_action = 0xFFFFu, root_try = 0;
    int32_t root_score = 0;
    int32_t alpha = -kAlphaBetaWin - 1, beta = kAlphaBetaWin + 1;  // the root's window: its score is exact
    uint32_t level = 0;
    uint32_t it = 0, cur = 0, cur_f = 0, cur_slot = 0;  // unvisited pieces of the hand slot, unplayed destinations of the current piece
    bool done = false;
    {
        const AbScan sc = ab_scan(s_att, g);
        if (sc.wins) {
            best_action = ab_first_win(s_att, g);
            root_score = kAlphaBetaWin - 1;
            done = true;
        } else if (!sc.moves) {
            cur_slot = 1; cur = 3u; cur_f = kAbPassFrom;  // the two pass moves are the children
        } else {
            it = g.op | g.ok;
        }
    }
    while (!done) {
        bool fin = false;  // the node at `level` is finished with value v
        int32_t v = 0;
        // (1) find the next move: advance over pieces and hand slots; light, so that step (2) runs on all lanes together
        while (cur == 0) {
            if (it) {
                const int f = __ffs(it) - 1;
                it &= it - 1;
                cur = s_att[(g.side * 16u + card_at(g.cards, g.side * 2u + cur_slot)) * 25u + f] & ~(g.op | g.ok);
                cur_f = (uint32_t)f;
            } else if (cur_slot == 0) {
                cur_slot = 1;
                it = g.op | g.ok;
            } else {  // every child was searched without a cut-off
                fin = true;
                v = alpha;
                break;
            }
        }
        if (!fin) {
            // (2) play one move
            const uint32_t to = __ffs(cur) - 1;
            cur &= cur - 1;
            const uint32_t action = cur_f == kAbPassFrom ? (kPassBit | ((g.side * 2u + to) << 10))
                                                         : make_action(g.side * 2u + cur_slot, cur_f, to, ((g.op >> cur_f) & 1u) ^ 1u);
            RelGame ch = g;
            apply_move_rel(ch, action);  // never a win: a node with a winning move is not expanded
            if (level == 0) root_try = action;
            if (level + 1 == (uint32_t)depth) {  // the child is a leaf
                ++nodes;
                const int32_t s = -eval_position(ch);
                if (s > alpha) {
                    alpha = s;
                    if (level == 0) best_action = action;
                }
                if (alpha >= beta) { fin = true; v = beta; }
            } else {  // descend: save this node, the child becomes the current node
                uint32_t* p = s_stk + (level * kAbWords) * kAbThreads + threadIdx.x;
                p[0 * kAbThreads] = g.op; p[1 * kAbThreads] = g.ok; p[2 * kAbThreads] = g.ep; p[3 * kAbThreads] = g.ek;
                p[4 * kAbThreads] = g.cards | (g.side << 20) | (cur_slot << 21);
                p[5 * kAbThreads] = it;
                p[6 * kAbThreads] = cur | (cur_f << 25);
                p[7 * kAbThreads] = (uint32_t)alpha;
                p[8 * kAbThreads] = (uint32_t)beta;
                ++level;
                g = ch;
                const int32_t a2 = -beta;
                beta = -alpha;
                alpha = a2;
                ++nodes;
                const AbScan sc = ab_scan(s_att, g);
                it = 0; cur = 0; cur_f = 0; cur_slot = 0;
                if (sc.wins) {
                    fin = true;
                    v = kAlphaBetaWin - (int32_t)(level + 1);
                } else if (!sc.moves) {
                    cur_slot = 1; cur = 3u; cur_f = kAbPassFrom;
                } else {
                    it = g.op | g.ok;
                }
            }
        }
        // (3) hand finished nodes' values up; a parent that cuts off is finished too (fail-hard: it returns beta)
        while (fin) {
            if (level == 0) {
                root_score = v;
                done = true;
                break;
            }
            --level;
            const uint32_t* p = s_stk + (level * kAbWords) * kAbThreads + threadIdx.x;
            g.op = p[0 * kAbThreads]; g.ok = p[1 * kAbThreads]; g.ep = p[2 * kAbThreads]; g.ek = p[3 * kAbThreads];
            const uint32_t cs = p[4 * kAbThreads];
            g.cards = cs & 0xFFFFFu; g.side = (cs >> 20) & 1u; cur_slot = (cs >> 21) & 1u;
            it = p[5 * kAbThreads];
            const uint32_t cw = p[6 * kAbThreads];
            cur = cw & kAll25; cur_f = cw >> 25;
            alpha = (int32_t)p[7 * kAbThreads];
            beta = (int32_t)p[8 * kAbThreads];
            const int32_t s = -v;
            if (s > alpha) {
                alpha = s;
                if (level == 0) best_action = root_try;
            }
            if (alpha >= beta) v = beta;
            else fin = false;
        }
    }
    out[game] = (uint16_t)best_action;
    if (score_out) score_out[game] = root_score;
    if (nodes_out) nodes_out[game] = nodes;
}

cudaError_t launch_alphabeta(Ctx* c, int depth, const int32_t* d_games, int64_t m, uint16_t* d_out, int32_t* d_score, unsigned long long* d_nodes) {
    if (m <= 0) return cudaSuccess;
    k_alphabeta<<<(unsigned)((m + kAbThreads - 1) / kAbThreads), kAbThreads, 0, c->stream>>>(c->d_states, d_games, m, depth, d_out, d_score, d_nodes);
    return cudaGetLastError();
}

}  // namespace onb
