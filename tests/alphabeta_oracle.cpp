// =====================================================================================
// tests/alphabeta_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of the alpha-beta arena opponent (ONB_AGENT_ALPHABETA, DESIGN.md §5d) in the shape of the reference's
// onitama-game/src/ai/alpha_beta/mod.rs: a recursive negamax over State with generate_all_legal_moves and heap move vectors,
// make_move on a copy standing in for GameState::progress / undo. The rules come from the CPU oracle (oracle/onb_oracle.cpp,
// included below); the evaluation is restated here square by square and shares no code with the CUDA kernel's popcount form
// (csrc/onb_rules.cuh, eval_position).
//
// orc_alphabeta_batch: the search as defined (fail-hard alpha-beta); orc_minimax_batch: the same tree without pruning, the
// check on the pruning itself (same best move and score at the root, never more positions entered).
// =====================================================================================
#include "../oracle/onb_oracle.cpp"

namespace orc_ab {
using namespace orc;

static const int32_t WIN = 1000000;
static const uint16_t ACTION_NONE = 0xFFFF;

// V(color): pawns 100 + 4 * rows advanced from the own home row + 2 * (2 - |col - 2|); kings 6 * (6 - manhattan(king, enemy temple))
static int32_t side_value(const State& st, int color) {
    int32_t v = 0;
    const unsigned temple = color == RED ? BLUE_TEMPLE : RED_TEMPLE;  // Red marches on Blue's temple (square 2) and vice versa
    for (unsigned n = 0; n < 25; ++n) {
        const int row = (int)n / 5, col = (int)n % 5;
        const int centre = 2 - std::abs(col - 2);
        if (get_bit(st.pawns[color], n)) {
            const int advance = color == RED ? 4 - row : row;
            v += 100 + 4 * advance + 2 * centre;
        }
        if (get_bit(st.kings[color], n)) {
            const int dist = std::abs(row - (int)temple / 5) + std::abs(col - (int)temple % 5);
            v += 6 * (6 - dist);
        }
    }
    return v;
}
static int32_t evaluate(const State& st, int side_to_move) { return side_value(st, side_to_move) - side_value(st, enemy(side_to_move)); }

struct Search {
    bool prune;
    uint64_t nodes = 0;

    // returns the node's score from the view of `side`; *best (root only) = the chosen action
    int32_t negamax(const State& st, int side, int32_t alpha, int32_t beta, int depth, int ply, uint16_t* best) {
        ++nodes;
        if (depth == 0) return evaluate(st, side);
        std::vector<std::pair<unsigned, Move>> moves = st.generate_all_legal_moves(side);
        // a move that wins at once ends the search of this node: nothing scores higher
        for (const auto& cm : moves) {
            State child = st;
            if (is_win(child.make_move(cm.second, side, cm.first))) {
                if (best) *best = encode_action(cm.first, cm.second);
                return WIN - (ply + 1);
            }
        }
        std::vector<uint16_t> actions;
        if (moves.empty()) {  // no legal move: the two pass moves (DESIGN.md §2; the reference panics here)
            const unsigned base = side == RED ? 0u : 2u;
            actions.push_back(encode_pass(base));
            actions.push_back(encode_pass(base + 1));
        } else {
            for (const auto& cm : moves) actions.push_back(encode_action(cm.first, cm.second));
        }
        int32_t best_score = INT32_MIN;
        uint16_t best_action = ACTION_NONE;
        for (uint16_t a : actions) {
            State child = st;
            if (a & (1u << 13)) child.pass((a >> 10) & 3u);
            else { const DoneMove d = decode_action(a); child.make_move(d.mov, side, d.used_card_idx); }
            const int32_t score = -negamax(child, enemy(side), -beta, -alpha, depth - 1, ply + 1, nullptr);
            if (score > best_score) { best_score = score; best_action = a; }
            if (prune) {
                if (best_score > alpha) alpha = best_score;
                if (alpha >= beta) break;
            }
        }
        if (best) *best = best_action;
        if (!prune) return best_score;
        return alpha >= beta ? beta : alpha;  // fail-hard
    }
};

static void search_root(const orc_state& r, int depth, bool prune, uint16_t* best, int32_t* score, uint64_t* nodes) {
    const State st = to_state(r);
    if (r.result != 0 || st.current_state() != IN_PROGRESS) {  // a decided game is not searched
        *best = ACTION_NONE; *score = 0; *nodes = 0;
        return;
    }
    Search s{prune};
    uint16_t b = ACTION_NONE;
    *score = s.negamax(st, r.side, -WIN - 1, WIN + 1, depth, 0, &b);
    *best = b;
    *nodes = s.nodes;
}

static void batch(const orc_state* roots, int64_t n, int depth, int threads, bool prune, uint16_t* best, int32_t* score, uint64_t* nodes) {
    std::atomic<int64_t> next{0};
    auto work = [&]() {
        for (int64_t i; (i = next.fetch_add(1)) < n;) search_root(roots[i], depth, prune, best + i, score + i, nodes + i);
    };
    if (threads < 1) threads = 1;
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
}

}  // namespace orc_ab

extern "C" {
void orc_alphabeta_batch(const orc_state* roots, int64_t n, int depth, int threads, uint16_t* best, int32_t* score, uint64_t* nodes) {
    orc_ab::batch(roots, n, depth, threads, true, best, score, nodes);
}
void orc_minimax_batch(const orc_state* roots, int64_t n, int depth, int threads, uint16_t* best, int32_t* score, uint64_t* nodes) {
    orc_ab::batch(roots, n, depth, threads, false, best, score, nodes);
}
// eval of each position from the view of its side to move
void orc_ab_eval(const orc_state* g, int64_t n, int32_t* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = orc_ab::evaluate(orc::to_state(g[i]), g[i].side);
}
}
