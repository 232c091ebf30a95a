// =====================================================================================
// tests/solver_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of the MCTS solver (onb_mcts_set_solver, include/onb.h, DESIGN.md §5k) on the CPU oracle's MctsArena, through
// tests/tb_search_oracle.cpp's descent and leaf rule (one descent per simulation; tablebase leaves optional). Proofs are kept in a
// per-node byte next to the arena: WIN = the side that moved into the node wins with best play, LOSS = it loses. Immediate wins are
// found by playing each new child's move on a copy of the leaf's State (State::make_move's own test), not by the kernels' square test.
// =====================================================================================
#include "tb_search_oracle.cpp"

namespace orc_sol {
using namespace orc;

static const uint8_t WIN = 8, LOSS = 16;

// the propagation rule from node x, just proven (proof[x] != 0), up the parent chain; stops at the first level that does not change
static void propagate(const std::vector<int64_t>& parent, const std::vector<std::vector<uint32_t>>& children, std::vector<uint8_t>& proof, uint32_t x) {
    for (;;) {
        const int64_t y = parent[x];
        if (y < 0 || proof[y]) return;
        uint8_t fy = LOSS;
        if (proof[x] != WIN) {
            for (uint32_t c : children[y])
                if (proof[c] != LOSS) return;
            fy = WIN;
        }
        proof[y] = fy;
        x = (uint32_t)y;
    }
}

struct SolverArena : orc_tbs::TbArena {
    bool solver, table;
    std::vector<uint8_t> proof;

    SolverArena(const State& s, int color, double c, uint32_t sims, eval_fn e, bool solver_, bool table_, const orc_tbs::Table& t)
        : TbArena(s, color, c, sims, e, nullptr, 1, 1.0, t), solver(solver_), table(table_), proof(1, 0) {}

    // MctsArena::select (eval mode) over the children not proven LOSS: the last maximal one
    uint32_t select_solver(uint32_t x) const {
        const MctsNode& parent = arena[x];
        auto uct = [&](const MctsNode& child) {
            return child.winrate + exploration_c * child.probability * (std::sqrt((double)parent.visits) / (double)(child.visits + 1));
        };
        int64_t best = -1;
        for (uint32_t c : parent.children) {
            if (proof[c] == LOSS) continue;
            if (best < 0 || total_key(uct(arena[c])) >= total_key(uct(arena[best]))) best = c;
        }
        return (uint32_t)best;
    }

    struct Leaf {
        uint32_t node;
        int result, color;
        int16_t v;
        State st;
        EvaluationResult ev;
    };

    Leaf descend() {
        State st = root_state;
        int color = root_color;
        uint32_t x = 0;
        while (arena[x].is_expanded && !arena[x].is_terminal && !(solver && proof[x])) {
            x = solver ? select_solver(x) : select(arena[x]);
            if (arena[x].has_mov) {
                const int64_t parent = arena[x].parent;
                const DoneMove& mv = arena[x].mov;
                const int r = arena[x].is_pass ? st.pass(mv.used_card_idx) : st.make_move(mv.mov, arena[parent].player_color, mv.used_card_idx);
                color = enemy(color);
                if (is_win(r)) {
                    arena[x].is_terminal = true;
                    if (solver) proof[x] = WIN;
                }
            }
        }
        Leaf l;
        l.node = x;
        l.result = st.current_state();
        l.color = color;
        l.v = table && !is_win(l.result) ? T.value(st, color) : orc_tbs::NONE;
        l.st = st;
        l.ev = evaluate(st, color);
        return l;
    }

    void finish(const Leaf& l) {
        const uint32_t x = l.node;
        const bool tleaf = l.v != orc_tbs::NONE;
        if (!(tleaf && x != 0) && !arena[x].is_expanded && !arena[x].is_terminal) {
            expand(x, l.ev);
            proof.resize(arena.size(), 0);
            if (solver) {
                bool born = false;
                for (uint32_t c : arena[x].children) {
                    State s2 = l.st;
                    const DoneMove& mv = arena[c].mov;
                    const int r = arena[c].is_pass ? s2.pass(mv.used_card_idx) : s2.make_move(mv.mov, arena[x].player_color, mv.used_card_idx);
                    if (is_win(r)) {
                        arena[c].is_terminal = true;
                        proof[c] = WIN;
                        born = true;
                    }
                }
                if (born) proof[x] = LOSS;
            }
        }
        if (solver && tleaf && x != 0 && l.v != 0) proof[x] = l.v > 0 ? LOSS : WIN;
        const int64_t parent = arena[x].parent >= 0 ? arena[x].parent : 0;
        const int reward_color = arena[parent].player_color;
        double reward;
        if (solver && proof[x]) {  // a decided leaf whose winner is the proven winner
            const int winner = proof[x] == WIN ? enemy(l.color) : l.color;
            reward = reward_fn(winner == RED ? RED_WIN : BLUE_WIN, reward_color);
        } else {
            reward = tleaf ? orc_tbs::tb_reward(l.v, l.color, reward_color) : is_win(l.result) ? reward_fn(l.result, reward_color) : l.ev.value;
        }
        back_propagate(x, reward);
        if (solver && proof[x] && x != 0) {
            std::vector<int64_t> par(arena.size());
            std::vector<std::vector<uint32_t>> ch(arena.size());
            for (size_t i = 0; i < arena.size(); ++i) {
                par[i] = arena[i].parent;
                ch[i] = arena[i].children;
            }
            propagate(par, ch, proof, x);
        }
    }

    uint32_t search(float pi[50]) {
        while (playouts < max_playouts) {
            finish(descend());
            playouts += 1;
        }
        uint32_t best = MctsArena::search(pi);  // pi, and the visit rule
        const auto& ch = arena[0].children;
        if (!solver || ch.empty()) return best;
        for (uint32_t c : ch)
            if (arena[c].is_terminal && proof[c] == WIN) return c;
        bool any_win = false, any_open = false;
        for (uint32_t c : ch) {
            any_win |= proof[c] == WIN;
            any_open |= proof[c] != LOSS;
        }
        int64_t b = -1;
        for (uint32_t c : ch) {
            const bool ok = any_win ? proof[c] == WIN : any_open ? proof[c] != LOSS : true;
            if (!ok) continue;
            const double a = (double)arena[c].visits / (double)arena[0].visits;
            if (b < 0 || total_key(a) >= total_key((double)arena[b].visits / (double)arena[0].visits)) b = c;
        }
        return (uint32_t)b;
    }
};

}  // namespace orc_sol

extern "C" {

// searches of n roots; solver: the switch; table != 0: tablebase leaves with cards / max_pawns / 25 class pointers / orc_tb_probe.
// Outputs as orc_tbs_search_batch's, plus proof [n] (+1 root LOSS, -1 root WIN, 0) and the dumped tree's flags with the proof bits.
void orc_sol_search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, int threads, int solver, int table,
                          const uint8_t* cards, int max_pawns, int16_t* const* tables, orc_tbs::probe_fn probe, uint16_t* best_actions, float* pi50,
                          uint32_t* root_visits, double* root_q, uint32_t* child_visits40, int64_t* n_nodes, int8_t* proof, int64_t dump_tree,
                          orc_tree_dump* dump, int64_t cap) {
    const orc_tbs::Table T{cards, max_pawns, tables, probe};
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : orc::hash_eval;
            orc_sol::SolverArena a(orc::to_state(roots[i]), roots[i].side, c_puct, sims, e, solver != 0, table != 0, T);
            float pi[50];
            const uint32_t best = a.search(pi);
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = ch.empty() ? 0xFFFF : orc_vl::node_action(a.arena[best]);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (proof) proof[i] = a.proof[0] == orc_sol::LOSS ? 1 : a.proof[0] == orc_sol::WIN ? -1 : 0;
            if (dump && i == dump_tree && cap >= (int64_t)a.arena.size()) {
                orc_vl::dump_arena(a, dump);
                for (size_t j = 0; j < a.arena.size(); ++j) dump->flags[j] |= a.proof[j];
            }
        }
    };
    if (threads <= 1) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}

// the propagation rule on a hand-built tree of m nodes (parent[i] < 0 for the root; children of i: [first_child[i], + n_child[i])):
// proof [m] (0 / 8 / 16) is updated in place from node x, whose proof is already set
void orc_sol_propagate(int64_t m, const int32_t* parent, const uint32_t* first_child, const uint32_t* n_child, uint8_t* proof, uint32_t x) {
    std::vector<int64_t> par(m);
    std::vector<std::vector<uint32_t>> ch(m);
    std::vector<uint8_t> pr(proof, proof + m);
    for (int64_t i = 0; i < m; ++i) {
        par[i] = parent[i];
        for (uint32_t c = 0; c < n_child[i]; ++c) ch[i].push_back(first_child[i] + c);
    }
    orc_sol::propagate(par, ch, pr, x);
    memcpy(proof, pr.data(), (size_t)m);
}

}  // extern "C"
