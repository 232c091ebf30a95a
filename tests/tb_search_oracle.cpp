// =====================================================================================
// tests/tb_search_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of tablebase leaves (onb_mcts_set_tablebase, DESIGN.md §5i) on the CPU oracle's MctsArena (oracle/onb_oracle.cpp,
// included unchanged through tests/vl_oracle.cpp, whose rounds the virtual-loss mode follows). A leaf below the root whose position
// the table holds is not expanded and backs up the reward of a decided leaf whose winner is the table's winner; the root is expanded
// as always and backs up the table's reward. The table is probed through tests/tablebase_oracle.cpp's index: the caller passes that
// library's orc_tb_probe and the tables as 25 class pointers (solved by orc_tb_solve or copied from the device).
// =====================================================================================
#include "vl_oracle.cpp"

namespace orc_tbs {
using namespace orc;

static const int16_t NONE = -32768;
// tests/tablebase_oracle.cpp's orc_tb_probe: the value of each game as onb_tb_probe defines it
typedef void (*probe_fn)(const uint8_t* cards, int max_pawns, int16_t* const* tables, const orc_state* g, int64_t n, int16_t* out);

struct Table {
    const uint8_t* cards;
    int max_pawns;
    int16_t* const* tables;
    probe_fn probe;
    int16_t value(const State& st, int color) const {
        orc_state g;
        memset(&g, 0, sizeof(g));
        from_state(st, g);
        g.side = (uint8_t)color;
        int16_t v = NONE;
        probe(cards, max_pawns, tables, &g, 1, &v);
        return v;
    }
};

// the reward a leaf of table value v != NONE backs up: a decided leaf's reward (reward_fn) whose winner is the table's winner -- the
// side to move at the leaf (leaf_color) if v > 0, the other side if v < 0 -- and 0 for a draw. reward_color: the colour of the leaf's
// parent, the root's own colour at the root.
static double tb_reward(int16_t v, int leaf_color, int reward_color) {
    if (v == 0) return 0.0;
    const int winner = v > 0 ? leaf_color : enemy(leaf_color);
    return reward_fn(winner == RED ? RED_WIN : BLUE_WIN, reward_color);
}

struct TbArena : orc_vl::VlArena {
    Table T;

    TbArena(const State& s, int color, double c, uint32_t sims, eval_fn e, void* u, uint32_t k, double vl_, const Table& t)
        : VlArena(s, color, c, sims, e, u, k, vl_), T(t) {}

    struct Leaf {
        uint32_t node;
        int result, color;
        int16_t v;
        EvaluationResult ev;
    };

    // from the root to a leaf: MctsArena::playout's descent, or vl_oracle's on virtual statistics (v != nullptr)
    Leaf descend(std::map<uint32_t, uint32_t>* v) {
        State st = root_state;
        int color = root_color;
        uint32_t node_idx = 0;
        std::vector<uint32_t> path(1, 0u);
        while (arena[node_idx].is_expanded && !arena[node_idx].is_terminal) {
            node_idx = v ? select_vl(node_idx, *v) : select(arena[node_idx]);
            if (arena[node_idx].has_mov) {
                int64_t parent = arena[node_idx].parent;
                const DoneMove& mv = arena[node_idx].mov;
                int r = arena[node_idx].is_pass ? st.pass(mv.used_card_idx) : st.make_move(mv.mov, arena[parent].player_color, mv.used_card_idx);
                color = enemy(color);
                if (is_win(r)) arena[node_idx].is_terminal = true;
            }
            path.push_back(node_idx);
        }
        if (v)
            for (uint32_t p : path) (*v)[p] += 1;
        Leaf l;
        l.node = node_idx;
        l.result = st.current_state();
        l.color = color;
        l.v = is_win(l.result) ? NONE : T.value(st, color);
        l.ev = evaluate(st, color);  // every leaf is evaluated, as every row goes through the evaluator; a table leaf's is ignored
        return l;
    }

    // expansion and backup of one leaf under the rule
    void finish(const Leaf& l) {
        const bool table = l.v != NONE;
        if (!(table && l.node != 0) && !arena[l.node].is_expanded && !arena[l.node].is_terminal) expand(l.node, l.ev);
        int64_t parent = arena[l.node].parent >= 0 ? arena[l.node].parent : 0;
        int reward_color = arena[parent].player_color;
        back_propagate(l.node, table ? tb_reward(l.v, l.color, reward_color) : is_win(l.result) ? reward_fn(l.result, reward_color) : l.ev.value);
    }

    uint32_t search(float pi[50]) {
        uint32_t done = 0;
        while (done < max_playouts) {
            const uint32_t b = leaves <= 1 ? 1u : done == 0 ? 1u : std::min(leaves, max_playouts - done);
            if (leaves <= 1) {
                finish(descend(nullptr));
            } else {  // vl_oracle's round: b descents on virtual statistics, then the leaves in descent order
                std::map<uint32_t, uint32_t> v;
                std::vector<Leaf> lv;
                for (uint32_t j = 0; j < b; ++j) lv.push_back(descend(&v));
                for (const Leaf& l : lv) finish(l);
            }
            done += b;
            rounds += 1;
        }
        playouts = done;
        return MctsArena::search(pi);
    }
};

}  // namespace orc_tbs

extern "C" {

// searches of n roots with tablebase leaves: leaves <= 1 one descent per simulation, K >= 2 virtual loss vl in rounds of K; the
// table: cards, max_pawns, 25 class pointers and tests/tablebase_oracle.cpp's orc_tb_probe. Outputs as orc_vl_search_batch's.
void orc_tbs_search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, int threads, uint32_t leaves, double vl,
                          const uint8_t* cards, int max_pawns, int16_t* const* tables, orc_tbs::probe_fn probe, uint16_t* best_actions, float* pi50,
                          uint32_t* root_visits, double* root_q, uint32_t* child_visits40, int64_t* n_nodes, int64_t dump_tree, orc_tree_dump* dump,
                          int64_t cap) {
    const orc_tbs::Table T{cards, max_pawns, tables, probe};
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : orc::hash_eval;
            orc_tbs::TbArena a(orc::to_state(roots[i]), roots[i].side, c_puct, sims, e, nullptr, leaves, vl, T);
            float pi[50];
            const uint32_t best = a.search(pi);
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = ch.empty() ? 0xFFFF : orc_vl::node_action(a.arena[best]);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (dump && i == dump_tree && cap >= (int64_t)a.arena.size()) orc_vl::dump_arena(a, dump);
        }
    };
    if (threads <= 1) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}

// the rule's reward of a leaf of table value v (!= NONE) at depth `depth` whose side to move is leaf_color
double orc_tbs_reward(int16_t v, int depth, int leaf_color) {
    return orc_tbs::tb_reward(v, leaf_color, depth ? orc::enemy(leaf_color) : leaf_color);
}

}  // extern "C"
