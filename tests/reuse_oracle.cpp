// =====================================================================================
// tests/reuse_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of search-tree reuse between moves (onb_mcts_set_reuse, DESIGN.md §5e) on top of the CPU oracle's MctsArena
// (oracle/onb_oracle.cpp, included below unchanged):
//   * match: a child of the remembered root is kept when the game is undecided and the position the child's move leads to
//     (boards, five card slots, side to move) equals the game's current state;
//   * reroot: the kept subtree is the child and all its descendants, filtered from the arena in arena order (parent and children
//     renumbered, the new root has no parent, every other field unchanged);
//   * continue: max_playouts = the visit target, playouts = the new root's visits, then MctsArena::search as it is.
// A ReuseSet holds one remembered arena per game, like a context's pools.
// =====================================================================================
#include <memory>

#include "../oracle/onb_oracle.cpp"

namespace orc_reuse {
using namespace orc;

static uint16_t node_action(const MctsNode& nd) {
    return !nd.has_mov ? 0xFFFF : nd.is_pass ? encode_pass(nd.mov.used_card_idx) : encode_action(nd.mov.used_card_idx, nd.mov.mov);
}

// position the move of child `c` of the root leads to
static bool child_matches(const MctsArena& a, uint32_t c, const orc_state& cur) {
    State st = a.root_state;
    const MctsNode& nd = a.arena[c];
    if (nd.is_pass) st.pass(nd.mov.used_card_idx);
    else st.make_move(nd.mov.mov, a.root_color, nd.mov.used_card_idx);
    if ((int)cur.side != enemy(a.root_color)) return false;
    for (int k = 0; k < 5; ++k)
        if (st.deck[k] != cur.cards[k]) return false;
    return st.pawns[0] == cur.pawns[0] && st.pawns[1] == cur.pawns[1] && st.kings[0] == cur.kings[0] && st.kings[1] == cur.kings[1];
}

// the arena-order filter: nodes keep..end whose parent is kept, renumbered in order
static void reroot(MctsArena& a, uint32_t keep, const orc_state& cur) {
    const size_t size = a.arena.size();
    std::vector<int64_t> map(size, -1);
    std::vector<MctsNode> out;
    for (size_t i = keep; i < size; ++i) {
        const MctsNode& nd = a.arena[i];
        if (i != keep && (nd.parent < (int64_t)keep || map[(size_t)nd.parent] < 0)) continue;
        map[i] = (int64_t)out.size();
        out.push_back(nd);
    }
    for (size_t k = 0; k < out.size(); ++k) {
        MctsNode& nd = out[k];
        nd.parent = k == 0 ? -1 : map[(size_t)nd.parent];
        for (uint32_t& ch : nd.children) ch = (uint32_t)map[ch];
        nd.idx = (uint32_t)k;
    }
    a.arena.swap(out);
    a.root_state = to_state(cur);
    a.root_color = cur.side;
    a.pass_seen = false;
}

struct ReuseSet {
    std::vector<std::unique_ptr<MctsArena>> trees;
};

// one search of game i to `sims` root visits, keeping what the remembered tree allows; returns 1 if a child was kept
static int search_one(ReuseSet& rs, int64_t i, const orc_state& cur, double c_puct, uint32_t sims, eval_fn e, void* user, float pi[50], uint32_t* best,
                      uint32_t* sims_run) {
    std::unique_ptr<MctsArena>& t = rs.trees[(size_t)i];
    int kept = 0;
    if (t && cur.result == 0) {
        for (uint32_t c : t->arena[0].children)
            if (child_matches(*t, c, cur)) {
                reroot(*t, c, cur);
                kept = 1;
                break;
            }
    }
    if (!kept) t.reset(new MctsArena(to_state(cur), cur.side, c_puct, sims, e, user));
    t->exploration_c = c_puct;
    t->eval = e;
    t->user = user;
    apply_noise_cfg(*t, (uint64_t)i);
    t->max_playouts = sims;
    t->playouts = t->arena[0].visits;
    const uint32_t before = t->playouts;
    *best = t->search(pi);
    *sims_run = t->playouts > before ? t->playouts - before : 0u;
    return kept;
}

static uint16_t best_code(const MctsArena& a, uint32_t best) {
    if (a.arena[0].children.empty()) return 0xFFFF;
    return node_action(a.arena[best]);
}

}  // namespace orc_reuse

extern "C" {

void* orc_reuse_new(int64_t n) {
    orc_reuse::ReuseSet* rs = new orc_reuse::ReuseSet();
    rs->trees.resize((size_t)n);
    return rs;
}
void orc_reuse_free(void* h) { delete static_cast<orc_reuse::ReuseSet*>(h); }

// per game: reroot (or start fresh) and search to `sims` root visits. evaluator: 0 uniform, 1 hash, 2 the callback `cb` (run with
// threads = 1). Any output may be NULL.
void orc_reuse_search(void* h, const orc_state* states, int64_t n, double c_puct, uint32_t sims, int evaluator, orc::eval_fn cb, void* user, int threads,
                      uint16_t* best_actions,
                      float* pi50, uint32_t* root_visits, double* root_q, uint32_t* child_visits40, int64_t* n_nodes, int32_t* kept,
                      uint32_t* sims_run) {
    orc_reuse::ReuseSet& rs = *static_cast<orc_reuse::ReuseSet*>(h);
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            float pi[50];
            uint32_t best = 0, run = 0;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : evaluator == 1 ? orc::hash_eval : cb;
            const int k = orc_reuse::search_one(rs, i, states[i], c_puct, sims, e, user, pi, &best, &run);
            const orc::MctsArena& a = *rs.trees[(size_t)i];
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = orc_reuse::best_code(a, best);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (kept) kept[i] = k;
            if (sims_run) sims_run[i] = run;
        }
    };
    if (threads <= 1) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}

// the remembered tree of game i (same layout as orc_mcts_search's dump); returns the node count (0: no tree)
int64_t orc_reuse_dump(void* h, int64_t i, orc_tree_dump* dump, int64_t cap) {
    orc_reuse::ReuseSet& rs = *static_cast<orc_reuse::ReuseSet*>(h);
    if (!rs.trees[(size_t)i]) return 0;
    const orc::MctsArena& a = *rs.trees[(size_t)i];
    const int64_t nn = (int64_t)a.arena.size();
    if (dump && cap >= nn) {
        for (int64_t k = 0; k < nn; ++k) {
            const orc::MctsNode& nd = a.arena[(size_t)k];
            dump->visits[k] = nd.visits; dump->reward[k] = nd.reward; dump->winrate[k] = nd.winrate; dump->prior[k] = nd.probability;
            dump->action[k] = orc_reuse::node_action(nd);
            dump->parent[k] = (int32_t)nd.parent;
            dump->first_child[k] = nd.children.empty() ? 0u : nd.children[0];
            dump->n_child[k] = (uint32_t)nd.children.size();
            dump->flags[k] = (uint8_t)((nd.is_expanded ? 1 : 0) | (nd.is_terminal ? 2 : 0) | (nd.is_pass ? 4 : 0));
        }
    }
    return nn;
}

// whole games from the given start states, one search per ply (to `sims` root visits; reuse = 0: a fresh tree every ply), the
// best move played, until a win or max_plies + 2 plies (train.rs:74-79). Per game and ply (stride max_plies + 2): pi [50], side to
// move; per game: plies, result, simulations run.
void orc_reuse_play_games(const orc_state* starts, int64_t n, double c_puct, uint32_t sims, int evaluator, uint32_t max_plies, int reuse, int threads,
                          float* pi_out, uint8_t* color_out, int32_t* plies_out, uint8_t* result_out, uint64_t* sims_out) {
    const int64_t stride = (int64_t)max_plies + 2;
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            orc_reuse::ReuseSet rs;
            rs.trees.resize((size_t)i + 1);
            orc_state g = starts[i];
            int32_t ply = 0;
            uint64_t total = 0;
            while (g.result == 0 && ply < stride) {
                if (!reuse) rs.trees[(size_t)i].reset();
                float pi[50];
                uint32_t best = 0, run = 0;
                orc_reuse::search_one(rs, i, g, c_puct, sims, evaluator == 0 ? orc::uniform_eval : orc::hash_eval, nullptr, pi, &best, &run);
                total += run;
                memcpy(pi_out + (i * stride + ply) * 50, pi, sizeof(pi));
                color_out[i * stride + ply] = g.side;
                orc::apply_action(g, orc_reuse::best_code(*rs.trees[(size_t)i], best));
                ++ply;
            }
            plies_out[i] = ply;
            result_out[i] = g.result;
            sims_out[i] = total;
        }
    };
    if (threads <= 1) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}

}  // extern "C"
