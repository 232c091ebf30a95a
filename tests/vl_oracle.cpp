// =====================================================================================
// tests/vl_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h) on the CPU oracle's MctsArena
// (oracle/onb_oracle.cpp, included below unchanged): the search runs in rounds; a round takes its b descents one after the other
// on virtual statistics kept in a map of pending descents, evaluates every leaf through the oracle's evaluator callbacks, then
// expands and backs up the leaves in descent order.
// =====================================================================================
#include <map>

#include "../oracle/onb_oracle.cpp"

namespace orc_vl {
using namespace orc;

// The choice at a node x with k children (DESIGN.md §5h): P the priors, N the visits, W the reward sums, V the pending descents of the
// round, np = N(x) + v(x). u = q' + (c P) (sqrt(np) / (N' + 1)), N' = N + V, W' = W (V = 0) or W - vl V, q' = W' / N' (0 if N' = 0);
// returns the position of the LAST maximal child under f64::total_cmp.
static size_t vl_choice(size_t k, const double* P, const uint32_t* N, const double* W, const uint32_t* V, uint32_t np, double c, double vl) {
    auto u = [&](size_t a) {
        const uint32_t n = N[a] + V[a];
        const double w = V[a] ? W[a] - vl * (double)V[a] : W[a];
        const double q = n ? w / (double)n : 0.0;
        return q + c * P[a] * (std::sqrt((double)np) / (double)(n + 1));
    };
    size_t best = 0;
    for (size_t a = 1; a < k; ++a)
        if (total_key(u(a)) >= total_key(u(best))) best = a;
    return best;
}

static uint16_t node_action(const MctsNode& nd) {
    return !nd.has_mov ? 0xFFFF : nd.is_pass ? encode_pass(nd.mov.used_card_idx) : encode_action(nd.mov.used_card_idx, nd.mov.mov);
}

struct VlArena : MctsArena {
    uint32_t leaves;  // K: descents per round after round 0 (1 gives the oracle's one-playout rounds)
    double vl;
    uint32_t rounds = 0;

    VlArena(const State& s, int color, double c, uint32_t sims, eval_fn e, void* u, uint32_t k, double vl_)
        : MctsArena(s, color, c, sims, e, u), leaves(k), vl(vl_) {}

    uint32_t select_vl(uint32_t x, std::map<uint32_t, uint32_t>& v) const {
        const auto& ch = arena[x].children;
        const size_t k = ch.size();
        std::vector<double> P(k), W(k);
        std::vector<uint32_t> N(k), V(k);
        for (size_t a = 0; a < k; ++a) {
            P[a] = arena[ch[a]].probability;
            N[a] = arena[ch[a]].visits;
            W[a] = arena[ch[a]].reward;
            V[a] = v.count(ch[a]) ? v[ch[a]] : 0u;
        }
        const uint32_t np = arena[x].visits + (v.count(x) ? v[x] : 0u);
        return ch[vl_choice(k, P.data(), N.data(), W.data(), V.data(), np, exploration_c, vl)];
    }

    struct Leaf {
        uint32_t node;
        int result;
        EvaluationResult ev;
    };

    void round(uint32_t b) {
        std::map<uint32_t, uint32_t> v;  // pending descents of this round per arena position
        std::vector<Leaf> lv(b);
        for (uint32_t j = 0; j < b; ++j) {
            State st = root_state;
            int color = root_color;
            uint32_t node_idx = 0;
            std::vector<uint32_t> path(1, 0u);
            while (arena[node_idx].is_expanded && !arena[node_idx].is_terminal) {
                node_idx = select_vl(node_idx, v);
                if (arena[node_idx].has_mov) {
                    int64_t parent = arena[node_idx].parent;
                    const DoneMove& mv = arena[node_idx].mov;
                    int r = arena[node_idx].is_pass ? st.pass(mv.used_card_idx) : st.make_move(mv.mov, arena[parent].player_color, mv.used_card_idx);
                    color = enemy(color);
                    if (is_win(r)) arena[node_idx].is_terminal = true;
                }
                path.push_back(node_idx);
            }
            for (uint32_t p : path) v[p] += 1;
            lv[j].node = node_idx;
            lv[j].result = st.current_state();
            lv[j].ev = evaluate(st, color);  // every leaf is evaluated, as every row goes through the network
        }
        for (uint32_t j = 0; j < b; ++j) {  // in descent order
            const uint32_t node_idx = lv[j].node;
            if (!arena[node_idx].is_expanded && !arena[node_idx].is_terminal) expand(node_idx, lv[j].ev);
            int64_t parent = arena[node_idx].parent >= 0 ? arena[node_idx].parent : 0;
            int reward_color = arena[parent].player_color;
            back_propagate(node_idx, is_win(lv[j].result) ? reward_fn(lv[j].result, reward_color) : lv[j].ev.value);
        }
    }

    // the rounds, then MctsArena::search's tail (pi and best, unchanged)
    uint32_t search(float pi[50]) {
        uint32_t done = 0;
        while (done < max_playouts) {
            const uint32_t b = done == 0 ? 1u : std::min(leaves, max_playouts - done);
            round(b);
            done += b;
            rounds += 1;
        }
        playouts = done;
        return MctsArena::search(pi);
    }
};

static void dump_arena(const MctsArena& a, orc_tree_dump* dump) {
    for (size_t i = 0; i < a.arena.size(); ++i) {
        const MctsNode& nd = a.arena[i];
        dump->visits[i] = nd.visits; dump->reward[i] = nd.reward; dump->winrate[i] = nd.winrate; dump->prior[i] = nd.probability;
        dump->action[i] = node_action(nd);
        dump->parent[i] = (int32_t)nd.parent;
        dump->first_child[i] = nd.children.empty() ? 0u : nd.children[0];
        dump->n_child[i] = (uint32_t)nd.children.size();
        dump->flags[i] = (uint8_t)((nd.is_expanded ? 1 : 0) | (nd.is_terminal ? 2 : 0) | (nd.is_pass ? 4 : 0));
    }
}

}  // namespace orc_vl

extern "C" {

// searches of n roots with K = leaves descents per round and virtual loss vl. evaluator: 0 uniform, 1 hash, 2 the callback `cb` (run
// with threads = 1). Outputs per tree (any may be NULL): best action, pi [50], root visits, root q, child visits [40], node count,
// rounds. dump (optional, with cap) receives tree `dump_tree`.
void orc_vl_search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, orc::eval_fn cb, void* user, int threads,
                         uint32_t leaves, double vl, uint16_t* best_actions, float* pi50, uint32_t* root_visits, double* root_q,
                         uint32_t* child_visits40, int64_t* n_nodes, uint32_t* rounds, int64_t dump_tree, orc_tree_dump* dump, int64_t cap) {
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : evaluator == 1 ? orc::hash_eval : cb;
            orc_vl::VlArena a(orc::to_state(roots[i]), roots[i].side, c_puct, sims, e, user, leaves, vl);
            float pi[50];
            const uint32_t best = a.search(pi);
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = ch.empty() ? 0xFFFF : orc_vl::node_action(a.arena[best]);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (rounds) rounds[i] = a.rounds;
            if (dump && i == dump_tree && cap >= (int64_t)a.arena.size()) orc_vl::dump_arena(a, dump);
        }
    };
    if (threads <= 1 || evaluator == 2) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}
// vl_choice of n nodes: node i has children [off[i], off[i + 1]) of P / N / W / V and the parent count np[i]; out[i] = the child's position
void orc_vl_choice(int64_t n, const int64_t* off, const double* P, const uint32_t* N, const double* W, const uint32_t* V, const uint32_t* np,
                   double c, double vl, int64_t* out) {
    for (int64_t i = 0; i < n; ++i)
        out[i] = (int64_t)orc_vl::vl_choice((size_t)(off[i + 1] - off[i]), P + off[i], N + off[i], W + off[i], V + off[i], np[i], c, vl);
}

}  // extern "C"
