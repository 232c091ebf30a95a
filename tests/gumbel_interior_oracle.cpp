// =====================================================================================
// tests/gumbel_interior_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of Gumbel MuZero's interior selection (onb_gumbel_config.interior, DESIGN.md §5f.1) on top of the Gumbel-search
// oracle (tests/gumbel_oracle.cpp, included below unchanged): below the root, interior_choice over a node's children replaces the
// oracle's PUCT select, and every playout that expands a node stores r_x, the reward it backed up into that node.
// =====================================================================================
#include "gumbel_oracle.cpp"

namespace orc_gumbel {

// Interior selection at a node with k children (DESIGN.md §5f): P the stored priors, N the visits, Q = W / N (read where N > 0), r_x
// the reward the expanding simulation backed up into the node. Returns the chosen child's position.
static size_t interior_choice(size_t k, const double* P, const uint32_t* N, const double* Q, double r_x, double c_visit, double c_scale) {
    double sP = 0.0;
    for (size_t a = 0; a < k; ++a) sP += P[a];
    const bool uni = !(sP > 0.0);  // every prior 0: every P counts as 1
    const double tot = uni ? (double)k : sP;
    std::vector<double> p(k), logit(k), qh(k), z(k);
    for (size_t a = 0; a < k; ++a) {
        const double Pa = uni ? 1.0 : P[a];
        p[a] = std::max(DBL_MIN, Pa / tot);
        logit[a] = Pa > 0.0 ? onb_log(Pa) : -INFINITY;
    }
    uint32_t sum_n = 0, max_n = 0;
    double spq = 0.0, sp = 0.0;
    for (size_t a = 0; a < k; ++a) {
        if (N[a] == 0) continue;
        spq += p[a] * Q[a];
        sp += p[a];
        sum_n += N[a];
        max_n = std::max(max_n, N[a]);
    }
    const double wq = sp > 0.0 ? spq / sp : 0.0;
    const double v_mix = (-r_x + (double)sum_n * wq) / (double)(sum_n + 1);
    double lo = INFINITY, hi = -INFINITY;
    for (size_t a = 0; a < k; ++a) {
        qh[a] = N[a] ? Q[a] : v_mix;
        lo = std::min(lo, qh[a]);
        hi = std::max(hi, qh[a]);
    }
    const double range = std::max(hi - lo, 1e-8);
    const double coef = (c_visit + (double)max_n) * c_scale;
    double zmax = -INFINITY;
    for (size_t a = 0; a < k; ++a) {
        z[a] = logit[a] + coef * ((qh[a] - lo) / range);
        zmax = std::max(zmax, z[a]);
    }
    double se = 0.0;
    for (size_t a = 0; a < k; ++a) {
        z[a] = onb_exp(z[a] - zmax);
        se += z[a];
    }
    size_t best = 0;
    double bs = -INFINITY;
    for (size_t a = 0; a < k; ++a) {
        const double sc = z[a] / se - (double)N[a] / (double)(sum_n + 1);
        if (sc > bs) { bs = sc; best = a; }
    }
    return best;
}

struct InteriorArena : GumbelArena {
    std::vector<double> rx;  // r_x by arena position, written when a playout expands the node

    using GumbelArena::GumbelArena;

    uint32_t select_interior(uint32_t x) const {
        const auto& ch = arena[x].children;
        const size_t k = ch.size();
        std::vector<double> P(k), Q(k);
        std::vector<uint32_t> N(k);
        for (size_t a = 0; a < k; ++a) {
            P[a] = arena[ch[a]].probability;
            N[a] = arena[ch[a]].visits;
            Q[a] = arena[ch[a]].winrate;
        }
        return ch[interior_choice(k, P.data(), N.data(), Q.data(), rx[x], g.c_visit, g.c_scale)];
    }

    // GumbelArena::playout with interior_choice below the root and r_x stored at expansion
    void playout() {
        State st = root_state;
        int color = root_color;
        uint32_t node_idx = 0;
        while (arena[node_idx].is_expanded && !arena[node_idx].is_terminal) {
            node_idx = node_idx == 0 ? select_root() : select_interior(node_idx);
            if (arena[node_idx].has_mov) {
                int64_t parent = arena[node_idx].parent;
                const DoneMove& mv = arena[node_idx].mov;
                int r = arena[node_idx].is_pass ? st.pass(mv.used_card_idx) : st.make_move(mv.mov, arena[parent].player_color, mv.used_card_idx);
                color = enemy(color);
                if (is_win(r)) arena[node_idx].is_terminal = true;
            }
        }
        bool need_expand = !arena[node_idx].is_expanded && !arena[node_idx].is_terminal;
        EvaluationResult ev;
        ev.value = 0.;
        int result = st.current_state();
        if (need_expand || !is_win(result)) ev = evaluate(st, color);
        if (need_expand) expand(node_idx, ev);
        int64_t parent = arena[node_idx].parent >= 0 ? arena[node_idx].parent : 0;
        int reward_color = arena[parent].player_color;
        const double reward = is_win(result) ? reward_fn(result, reward_color) : ev.value;
        if (need_expand) {
            rx.resize(arena.size(), 0.0);
            rx[node_idx] = reward;
        }
        back_propagate(node_idx, reward);
    }

    // the playouts with this playout, then GumbelArena::search's tail (best and pi, unchanged)
    uint32_t search(float pi[50]) {
        while (playouts < max_playouts) {
            playout();
            if (playouts == 0) r0 = arena[0].reward;
            playouts += 1;
        }
        return GumbelArena::search(pi);
    }
};


template <class Arena>
static void search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, orc::eval_fn cb, void* user, int threads,
                         const Cfg& cfg, uint64_t game0, uint16_t* best_actions, float* pi50, uint32_t* root_visits, double* root_q,
                         uint32_t* child_visits40, int64_t* n_nodes, double* r0_out, int64_t dump_tree, orc_tree_dump* dump, int64_t cap) {
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : evaluator == 1 ? orc::hash_eval : cb;
            Arena a(orc::to_state(roots[i]), roots[i].side, c_puct, sims, e, user, cfg, game0 + (uint64_t)i);
            float pi[50];
            const uint32_t best = a.search(pi);
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = ch.empty() ? 0xFFFF : node_action(a.arena[best]);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (r0_out) r0_out[i] = a.r0;
            if (dump && i == dump_tree && cap >= (int64_t)a.arena.size()) dump_arena(a, dump);
        }
    };
    if (threads <= 1 || evaluator == 2) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}
}  // namespace orc_gumbel

extern "C" {

// orc_gumbel_search_batch's arguments and outputs plus `interior`: 1 = Gumbel MuZero (interior selection below the root), 0 = the
// root-only search through this file's batch loop
void orc_gumbel_interior_search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, orc::eval_fn cb, void* user,
                                      int threads, uint32_t m, double c_visit, double c_scale, double scale, uint64_t seed, uint32_t step, uint64_t game0,
                                      uint16_t* best_actions, float* pi50, uint32_t* root_visits, double* root_q, uint32_t* child_visits40,
                                      int64_t* n_nodes, double* r0_out, int64_t dump_tree, orc_tree_dump* dump, int64_t cap, int interior) {
    const orc_gumbel::Cfg cfg{m, c_visit, c_scale, scale, seed, step};
    if (interior)
        orc_gumbel::search_batch<orc_gumbel::InteriorArena>(roots, n, c_puct, sims, evaluator, cb, user, threads, cfg, game0, best_actions, pi50,
                                                            root_visits, root_q, child_visits40, n_nodes, r0_out, dump_tree, dump, cap);
    else
        orc_gumbel::search_batch<orc_gumbel::GumbelArena>(roots, n, c_puct, sims, evaluator, cb, user, threads, cfg, game0, best_actions, pi50,
                                                          root_visits, root_q, child_visits40, n_nodes, r0_out, dump_tree, dump, cap);
}
// interior_choice of n nodes: node i has children [off[i], off[i + 1]) of P / N / Q and the reward rx[i]; out[i] = the child's position
void orc_gumbel_interior_choice(int64_t n, const int64_t* off, const double* P, const uint32_t* N, const double* Q, const double* rx, double c_visit,
                                double c_scale, int64_t* out) {
    for (int64_t i = 0; i < n; ++i)
        out[i] = (int64_t)orc_gumbel::interior_choice((size_t)(off[i + 1] - off[i]), P + off[i], N + off[i], Q + off[i], rx[i], c_visit, c_scale);
}

}  // extern "C"
