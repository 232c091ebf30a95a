// =====================================================================================
// tests/gumbel_oracle.cpp  --  TEST INFRASTRUCTURE ONLY (never linked into / imported by the product).
//
// CPU restatement of the Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f) on top of the CPU oracle's MctsArena
// (oracle/onb_oracle.cpp, included below unchanged), in the reference's shape: a sequential loop over the root's children vector
// replaces MctsArena::select at the root and the tail of search(); below the root the oracle's PUCT select runs as it is.
// onb_log / onb_exp and the sequential-halving table come from the product's onb_gumbel.cuh (compiled here with
// -ffp-contract=off, so the host build uses the same IEEE operations as the kernels).
// =====================================================================================
#include <cfloat>

#include "../oracle/onb_oracle.cpp"
#include "../onitama_alphazero_b200/csrc/onb_gumbel.cuh"

namespace orc_gumbel {
using namespace orc;
using onb_gumbel::onb_exp;
using onb_gumbel::onb_log;

struct Cfg {
    uint32_t m;
    double c_visit, c_scale, scale;
    uint64_t seed;
    uint32_t step;
};

static uint16_t node_action(const MctsNode& nd) {
    return !nd.has_mov ? 0xFFFF : nd.is_pass ? encode_pass(nd.mov.used_card_idx) : encode_action(nd.mov.used_card_idx, nd.mov.mov);
}

struct GumbelArena : MctsArena {
    Cfg g;
    uint64_t game;
    double r0 = 0.0;  // the reward the root's own evaluation (playout 0) backed up into the root
    std::vector<double> c_logit, c_base, c_p;  // priors() of the expanded root (the priors never change afterwards)
    std::vector<uint32_t> c_seq;               // seq(m_eff, sims - 1)

    GumbelArena(const State& s, int color, double c, uint32_t sims, eval_fn e, void* u, const Cfg& cfg, uint64_t game_id)
        : MctsArena(s, color, c, sims, e, u), g(cfg), game(game_id) {}

    // logit(a), base(a) = g(a) + (logit(a) - L), p(a)
    void priors(std::vector<double>& logit, std::vector<double>& base, std::vector<double>& p) const {
        const auto& ch = arena[0].children;
        const size_t k = ch.size();
        double sp = 0.0;
        for (uint32_t c : ch) sp += arena[c].probability;
        const bool uni = !(sp > 0.0);  // every prior 0: every P counts as 1
        if (uni) sp = (double)k;
        logit.assign(k, 0.0);
        base.assign(k, 0.0);
        p.assign(k, 0.0);
        double L = -INFINITY;
        for (size_t a = 0; a < k; ++a) {
            const double P = uni ? 1.0 : arena[ch[a]].probability;
            logit[a] = P > 0.0 ? onb_log(P) : -INFINITY;
            if (logit[a] > L) L = logit[a];
        }
        for (size_t a = 0; a < k; ++a) {
            const double u = ((double)rand_u32(g.seed, game, g.step, onb_gumbel::kGumbelDraw + (uint32_t)a) + 0.5) * 0x1p-32;
            const double gum = g.scale * -onb_log(-onb_log(u));
            base[a] = gum + (logit[a] - L);
            const double P = uni ? 1.0 : arena[ch[a]].probability;
            p[a] = std::max(DBL_MIN, P / sp);
        }
    }

    // completed Q (qtransform_completed_by_mix_value): sigma(a) for every child
    std::vector<double> sigma(const std::vector<double>& p, uint32_t* max_n_out) const {
        const auto& ch = arena[0].children;
        const size_t k = ch.size();
        uint32_t sum_n = 0, max_n = 0;
        double spq = 0.0, sp = 0.0;
        for (size_t a = 0; a < k; ++a) {
            const MctsNode& c = arena[ch[a]];
            if (c.visits == 0) continue;
            spq += p[a] * c.winrate;
            sp += p[a];
            sum_n += c.visits;
            max_n = std::max(max_n, c.visits);
        }
        const double wq = sp > 0.0 ? spq / sp : 0.0;
        const double v_mix = (-r0 + (double)sum_n * wq) / (double)(sum_n + 1);
        std::vector<double> qh(k);
        double lo = INFINITY, hi = -INFINITY;
        for (size_t a = 0; a < k; ++a) {
            const MctsNode& c = arena[ch[a]];
            qh[a] = c.visits ? c.winrate : v_mix;
            lo = std::min(lo, qh[a]);
            hi = std::max(hi, qh[a]);
        }
        const double range = std::max(hi - lo, 1e-8);
        const double coef = (g.c_visit + (double)max_n) * g.c_scale;
        std::vector<double> s(k);
        for (size_t a = 0; a < k; ++a) s[a] = coef * ((qh[a] - lo) / range);
        if (max_n_out) *max_n_out = max_n;
        return s;
    }

    // the first child of maximal score among those with `visits` visits (child 0 if none)
    size_t pick(uint32_t visits) {
        if (c_base.empty()) priors(c_logit, c_base, c_p);
        const std::vector<double>& base = c_base;
        const std::vector<double> s = sigma(c_p, nullptr);
        const auto& ch = arena[0].children;
        size_t best = 0;
        double bs = -INFINITY;
        for (size_t a = 0; a < ch.size(); ++a) {
            if (arena[ch[a]].visits != visits) continue;
            const double sc = std::max(-1e9, base[a] + s[a]);
            if (sc > bs) { bs = sc; best = a; }
        }
        return best;
    }

    uint32_t select_root() {
        const auto& ch = arena[0].children;
        const uint32_t m_eff = std::min<uint32_t>(g.m, (uint32_t)ch.size());
        const uint32_t n = max_playouts - 1, i = arena[0].visits - 1;
        if (c_seq.size() != n) {
            c_seq.assign(n, 0);
            onb_gumbel::seq_halving(m_eff, n, c_seq.data());
        }
        return ch[pick(c_seq[i < n ? i : n - 1])];
    }

    // MctsArena::playout (mcts_arena.rs:127-177) with the root's select replaced
    void playout() {
        State st = root_state;
        int color = root_color;
        uint32_t node_idx = 0;
        while (arena[node_idx].is_expanded && !arena[node_idx].is_terminal) {
            node_idx = node_idx == 0 ? select_root() : select(arena[node_idx]);
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
        if (is_win(result)) back_propagate(node_idx, reward_fn(result, reward_color));
        else back_propagate(node_idx, ev.value);
    }

    // search(): the playouts, then best = pick(max N) and pi = softmax(logit + sigma) per policy index. Returns the best child's
    // arena index (0 without children).
    uint32_t search(float pi[50]) {
        while (playouts < max_playouts) {
            playout();
            if (playouts == 0) r0 = arena[0].reward;
            playouts += 1;
        }
        for (int i = 0; i < 50; ++i) pi[i] = 0.f;
        const auto& ch = arena[0].children;
        if (ch.empty()) return 0;
        std::vector<double> logit, base, p;
        priors(logit, base, p);
        uint32_t max_n = 0;
        const std::vector<double> s = sigma(p, &max_n);
        std::vector<double> z(ch.size());
        double zmax = -INFINITY;
        for (size_t a = 0; a < ch.size(); ++a) {
            z[a] = logit[a] + s[a];
            zmax = std::max(zmax, z[a]);
        }
        double se = 0.0;
        for (size_t a = 0; a < ch.size(); ++a) {
            z[a] = onb_exp(z[a] - zmax);
            se += z[a];
        }
        double pd[50] = {0.0};
        for (size_t a = 0; a < ch.size(); ++a) {
            const MctsNode& c = arena[ch[a]];
            pd[(c.mov.used_card_idx & 1u) * 25 + (c.is_pass ? 0 : c.mov.mov.to)] += z[a] / se;
        }
        for (int i = 0; i < 50; ++i) pi[i] = (float)pd[i];
        return ch[pick(max_n)];
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

}  // namespace orc_gumbel

extern "C" {

void orc_gumbel_log(const double* x, int64_t n, double* out) { for (int64_t i = 0; i < n; ++i) out[i] = onb_gumbel::onb_log(x[i]); }
void orc_gumbel_exp(const double* x, int64_t n, double* out) { for (int64_t i = 0; i < n; ++i) out[i] = onb_gumbel::onb_exp(x[i]); }
void orc_gumbel_seq(uint32_t m, uint32_t n, uint32_t* out) { onb_gumbel::seq_halving(m, n, out); }

// Gumbel searches of n roots (tree i searches global game game0 + i). evaluator: 0 uniform, 1 hash, 2 the callback `cb` (run with
// threads = 1). Outputs per tree (any may be NULL): best action, pi [50], root visits, root q, child visits [40], node count, r0.
// dump (optional, with cap) receives tree `dump_tree`.
void orc_gumbel_search_batch(const orc_state* roots, int64_t n, double c_puct, uint32_t sims, int evaluator, orc::eval_fn cb, void* user, int threads,
                             uint32_t m, double c_visit, double c_scale, double scale, uint64_t seed, uint32_t step, uint64_t game0, uint16_t* best_actions,
                             float* pi50, uint32_t* root_visits, double* root_q, uint32_t* child_visits40, int64_t* n_nodes, double* r0_out,
                             int64_t dump_tree, orc_tree_dump* dump, int64_t cap) {
    const orc_gumbel::Cfg cfg{m, c_visit, c_scale, scale, seed, step};
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t i = next.fetch_add(1);
            if (i >= n) break;
            const orc::eval_fn e = evaluator == 0 ? orc::uniform_eval : evaluator == 1 ? orc::hash_eval : cb;
            orc_gumbel::GumbelArena a(orc::to_state(roots[i]), roots[i].side, c_puct, sims, e, user, cfg, game0 + (uint64_t)i);
            float pi[50];
            const uint32_t best = a.search(pi);
            const auto& ch = a.arena[0].children;
            if (best_actions) best_actions[i] = ch.empty() ? 0xFFFF : orc_gumbel::node_action(a.arena[best]);
            if (pi50) memcpy(pi50 + 50 * i, pi, sizeof(pi));
            if (root_visits) root_visits[i] = a.arena[0].visits;
            if (root_q) root_q[i] = a.arena[0].winrate;
            if (child_visits40) for (size_t c = 0; c < 40; ++c) child_visits40[i * 40 + c] = c < ch.size() ? a.arena[ch[c]].visits : 0u;
            if (n_nodes) n_nodes[i] = (int64_t)a.arena.size();
            if (r0_out) r0_out[i] = a.r0;
            if (dump && i == dump_tree && cap >= (int64_t)a.arena.size()) orc_gumbel::dump_arena(a, dump);
        }
    };
    if (threads <= 1 || evaluator == 2) { work(); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(work);
    for (auto& th : pool) th.join();
}

}  // extern "C"
