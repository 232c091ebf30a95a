// The `AlphaBeta` agent of the C++ host mirror (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "n depth", then n positions "pawn_red pawn_blue king_red king_blue card0 .. card4 side" (reference bit layout).
// stdout: one line per position "action score" (the agent's move as an onb_action code and its score), then the arena checks and
// "ALL OK". Exit code 0 on success.
#include <cstdio>
#include <memory>
#include "onitama_b200.hpp"

using namespace onitama;
static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

int main() {
    try {
        long n = 0, depth = 0;
        if (std::scanf("%ld %ld", &n, &depth) != 2) return 3;
        AlphaBeta agent((int32_t)depth);
        CHECK(agent.id() == (uint64_t)depth && std::string(agent.name()) == "AlphaBeta AI");
        for (long i = 0; i < n; ++i) {
            unsigned v[10];
            for (unsigned& x : v)
                if (std::scanf("%u", &x) != 1) return 3;
            onb_state o{};
            o.pawns[0] = v[0]; o.pawns[1] = v[1]; o.kings[0] = v[2]; o.kings[1] = v[3];
            for (int k = 0; k < 5; ++k) o.cards[k] = (uint8_t)v[4 + k];
            GameState gs = GameState::with_deck(Deck());
            gs.state.from_onb(o);
            gs.curr_player_color = v[9] ? PlayerColor::Blue : PlayerColor::Red;
            auto mv = agent.generate_move(gs);
            std::printf("%u %.0f\n", (unsigned)to_action(mv.first), mv.second);
        }
        // fight(): the reference's sequential arena loop with the agent on one side
        EvaluatorConfig ec;
        ec.game_amnt = 2;
        ec.max_plies = 30;
        ec.seed = 4;
        FightStatistics fs = fight(ec, std::make_unique<AlphaBeta>(2), std::make_unique<Random>(5));
        CHECK(fs.wins + fs.losses + fs.draws == 2 && fs.games_red == 1 && fs.games_blue == 1);
        // fight_device(): the same agent inside the library's arena, on an engine without search-tree pools
        Engine e(32, 0, 9, 0, false);
        EvaluatorConfig ed;
        ed.game_amnt = 32;
        onb_agent ab{ONB_AGENT_ALPHABETA, 0, 0, 3, 0., 0, 0}, rnd{ONB_AGENT_RANDOM, 0, 0, 0, 0., 0, 0};
        FightStatistics d = fight_device(e, ed, ab, rnd);
        CHECK(d.wins + d.losses + d.draws == 32 && d.wins > d.losses);
        bool threw = false;
        onb_agent bad = ab;
        bad.sims = ONB_ALPHABETA_MAX_DEPTH + 1;
        try { fight_device(e, ed, bad, rnd); } catch (const Error& err) { threw = err.code == ONB_E_INVALID; }
        CHECK(threw);
    } catch (const Error& e) {
        std::printf("FAIL exception %d: %s\n", e.code, e.what());
        return 2;
    }
    if (failures) { std::printf("%d FAILURES\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
