// The MCTS solver (AlphaZeroMctsConfig::solver) and ONB_AGENT_PUCT_SOLVER in fight_device, in the C++ host mirror
// (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "plies playouts games fight_plies", then one position "pawn_red pawn_blue king_red king_blue card0 .. card4 side"
// (reference bit layout).
// stdout: the chosen moves as onb_action codes, one per line, with the device evaluator and then with the same evaluator as a
// HostEvaluator; then "FIGHT w l d" and the per-game results of fight_device (PUCT_SOLVER against PUCT, dealt decks, seed 0), one
// line; then "ALL OK". Exit code 0 on success.
#include <cstdio>
#include <string>
#include "onitama_b200.hpp"

using namespace onitama;
static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

int main() {
    try {
        long plies = 0, playouts = 0, games = 0, fight_plies = 0;
        if (std::scanf("%ld %ld %ld %ld", &plies, &playouts, &games, &fight_plies) != 4) return 3;
        unsigned v[10];
        for (unsigned& x : v)
            if (std::scanf("%u", &x) != 1) return 3;
        onb_state o{};
        o.pawns[0] = v[0]; o.pawns[1] = v[1]; o.kings[0] = v[2]; o.kings[1] = v[3];
        for (int k = 0; k < 5; ++k) o.cards[k] = (uint8_t)v[4 + k];
        for (int host = 0; host < 2; ++host) {
            GameState gs = GameState::with_deck(Deck());
            gs.state.from_onb(o);
            gs.curr_player_color = v[9] ? PlayerColor::Blue : PlayerColor::Red;
            AlphaZeroMcts agent;
            agent.config.max_playouts = (uint32_t)playouts;
            agent.config.exploration_c = 2.0;
            agent.config.solver = true;
            agent.device_evaluator = ONB_EVAL_UNIFORM;
            if (host)  // the uniform evaluator on the host: every row gets policy 1/50 and value 0
                agent.model = [](const float*, int64_t n, float* policy, float* value) {
                    for (int64_t i = 0; i < n * 50; ++i) policy[i] = 1.0f / 50.0f;
                    for (int64_t i = 0; i < n; ++i) value[i] = 0.f;
                };
            for (long p = 0; p < plies; ++p) {
                auto mv = agent.generate_move(gs);
                std::printf("%u\n", (unsigned)to_action(mv.first));
                const MoveResult r = gs.state.make_move(mv.first.mov, gs.curr_player_color, mv.first.used_card_idx);
                gs.curr_player_color = gs.curr_player_color == PlayerColor::Red ? PlayerColor::Blue : PlayerColor::Red;
                if (r == MoveResult::RedWin || r == MoveResult::BlueWin) break;
            }
        }
        // the solver does not combine with tree reuse
        bool threw = false;
        TrainingAlphaZeroMcts mcts;
        mcts.config.max_playouts = (uint32_t)playouts;
        mcts.config.solver = true;
        mcts.config.reuse = true;
        State s;
        s.from_onb(o);
        try { mcts.generate_move_tensor(s, v[9] ? PlayerColor::Blue : PlayerColor::Red); } catch (const Error& err) { threw = err.code == ONB_E_STATE; }
        CHECK(threw);
        mcts.config.reuse = false;  // and the next search of the shared engine runs as usual
        mcts.generate_move_tensor(s, v[9] ? PlayerColor::Blue : PlayerColor::Red);
        mcts.config.solver = false;  // switching it off again is applied too
        mcts.generate_move_tensor(s, v[9] ? PlayerColor::Blue : PlayerColor::Red);
        CHECK(!Engine::single(mcts.config.max_playouts).solver_applied);

        // fight_device: ONB_AGENT_PUCT_SOLVER against ONB_AGENT_PUCT, agent A red in the even games
        EvaluatorConfig ec;
        ec.game_amnt = (size_t)games;
        ec.max_plies = fight_plies;
        Engine e(games, (uint32_t)playouts, 0, 0, false);
        onb_agent sol = puct_solver_agent((uint32_t)playouts, 2.0, ONB_EVAL_UNIFORM);
        onb_agent puct{};
        puct.kind = ONB_AGENT_PUCT;
        puct.evaluator = ONB_EVAL_UNIFORM;
        puct.sims = (uint32_t)playouts;
        puct.c = 2.0;
        FightStatistics st = fight_device(e, ec, sol, puct);
        CHECK(st.wins + st.losses + st.draws == (size_t)games);
        CHECK(!e.solver_applied);
        std::printf("FIGHT %zu %zu %zu\n", st.wins, st.losses, st.draws);
        for (uint8_t r : e.last_fight_results) std::printf("%u ", (unsigned)r);
        std::printf("\n");
    } catch (const Error& e) {
        std::printf("FAIL exception %d: %s\n", e.code, e.what());
        return 2;
    }
    if (failures) { std::printf("%d FAILURES\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
