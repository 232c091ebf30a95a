// Gumbel MuZero (the GumbelMuZero agent's configuration: AlphaZeroMctsConfig::gumbel with interior = 1) in the C++ host mirror (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "plies playouts m seed", then one position "pawn_red pawn_blue king_red king_blue card0 .. card4 side" (reference bit layout).
// stdout: one line per ply with the chosen move as an onb_action code (the move is then played; consecutive moves take steps 0, 1, ...),
// then "ALL OK". Exit code 0 on success.
#include <cstdio>
#include <string>
#include "onitama_b200.hpp"

using namespace onitama;
static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

int main() {
    try {
        long plies = 0, playouts = 0, m = 0;
        unsigned long long seed = 0;
        if (std::scanf("%ld %ld %ld %llu", &plies, &playouts, &m, &seed) != 4) return 3;
        unsigned v[10];
        for (unsigned& x : v)
            if (std::scanf("%u", &x) != 1) return 3;
        onb_state o{};
        o.pawns[0] = v[0]; o.pawns[1] = v[1]; o.kings[0] = v[2]; o.kings[1] = v[3];
        for (int k = 0; k < 5; ++k) o.cards[k] = (uint8_t)v[4 + k];
        GameState gs = GameState::with_deck(Deck());
        gs.state.from_onb(o);
        gs.curr_player_color = v[9] ? PlayerColor::Blue : PlayerColor::Red;
        const GumbelMuZero agent((uint32_t)m, 0.1, seed);
        CHECK(agent.config.gumbel.interior == 1 && std::string(agent.name()) == "Gumbel MuZero AI");
        TrainingAlphaZeroMcts mcts;
        mcts.config = agent.config;
        mcts.config.max_playouts = (uint32_t)playouts;
        mcts.config.exploration_c = 2.0;
        mcts.device_evaluator = ONB_EVAL_HASH;
        for (long p = 0; p < plies; ++p) {
            auto mv = mcts.generate_move_tensor(gs.state, gs.curr_player_color);
            float sum = 0.f;
            for (float x : mv.second) sum += x;
            CHECK(sum > 0.999f && sum < 1.001f);  // the improved policy
            std::printf("%u\n", (unsigned)to_action(mv.first));
            const MoveResult r = gs.state.make_move(mv.first.mov, gs.curr_player_color, mv.first.used_card_idx);
            gs.curr_player_color = gs.curr_player_color == PlayerColor::Red ? PlayerColor::Blue : PlayerColor::Red;
            if (r == MoveResult::RedWin || r == MoveResult::BlueWin) break;
        }
        // Gumbel MuZero does not combine with train-mode noise
        bool threw = false;
        mcts.config.train = true;
        try { mcts.generate_move_tensor(gs.state, gs.curr_player_color); } catch (const Error& err) { threw = err.code == ONB_E_STATE; }
        CHECK(threw);
    } catch (const Error& e) {
        std::printf("FAIL exception %d: %s\n", e.code, e.what());
        return 2;
    }
    if (failures) { std::printf("%d FAILURES\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
