// Tree reuse (AlphaZeroMctsConfig::reuse) in the C++ host mirror (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "plies playouts", then one position "pawn_red pawn_blue king_red king_blue card0 .. card4 side" (reference bit layout).
// stdout: one line per ply with the chosen move as an onb_action code (the move is then played), then the reuse counters and
// "ALL OK". Exit code 0 on success.
#include <cstdio>
#include "onitama_b200.hpp"

using namespace onitama;
static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

int main() {
    try {
        long plies = 0, playouts = 0;
        if (std::scanf("%ld %ld", &plies, &playouts) != 2) return 3;
        unsigned v[10];
        for (unsigned& x : v)
            if (std::scanf("%u", &x) != 1) return 3;
        onb_state o{};
        o.pawns[0] = v[0]; o.pawns[1] = v[1]; o.kings[0] = v[2]; o.kings[1] = v[3];
        for (int k = 0; k < 5; ++k) o.cards[k] = (uint8_t)v[4 + k];
        GameState gs = GameState::with_deck(Deck());
        gs.state.from_onb(o);
        gs.curr_player_color = v[9] ? PlayerColor::Blue : PlayerColor::Red;
        TrainingAlphaZeroMcts mcts;
        mcts.config.max_playouts = (uint32_t)playouts;
        mcts.config.exploration_c = 2.0;
        mcts.config.reuse = true;
        mcts.device_evaluator = ONB_EVAL_HASH;
        Engine& e = Engine::single(mcts.config.max_playouts);
        e.check(onb_mcts_reuse_stats(e.ctx(), nullptr, 1));
        for (long p = 0; p < plies; ++p) {
            auto mv = mcts.generate_move_tensor(gs.state, gs.curr_player_color);
            std::printf("%u\n", (unsigned)to_action(mv.first));
            const MoveResult r = gs.state.make_move(mv.first.mov, gs.curr_player_color, mv.first.used_card_idx);
            gs.curr_player_color = gs.curr_player_color == PlayerColor::Red ? PlayerColor::Blue : PlayerColor::Red;
            if (r == MoveResult::RedWin || r == MoveResult::BlueWin) break;
        }
        uint64_t st[4];
        e.check(onb_mcts_reuse_stats(e.ctx(), st, 0));
        std::printf("stats %llu %llu %llu %llu\n", (unsigned long long)st[0], (unsigned long long)st[1], (unsigned long long)st[2],
                    (unsigned long long)st[3]);
        CHECK(st[ONB_REUSE_KEPT] > 0 && st[ONB_REUSE_SIMS] < st[ONB_REUSE_TREES] * (uint64_t)playouts);
        // a host network cannot drive a reuse search
        bool threw = false;
        mcts.model = [](const float*, int64_t n, float* pol, float* val) {
            for (int64_t i = 0; i < n * 50; ++i) pol[i] = 0.02f;
            for (int64_t i = 0; i < n; ++i) val[i] = 0.f;
        };
        try { mcts.generate_move_tensor(gs.state, gs.curr_player_color); } catch (const Error& err) { threw = err.code == ONB_E_INVALID; }
        CHECK(threw);
    } catch (const Error& e) {
        std::printf("FAIL exception %d: %s\n", e.code, e.what());
        return 2;
    }
    if (failures) { std::printf("%d FAILURES\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
