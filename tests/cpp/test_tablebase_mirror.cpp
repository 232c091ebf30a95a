// The `Tablebase` agent of the C++ host mirror (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "n card0 .. card4", then n positions "pawn_red pawn_blue king_red king_blue card0 .. card4 side" (reference bit layout).
// stdout: one line per position, the agent's move as an onb_action code, then the checks and "ALL OK". Exit code 0 on success.
#include <cstdio>
#include <memory>
#include "onitama_b200.hpp"

using namespace onitama;
static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

int main() {
    try {
        long n = 0;
        unsigned c[5];
        if (std::scanf("%ld %u %u %u %u %u", &n, &c[0], &c[1], &c[2], &c[3], &c[4]) != 6) return 3;
        Tablebase agent({(uint8_t)c[0], (uint8_t)c[1], (uint8_t)c[2], (uint8_t)c[3], (uint8_t)c[4]}, 1);
        CHECK(std::string(agent.name()) == "Tablebase AI");
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
            std::printf("%u\n", (unsigned)to_action(mv.first));
        }
        // a position outside the table (the start position has eight pawns) is refused
        bool threw = false;
        GameState start = GameState::with_deck(Deck());
        try { agent.generate_move(start); } catch (const Error& err) { threw = err.code == ONB_E_STATE; }
        CHECK(threw);
    } catch (const Error& e) {
        std::printf("FAIL exception %d: %s\n", e.code, e.what());
        return 2;
    }
    if (failures) { std::printf("%d FAILURES\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
