// The self-play move protocol (TrainConfig::temp_plies / temperature / resign_below / resign_holdout) in the C++ host mirror
// (include/onitama_b200.hpp) on the GPU through libonb.so.
// stdin: "slots games sims temp_plies temperature resign_below resign_holdout seed".
// stdout: the sample count, then one line "z colour" per sample (ply-major, as self_play_continuous returns them), then "ALL OK".
// Exit code 0 on success.
#include <cstdio>
#include "onitama_b200.hpp"

using namespace onitama;

int main() {
    try {
        long slots = 0, games = 0, sims = 0, temp_plies = 0;
        double temperature = 0, resign_below = 0, holdout = 0;
        unsigned long long seed = 0;
        if (std::scanf("%ld %ld %ld %ld %lf %lf %lf %llu", &slots, &games, &sims, &temp_plies, &temperature, &resign_below, &holdout, &seed) != 8) return 3;
        Engine e(slots, (uint32_t)sims, seed);
        TrainingAlphaZeroMcts mcts;
        mcts.config.max_playouts = (uint32_t)sims;
        mcts.config.exploration_c = 2.0;
        mcts.device_evaluator = ONB_EVAL_UNIFORM;
        TrainConfig cfg;
        cfg.self_play_game_amnt = (size_t)games;
        cfg.seed = seed;
        cfg.temp_plies = (uint32_t)temp_plies;
        cfg.temperature = temperature;
        cfg.resign_below = resign_below;
        cfg.resign_holdout = holdout;
        const std::vector<SelfPlayData> data = self_play_continuous(e, mcts, cfg);
        std::printf("%zu\n", data.size());
        for (const SelfPlayData& d : data) std::printf("%.1f %d\n", d.z, (int)d.player_color);
        // an invalid setting is refused through the mirror too
        cfg.temperature = 0.0;
        bool refused = false;
        try {
            self_play_continuous(e, mcts, cfg);
        } catch (const Error& err) {
            refused = err.code == ONB_E_INVALID;
        }
        if (!refused) {
            std::printf("FAIL: temperature 0 was not refused\n");
            return 1;
        }
        std::printf("ALL OK\n");
        return 0;
    } catch (const std::exception& ex) {
        std::printf("EXCEPTION %s\n", ex.what());
        return 2;
    }
}
