// Plays two pairings through the C++ mirror's player overload of evaluate (include/az_b200.hpp) with the match's evaluation cache
// under the synthetic evaluator and prints their winrates as JSON lines for tests/test_match_cache_gpu.py, which compares them with
// evaluation.evaluate() of the same players.
#include <cstdio>
#include <cstdlib>
#include "az_b200.hpp"

using namespace az;

static void print(const char* name, const EvaluationResult& r) {
    std::printf("{\"pairing\": \"%s\", \"winrate\": %.9g, \"drawrate\": %.9g, \"p2_winrate\": %.9g}\n", name, r.winrate, r.drawrate, r.lossrate);
}

int main(int argc, char** argv) {
    const uint64_t stub_seed = argc > 1 ? std::strtoull(argv[1], nullptr, 10) : 17;
    az_config cfg = Engine::default_config();
    cfg.max_games = 8; cfg.max_batch = 64; cfg.num_simulations = 16;
    Engine eng(cfg);
    if (az_set_evaluator_stub(eng.handle(), 1, stub_seed) != AZ_OK) return 3;
    AlphaZero model(eng);
    const az_match_player mcts{AZ_PLAYER_MCTS, 0, 16, 2, 1.0f};
    const az_match_player mcts8{AZ_PLAYER_MCTS, 1, 8, 1, 1.0f};
    const az_match_player rnd{AZ_PLAYER_RANDOM, 0, 0, 0, 0.0f};
    print("mcts16_mcts8", evaluate(model, mcts, mcts8, 12, 15, 4, 100, 0, 256, 16));
    print("mcts_random", evaluate(model, mcts, rnd, 12, 15, 4, 100, 0, 256, 16));
    return 0;
}
