// Plays one match through the C++ mirror's evaluate (include/az_b200.hpp) under the synthetic evaluator and prints its winrates
// as a JSON line for tests/test_match_gpu.py, which compares them with evaluation.evaluate_on_device.
#include <cstdio>
#include <cstdlib>
#include "az_b200.hpp"

using namespace az;

int main(int argc, char** argv) {
    const uint64_t stub_seed = argc > 1 ? std::strtoull(argv[1], nullptr, 10) : 17;
    az_config cfg = Engine::default_config();
    cfg.max_games = 8; cfg.max_batch = 64; cfg.num_simulations = 16;
    Engine eng(cfg);
    if (az_set_evaluator_stub(eng.handle(), 1, stub_seed) != AZ_OK) return 3;
    AlphaZero model(eng);
    const EvaluationResult r = evaluate(model, 0, 1, 12, 15, 4, 100, 16, 2, 1.0f, false, 8);
    std::printf("{\"winrate\": %.9g, \"drawrate\": %.9g, \"p2_winrate\": %.9g}\n", r.winrate, r.drawrate, r.lossrate);
    return 0;
}
