// Drives the leaf-parallel overload of run_all_episodes in the C++ mirror (include/az_b200.hpp) and prints per-run totals as JSON
// lines for tests/test_selfplay_vl_gpu.py: K = 1 next to the default overload, and K = 4 for the test restatement.
#include <cstdio>
#include <cstdlib>
#include "az_b200.hpp"

using namespace az;

static void report(const char* name, const std::pair<float, std::vector<EpisodeStep>>& r) {
    double vsum = 0;
    std::size_t dsum = 0;
    for (auto& s : r.second) { vsum += s.final_value; dsum += s.search_depth; }
    std::printf("{\"test\": \"%s\", \"steps\": %zu, \"value_sum\": %.6f, \"depth_sum\": %zu, \"avg_batch\": %.3f}\n", name, r.second.size(),
                vsum, dsum, r.first);
}

int main(int argc, char** argv) {
    const uint64_t stub_seed = argc > 1 ? std::strtoull(argv[1], nullptr, 10) : 5;
    az_config cfg = Engine::default_config();
    cfg.max_games = 4; cfg.max_batch = 16; cfg.num_simulations = 16; cfg.seed = 42;
    Engine eng(cfg);
    if (az_set_evaluator_stub(eng.handle(), 1, stub_seed) != AZ_OK) return 3;
    AlphaZero model(eng);
    report("default", run_all_episodes(model, 4, 0, 16));
    report("k1", run_all_episodes(model, 4, 0, 16, 1, 1.0f));
    report("k4", run_all_episodes(model, 4, 0, 16, 4, 1.0f));
    return 0;
}
