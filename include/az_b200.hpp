// az_b200.hpp — C++ host-side mirror of the reference's interface for the self-play hot path, over the C ABI (az_b200.h).
//
// The reference is Rust; no Rust toolchain exists in the build image, so the host side above the C ABI is C++ (header
// only) with the reference's own names and argument meaning:
//   GameState, GameResult, play_move, move_to_index, index_to_move, to_tensor      chess.rs:13-63, 73-171, 191-245
//   AlphaZero::forward                                                               agent.rs:112-144
//   MCTree::init / monte_carlo_tree_search / traverse_new / max_subtree_depth        tree.rs:37-64, 106-115, 239-269
//   process_batch, run_all_episodes, EpisodeStep                                     training.rs:15-20, 340-422
// Error behaviour: where the reference returns Err("Illegal move") the mirror returns GameResult::Illegal / nullopt;
// where it panics, az::Error is thrown with the engine's message.  One Engine per GPU; calls are not thread safe.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "az_b200.h"

namespace az {

constexpr std::size_t ACTION_SPACE = AZ_ACTION_SPACE;  // parameters.rs:3
using Position = az_position;                          // shakmaty::Chess as plain data
using Move = az_move;
using Policy = std::array<float, ACTION_SPACE>;        // Box<[f32; ACTION_SPACE]>

struct Error : std::runtime_error {
    int status;
    Error(int s, const std::string& what) : std::runtime_error(what), status(s) {}
};

enum class GameResult { Ongoing = AZ_RESULT_ONGOING, Draw = AZ_RESULT_DRAW, WhiteWins = AZ_RESULT_WHITE_WINS, BlackWins = AZ_RESULT_BLACK_WINS,
                        Illegal = AZ_RESULT_ILLEGAL };

class Engine {
public:
    explicit Engine(const az_config& cfg) : cfg_(cfg) {
        az_engine* h = nullptr;
        const int rc = az_engine_create(&cfg, &h);
        if (rc != AZ_OK) {
            std::string msg = h ? az_last_error(h) : "az_engine_create failed";
            if (h) az_engine_destroy(h);
            throw Error(rc, msg);
        }
        h_.reset(h);
    }
    static az_config default_config() { az_config c; az_config_default(&c); return c; }
    az_engine* handle() const { return h_.get(); }
    const az_config& config() const { return cfg_; }
    void check(int rc, const char* what) const {
        if (rc != AZ_OK) throw Error(rc, std::string(what) + ": " + az_last_error(h_.get()));
    }

private:
    struct Deleter { void operator()(az_engine* e) const { az_engine_destroy(e); } };
    std::unique_ptr<az_engine, Deleter> h_;
    az_config cfg_;
};

// ---- chess.rs ---------------------------------------------------------------------------------------------------
struct GameState {                       // chess.rs:13-27
    Position position;
    std::vector<Position> pos_count;     // every counted position (the reference's HashMap<Chess, usize> with multiplicity)
    GameState() { az_position_start(&position); pos_count.push_back(position); }
    explicit GameState(const Position& p) : position(p) { pos_count.push_back(p); }
};

// play_move(&mut GameState, action) driven by a policy index as the tree does (tree.rs:211-212)
inline GameResult play_move(Engine& e, GameState& st, std::size_t action_index) {
    const uint32_t offs[2] = {0, (uint32_t)st.pos_count.size()};
    const uint16_t idx = (uint16_t)action_index;
    int32_t res = AZ_RESULT_ILLEGAL;
    Position p = st.position;
    e.check(az_play_move(e.handle(), 1, &p, st.pos_count.data(), offs, &idx, &res), "az_play_move");
    if (res == AZ_RESULT_ILLEGAL) return GameResult::Illegal;
    st.position = p;
    // chess.rs:52-53 counts the new position unless shakmaty's outcome() already ended the game; a draw by the counting
    // rules is counted too, which no longer matters because the game is over either way
    if (res == AZ_RESULT_ONGOING || res == AZ_RESULT_DRAW) st.pos_count.push_back(p);
    return (GameResult)res;
}
inline std::vector<Move> legal_moves(Engine& e, const Position& p, std::vector<uint16_t>* indices = nullptr) {
    std::vector<Move> mv(AZ_MAX_MOVES);
    std::vector<uint16_t> ix(AZ_MAX_MOVES);
    int32_t n = 0;
    e.check(az_movegen(e.handle(), 1, &p, mv.data(), ix.data(), &n), "az_movegen");
    mv.resize(n);
    ix.resize(n);
    if (indices) *indices = std::move(ix);
    return mv;
}
inline std::size_t move_to_index(Engine& e, const Position& p, Move m) {
    uint16_t idx = 0;
    e.check(az_move_to_index(e.handle(), 1, &p, &m, &idx), "az_move_to_index");
    return idx;
}
inline std::optional<Move> index_to_move(Engine& e, std::size_t index, const Position& p) {
    const uint16_t idx = (uint16_t)index;
    Move m = AZ_MOVE_NONE;
    e.check(az_index_to_move(e.handle(), 1, &p, &idx, &m), "az_index_to_move");
    if (m == AZ_MOVE_NONE) return std::nullopt;
    return m;
}
inline std::vector<float> to_tensor(Engine& e, const Position& p) {  // [1, 19, 8, 8]
    std::vector<float> planes(AZ_NUM_PLANES * 64);
    e.check(az_encode(e.handle(), 1, &p, planes.data()), "az_encode");
    return planes;
}

// ---- agent.rs ---------------------------------------------------------------------------------------------------
class AlphaZero {
public:
    explicit AlphaZero(Engine& e) : e_(e) {}
    // load_model (main.rs:109-116): 144 tensors in az_weight_name order
    void load(const std::vector<const float*>& arrays) { e_.check(az_load_weights(e_.handle(), arrays.data(), (int)arrays.size()), "az_load_weights"); }
    // a second network for matches (az_load_network): slot 1 is searched by MCTree::monte_carlo_tree_search(.., network)
    void load(const std::vector<const float*>& arrays, int network) {
        e_.check(az_load_network(e_.handle(), network, arrays.data(), (int)arrays.size()), "az_load_network");
    }
    // forward(Tensor<B,4>[N,19,8,8]) -> (Tensor<B,2>[N,4096], Tensor<B,1>[N])
    std::pair<std::vector<float>, std::vector<float>> forward(const float* planes, int n) const {
        std::vector<float> policy((std::size_t)n * ACTION_SPACE), value(n);
        e_.check(az_forward_planes(e_.handle(), n, planes, policy.data(), value.data()), "az_forward_planes");
        return {std::move(policy), std::move(value)};
    }
    Engine& engine() const { return e_; }

private:
    Engine& e_;
};

// process_batch (training.rs:380-422): positions in, (policy row, value) per request out; returns the batch size
struct InferenceResult { Policy policy; float value; };
inline float process_batch(const std::vector<Position>& requests, const AlphaZero& model, std::vector<InferenceResult>& out) {
    const int n = (int)requests.size();
    std::vector<float> policy((std::size_t)n * ACTION_SPACE), value(n);
    model.engine().check(az_forward(model.engine().handle(), n, requests.data(), policy.data(), value.data()), "az_forward");
    out.resize(n);
    for (int i = 0; i < n; i++) {
        std::copy(policy.begin() + (std::size_t)i * ACTION_SPACE, policy.begin() + (std::size_t)(i + 1) * ACTION_SPACE, out[i].policy.begin());
        out[i].value = value[i];
    }
    return (float)n;
}

// ---- tree.rs ----------------------------------------------------------------------------------------------------
// The tree itself lives in GPU memory for the duration of a search; like the reference (no tree reuse, tree.rs:239-256)
// nothing but the root state survives a move.
class MCTree {
public:
    // MCTree::init(model, state, apply_noise); (noise_game, noise_ply) key the project's counter-based generator
    static MCTree init(AlphaZero& model, GameState state, bool apply_noise, uint64_t noise_game = 0, uint32_t noise_ply = 0) {
        return MCTree(model, std::move(state), apply_noise, noise_game, noise_ply);
    }
    // NUM_SIMULATIONS simulations from the root; returns visits^(1/T)/sum with T = 1 (tree.rs:106-115)
    Policy monte_carlo_tree_search(int num_simulations = 0) {
        Engine& e = model_->engine();
        const int sims = num_simulations > 0 ? num_simulations : e.config().num_simulations;
        const uint32_t offs[2] = {0, (uint32_t)state.pos_count.size()};
        Policy visits;
        int32_t depth = 0;
        e.check(az_search(e.handle(), 1, &state.position, state.pos_count.data(), offs, sims, noise_ ? &noise_game_ : nullptr,
                          noise_ ? &noise_ply_ : nullptr, visits.data(), nullptr, &depth), "az_search");
        depth_ = (std::size_t)depth;
        float sum = 0.0f;
        for (float v : visits) sum += v;
        if (sum > 0.0f) for (float& v : visits) v = v / sum;
        return visits;
    }
    // NOT IN THE REFERENCE: the same search with up to leaves_per_root leaves per network round and virtual loss
    // (az_search_vl); leaves_per_root = 1 is the overload above bit for bit
    Policy monte_carlo_tree_search(int num_simulations, int leaves_per_root, float virtual_loss) {
        Engine& e = model_->engine();
        const int sims = num_simulations > 0 ? num_simulations : e.config().num_simulations;
        const uint32_t offs[2] = {0, (uint32_t)state.pos_count.size()};
        Policy visits;
        int32_t depth = 0;
        e.check(az_search_vl(e.handle(), 1, &state.position, state.pos_count.data(), offs, sims, leaves_per_root, virtual_loss,
                             noise_ ? &noise_game_ : nullptr, noise_ ? &noise_ply_ : nullptr, visits.data(), nullptr, &depth, nullptr),
                "az_search_vl");
        depth_ = (std::size_t)depth;
        float sum = 0.0f;
        for (float v : visits) sum += v;
        if (sum > 0.0f) for (float& v : visits) v = v / sum;
        return visits;
    }
    // the same with the network in slot `network` of the model's engine (az_search_networks); network 0 is the overload above
    Policy monte_carlo_tree_search(int num_simulations, int leaves_per_root, float virtual_loss, int network) {
        Engine& e = model_->engine();
        const int sims = num_simulations > 0 ? num_simulations : e.config().num_simulations;
        const uint32_t offs[2] = {0, (uint32_t)state.pos_count.size()};
        const uint8_t net = (uint8_t)network;
        if (network < 0 || network >= AZ_MAX_NETWORKS) throw Error(AZ_ERR_INVALID_ARGUMENT, "network must be in [0, AZ_MAX_NETWORKS)");
        Policy visits;
        int32_t depth = 0;
        e.check(az_search_networks(e.handle(), 1, &state.position, state.pos_count.data(), offs, sims, leaves_per_root, virtual_loss, &net,
                                   noise_ ? &noise_game_ : nullptr, noise_ ? &noise_ply_ : nullptr, visits.data(), nullptr, &depth, nullptr),
                "az_search_networks");
        depth_ = (std::size_t)depth;
        float sum = 0.0f;
        for (float v : visits) sum += v;
        if (sum > 0.0f) for (float& v : visits) v = v / sum;
        return visits;
    }
    std::size_t max_subtree_depth() const { return depth_; }   // of the last search (tree.rs:258-269)
    // traverse_new(action, apply_noise): the played move must be legal and the game ongoing (the reference panics otherwise)
    MCTree traverse_new(std::size_t action, bool apply_noise) && {
        GameState next = std::move(state);
        const GameResult r = play_move(model_->engine(), next, action);
        if (r != GameResult::Ongoing) throw Error(AZ_ERR_STATE, "Attempted to traverse to a non-existent child node.");
        return MCTree(*model_, std::move(next), apply_noise, noise_game_, noise_ply_ + 1);
    }
    GameState state;

private:
    MCTree(AlphaZero& m, GameState s, bool noise, uint64_t g, uint32_t p)
        : state(std::move(s)), model_(&m), noise_(noise), noise_game_(g), noise_ply_(p) {}
    AlphaZero* model_;
    bool noise_;
    uint64_t noise_game_;
    uint32_t noise_ply_;
    std::size_t depth_ = 0;
};

// ---- training.rs ------------------------------------------------------------------------------------------------
struct EpisodeStep {            // training.rs:15-20
    Position state;
    Policy improved_policy;
    float final_value;
    std::size_t search_depth;
};

namespace detail {
// the games first_game_id .. first_game_id + n_games - 1 of the self-play just begun, each played to completion
// (training.rs:352-361,376-377); returns (avg_batch_size, steps of the finished games)
inline std::pair<float, std::vector<EpisodeStep>> collect_episodes(Engine& e, int n_games, uint64_t first_game_id, int waves_per_call) {
    std::vector<EpisodeStep> steps;
    std::vector<az_sample> buf((std::size_t)std::max(n_games * 128, 1 << 16));
    const float sims = (float)e.config().num_simulations;
    az_selfplay_stats st{};
    double batches = 0.0, evals = 0.0;
    std::vector<char> finished((std::size_t)n_games, 0);
    int n_finished = 0;
    for (;;) {
        e.check(az_selfplay_step(e.handle(), waves_per_call, &st), "az_selfplay_step");
        batches += waves_per_call;
        evals = (double)st.evaluations;
        if (st.pending_samples) {
            int n = 0;
            e.check(az_selfplay_drain(e.handle(), buf.data(), (int)buf.size(), &n), "az_selfplay_drain");
            for (int i = 0; i < n; i++) {
                char& f = finished[(std::size_t)(buf[i].game_id - first_game_id)];
                if (!f) { f = 1; n_finished++; }
                EpisodeStep s;
                s.state = buf[i].position;
                s.improved_policy.fill(0.0f);
                for (int k = 0; k < buf[i].n_visits; k++) s.improved_policy[buf[i].index[k]] = (float)buf[i].count[k] / sims;  // T = 1
                s.final_value = buf[i].final_value;
                s.search_depth = (std::size_t)buf[i].search_depth;
                steps.push_back(s);
            }
        }
        if (st.active_games == 0 && st.pending_samples == 0) break;  // every slot is idle: all n_games episodes are complete
    }
    return {(float)(evals / batches), std::move(steps)};
}
}  // namespace detail

// run_all_episodes(model): `n_games` self-play games on the device; returns (avg_batch_size, steps of the finished games)
inline std::pair<float, std::vector<EpisodeStep>> run_all_episodes(AlphaZero& model, int n_games, uint64_t first_game_id = 0,
                                                                   int waves_per_call = 64) {
    Engine& e = model.engine();
    e.check(az_selfplay_begin_n(e.handle(), n_games, first_game_id, (uint64_t)n_games), "az_selfplay_begin_n");
    return detail::collect_episodes(e, n_games, first_game_id, waves_per_call);
}

// NOT IN THE REFERENCE: the same games with every ply searched leaf-parallel, up to leaves_per_game leaves per game and network
// round under virtual loss (az_selfplay_begin_vl); leaves_per_game = 1 plays the overload above's games record for record
inline std::pair<float, std::vector<EpisodeStep>> run_all_episodes(AlphaZero& model, int n_games, uint64_t first_game_id, int waves_per_call,
                                                                   int leaves_per_game, float virtual_loss) {
    Engine& e = model.engine();
    e.check(az_selfplay_begin_vl(e.handle(), n_games, first_game_id, (uint64_t)n_games, leaves_per_game, virtual_loss),
            "az_selfplay_begin_vl");
    return detail::collect_episodes(e, n_games, first_game_id, waves_per_call);
}

// ---- validation.rs ------------------------------------------------------------------------------------------------
struct EvaluationResult {       // what evaluate (validation.rs:155-282) returns, from player 1's side
    float winrate;              // (wins + draws / 2) / n_games
    float drawrate;
    float lossrate;             // player 2's wins
};

// evaluate(model, network_1, network_2): n_games games between the model's network slots network_1 (player 1, White in even games)
// and network_2, both Player::MctsModel with num_simulations (0: the config's), or both Player::BaseModel when base_model is set;
// played resident on the device (az_match_*), move sampling keyed by (seed, game, ply).  leaves_per_root > 1 (NOT IN THE
// REFERENCE) searches with virtual loss as az_search_vl.  Games still on after max_plies plies count as draws.  n_concurrent = 0
// plays as many games at once as max_games and the two network ranges (2 x round4(slots x K) <= max_batch) allow.
inline EvaluationResult evaluate(AlphaZero& model, int network_1, int network_2, uint32_t n_games = 256, uint32_t num_stochastic_moves = 15,
                                 uint64_t seed = 0, uint32_t max_plies = 450, int num_simulations = 0, int leaves_per_root = 1,
                                 float virtual_loss = 1.0f, bool base_model = false, int n_concurrent = 0, int waves_per_call = 256) {
    Engine& e = model.engine();
    az_match_config c{};
    c.player_kind = base_model ? 1 : 0;
    c.network[0] = (uint8_t)network_1;
    c.network[1] = (uint8_t)network_2;
    c.num_simulations = num_simulations;
    c.leaves_per_root = leaves_per_root;
    c.virtual_loss = virtual_loss;
    c.num_stochastic_moves = num_stochastic_moves;
    c.max_plies = max_plies;
    c.seed = seed;
    if (n_concurrent <= 0) {
        const int k = base_model ? 1 : std::max(leaves_per_root, 1);
        const int max_batch = std::max(e.config().max_batch, e.config().max_games);
        n_concurrent = std::min<int64_t>({(int64_t)n_games, (int64_t)e.config().max_games, (int64_t)((max_batch / 2) / 4 * 4 / k)});
    }
    e.check(az_match_begin(e.handle(), n_concurrent, 0, n_games, &c), "az_match_begin");
    az_match_stats st{};
    do e.check(az_match_step(e.handle(), waves_per_call, &st), "az_match_step");
    while (st.active_games);
    std::vector<int8_t> white(n_games);
    std::vector<uint16_t> plies(n_games);
    std::vector<uint8_t> finished(n_games);
    e.check(az_match_results(e.handle(), white.data(), plies.data(), finished.data(), nullptr), "az_match_results");
    float wins = 0.0f, draws = 0.0f;
    for (uint32_t g = 0; g < n_games; g++) {
        const int p1 = g % 2 == 0 ? white[g] : -white[g];   // validation.rs:196-200
        wins += p1 == 1 ? 1.0f : 0.0f;
        draws += p1 == 0 ? 1.0f : 0.0f;
    }
    const float n = (float)n_games;
    return {(wins + draws / 2.0f) / n, draws / n, (n - wins - draws) / n};
}

// ---- memory.rs ----------------------------------------------------------------------------------------------------
struct TrainingBatch {          // what ReplayBuffer::sample hands to train() (training.rs:150-172), already stacked
    std::size_t n = 0;
    std::vector<float> planes;  // [n][19][8][8]
    std::vector<float> policy;  // [n][4096]
    std::vector<float> value;   // [n]
};

class ReplayBuffer {            // memory.rs:26-118, device resident
public:
    ReplayBuffer(Engine& e, int capacity = 100000, int max_batch = 512) : eng_(&e), max_batch_(max_batch) {
        az_replay* h = nullptr;
        e.check(az_replay_create(e.handle(), capacity, max_batch, &h), "az_replay_create");
        h_.reset(h);
    }
    // add(step) for a batch of self-play records, in order; returns the number of new unique positions (memory.rs:41-76)
    std::size_t add(const std::vector<az_sample>& steps) {
        int nu = 0;
        eng_->check(az_replay_add(h_.get(), steps.data(), (int)steps.size(), &nu), "az_replay_add");
        return (std::size_t)nu;
    }
    // the finished games still in device memory (no host round trip); returns (steps, new unique positions)
    std::pair<std::size_t, std::size_t> add_pending() {
        int n = 0, nu = 0;
        eng_->check(az_replay_add_pending(h_.get(), &n, &nu), "az_replay_add_pending");
        return {(std::size_t)n, (std::size_t)nu};
    }
    std::size_t len() const {
        int n = 0;
        eng_->check(az_replay_len(h_.get(), &n), "az_replay_len");
        return (std::size_t)n;
    }
    TrainingBatch sample(std::size_t batch_size, uint64_t seed) const {   // memory.rs:78-97
        TrainingBatch b;
        b.planes.resize(batch_size * AZ_NUM_PLANES * 64);
        b.policy.resize(batch_size * ACTION_SPACE);
        b.value.resize(batch_size);
        int n = 0;
        eng_->check(az_replay_sample(h_.get(), (int)batch_size, seed, b.planes.data(), b.policy.data(), b.value.data(), &n), "az_replay_sample");
        b.n = (std::size_t)n;
        b.planes.resize(b.n * AZ_NUM_PLANES * 64); b.policy.resize(b.n * ACTION_SPACE); b.value.resize(b.n);
        return b;
    }
    az_replay* handle() const { return h_.get(); }

private:
    struct Deleter { void operator()(az_replay* r) const { az_replay_destroy(r); } };
    Engine* eng_;
    int max_batch_;
    std::unique_ptr<az_replay, Deleter> h_;
};

// ---- chess.rs:295-318 -----------------------------------------------------------------------------------------------
// get_best_move(pos, depth): the reference picks uniformly among the best-scoring moves with thread_rng; here the caller
// supplies the random number (u in [0,1)) so that a match is reproducible.  None when there is no legal move.
inline std::optional<Move> get_best_move(Engine& e, const Position& pos, uint32_t depth, double u = 0.0) {
    std::vector<int32_t> scores(AZ_MAX_MOVES);
    int32_t count = 0;
    e.check(az_minimax(e.handle(), 1, &pos, (int)depth, scores.data(), &count), "az_minimax");
    if (count == 0) return std::nullopt;
    std::vector<Move> moves = legal_moves(e, pos);
    int32_t best = scores[0];
    for (int i = 1; i < count; i++) best = std::max(best, scores[i]);
    std::vector<Move> best_moves;
    for (int i = 0; i < count; i++) if (scores[i] == best) best_moves.push_back(moves[(std::size_t)i]);
    return best_moves[std::min(best_moves.size() - 1, (std::size_t)(u * (double)best_moves.size()))];
}

}  // namespace az
