/* az_b200.h — C ABI of the B200-native self-play engine.
 *
 * Drop-in boundary for the hot path of AlexandreGac/alphazero-chess (reference: /root/reference/src).
 * The reference has no FFI of its own; every entry point below names the Rust item it replaces so that a thin
 * `-sys` crate can bind it 1:1 (see INTEGRATION.md).  Conventions: every function returns 0 on success or a negative
 * az_status (never aborts, where the reference panics); buffers are caller-owned, flat, host memory unless the name
 * ends in `_dev`; one engine per GPU, calls on one engine must be serialised by the caller.
 * All compute runs in hand-written sm_100a CUDA kernels; there is no CPU fallback.
 */
#ifndef AZ_B200_H
#define AZ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZ_ACTION_SPACE 4096 /* parameters.rs:3 */
#define AZ_MAX_MOVES 256     /* shakmaty MoveList capacity */
#define AZ_NUM_PLANES 19     /* chess.rs:176-189 */
#define AZ_NUM_WEIGHT_ARRAYS 144
#define AZ_MAX_NETWORKS 2    /* network slots of an engine (az_load_network) */

typedef enum az_status {
    AZ_OK = 0,
    AZ_ERR_INVALID_ARGUMENT = -1,
    AZ_ERR_CUDA = -2,
    AZ_ERR_NO_DEVICE = -3,
    AZ_ERR_OUT_OF_MEMORY = -4,
    AZ_ERR_NO_WEIGHTS = -5,
    AZ_ERR_CAPACITY = -6,      /* a per-game node/edge pool or a batch limit was exceeded */
    AZ_ERR_ILLEGAL_MOVE = -7,  /* reference: panic "Illegal move!" (tree.rs:211) */
    AZ_ERR_STATE = -8
} az_status;

/* GameResult (chess.rs:29-34); AZ_RESULT_ILLEGAL mirrors Err("Illegal move") of play_move (chess.rs:38-40) */
enum { AZ_RESULT_ONGOING = 0, AZ_RESULT_DRAW = 1, AZ_RESULT_WHITE_WINS = 2, AZ_RESULT_BLACK_WINS = 3, AZ_RESULT_ILLEGAL = -1 };

/* shakmaty::Chess as plain data (squares a1 = 0 ... h8 = 63) */
typedef struct az_position {
    uint64_t roles[6];  /* pawn, knight, bishop, rook, queen, king */
    uint64_t colors[2]; /* white, black */
    uint8_t turn;       /* 0 white, 1 black */
    uint8_t castling;   /* bit0 white king-side, bit1 white queen-side, bit2 black king-side, bit3 black queen-side */
    int8_t ep_square;   /* -1, or the square passed over by the last double push (kept after every double push) */
    uint8_t reserved;
    uint16_t halfmoves;
    uint16_t fullmoves;
} az_position; /* 72 bytes */

/* Move on the wire: from | to<<6 | promotion<<12 (0 none, 1 knight, 2 bishop, 3 rook, 4 queen) | special<<15.
 * special marks castling (shakmaty encoding: from = king, to = own rook) and en passant. 0xFFFF = None. */
typedef uint16_t az_move;
#define AZ_MOVE_NONE 0xFFFFu

/* parameters.rs as runtime configuration */
typedef struct az_config {
    int32_t device;                 /* CUDA ordinal */
    int32_t max_games;              /* concurrent games / search roots resident on the GPU */
    int32_t max_batch;              /* largest n accepted by the batched entry points (0: max_games) */
    int32_t num_simulations;        /* NUM_SIMULATIONS (256) */
    float c_puct;                   /* C_PUCT (3.0) */
    float dirichlet_alpha;          /* DIRICHLET_ALPHA (0.3) */
    float dirichlet_epsilon;        /* DIRICHLET_EPSILON (0.25) */
    uint32_t temperature_annealing; /* TEMPERATURE_ANNEALING (15) */
    uint32_t num_halfmoves;         /* chess.rs:9 (100) */
    uint32_t num_fullmoves;         /* chess.rs:10 (200) */
    uint32_t repetitions;           /* chess.rs:11 (3) */
    uint64_t seed;                  /* SEED (42): keys the counter-based noise / move-sampling generator */
    int32_t precision;              /* 0: bf16 tensor-core network (tcgen05), 1: fp32 network (parity mode) */
    int32_t cache_log2;             /* log2 slots of the GPU position->evaluation cache (0 disables; training.rs:342) */
    int32_t edge_capacity_per_node; /* average edge-pool budget per tree node (0: 96); overflow -> AZ_ERR_CAPACITY */
    float temperature;              /* TEMPERATURE (1.0): improved policy = visits^(1/T) / sum (tree.rs:173-177) */
} az_config;

typedef struct az_engine az_engine;

void az_config_default(az_config* cfg);
int az_engine_create(const az_config* cfg, az_engine** out); /* replaces the setup in train() (training.rs:40-63) */
void az_engine_destroy(az_engine* eng);
const char* az_last_error(const az_engine* eng);
const char* az_version(void);

/* ---- positions (host helpers, no device work) ------------------------------------------------------------------ */
void az_position_start(az_position* out);                    /* Chess::new() (chess.rs:21) */
int az_position_from_fen(const char* fen, az_position* out); /* test/bench convenience */

/* ---- network (agent.rs) ------------------------------------------------------------------------------------------
 * az_load_weights replaces load_model (main.rs:109-116): `arrays` holds AZ_NUM_WEIGHT_ARRAYS host f32 tensors in burn's
 * layout, in the order returned by az_weight_name(i):
 *   input_conv.{weight[128,19,3,3],bias}, input_bn.{gamma,beta,running_mean,running_var},
 *   res_blocks.N.{conv1.{weight,bias},bn1.{4},conv2.{weight,bias},bn2.{4}} for N = 0..9,
 *   policy_conv_1.{weight[32,128,1,1],bias}, policy_bn.{4}, policy_conv_2.{weight[64,32,1,1],bias},
 *   value_conv.{weight[8,128,1,1],bias}, value_bn.{4}, value_linear_1.{weight[512,64],bias}, value_linear_2.{weight[64,1],bias} */
const char* az_weight_name(int i);
int64_t az_weight_size(int i);
int az_load_weights(az_engine* eng, const float* const* arrays, int n_arrays);
/* same, from device f32 pointers (e.g. the buffer an NCCL broadcast just filled) */
int az_load_weights_dev(az_engine* eng, const float* const* arrays_dev, int n_arrays);
/* Network slots: an engine holds up to AZ_MAX_NETWORKS networks, which the batched calls below select per board or root (the
 * two players of a match, validation.rs:155-282, SURVEY section 8(f) #3).  Slot 0 is what az_load_weights loads; az_load_network
 * loads host arrays (as az_load_weights, same validation and BatchNorm folding) into slot `network`: az_load_network(e, 0, ...)
 * is az_load_weights.  The weights of slot 1 are allocated by its first load; activations and every other buffer are shared. */
int az_load_network(az_engine* eng, int network, const float* const* arrays, int n_arrays);
/* AlphaZero::forward (agent.rs:112-144) on planes [n][19][8][8] -> policy [n][4096] (softmax over ALL indices), value [n] */
int az_forward_planes(az_engine* eng, int n, const float* planes, float* policy_out, float* value_out);
/* to_tensor + forward: what process_batch does per request (training.rs:383-397) */
int az_forward(az_engine* eng, int n, const az_position* pos, float* policy_out, float* value_out);
/* az_forward with a network per board (network[i] < AZ_MAX_NETWORKS, any order): both networks run in the same launches,
 * and every row is bit-identical to az_forward of that board on an engine holding only its network.  AZ_ERR_INVALID_ARGUMENT
 * for an id >= AZ_MAX_NETWORKS, AZ_ERR_NO_WEIGHTS for a network never loaded, AZ_ERR_CAPACITY when the sum over networks of
 * their board counts rounded up to a multiple of 4 exceeds az_config.max_batch.  The bf16 path needs the default AZ_TOWER_*,
 * AZ_INPUT_* and AZ_HEADS_TC configuration (else AZ_ERR_STATE); the fp32 path (precision 1) runs the networks in turn. */
int az_forward_networks(az_engine* eng, int n, const az_position* pos, const uint8_t* network, float* policy_out, float* value_out);

/* ---- chess.rs ------------------------------------------------------------------------------------------------- */
/* Chess::legal_moves() (tree.rs:39,86): moves_out [n][256], index_out [n][256] = move_to_index of each (nullable) */
int az_movegen(az_engine* eng, int n, const az_position* pos, az_move* moves_out, uint16_t* index_out, int32_t* count_out);
/* perft(depth) per root, breadth-first on the GPU (BASELINE config 2) */
int az_perft(az_engine* eng, int n, const az_position* pos, int depth, uint64_t* nodes_out);
/* get_best_move up to its random tie-break (chess.rs:295-318; Player::MiniMax(depth), validation.rs:113,352): the full-width
 * negamax score -negamax(child, depth-1) of every legal move of each root, in az_movegen order.  scores_out [n][256],
 * count_out [n] (0 = no legal move: the reference returns None).  Mate is +-(20000 + remaining depth), draws 0, the
 * horizon is material (100/320/330/500/900) from the mover's side (chess.rs:247-292).  1 <= depth <= 8. */
int az_minimax(az_engine* eng, int n, const az_position* pos, int depth, int32_t* scores_out, int32_t* count_out);
/* play_move (chess.rs:36-63) driven by a policy index as in tree.rs:211-212.  history is the concatenation of every
 * position already counted in GameState::pos_count (including the current one), hist_offsets[n+1] delimits games. */
int az_play_move(az_engine* eng, int n, az_position* pos_inout, const az_position* history, const uint32_t* hist_offsets,
                 const uint16_t* action_index, int32_t* result_out);
/* move_to_index (chess.rs:73-116) */
int az_move_to_index(az_engine* eng, int n, const az_position* pos, const az_move* moves, uint16_t* index_out);
/* index_to_move (chess.rs:118-171): AZ_MOVE_NONE where the reference returns None */
int az_index_to_move(az_engine* eng, int n, const az_position* pos, const uint16_t* index, az_move* moves_out);
/* to_tensor (chess.rs:191-245): planes_out [n][19][8][8] f32 */
int az_encode(az_engine* eng, int n, const az_position* pos, float* planes_out);

/* ---- tree.rs ---------------------------------------------------------------------------------------------------
 * MCTree::init + monte_carlo_tree_search (tree.rs:37-64,106-115) for n roots at once: one simulation in flight per
 * game (F5), batch = games.  visits_out [n][4096] are raw visit counts (improved policy = visits / sims at T = 1),
 * depth_out = max_subtree_depth (tree.rs:258-269).  noise_game_ids (nullable) enables root Dirichlet noise keyed by
 * (seed, game id, noise_ply).  history/hist_offsets as in az_play_move (nullable: GameState::new semantics). */
int az_search(az_engine* eng, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
              int num_simulations, const uint64_t* noise_game_ids, const uint32_t* noise_plies, float* visits_out,
              float* scores_out, int32_t* depth_out);

/* NOT IN THE REFERENCE: leaf-parallel search with virtual loss for callers with few roots (a non-parity mode, except at
 * leaves_per_root = 1, where results are bit-identical to az_search).  Each root runs its simulations in batches of up to
 * leaves_per_root (K) leaves that share one network round: descents score every edge with N' = N + V and W' = W -
 * virtual_loss * V, V being the descents of the current batch through the edge; a descent ending on an edge another descent of
 * the batch already took (a collision) ends the root's batch.  Leaves are expanded as in tree.rs and backed up in gather
 * order, so results are deterministic.  Exactly num_simulations visits per non-terminal root.  n * K <= az_config.max_batch
 * (else AZ_ERR_CAPACITY); K >= 1 and a finite virtual_loss >= 0 (else AZ_ERR_INVALID_ARGUMENT).  The other arguments are
 * those of az_search.  The in-flight counts (4 bytes per edge of the pool) and per-leaf paths (8 bytes x (num_simulations + 2)
 * per max_batch slot) are allocated by the first call. */
typedef struct az_search_stats {
    uint64_t waves;           /* network rounds */
    uint64_t evaluations;     /* boards sent to the network */
    uint64_t terminal_leaves;
    uint64_t collisions;      /* descents discarded because their leaf edge was already taken in the batch */
} az_search_stats;
int az_search_vl(az_engine* eng, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                 int num_simulations, int leaves_per_root, float virtual_loss, const uint64_t* noise_game_ids,
                 const uint32_t* noise_plies, float* visits_out, float* scores_out, int32_t* depth_out,
                 az_search_stats* stats_out /* nullable */);

/* az_search_vl with a network per root (network[i] < AZ_MAX_NETWORKS): the match ply of evaluate (validation.rs:155-282) with
 * both players' roots in one call, so that they share every network round.  The same semantics as az_search_vl -- a parity
 * mode only at leaves_per_root = 1, where each root's results equal az_search of that root on an engine holding its network --
 * and the same errors, plus: AZ_ERR_INVALID_ARGUMENT for an id >= AZ_MAX_NETWORKS, AZ_ERR_NO_WEIGHTS for a network never loaded
 * (not under the synthetic evaluator, where network s uses seed + s), AZ_ERR_CAPACITY when the sum over networks of
 * (roots x leaves_per_root) rounded up to a multiple of 4 exceeds az_config.max_batch. */
int az_search_networks(az_engine* eng, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                       int num_simulations, int leaves_per_root, float virtual_loss, const uint8_t* network,
                       const uint64_t* noise_game_ids, const uint32_t* noise_plies, float* visits_out, float* scores_out,
                       int32_t* depth_out, az_search_stats* stats_out /* nullable */);

/* test hook: replace the network by the deterministic synthetic evaluator shared with the oracle (kind 1) or
 * restore the network (kind 0) */
int az_set_evaluator_stub(az_engine* eng, int kind, uint64_t seed);

/* ---- training.rs run_episode / run_all_episodes ------------------------------------------------------------------
 * Self-play is resident on the device: az_selfplay_begin resets n_games games to the start position (game ids
 * first_game_id ...), az_selfplay_step advances every game by `waves` network evaluations, finished games restart with
 * fresh ids, az_selfplay_drain copies finished EpisodeSteps (training.rs:15-20) to the host in a sparse format. */
typedef struct az_selfplay_stats {
    uint64_t simulations;     /* async_simulation calls from a root (tree.rs:180) */
    uint64_t positions;       /* EpisodeSteps produced (training.rs:303) */
    uint64_t evaluations;     /* network forwards requested */
    uint64_t cache_hits;      /* CACHE_HITS (training.rs:12) */
    uint64_t terminal_leaves; /* simulations that ended in a terminal position */
    uint64_t games_finished;
    uint64_t sum_leaf_depth;  /* for the measured mean descent depth */
    uint64_t sum_edges;       /* edges visited by selection (bytes model of DESIGN.md) */
    uint64_t waves;
    uint64_t pending_samples; /* samples waiting for az_selfplay_drain */
    uint64_t active_games;    /* slots still playing (az_selfplay_begin_n: 0 once every game of the generation has ended) */
    uint64_t parked_games;    /* finished games waiting for room in the sample queue (drain to let them publish) */
    uint64_t cache_evictions; /* cache entries replaced by newer ones (capacity management, parameters.rs:4) */
    uint64_t sum_search_depth; /* sum of EpisodeStep::search_depth over `positions`: avg_search_depth of training.rs:91-97 */
} az_selfplay_stats;

typedef struct az_sample {
    az_position position;   /* EpisodeStep::state */
    float final_value;      /* EpisodeStep::final_value */
    int32_t search_depth;   /* EpisodeStep::search_depth */
    uint64_t game_id;
    uint32_t ply;
    uint16_t action;        /* policy index actually played */
    uint16_t n_visits;      /* number of (index, count) pairs: improved_policy[index] = count / sims */
    uint16_t index[AZ_MAX_MOVES];
    uint16_t count[AZ_MAX_MOVES];
} az_sample;

int az_selfplay_begin(az_engine* eng, int n_games, uint64_t first_game_id);
/* run_all_episodes (training.rs:340-378) plays exactly NUM_EPISODES games to completion: n_concurrent slots play the games
 * first_game_id .. first_game_id + total_games - 1; a slot whose game ends takes the next unplayed id or goes idle, and
 * stats.active_games reaches 0 when the generation is complete.  total_games = 0: games restart forever (az_selfplay_begin). */
int az_selfplay_begin_n(az_engine* eng, int n_concurrent, uint64_t first_game_id, uint64_t total_games);
/* NOT IN THE REFERENCE: az_selfplay_begin_n with the search of every ply run as in az_search_vl (a non-parity mode, except at
 * leaves_per_game = 1, where every record is byte-identical to az_selfplay_begin_n's).  Each game puts up to leaves_per_game (K)
 * leaves into every network round (virtual loss, collisions end a game's batch, expansion after the gather, backups in leaf
 * order); a game whose search is complete plays its move and gathers the first batch of its next ply in the same wave.  Root
 * priors, noise, move choice, exactly-N / endless generations, parking and draining are those of az_selfplay_begin_n, and a
 * game's records depend only on (config, seed, game id, K, virtual_loss, network), not on the slots or the other games.
 * az_selfplay_step then runs these waves, with stats as documented above except: evaluations = boards sent to the network,
 * cache_hits = 0, sum_edges = 0.  Errors (the engine stays usable): AZ_ERR_INVALID_ARGUMENT for K < 1 or a negative or
 * non-finite virtual_loss, AZ_ERR_CAPACITY when n_concurrent x K > az_config.max_batch, AZ_ERR_STATE with the evaluation cache
 * (cache_log2 > 0), AZ_ERR_NO_WEIGHTS as az_selfplay_begin_n.  Uses the buffers of az_search_vl (allocated by the first call of
 * either).  A later az_selfplay_begin_n or az_search* call returns the engine to the default path. */
int az_selfplay_begin_vl(az_engine* eng, int n_concurrent, uint64_t first_game_id, uint64_t total_games, int leaves_per_game,
                         float virtual_loss);
/* since az_selfplay_begin_vl: waves (network rounds of az_selfplay_step), leaf evaluations (the start-position forward is not
 * counted), terminal leaves and collisions.  AZ_ERR_STATE when no az_selfplay_begin_vl self-play is in progress. */
int az_selfplay_vl_stats(az_engine* eng, az_search_stats* stats_out);
int az_selfplay_step(az_engine* eng, int waves, az_selfplay_stats* stats_out);
int az_selfplay_drain(az_engine* eng, az_sample* out, int max_samples, int* n_out);
/* same, into DEVICE memory (e.g. the send buffer of an NCCL gather): no host hop between self-play and the replay buffer */
int az_selfplay_drain_dev(az_engine* eng, az_sample* out_dev, int max_samples, int* n_out);

/* ---- validation.rs evaluate (validation.rs:155-282) ----------------------------------------------------------------
 * A match is resident on the device: az_match_begin sets up n_games games (game indices first_game .. first_game + n_games - 1)
 * on n_concurrent slots, az_match_step advances every slot by `waves` network rounds, az_match_results copies each game's result
 * and moves to the host.  Both players live on this engine (network slots network[0] for player 1, network[1] for player 2,
 * equal or not) and share every network round.  Player 1 is White in even games (validation.rs:196-200).  Each ply searches a
 * fresh root (MCTree::init(model, state, false): no tree reuse, no noise) with the game's whole history, with az_search_vl
 * semantics at leaves_per_root K (K = 1: az_search) -- or, for BaseModel players, takes the root's priors of the legal moves.
 * The mover samples while the position's fullmove number <= num_stochastic_moves and otherwise takes the last maximum, over the
 * weights visits / sum(visits) (MCTS, temperature ignored) or the priors (BaseModel) in policy-index order: f32 cumulative sums,
 * the first one > f32(u) x total, u = (mix(seed, game, ply) >> 11) x 2^-53 with the splitmix-style mix of
 * alphazero-chess_b200/evaluation.py (not the engine's generator).  Moves are played through the rules of az_play_move.  A game
 * still on after max_plies plies is unfinished, with result 0.  A game's moves and result depend only on (config, seed, game
 * index, the players' settings, the two networks), never on the slots or the other games, and equal those of evaluation.py's
 * host loop `evaluate`.  NOT IN THE REFERENCE: the reference samples from an unseeded thread_rng, and leaves_per_root > 1 is a
 * non-parity mode as in az_search_vl. */
typedef struct az_match_config {
    int32_t player_kind;           /* 0: Player::MctsModel for both sides, 1: Player::BaseModel for both sides */
    uint8_t network[2];            /* network slot of player 1 and of player 2 */
    int32_t num_simulations;       /* MCTS: 1 .. az_config.num_simulations (0: az_config.num_simulations) */
    int32_t leaves_per_root;       /* MCTS: K >= 1 (1: az_search semantics) */
    float virtual_loss;            /* MCTS: finite, >= 0 */
    uint32_t num_stochastic_moves; /* TEMPERATURE_ANNEALING (parameters.rs:31: 15) */
    uint32_t max_plies;            /* >= 1 (450 in evaluation.py) */
    uint64_t seed;
} az_match_config;
typedef struct az_match_stats {   /* totals since az_match_begin */
    uint64_t waves;                /* network rounds */
    uint64_t evaluations[AZ_MAX_NETWORKS]; /* boards sent to each network: roots and non-terminal leaves */
    uint64_t leaves;               /* leaves gathered by the searches */
    uint64_t terminal_leaves;
    uint64_t collisions;
    uint64_t plies;                /* moves played */
    uint64_t games_finished;       /* games with a recorded result: ended by the rules or cut at max_plies */
    uint64_t active_games;         /* games in progress (0: the match is complete) */
    uint64_t cache_hits[AZ_MAX_NETWORKS]; /* az_match_players_config.cache_log2 > 0: roots and leaves of each network taken from the
                                             match's evaluation cache instead of the network (evaluations + cache_hits = the
                                             evaluations of the same match without the cache) */
} az_match_stats;
/* Errors (the engine stays usable): AZ_ERR_INVALID_ARGUMENT for an unknown player_kind, a network id >= AZ_MAX_NETWORKS, and for
 * MCTS players K < 1, a negative or non-finite virtual_loss or num_simulations out of range; also for n_concurrent < 1, n_games
 * = 0 or max_plies = 0.  AZ_ERR_NO_WEIGHTS for a network slot never loaded (not under the synthetic evaluator, where network s
 * uses seed + s).  AZ_ERR_CAPACITY when n_concurrent > az_config.max_games or the two network ranges do not fit
 * az_config.max_batch: network 0's range holds n_concurrent x K boards from board 0, network 1's as many from
 * round4(n_concurrent x K), and round4(n_concurrent x K) x 2 must fit (K = 1 for BaseModel players).  AZ_ERR_STATE for a bf16
 * engine with non-default AZ_TOWER_* / AZ_INPUT_* / AZ_HEADS_TC settings, as az_forward_networks.  Within max_games,
 * n_concurrent > n_games plays on n_games slots.  The match uses the search buffers of az_search_vl (allocated by the first call of either), so a later
 * az_selfplay_begin* or az_search* call ends it; az_engine_create's footprint is unchanged. */
int az_match_begin(az_engine* eng, int n_concurrent, uint32_t first_game, uint32_t n_games, const az_match_config* config);

/* Mixed pairings: each player has its own kind and settings (evaluation.py's MctsPlayer, BasePlayer and RandomPlayer).  The match
 * plays the games evaluation.py's `evaluate` plays for those players on this engine, bit for bit, as az_match_begin does for two
 * equal players (az_match_begin is this call with two players of its kind and settings).  An MCTS player searches each of its
 * plies with its own num_simulations S, leaves_per_root K and virtual_loss on its network slot; a BaseModel player takes its
 * network's priors of the legal moves; both choose as az_match_begin describes.  A Random player plays
 * index[int(u x count)] of az_movegen's legal moves (az_movegen order, under-promotions included), u = (mix(seed ^ 0x5151, game,
 * ply) >> 11) x 2^-53 and the product in double, whatever the fullmove number.  A Random ply needs no network round: the slot
 * plays it in the wave in which its root is set up and goes on with the next ply, so Random vs Random needs no weights and makes
 * no evaluation.  A Random ply counts in az_match_stats.plies and in no evaluations[]. */
#define AZ_PLAYER_MCTS 0         /* Player::MctsModel */
#define AZ_PLAYER_BASE_MODEL 1   /* Player::BaseModel */
#define AZ_PLAYER_RANDOM 2       /* Player::Random */
typedef struct az_match_player {
    int32_t kind;                  /* AZ_PLAYER_* */
    uint8_t network;               /* MCTS and BaseModel: network slot (ignored for Random) */
    int32_t num_simulations;       /* MCTS: 1 .. az_config.num_simulations (0: az_config.num_simulations) */
    int32_t leaves_per_root;       /* MCTS: K >= 1 (1: az_search semantics) */
    float virtual_loss;            /* MCTS: finite, >= 0 */
} az_match_player;
typedef struct az_match_players_config {
    az_match_player player[2];     /* player 1 (White in even games) and player 2 */
    uint32_t num_stochastic_moves; /* TEMPERATURE_ANNEALING (parameters.rs:31: 15) */
    uint32_t max_plies;            /* >= 1 (450 in evaluation.py) */
    uint64_t seed;
    int32_t cache_log2;            /* 0: no evaluation cache.  1 .. 26: the match gets its own cache of 2^cache_log2 slots of 1 KiB
                                      each (cache_log2 = 20: 1 GiB of device memory), allocated by the first match that needs it,
                                      kept for later ones and emptied by every begin call */
} az_match_players_config;
/* The evaluation cache (cache_log2 > 0) is the one self-play uses (az_config.cache_log2, training.rs:342) with the network slot in
 * its key: a root or leaf whose position (FEN identity: board, turn, castling, pseudo-legal ep, both move counters) was evaluated
 * earlier in the match by the same network takes that evaluation's priors and value instead of a network round.  Network rows
 * are batch-invariant, so the games, the moves and every search are those of the match without the cache, bit for bit; only the
 * boards sent to the network drop, by az_match_stats.cache_hits.  Hit counts may differ between runs (slots race to insert
 * within a wave); the games do not.  The engine's self-play cache is neither used nor changed.
 * Errors (the engine stays usable): AZ_ERR_INVALID_ARGUMENT for an unknown kind (MiniMax included), a network id >=
 * AZ_MAX_NETWORKS of an MCTS or BaseModel player, for an MCTS player's K < 1, negative or non-finite virtual_loss or
 * num_simulations out of range, for cache_log2 < 0 or > 26, and for n_concurrent < 1, n_games = 0 or max_plies = 0.
 * AZ_ERR_OUT_OF_MEMORY when the cache cannot be allocated.  AZ_ERR_NO_WEIGHTS for a network slot
 * never loaded that an MCTS or BaseModel player uses (not under the synthetic evaluator).  AZ_ERR_CAPACITY when n_concurrent >
 * az_config.max_games or the network ranges do not fit az_config.max_batch: each network used by a player gets
 * round4(slots x K) boards, K the largest leaves_per_root of its players (1 for BaseModel), network 0's range from board 0 and
 * network 1's right after it; a network no player uses reserves nothing.  AZ_ERR_STATE as az_match_begin, when a network is
 * used.  az_match_step, az_match_stats and az_match_results serve both begin calls. */
int az_match_begin_players(az_engine* eng, int n_concurrent, uint32_t first_game, uint32_t n_games, const az_match_players_config* config);
/* AZ_ERR_STATE when no match is in progress; AZ_ERR_CAPACITY when a search pool overflowed (raise edge_capacity_per_node) */
int az_match_step(az_engine* eng, int waves, az_match_stats* stats_out /* nullable */);
/* per game of the last match begun, in game-index order: result from White's side (1, 0, -1), plies played, 1 if the game ended
 * by the rules (0: cut at max_plies, or still in progress), and moves_out [n_games][max_plies] the policy indices played
 * (AZ_MOVE_NONE after the last).  Readable until the next az_match_begin* call that passes its argument checks (one that then
 * fails to allocate leaves no match and no results), also after a later search or self-play call ended the match; AZ_ERR_STATE
 * before the first az_match_begin. */
int az_match_results(az_engine* eng, int8_t* result_out, uint16_t* plies_out, uint8_t* finished_out, uint16_t* moves_out /* nullable */);

/* ---- memory.rs: ReplayBuffer (SURVEY section 8(f) #1, the consumer of self-play output) ---------------------------
 * Device resident.  az_replay_add mirrors ReplayBuffer::add (memory.rs:41-76) for a batch of EpisodeSteps applied in
 * order: positions are de-duplicated by their FEN identity (pseudo-legal ep, counters), policy/value become running
 * means, the oldest unique position is evicted at capacity; *new_unique_out is the sum of add()'s return values.
 * az_replay_add_pending consumes the finished-game samples self-play left in device memory (no host round trip).
 * az_replay_sample mirrors ReplayBuffer::sample (memory.rs:78-97): min(batch, len) distinct entries, uniformly, returned as
 * to_tensor planes [n][19][8][8], policy [n][4096] and value [n].
 * az_replay_export / az_replay_import move pages (<= max_batch entries) of {position, policy[4096], value, visit_count} in
 * FIFO order (oldest first) for ReplayBuffer::save / load (memory.rs:100-115); the bincode framing of the reference's file
 * is host-side (alphazero-chess_b200/replay_io.py).  Imported entries are appended as the newest ones. */
typedef struct az_replay az_replay;
int az_replay_create(az_engine* eng, int capacity, int max_batch, az_replay** out);
void az_replay_destroy(az_replay* rp);
int az_replay_add(az_replay* rp, const az_sample* samples, int n, int* new_unique_out);
int az_replay_add_pending(az_replay* rp, int* n_added_out, int* new_unique_out);
/* az_replay_add for samples already in device memory (what an NCCL gather delivered) */
int az_replay_add_dev(az_replay* rp, const az_sample* samples_dev, int n, int* new_unique_out);
int az_replay_len(az_replay* rp, int* len_out);
int az_replay_sample(az_replay* rp, int batch_size, uint64_t seed, float* planes_out, float* policy_out, float* value_out, int* n_out);
/* the same batch into DEVICE memory (the trainer's input tensors): no host hop between the replay buffer and the training step */
int az_replay_sample_dev(az_replay* rp, int batch_size, uint64_t seed, float* planes_dev, float* policy_dev, float* value_dev, int* n_out);
int az_replay_export(az_replay* rp, int first, int n, az_position* pos_out, float* policy_out, float* value_out, uint32_t* visits_out,
                     int* n_out);
int az_replay_import(az_replay* rp, int n, const az_position* pos, const float* policy, const float* value, const uint32_t* visits);
/* test hook: the entry stored for one position (visit_count 0 if absent) */
int az_replay_get(az_replay* rp, const az_position* pos, float* policy_out, float* value_out, uint32_t* visit_count_out);

/* ---- measurement hooks (bench.py) -------------------------------------------------------------------------------
 * az_timer_*: CUDA events on the engine's own stream.  az_profile_enable(k): every k-th network forward brackets the
 * 20 tower convolutions with events and records the batch size; az_profile_read sums what has completed. */
typedef struct az_profile {
    double tower_ms;        /* summed duration of the sampled 20-convolution towers */
    uint64_t tower_samples; /* number of sampled forwards */
    uint64_t tower_boards;  /* summed batch sizes of the sampled forwards */
    double input_ms;        /* input convolution of the sampled forwards */
    double heads_ms;        /* policy/value heads of the sampled forwards */
    double advance_ms;      /* search kernel (k_advance) that produced the sampled batches (0 outside search/self-play) */
    uint64_t tower_launches; /* tower kernel launches inside the sampled forwards (one per L2-sized board range) */
} az_profile;
int az_timer_start(az_engine* eng);
int az_timer_stop(az_engine* eng, float* ms_out);
int az_profile_enable(az_engine* eng, int every_n_forwards);
int az_profile_read(az_engine* eng, az_profile* out);
uint64_t az_launch_count(const az_engine* eng); /* kernels launched by this engine so far */

/* ---- unit-test entry points (device pointers) ------------------------------------------------------------------ */
/* legal moves through the warp-cooperative generator of the search kernel (one warp per position) */
int az_dbg_movegen_warp(az_engine* eng, int n, const az_position* pos, az_move* moves_out, int32_t* count_out);
/* the EpisodeSteps staged so far by the unfinished game in slot `slot` (published to the sample queue when it ends) */
int az_dbg_selfplay_staged(az_engine* eng, int slot, az_sample* out, int max_samples, int* n_out);
int az_dbg_conv3x3_tc(const void* in_bf16, int cin, const void* w_bf16, const float* bias, const void* residual,
                      void* out_bf16, int n_boards, int relu, int iters, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* AZ_B200_H */
