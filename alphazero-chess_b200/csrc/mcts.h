// Device-resident PUCT search and self-play (tree.rs:25-289, training.rs:294-378).
#pragma once
#include "engine.h"
#include <cuda_bf16.h>

namespace azb {

constexpr int HIST_CAP = 512;     // positions kept per game (a game ends by fullmove 200 => < 400 plies)
constexpr int MAX_SAMPLE_PLIES = 512;

struct __align__(16) GameCtl {
    unsigned long long game_id;
    uint32_t n_nodes, n_edges;
    uint32_t sims_done, ply;
    uint32_t hist_len;
    int32_t pending_node;   // node waiting for its evaluation (-1 none)
    int32_t pending_slot;
    uint32_t path_len;      // edges on the path of the pending simulation
    uint32_t max_depth;
    uint32_t status;        // 0 active, 1 search finished / slot idle, 2 capacity error, 3 illegal state, 4 parked: the game is over
                            //   and its samples wait for room in the sample queue (park_scale = result x decay)
    uint32_t noise_ply;
    uint32_t flags;         // bit0: Dirichlet noise at the root; bits 8-15: number of edges of the root (its offset is 0)
    uint32_t n_samples;
    uint32_t park_scale;    // f32 bits
};

struct SearchParams {
    int n_games;
    int S;
    float c_puct, alpha, eps;
    uint32_t anneal;
    int num_halfmoves, num_fullmoves, repetitions;
    unsigned long long seed;
    int node_cap, edge_cap;
    int mode;        // 0: az_search (stop after S simulations), 1: self-play
    int max_iters;   // simulations a game may complete per wave without needing the network
    int fp32_planes; // 1: requests are written as f32 NCHW planes, 0: bf16 NHWC
    int plane_ch;    // channel pitch of the bf16 plane buffer (32; 64 with AZ_INPUT_K32=0)
    int sample_cap;
    uint32_t cache_mask;  // slots - 1 (0: cache disabled)
    int priors_scattered; // 1: the evaluator already wrote the legal-move priors into edge_P (fused heads)
    unsigned long long last_game_id;  // self-play: game ids >= this are not started (0: games restart forever)
    float inv_temperature;            // 1 / TEMPERATURE as f32 (tree.rs:174)
    uint32_t cache_epoch;             // coarse clock (one tick per ply of self-play) used to age cache entries, 6 bits
    int consume;                      // 1: first k_advance pass of a wave (evaluations of the previous wave are consumed);
                                      // 0: an extra pass -- only games that still have no request in flight run
};

// Position -> (legal-move priors, value) cache: the moka Cache<Fen, CacheEntry> of training.rs:342 / tree.rs:214-218.
// Key = everything Fen::from_position(.., EnPassantMode::PseudoLegal) contains (board, turn, castling, pseudo-legal ep,
// halfmove clock, fullmove number), compared exactly.  A published entry is immutable until it is evicted.
//
// Slot state word: [1:0] 0 empty / 1 being written / 2 published, [7:2] epoch of the last insertion or hit, [13:8] rewrite
// sequence of the slot, [31:14] 18 tag bits of the key's hash.  Capacity management (moka's role, parameters.rs:4): when the
// 8 probed slots are all taken, the entry that has not been inserted or hit for the most epochs (at least CACHE_MIN_AGE)
// is replaced.  Readers are seqlock style: observe the word (acquire), compare the key, copy, fence, observe the word again;
// any change other than the epoch bits discards the hit, so a reader never uses a half-replaced entry.
constexpr int CACHE_MAX_PRIORS = 238;
constexpr uint32_t CACHE_EPOCH_MASK = 63u << 2;
constexpr int CACHE_MIN_AGE = 2;
struct __align__(16) CacheEntry {
    DPos key;
    float value;
    uint32_t n_priors;
    float prior[CACHE_MAX_PRIORS];
};
static_assert(sizeof(CacheEntry) == 1024, "one cache slot is 1 KiB: with cudaMalloc's 256-byte alignment no two entries share a 128-byte line");

struct Counters {
    unsigned long long simulations, positions, evaluations, cache_hits, terminal_leaves, games_finished, sum_leaf_depth, sum_edges,
        next_game_id, samples_out, errors;
};

constexpr unsigned long long EDGE_NO_CHILD = ~0ULL;
constexpr int STAT_STRIPES = 64;
constexpr int STAT_WIDTH = 40;    // per stripe: 0..7 the statistics fields of Counters, 8..15 AZ_ADV_TIMING phase clocks, 16 cache evictions, 17 sum of search depths,
                                  // 24..39 AZ_ADV_TIMING histogram of a warp's time in k_advance (buckets of 4096 clocks)

struct SearchPtrs {
    // nodes [G * node_cap]
    DPos* node_pos;
    uint32_t* node_edge_off;
    uint16_t* node_nedges;
    uint16_t* node_nmoves;
    uint16_t* node_depth;
    // edges [G * edge_cap]
    float* edge_P;
    float* edge_N;
    float* edge_W;
    unsigned long long* edge_link;   // child node id | its edge count << 16 | its edge offset << 24 (EDGE_NO_CHILD: none): selection
                                     // walks from edges to edges without a dependent load of the child's node record
    uint32_t* edge_mv;   // wire move | policy index << 16
    // per game
    GameCtl* ctl;
    uint2* path;         // [G][node_cap]: x = node | edge << 16, y = the edge's index in the game's edge pool (saves backup a lookup)
    DPos* hist;          // [G][HIST_CAP]
    // evaluation requests / results
    int* batch_count;          // this wave's request counter (one of two: run_wave alternates, see batch_zero)
    int* batch_zero;           // the other counter: k_advance clears it for the next wave (no memset launch per wave); may be null
    DPos* req_pos;             // [max_batch]
    __nv_bfloat16* req_bf16;   // [max_batch][64][plane_ch]
    float* req_f32;            // [max_batch][19][64]
    unsigned long long* req_edge_off;  // [max_batch] first edge (global index) of the node each request will fill
    int* req_nedges;           // [max_batch]
    const float* res_policy;   // [max_batch][4096]
    const float* res_value;    // [max_batch]
    // self-play
    az_sample* game_samples;   // [G][MAX_SAMPLE_PLIES]
    az_sample* out_samples;    // [sample_cap]
    float* start_prior;        // [32] priors of the start position's legal moves (move order)
    uint32_t* cache_state;     // [slots] 0 empty, 1 being written, (tag << 2) | 2 published
    CacheEntry* cache_entry;   // [slots]
    Counters* counters;
    unsigned long long* stats;         // [STAT_STRIPES][STAT_WIDTH]: the statistics fields of Counters, striped by block to spread the atomics
};

// The session-bound calls an engine accepts.  az_selfplay_begin_n / az_selfplay_begin_vl / az_match_begin start a session once
// their arguments are accepted; every az_search* call that gets past its argument checks ends it.
enum class Session { none, selfplay, selfplay_vl, match };

// az_selfplay_begin_vl: leaves per game of the self-play in progress, its virtual loss and the waves run since the begin call
struct SelfplayVL {
    int K = 0;
    float lambda = 0.0f;
    unsigned long long waves = 0;
};

// a device buffer that grows only when a larger one is needed (its owner frees `p`)
template <class T>
struct GrowBuf {
    T* p = nullptr;
    size_t cap = 0;   // elements
};

// az_match_*: the match in progress and the results of the last one begun (readable after a search has ended the match).
// The result buffers belong to the match; the search buffers are shared with az_search_vl
struct MatchState {
    uint32_t games = 0;                    // games of the last az_match_begin (0: none yet)
    int K = 1;                             // leaves per root per wave (1 for BaseModel players)
    uint32_t row = 0;                      // moves stored per game on the device (<= HIST_CAP: a game ends by then)
    unsigned long long first = 0;          // the first game index
    int first_wave = 0;                    // 1 until the first wave has run: every slot starts a game
    unsigned long long waves = 0;
    unsigned long long* next = nullptr;    // [1] next game index to start
    unsigned long long* stats = nullptr;   // [4] evaluations of network 0, of network 1, plies, games ended
    GrowBuf<int8_t> result;                // [games]
    GrowBuf<uint16_t> plies;
    GrowBuf<uint8_t> finished;
    GrowBuf<uint16_t> moves;               // [games][row]
    az_match_config cfg{};
    az_position startpos{};
};

struct SearchState {
    SearchParams prm;
    SearchPtrs ptr;
    int G = 0;
    Session session = Session::none;
    unsigned long long cache_evictions = 0;
    unsigned long long sum_search_depth = 0;
    int adv_passes = 1;                    // k_advance launches per wave (AZ_ADV_PASSES, see run_wave)
    int* batch_base = nullptr;             // [8] ints: two alternating request counters, then four flag words
    int batch_parity = 0;
    unsigned long long wave_counter = 0;   // self-play waves since az_selfplay_begin (cache epoch = wave_counter / S)
    unsigned long long* d_noise_ids = nullptr;  // [max_games] az_search staging (no allocation per call)
    uint32_t* d_noise_plies = nullptr;
    SelfplayVL sp_vl;
    // az_search_vl and az_selfplay_begin_vl, allocated by the first such call (az_engine_create's footprint does not include them)
    uint32_t* vl_V = nullptr;              // [G * edge_cap] descents of the current batch through each edge
    uint2* vl_path = nullptr;              // [max_batch][node_cap] one descent per leaf
    int* vl_len = nullptr;                 // [max_batch]
    int* vl_slot = nullptr;                // [max_batch]
    float* vl_value = nullptr;             // [max_batch]
    int* vl_count = nullptr;               // [G]
    unsigned long long* vl_stats = nullptr; // [4]
    uint8_t* d_net = nullptr;              // [G] az_search_networks: network of each root (allocated on its first call)
    MatchState match;
    std::vector<void*> allocs;
};

int search_create(az_engine* e);
// finished-game samples waiting in device memory (what az_selfplay_drain would copy out); clearing resets the queue
int search_pending_samples(az_engine* e, const az_sample** d_samples, int* n);
int search_clear_pending(az_engine* e);
void search_destroy(az_engine* e);

}  // namespace azb
