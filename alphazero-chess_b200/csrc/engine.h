// Internal engine state shared by the translation units of libaz_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <string>
#include <vector>
#include "../../include/az_b200.h"
#include "chess.cuh"

namespace azb {

struct NetWeights;   // nn_weights.cu
struct SearchState;  // mcts.cu

struct RuleParams {
    int num_halfmoves, num_fullmoves, repetitions;
};

}  // namespace azb

struct az_engine {
    az_config cfg;
    cudaStream_t stream = nullptr;
    std::string err;
    int max_batch = 0;
    int sm_count = 148;

    // staging for the batched chess.rs entry points (device)
    az_position* d_wire = nullptr;     // [max_batch]
    az_position* d_hist = nullptr;     // history staging (grown on demand)
    size_t hist_cap = 0;
    uint32_t* d_hist_off = nullptr;    // [max_batch + 1]
    uint16_t* d_moves = nullptr;       // [max_batch][256]
    uint16_t* d_index = nullptr;       // [max_batch][256]
    int32_t* d_count = nullptr;        // [max_batch]
    uint16_t* d_u16a = nullptr;        // [max_batch]
    uint16_t* d_u16b = nullptr;        // [max_batch]
    float* d_planes = nullptr;         // [max_batch][19*64]
    float* d_policy = nullptr;         // [max_batch][4096]
    float* d_value = nullptr;          // [max_batch]
    float* d_scores = nullptr;         // [max_batch][4096] (az_search scores export, lazy)

    // perft level buffers (allocated lazily)
    std::vector<azb::DPos*> perft_pos;
    std::vector<uint32_t*> perft_root;
    unsigned long long* d_perft_count = nullptr;
    unsigned long long* d_perft_nodes = nullptr;
    size_t perft_cap = 0;
    // minimax (az_minimax): per-level score arrays beside the perft level buffers, root bookkeeping
    std::vector<int*> mm_score;
    unsigned int* d_mm_first = nullptr;  // [max_batch]
    int* d_mm_nchild = nullptr;          // [max_batch]
    int* d_mm_out = nullptr;             // [max_batch][256]
    int* d_mm_count = nullptr;           // [max_batch]

    // measurement
    uint64_t n_launches = 0;
    cudaEvent_t timer0 = nullptr, timer1 = nullptr;
    int prof_every = 0;
    uint64_t prof_counter = 0;
    struct ProfSample { cudaEvent_t adv, in0, a, b, h1; int slot; };  // advance start, input conv start, tower start/end, heads end
    cudaEvent_t prof_adv_event = nullptr;  // recorded before k_advance when the coming forward will be sampled
    std::vector<ProfSample> prof_pending;
    int* prof_counts_host = nullptr;   // pinned ring of batch sizes
    int prof_slot = 0;
    double prof_ms = 0.0, prof_input_ms = 0.0, prof_heads_ms = 0.0, prof_adv_ms = 0.0;
    uint64_t prof_samples = 0, prof_boards = 0, prof_launches = 0;

    // tuning switches (DESIGN.md section 8): read from the environment ONCE, when the engine is created, and kept per engine
    // (no process-wide statics shared by engines / devices)
    struct Knobs {
        int tower_fused = 1;       // AZ_TOWER_FUSED
        int tower_split = 0;       // AZ_TOWER_SPLIT (0: automatic)
        int tower_inkernel = 1;    // AZ_TOWER_INKERNEL
        int tc_release_arrive = 0; // AZ_TC_RELEASE_ARRIVE
        int tower_grid = 0;        // AZ_TOWER_GRID (0: every SM; the SM-partition experiment of profiles/)
        int tower_wide = 2;        // AZ_TOWER_WIDE: ONE TMA box per channel half serves the three horizontal taps of the tower; 2 (default) = 10-file boxes, three stages; 1 = 16-file boxes, two stages; 0 = one 8-file box per tap (round 1)
        int tower_l2hint = 1;      // AZ_TOWER_L2HINT (default 1): L2::evict_last on the tower's activation stores (1), residual loads (2), TMA loads (4)
        int input_epi2 = 0;        // AZ_INPUT_EPI2: the input convolution runs two sets of epilogue warps on alternate tiles
        int heads_tc = 1;          // AZ_HEADS_TC (default 1): policy/value heads on tcgen05 (nn_heads_tc.cu); 0 = warp-level mma.sync kernel (nn_heads.cu)
        int input_k32 = 1;         // AZ_INPUT_K32 (default 1): 32-channel plane layout (K padded to 32 instead of 64 in the input convolution); 0 = 64 channels
    } knobs;

    azb::NetWeights* net = nullptr;
    azb::NetWeights* net1 = nullptr;   // network slot 1 (az_load_network): weights only, allocated by its first load
    // az_forward_networks (allocated on its first call): boards per network, the slot of each board, its gathered value
    int* d_net_counts = nullptr;       // [AZ_MAX_NETWORKS]
    int* d_net_slot = nullptr;         // [max_batch]
    float* d_net_value = nullptr;      // [max_batch]
    azb::SearchState* search = nullptr;
    int stub_kind = 0;
    uint64_t stub_seed = 0;
};

namespace azb {

int set_err(az_engine* e, int code, const char* what);
int check_cuda(az_engine* e, cudaError_t r, const char* what);
#define AZ_CUDA(e, call) do { int _r = azb::check_cuda((e), (call), #call); if (_r) return _r; } while (0)

// chess_kernels.cu
void launch_movegen(cudaStream_t s, const az_position* wire, int n, uint16_t* moves, uint16_t* index, int32_t* count);
void launch_movegen_warp(cudaStream_t s, const az_position* wire, int n, uint16_t* moves, int32_t* count);
void launch_play_move(cudaStream_t s, az_position* wire, const az_position* hist, const uint32_t* hist_off, const uint16_t* action,
                      int32_t* result, int n, RuleParams rp);
void launch_move_to_index(cudaStream_t s, const az_position* wire, const uint16_t* moves, uint16_t* index, int n);
void launch_index_to_move(cudaStream_t s, const az_position* wire, const uint16_t* index, uint16_t* moves, int n);
void launch_encode_f32(cudaStream_t s, const az_position* wire, float* planes, int n);
void launch_wire_to_dpos(cudaStream_t s, const az_position* wire, DPos* out, uint32_t* root_ids, int n);
void launch_perft_expand(cudaStream_t s, const DPos* in, const uint32_t* in_root, int n_in, DPos* out, uint32_t* out_root,
                         unsigned long long* out_count);
void launch_perft_count(cudaStream_t s, const DPos* in, const uint32_t* in_root, int n_in, unsigned long long* nodes);
void launch_mm_expand(cudaStream_t s, const DPos* in, int n_in, int depth, int is_root, DPos* out, uint32_t* out_parent,
                      unsigned long long* out_count, int* score, unsigned int* first_child, int* n_child);
void launch_mm_leaf(cudaStream_t s, const DPos* in, int n_in, int* score);
void launch_mm_backup(cudaStream_t s, const int* child_score, const uint32_t* child_parent, int n_children, int* parent_score);
void launch_mm_root(cudaStream_t s, const unsigned int* first_child, const int* n_child, const int* child_score, int n_roots,
                    int* scores_out, int* count_out);

}  // namespace azb
