// Policy/value network (agent.rs) on the device: weight import with BatchNorm folding, the bf16 tensor-core path
// (tcgen05 convolutions + fused heads) and the fp32 parity path.
#pragma once
#include "engine.h"
#include <cuda_bf16.h>

namespace azb {

// Optional fused epilogue of the heads: write the priors of each board's legal moves straight into the search tree
// (edge_P[edge_off[b] + e] = softmax[policy index of edge e]) instead of materialising the 16 KB policy row.
struct HeadScatter {
    const unsigned long long* edge_off;  // [n] first edge of the node waiting for board b
    const int* n_edges;                  // [n]
    const uint32_t* edge_mv;             // wire move | policy index << 16
    float* edge_P;
};

// Multi-network batch (az_forward_networks, az_search_networks): network 0 (e->net) owns boards [0, counts_dev[0]), network 1
// (e->net1) owns [base1, base1 + counts_dev[1]); base1 is a multiple of 4 and base1 + the capacity of network 1's range <= cap
struct NetBatch {
    const int* counts_dev;   // [AZ_MAX_NETWORKS]
    int base1;
    int cap;
};

struct NetWeights {
    bool loaded = false;
    int max_boards = 0;
    int in_ch = 32;   // channel pitch of the bf16 plane buffer a_in: 32 (default: half the TMA bytes and MMAs of the input convolution) or 64 (AZ_INPUT_K32=0)
    // ---- fp32 parameters, BatchNorm folded: conv weights [co][ci][3][3], head matrices as documented in nn.cu
    float* f_w_in = nullptr;     // [128][19][9]
    float* f_b_in = nullptr;     // [128]
    float* f_w_tower = nullptr;  // [20][128][128][9]
    float* f_b_tower = nullptr;  // [20][128]
    float* f_w40t = nullptr;     // [128][40]  policy_conv_1 (32) + value_conv (8), transposed, BN folded
    float* f_b40 = nullptr;      // [40]
    float* f_wp2t = nullptr;     // [32][64]   policy_conv_2 transposed
    float* f_bp2 = nullptr;      // [64]
    float* f_wl1 = nullptr;      // [512][64]  value_linear_1 (burn layout [d_in][d_out])
    float* f_bl1 = nullptr;      // [64]
    float* f_wl2 = nullptr;      // [64]
    float* f_bl2 = nullptr;      // [1]
    // ---- bf16 tensor-core operands: [tap][co][ci]
    __nv_bfloat16* h_w_in = nullptr;     // [9][128][in_ch]  (19 channels zero-padded to in_ch)
    __nv_bfloat16* h_w_tower = nullptr;  // [20][9][128][128]
    __nv_bfloat16* h_w40 = nullptr;      // [40][128]  heads stage 1 (policy_conv_1 | value_conv), BN folded
    __nv_bfloat16* h_wp2 = nullptr;      // [64][32]   policy_conv_2
    __nv_bfloat16* h_wl1t = nullptr;     // [64][512]  value_linear_1 transposed
    CUtensorMap map_w_in;
    CUtensorMap map_w_tower[20];
    // ---- activations
    __nv_bfloat16* a_in = nullptr;       // [max_boards][64 squares][in_ch]
    __nv_bfloat16* a_buf[3] = {nullptr, nullptr, nullptr};  // [max_boards][64][128]
    CUtensorMap map_a_in;
    CUtensorMap map_a[3];
    CUtensorMap map_rows[3];             // a_buf[i] as [max_boards * 64][128] (heads on tcgen05)
    CUtensorMap* d_maps = nullptr;       // device copy {map_a[0..2], map_w_tower[0..19]} for the fused tower kernel
    float* g_buf[3] = {nullptr, nullptr, nullptr};          // fp32 path, NCHW [max_boards][128][64] (allocated lazily)
};

int net_create(az_engine* e);
void net_destroy(az_engine* e);

// Forward over boards whose bf16 NHWC planes are already in net->a_in (n read from n_dev when non-null).
// policy_out [n][4096] f32 (nullable), value_out [n] f32.  Returns the buffer index holding the tower output.
int net_forward_bf16(az_engine* e, const int* n_dev, int n_static, float* policy_out, float* value_out, const HeadScatter* scatter = nullptr,
                     const NetBatch* nb = nullptr);
// fp32 parity path from NCHW f32 planes [n][19][64]
int net_forward_fp32(az_engine* e, const float* planes, const int* n_dev, int n_static, float* policy_out, float* value_out,
                     const NetWeights* wts = nullptr /* the weights of another slot; activations are always e->net's */);
// fused heads on warp-level tensor-core MMAs (nn_heads.cu); tower = NHWC bf16 [n][64][128]
int launch_heads_mma(az_engine* e, const __nv_bfloat16* tower, const int* n_dev, int n_static, float* policy_out, float* value_out,
                     const HeadScatter* scatter);
// the same heads on tcgen05 (nn_heads_tc.cu, AZ_HEADS_TC=1): tiles of two boards, stage 1 and 2 as UMMA, softmax per pixel thread
int launch_heads_tc(az_engine* e, const CUtensorMap* act_rows_map, const int* n_dev, int n_static, float* policy_out, float* value_out,
                    const HeadScatter* scatter);
struct NetWeights;
// the heads of a multi-network batch on tcgen05 (k_heads_tc_nets): the CTAs are split between the networks
int launch_heads_tc_nets(az_engine* e, const NetWeights* w0, const NetWeights* w1, const CUtensorMap* act_rows_map, const int* counts_dev,
                         int base1, int n_max, float* policy_out, float* value_out, const HeadScatter* scatter);
// the forward of a multi-network batch: bf16 with the default configuration in one set of launches shared by the networks
// (net_forward_bf16 with nb), otherwise and on the fp32 path one network after the other over its range
int net_forward_networks(az_engine* e, const NetBatch& nb, const float* planes_f32, float* policy_out, float* value_out,
                         const HeadScatter* scatter = nullptr);
// AZ_ERR_STATE (with the engine's error message set) when the bf16 multi-network forward cannot run: it needs the default
// AZ_TOWER_*, AZ_INPUT_* and AZ_HEADS_TC configuration; AZ_OK otherwise (the fp32 path runs under any configuration)
int net_networks_supported(az_engine* e);
// network slot s (0: e->net, 1: e->net1, null until its first load)
NetWeights* net_slot(az_engine* e, int s);
// f32 NCHW planes -> bf16 NHWC (`ch` = 64 or 32 channels per square) into net->a_in
void launch_planes_to_bf16(cudaStream_t s, const float* planes, __nv_bfloat16* out, int n, int ch);
// positions -> bf16 NHWC planes (to_tensor fused with the layout the first convolution wants)
void launch_encode_bf16_wire(cudaStream_t s, const az_position* wire, __nv_bfloat16* out, int n, int ch);

// device helper used by the search kernels: writes the 64x64 bf16 plane tile of one position (one warp)
#ifdef __CUDACC__
__device__ __forceinline__ void encode_bf16_warp(const DPos& p, __nv_bfloat16* out /*[64][ch]*/, int lane, int ch = 64) {
    // to_tensor (chess.rs:191-245) in the layout the first convolution reads: [square][ch channels] bf16 (ch = 64 or 32), 19 used.
    // Each lane builds two squares: one piece plane at most, four constant castling planes, ep, two constant counters.
    // Channels 24..ch-1 of every square stay zero (zero-filled at allocation, never written).
    const int turn = meta_turn(p.meta);
    const u64 occ = occupied(p);
    const u64 ours = turn == 0 ? p.white : occ ^ p.white;
    const int pep = pseudo_legal_ep(p);
    const int c = meta_castling(p.meta);
    const int us_r = (c >> (turn * 2)) & 3, th_r = (c >> ((turn ^ 1) * 2)) & 3;
    const uint32_t ONE = 0x3F80u;  // bf16 1.0
    // planes 12..15 as two packed words (12|13, 14|15)
    const uint32_t castle_lo = ((us_r & 1) ? ONE : 0u) | ((us_r & 2) ? ONE << 16 : 0u);
    const uint32_t castle_hi = ((th_r & 1) ? ONE : 0u) | ((th_r & 2) ? ONE << 16 : 0u);
    __nv_bfloat16 hm = __float2bfloat16_rn(__fdiv_rn((float)meta_halfmoves(p.meta), 100.0f));
    __nv_bfloat16 fm = __float2bfloat16_rn(__fdiv_rn((float)meta_fullmoves(p.meta), 200.0f));
    const uint32_t hm_bits = *reinterpret_cast<unsigned short*>(&hm), fm_bits = *reinterpret_cast<unsigned short*>(&fm);
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const int sqc = lane + 32 * k;               // canonical square (rank flipped for Black)
        const int sq = turn ? (sqc ^ 56) : sqc;
        const u64 b = bit(sq);
        int plane = -1;
        if (occ & b) {
            const int role = (p.pawn & b) ? 0 : (p.knight & b) ? 1 : (p.bishop & b) ? 2 : (p.rook & b) ? 3 : (p.queen & b) ? 4 : 5;
            plane = role + ((ours & b) ? 0 : 6);
        }
        uint32_t w[10];
        const uint32_t pv = (plane & 1) ? ONE << 16 : ONE;
#pragma unroll
        for (int j = 0; j < 6; j++) w[j] = (plane >= 0 && (plane >> 1) == j) ? pv : 0u;   // planes 0..11 live in words 0..5
        w[6] = castle_lo;
        w[7] = castle_hi;
        w[8] = (sq == pep ? ONE : 0u) | (hm_bits << 16);                    // planes 16, 17
        w[9] = fm_bits;                                                    // plane 18 (19 is padding)
        uint4* o = reinterpret_cast<uint4*>(out) + sqc * (ch >> 3);
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
        o[2] = make_uint4(w[8], w[9], 0u, 0u);
    }
}
#endif

}  // namespace azb
