// Host-side interface of the tcgen05 convolution (nn_tc.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace azb {
// activations: NHWC bf16 [max_boards][8][8][channels], channels in {64, 128}
int tc_make_act_map(CUtensorMap* map, const void* base, int channels, int max_boards, int wide = 0);
// the same buffer as a matrix [max_boards * 64 pixel rows][128 channels] for the tcgen05 heads (nn_heads_tc.cu)
int tc_make_rows_map(CUtensorMap* map, const void* base, int max_boards);
// weights: bf16 [9 taps][128 out][cin], BatchNorm already folded
int tc_make_weight_map(CUtensorMap* map, const void* base, int cin);
// out = act( conv3x3(in) + bias (+ residual) ); the board count is read from n_boards_dev when non-null
int tc_conv3x3_launch(cudaStream_t stream, const CUtensorMap* in_map, const CUtensorMap* w_map, int cin, const float* bias,
                      const void* residual, void* out, const int* n_boards_dev, int n_boards_static, int relu, int grid, int dbg = 0);   // dbg bit 5 (32): hand accumulators back with a release arrive
// the 20-layer residual tower in one persistent launch; maps_dev = device array {act0, act1, act2, w[0..19]}
int tc_tower_launch(cudaStream_t stream, const CUtensorMap* maps_dev, const float* bias, void* const* act, const int* n_boards_dev,
                    int n_boards_static, int n_layers, int stem, int grid, int tile_lo = 0, int tile_hi = 0x7FFFFFFF, int range_tiles = 0,
                    int release_arrive = 0, int wide = 0, int l2_hint = 0);   // wide: one 16-file box per channel half (maps_dev[25..27])
// Multi-network batches (tc_conv.cuh, net_part): network 0 owns boards [0, counts_dev[0]), network 1 [base1, base1 + counts_dev[1]),
// base1 a multiple of 4.  The 32-channel input convolution (w_map0 / w_map1 and bias0 / bias1 of the two networks, output bias
// + ReLU) and the 10-file-box tower (maps0_dev / maps1_dev: the maps array of tc_tower_launch of each network).
int tc_conv3x3_nets_launch(cudaStream_t stream, const CUtensorMap* in_map, const CUtensorMap* w_map0, const CUtensorMap* w_map1,
                           const float* bias0, const float* bias1, void* out, const int* counts_dev, int base1, int grid, int dbg = 0);
int tc_tower_nets_launch(cudaStream_t stream, const CUtensorMap* maps0_dev, const CUtensorMap* maps1_dev, const float* bias0,
                         const float* bias1, void* const* act, const int* counts_dev, int base1, int grid, int release_arrive, int l2_hint);
}  // namespace azb
