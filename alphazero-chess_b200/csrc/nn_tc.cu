// 3x3 "same" convolutions of the policy/value network (agent.rs:22-23,36,40,74-76) as implicit GEMMs on the
// 5th-generation tensor cores: tcgen05.mma (cta_group::2) with TMEM accumulators, operands staged by TMA.
//
//   M = 256 rows  = 4 boards x 64 squares per CTA pair (128 rows per CTA); within a CTA row r <-> (rank r>>4, board (r>>3)&1, file r&7)
//   N = 128       = all output channels; each CTA of the pair keeps the weights of 64 of them resident in SMEM
//   K = 9 taps x Cin, consumed in 64-channel blocks
//
// Activations are NHWC bf16 [board][rank][file][C].  One TMA box {64 ch, 8 files, 2 boards, 10 ranks} is fetched per
// (channel half, dx): the dx shift and the rank halo are resolved by signed box coordinates (out-of-bounds elements are
// zero-filled = "same" padding), and because the box is laid out rank-major the three dy taps are just three
// 1024B-aligned row windows of the same SMEM stage.  So 6 boxes (120 KB) feed the 72 MMAs of a tile instead of 18.
// WIDE (the tower's default, AZ_TOWER_WIDE=2): ONE box {64 ch, 10 files (-1..8), 2 boards, 10 ranks} per channel half serves all
// nine taps -- the files outside the board are zero-filled like the ranks, the 8-row groups of the A operand are 10 rows = 1280
// bytes apart (the descriptor's stride byte offset) and tap (dx, dy) is the window starting dy * 2560 + dx * 128 bytes into the
// stage.  The start address is then not 1024-byte aligned; that is legal because the tensor core derives the 128-byte-swizzle
// XOR from the address bits (7..9), exactly as TMA wrote the tile.  2 boxes (51 KB written, 32 KB read from the L2) per tile.
// BatchNorm is folded into weights/bias on the host; the epilogue applies bias (+ residual) (+ ReLU) and writes bf16.
//
//   conv3x3_tc2_kernel<HALVES, KROW, WIDE>  one layer per launch (the 19->128 input convolution, and the tower with AZ_TOWER_FUSED=0)
//   conv_tower_kernel<WIDE>                 the 20 tower layers in one persistent launch
// The single-CTA first version (N = 64 per CTA, issue-bound) is described in profiles/r1_conv_ablation.md.
#include "tc_conv.cuh"
#include "nn_tc.h"
#include "device_once.h"
#include <cuda_bf16.h>
#include <cstdio>
#include <cstdlib>

namespace azb {

// defined before anything that prints, so that the module lists it where it has always been (first)
__device__ const char kTowerTimeoutMsg[] = "azb: tower epilogue wait timeout\n";

constexpr int kWTileBytes = 64 * 128;    // 64 output channels x 64 input channels bf16

// KROW = bytes per operand row in shared memory = input channels per K block x 2: 128 (64 channels, 128-byte swizzle) for the
// tower and the 64-channel plane layout, 64 (32 channels, 64-byte swizzle) for the 32-channel plane layout of the input convolution
// WIDE = 1 (experiment, AZ_DBG_CONV bit 6): ONE box per channel half serves all three horizontal taps.  The box spans files -1..14
// (16-row pitch per (rank, board), files outside the board zero-filled by TMA), so the tap dx is a window that starts dx rows
// (128 bytes) into every 8-row group: 8-row groups 2048 bytes apart, start address + dx * 128.
template <int HALVES, int KROW = 128, int WIDE = 0>
struct ConvSmem {
    static constexpr int kPitch = WIDE == 1 ? 16 : WIDE == 2 ? 10 : 8;   // rows (files) per (rank, board) group in a stage
    static constexpr int kStages = HALVES == 1 ? 6 : WIDE == 1 ? 2 : WIDE == 2 ? 3 : 4;
    static constexpr int kWTiles = HALVES * 9;
    static constexpr int kStageB = 20 * kPitch * KROW;
    static constexpr int kWTileB = 64 * KROW;
    static constexpr int kWBytes = kWTiles * kWTileB;
    static constexpr int kABytes = kStages * kStageB;
    static constexpr int kMisc = 2048;
    static constexpr int kTotal = kWBytes + kABytes + kMisc + 1024;  // + alignment slack
};

// ================================================================================================================
// CTA-pair version (cta_group::2): the two SMs of a pair compute one 256-row tile (4 boards) against all 128 output
// channels.  Each CTA stages its own 128 rows of A and keeps HALF of the weights (64 output channels) resident; the
// leader CTA issues M=256 x N=128 x K=16 MMAs that read both CTAs' shared memory.  Per SM this halves the TMA traffic
// and the shared-memory operand bandwidth of the single-CTA kernel and doubles the work per issued instruction
// (the single-CTA kernel was bound by the issue rate of its N=64 MMAs: profiles/r1_conv_ablation.md).
constexpr int kTmemCols2 = 256;  // 2 accumulator stages x 128 fp32 columns
// Epilogue warps per CTA: kEpiWarps / 4 per TMEM lane quarter, each owning 128 / (kEpiWarps / 4) accumulator columns of its 32 rows.
// Measured (profiles/r2_ab.md): 16 warps (32 columns = one tcgen05.ld each) make the tower 3.4 % SLOWER than 8 warps (64 columns) and leave
// the input convolution unchanged, so 8 is the default; -DAZ_EPI_WARPS=16 rebuilds the experiment.
#ifndef AZ_EPI_WARPS
#define AZ_EPI_WARPS 8
#endif
constexpr int kEpiWarps = AZ_EPI_WARPS;
constexpr int kEpiCols = 128 / (kEpiWarps / 4);   // accumulator columns per epilogue warp
constexpr int kEpiChunks = kEpiCols / 32;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreads2 = 64 + kEpiThreads;   // warp 0 TMA, warp 1 MMA/TMEM, then the epilogue warps
static_assert(kEpiWarps == 8 || kEpiWarps == 16, "epilogue warps: 8 or 16");

// GROUPS = 2 (the input convolution): two sets of epilogue warps take alternate tiles (set g always drains TMEM buffer g), so the
// epilogues of consecutive tiles overlap in time.  The layer is bound by the latency of one tile's epilogue (wait, tcgen05.ld,
// bias / ReLU / pack, stores), not by its width, which is why splitting one tile over 16 warps did not help (profiles/r2_ab.md 4).
// Which tiles a CTA pair computes, and with which weights.  ConvSched<false> is the single-network launch (its expressions are
// those the kernel has always had, so its code is unchanged); ConvSched<true> a multi-network batch (net_part in tc_conv.cuh).
struct ConvNets {
    const int* counts;   // device [2]: boards of each network
    int base1;           // first board of network 1
    const CUtensorMap* w_map1;
    const float* bias1;
};
template <bool NETS> struct ConvSched;
template <> struct ConvSched<false> {
    __device__ __forceinline__ explicit ConvSched(const ConvNets&) {}
    __device__ __forceinline__ int n_boards(const int* n_boards_ptr, int n_boards_static) const { return n_boards_ptr ? *n_boards_ptr : n_boards_static; }
    __device__ __forceinline__ int n_tiles(int n_boards) const { return (n_boards + 3) >> 2; }
    __device__ __forceinline__ int first_tile() const { return blockIdx.x >> 1; }
    __device__ __forceinline__ int tile_step() const { return gridDim.x >> 1; }
    __device__ __forceinline__ const CUtensorMap* w_map(const CUtensorMap* w0) const { return w0; }
    __device__ __forceinline__ const float* bias(const float* b0) const { return b0; }
};
template <> struct ConvSched<true> {
    NetPart np;
    const ConvNets& nets;
    __device__ __forceinline__ explicit ConvSched(const ConvNets& n) : np(net_part(n.counts, n.base1, gridDim.x >> 1, blockIdx.x >> 1, 4)), nets(n) {}
    __device__ __forceinline__ int n_boards(const int*, int) const { return np.end_board; }
    __device__ __forceinline__ int n_tiles(int) const { return np.first_tile + np.n_tiles; }
    __device__ __forceinline__ int first_tile() const { return np.first_tile + np.unit; }
    __device__ __forceinline__ int tile_step() const { return np.units; }
    __device__ __forceinline__ const CUtensorMap* w_map(const CUtensorMap* w0) const { return np.net ? nets.w_map1 : w0; }
    __device__ __forceinline__ const float* bias(const float* b0) const { return np.net ? nets.bias1 : b0; }
};

template <int HALVES, int KROW, int WIDE, int GROUPS, bool NETS>
__device__ __forceinline__ void conv3x3_tc2_body(const CUtensorMap& in_map, const CUtensorMap* w_map_p, const float* __restrict__ bias,
                                                 const __nv_bfloat16* __restrict__ residual, __nv_bfloat16* __restrict__ out,
                                                 const int* __restrict__ n_boards_ptr, int n_boards_static, int relu, int dbg,
                                                 const ConvNets& nets) {
    using S = ConvSmem<HALVES, KROW, WIDE>;
    constexpr int kStageBytes = S::kStageB, kWTileBytes = S::kWTileB;   // shadow the 128-byte-row constants of the tower
    constexpr int KSTEPS = KROW / 32;                                   // K = 16 elements = 32 bytes per MMA
    constexpr int NS = S::kStages;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* w_sm = smem;
    uint8_t* a_sm = smem + S::kWBytes;
    uint8_t* misc = a_sm + S::kABytes;
    float* bias_s = reinterpret_cast<float*>(misc);                     // 128 floats
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(misc + 512);       // NS        (leader's copy is the live one)
    uint64_t* empty_bar = full_bar + NS;                                // NS        (per CTA, multicast commit)
    uint64_t* wfull_bar = empty_bar + NS;                               // kWTiles   (leader)
    uint64_t* tfull_bar = wfull_bar + S::kWTiles;                       // 2         (per CTA, multicast commit)
    uint64_t* tempty_bar = tfull_bar + 2;                               // 2         (leader, 8 warp arrivals)
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const ConvSched<NETS> sched(nets);
    const int n_boards = sched.n_boards(n_boards_ptr, n_boards_static);
    const int n_tiles = sched.n_tiles(n_boards);
    const int first_tile = sched.first_tile(), tile_step = sched.tile_step();
    const CUtensorMap& w_map = *sched.w_map(w_map_p);
    bias = sched.bias(bias);

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&in_map);
        tma_prefetch_desc(&w_map);
        for (int i = 0; i < NS; i++) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < S::kWTiles; i++) mbar_init(&wfull_bar[i], 1);
        for (int i = 0; i < 2; i++) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * kEpiWarps); }
        fence_barrier_init();
    }
    if (threadIdx.x >= 64 && threadIdx.x < 192) bias_s[threadIdx.x - 64] = bias[threadIdx.x - 64];
    if (warp == 1) tmem2_alloc(tmem_ptr_s, kTmemCols2);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp == 0) {
        // ---------------------------------------------------------------- TMA producer (both CTAs, warp-uniform)
        int stage = 0; uint32_t phase = 0; bool first = true;
        for (int t = first_tile; t < n_tiles; t += tile_step) {
            if constexpr (WIDE) {
                for (int half = 0; half < HALVES; half++) {
                    if (first && elect_one()) {
                        for (int dxi = 0; dxi < 3; dxi++)
                            for (int dyi = 0; dyi < 3; dyi++) {
                                const int wt = (half * 3 + dxi) * 3 + dyi, tap = dyi * 3 + dxi;
                                if (rank == 0) mbar_arrive_expect_tx(&wfull_bar[wt], 2 * kWTileBytes);
                                tma2_load_2d(w_sm + wt * kWTileBytes, &w_map, &wfull_bar[wt], half * 64, tap * 128 + (int)rank * 64);
                            }
                    }
                    mbar_wait(&empty_bar[stage], phase ^ 1, 11);
                    if (elect_one()) {
                        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kStageBytes);
                        tma2_load_4d(a_sm + stage * kStageBytes, &in_map, &full_bar[stage], half * 64, -1, t * 4 + (int)rank * 2, -1);
                    }
                    __syncwarp();
                    if (++stage == NS) { stage = 0; phase ^= 1; }
                }
                first = false;
            } else {
            for (int half = 0; half < HALVES; half++)
                for (int dxi = 0; dxi < 3; dxi++) {
                    if (first && elect_one()) {
                        for (int dyi = 0; dyi < 3; dyi++) {
                            const int wt = (half * 3 + dxi) * 3 + dyi, tap = dyi * 3 + dxi;
                            if (rank == 0) mbar_arrive_expect_tx(&wfull_bar[wt], 2 * kWTileBytes);
                            tma2_load_2d(w_sm + wt * kWTileBytes, &w_map, &wfull_bar[wt], half * 64, tap * 128 + (int)rank * 64);
                        }
                    }
                    mbar_wait(&empty_bar[stage], phase ^ 1, 11);
                    if (elect_one()) {
                        if (dbg & 1) { if (rank == 0) mbar_arrive(&full_bar[stage]); }
                        else {
                            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kStageBytes);
                            tma2_load_4d(a_sm + stage * kStageBytes, &in_map, &full_bar[stage], half * 64, dxi - 1, t * 4 + (int)rank * 2, -1);
                        }
                    }
                    __syncwarp();
                    if (++stage == NS) { stage = 0; phase ^= 1; }
                }
            first = false;
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // ------------------------------------------------------------ MMA issuer (leader CTA, warp-uniform loop)
            constexpr uint32_t idesc = umma_idesc_bf16(256, 128);
            const uint64_t dbase = KROW == 128 ? umma_desc_base_sw128() : umma_desc_base_sw64();
            const uint32_t w_lo = (smem_u32(w_sm) & 0x3FFFF) >> 4;
            int stage = 0; uint32_t phase = 0; int lt = 0;
            for (int t = first_tile; t < n_tiles; t += tile_step, lt++) {
                const int acc = lt & 1; const uint32_t accphase = (lt >> 1) & 1;
                mbar_wait(&tempty_bar[acc], accphase ^ 1, 12);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 128;
                if constexpr (WIDE) {
                    for (int half = 0; half < HALVES; half++) {
                        mbar_wait(&full_bar[stage], phase, 13);
                        if (lt == 0)
                            for (int wt = 0; wt < 9; wt++) mbar_wait(&wfull_bar[half * 9 + wt], 0, 14);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t a_lo = (smem_u32(a_sm + stage * kStageBytes) & 0x3FFFF) >> 4;
                            // 8-row groups (one rank of one board) are kPitch rows apart
                            const uint64_t abase = ((uint64_t)1 << 16) | ((uint64_t)((S::kPitch * KROW) >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)(KROW == 128 ? 2 : 4) << 61);
#pragma unroll
                            for (int dxi = 0; dxi < 3; dxi++) {
                                const uint32_t b_lo = w_lo + (uint32_t)((half * 3 + dxi) * 3) * (kWTileBytes >> 4);
                                // dbg bit 7: tell the hardware that the window starts dx rows into the 1024-byte swizzle pattern
                                const uint64_t aoff = abase | ((dbg & 128) ? ((uint64_t)dxi << 49) : 0);
#pragma unroll
                                for (int dyi = 0; dyi < 3; dyi++) {
#pragma unroll
                                    for (int k = 0; k < KSTEPS; k++) {
                                        const uint64_t ad = aoff | (uint64_t)(a_lo + dyi * ((2 * S::kPitch * KROW) >> 4) + dxi * (KROW >> 4) + k * 2);
                                        const uint64_t bd = dbase | (uint64_t)(b_lo + dyi * (kWTileBytes >> 4) + k * 2);
                                        umma2_bf16(d_tmem, ad, bd, idesc, (half | dxi | dyi | k) != 0 ? 1u : 0u);
                                    }
                                }
                            }
                            umma2_commit_mc(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == NS) { stage = 0; phase ^= 1; }
                    }
                } else {
                for (int half = 0; half < HALVES; half++)
                    for (int dxi = 0; dxi < 3; dxi++) {
                        mbar_wait(&full_bar[stage], phase, 13);
                        if (lt == 0)
                            for (int dyi = 0; dyi < 3; dyi++) mbar_wait(&wfull_bar[(half * 3 + dxi) * 3 + dyi], 0, 14);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t a_lo = (smem_u32(a_sm + stage * kStageBytes) & 0x3FFFF) >> 4;
                            const uint32_t b_lo = w_lo + (uint32_t)((half * 3 + dxi) * 3) * (kWTileBytes >> 4);
#pragma unroll
                            for (int dyi = 0; dyi < 3; dyi++) {
#pragma unroll
                                for (int k = 0; k < KSTEPS; k++) {
                                    const uint64_t ad = dbase | (uint64_t)(a_lo + dyi * ((16 * KROW) >> 4) + k * 2);
                                    const uint64_t bd = dbase | (uint64_t)(b_lo + dyi * (kWTileBytes >> 4) + k * 2);
                                    if (!(dbg & 2)) umma2_bf16(d_tmem, ad, bd, idesc, (half | dxi | dyi | k) != 0 ? 1u : 0u);
                                }
                            }
                            umma2_commit_mc(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == NS) { stage = 0; phase ^= 1; }
                    }
                }
                if (elect_one()) umma2_commit_mc(&tfull_bar[acc]);
                __syncwarp();
            }
        }
    } else {
        // ------------------------------------------------ epilogue (TMEM lane quarter q, column group cg of kEpiCols columns)
        const int q = warp & 3;
        const int egrp = (warp - 2) / kEpiWarps;            // epilogue set (GROUPS = 2: alternate tiles)
        const int cg = ((warp - 2) % kEpiWarps) >> 2;
        const int row = q * 32 + lane;
        const int h = row >> 4, b = (row >> 3) & 1, w = row & 7;
        int lt = 0;
        for (int t = first_tile; t < n_tiles; t += tile_step, lt++) {
            if (GROUPS == 2 && (lt & 1) != egrp) continue;
            const int acc = lt & 1; const uint32_t accphase = (lt >> 1) & 1;
            const int board = t * 4 + (int)rank * 2 + b;
            const bool valid = board < n_boards;
            const size_t off = ((size_t)board * 64 + h * 8 + w) * 128 + cg * kEpiCols;
            if (dbg & 4) {
                mbar_wait(&tfull_bar[acc], accphase, 15);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { if (dbg & 32) mbar_arrive_cluster(&tempty_bar[acc], 0); else mbar_arrive_cluster_relaxed(&tempty_bar[acc], 0); }
                continue;
            }
            const bool has_res = residual != nullptr && valid && !(dbg & 8);
            // the residual part of the row is requested before waiting for the accumulator (32-byte loads in flight)
            uint32_t res[kEpiCols / 2];
            if (has_res) {
#pragma unroll
                for (int i = 0; i < kEpiCols / 16; i++) ld_global_v8(residual + off + i * 16, &res[i * 8]);
            }
            mbar_wait(&tfull_bar[acc], accphase, 15);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 128 + cg * kEpiCols;
#pragma unroll
            for (int chunk = 0; chunk < kEpiChunks; chunk++) {
                uint32_t r[32];
                tmem_ld32(taddr + chunk * 32, r);
                tmem_ld_wait();
                if (chunk == kEpiChunks - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { if (dbg & 32) mbar_arrive_cluster(&tempty_bar[acc], 0); else mbar_arrive_cluster_relaxed(&tempty_bar[acc], 0); }
                }
                if (valid) {
#pragma unroll
                    for (int v = 0; v < 2; v++) {  // 16 channels = 32 bytes per store
                        uint32_t packed[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const int c = v * 16 + j * 2;
                            const float2 bb = *reinterpret_cast<const float2*>(&bias_s[cg * kEpiCols + chunk * 32 + c]);
                            float x0 = __uint_as_float(r[c]) + bb.x;
                            float x1 = __uint_as_float(r[c + 1]) + bb.y;
                            if (has_res) {
                                const uint32_t rr = res[chunk * 16 + v * 8 + j];
                                x0 += __uint_as_float(rr << 16);
                                x1 += __uint_as_float(rr & 0xFFFF0000u);
                            }
                            if (relu) { x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f); }
                            __nv_bfloat162 pk = __floats2bfloat162_rn(x0, x1);
                            packed[j] = *reinterpret_cast<uint32_t*>(&pk);
                        }
                        if (dbg & 512) st_global_v8_hint(out + off + chunk * 32 + v * 16, packed, l2_policy_evict_last());
                        else if (!(dbg & 16)) st_global_v8(out + off + chunk * 32 + v * 16, packed);
                        else if (packed[0] == 0x12345678u && packed[7] == 0x9abcdef0u) st_global_v8(out + off, packed);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) { tc_fence_after(); tmem2_dealloc(tmem_base, kTmemCols2); }
}

template <int HALVES, int KROW, int WIDE = 0, int GROUPS = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + GROUPS * kEpiThreads, 1)
conv3x3_tc2_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ CUtensorMap w_map,
                   const float* __restrict__ bias, const __nv_bfloat16* __restrict__ residual,
                   __nv_bfloat16* __restrict__ out, const int* __restrict__ n_boards_ptr, int n_boards_static, int relu, int dbg) {
    conv3x3_tc2_body<HALVES, KROW, WIDE, GROUPS, false>(in_map, &w_map, bias, residual, out, n_boards_ptr, n_boards_static, relu, dbg,
                                                        ConvNets{nullptr, 0, nullptr, nullptr});
}

// the input convolution of a multi-network batch: the CTA pairs are split between the two networks' weights (ConvSched<true>)
template <int HALVES, int KROW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1)
conv3x3_tc2_nets_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ CUtensorMap w_map,
                        const __grid_constant__ CUtensorMap w_map1, const float* __restrict__ bias, const float* __restrict__ bias1,
                        __nv_bfloat16* __restrict__ out, const int* __restrict__ counts, int base1, int dbg) {
    conv3x3_tc2_body<HALVES, KROW, 0, 1, true>(in_map, &w_map, bias, nullptr, out, nullptr, 0, 1, dbg, ConvNets{counts, base1, &w_map1, bias1});
}

// ================================================================================================================
// Fused residual tower: all 20 3x3 convolutions (agent.rs:118-120) in ONE persistent launch.
// A convolution is local to a board, and a CTA pair keeps the same boards in every layer, so no grid-wide
// synchronisation is needed between layers: a pair runs layer after layer over its own tiles.  Only the weights change,
// so each CTA re-streams its 144 KB half of the next layer's weights through shared memory as soon as the last tile of
// the current layer has consumed them (per weight-group empty barriers), which keeps the MMA pipe busy across layer
// boundaries and removes 19 launch fill/drain phases.  Tile t of layer l+1 reads what this CTA's own epilogue wrote for
// tile t of layer l: the epilogue warps publish per-warp completion counters after a generic->async proxy fence and the
// TMA producer checks them (they are normally many tiles ahead).
struct TowerParams {
    const CUtensorMap* maps;   // device memory: [0..2] activation buffers, [3..22] weights of the 20 layers,
                               // [23] the 64-channel plane buffer, [24] the input convolution's weights
    const float* bias;         // [21][128]: 20 tower layers, then the input convolution
    __nv_bfloat16* act[3];
    const int* n_boards_ptr;
    int n_boards_static;
    int n_layers;              // 20
    int release_arrive;        // 1: hand accumulators back with a release arrive (AZ_TC_RELEASE_ARRIVE=1, the first version)
    int l2_hint;               // AZ_TOWER_L2HINT: bit 0 = activation stores, bit 1 = residual loads, bit 2 = activation TMA loads carry L2::evict_last
    int tile_lo, tile_hi;      // this launch covers tiles [tile_lo, min(all tiles, tile_hi)) (a tile = 4 boards) ...
    int range_tiles;           // ... as consecutive ranges of this many tiles: all layers of one range, then the next range
    int stem;                  // 1: run the input convolution (agent.rs:117; 64 padded channels -> act[0]) as a first layer
};


// WIDE = 1 (AZ_TOWER_WIDE): one TMA box per channel half serves the three horizontal taps (see ConvSmem): a third of the L2 -> shared
// memory traffic and of the TMA instructions; the activation maps are then maps[25..27] (16-file boxes) and there is no stem.
// Which tiles a CTA pair computes, in which ranges, with which weights (as ConvSched): TowerSched<false> is the single-network
// launch, TowerSched<true> a multi-network batch.  There a network's pairs walk its tiles in ranges of at most 7 rounds (>= 6 tiles
// per pair when it has them), the sizing of the single-network launch (net_forward_bf16), so that the ranges the two networks
// work on at the same time hold about as many boards as one range of the single-network launch and stay in the L2 together.
struct TowerNets {
    const int* counts;   // device [2]: boards of each network
    int base1;           // first board of network 1
    const CUtensorMap* maps1;   // network 1's device maps: the activation maps of TowerParams::maps and its own weights
    const float* bias1;
};
template <bool NETS> struct TowerSched;
template <> struct TowerSched<false> {
    __device__ __forceinline__ TowerSched(const TowerParams&, const TowerNets&) {}
    __device__ __forceinline__ int n_boards(const TowerParams& prm) const { return prm.n_boards_ptr ? *prm.n_boards_ptr : prm.n_boards_static; }
    __device__ __forceinline__ int n_tiles(const TowerParams& prm, int n_boards) const { return min((n_boards + 3) >> 2, prm.tile_hi); }
    __device__ __forceinline__ int tile_step() const { return gridDim.x >> 1; }
    __device__ __forceinline__ int tile_lo(const TowerParams& prm) const { return prm.tile_lo; }
    __device__ __forceinline__ int range_tiles(const TowerParams& prm) const { return prm.range_tiles; }
    __device__ __forceinline__ int pair() const { return blockIdx.x >> 1; }
    __device__ __forceinline__ const CUtensorMap* maps(const TowerParams& prm) const { return prm.maps; }
    __device__ __forceinline__ const float* bias(const TowerParams& prm) const { return prm.bias; }
};
template <> struct TowerSched<true> {
    NetPart np;
    int per;
    const TowerNets& nets;
    __device__ __forceinline__ TowerSched(const TowerParams&, const TowerNets& n)
        : np(net_part(n.counts, n.base1, gridDim.x >> 1, blockIdx.x >> 1, 4)), nets(n) {
        int nr = max(1, (np.n_tiles + 7 * np.units - 1) / (7 * np.units));
        if (np.n_tiles < 6 * np.units * nr) nr = max(1, np.n_tiles / (6 * np.units));
        per = max(1, (np.n_tiles + nr - 1) / nr);
    }
    __device__ __forceinline__ int n_boards(const TowerParams&) const { return np.end_board; }
    __device__ __forceinline__ int n_tiles(const TowerParams&, int) const { return np.first_tile + np.n_tiles; }
    __device__ __forceinline__ int tile_step() const { return np.units; }
    __device__ __forceinline__ int tile_lo(const TowerParams&) const { return np.first_tile; }
    __device__ __forceinline__ int range_tiles(const TowerParams&) const { return per; }
    __device__ __forceinline__ int pair() const { return np.unit; }
    __device__ __forceinline__ const CUtensorMap* maps(const TowerParams& prm) const { return np.net ? nets.maps1 : prm.maps; }
    __device__ __forceinline__ const float* bias(const TowerParams& prm) const { return np.net ? nets.bias1 : prm.bias; }
};

template <int WIDE, bool NETS>
__device__ __forceinline__ void conv_tower_body(const TowerParams& prm, const TowerNets& nets) {
    using S = ConvSmem<2, 128, WIDE>;
    constexpr int kStageBytes = S::kStageB;
    constexpr int NS = S::kStages;
    constexpr int kGroupBytes = 3 * kWTileBytes;  // the three dy taps of one (channel half, dx)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* w_sm = smem;
    uint8_t* a_sm = smem + S::kWBytes;
    uint8_t* misc = a_sm + S::kABytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(misc);             // NS   (leader)
    uint64_t* empty_bar = full_bar + NS;                                // NS   (per CTA)
    uint64_t* wfull_bar = empty_bar + NS;                               // 6    (leader)
    uint64_t* wempty_bar = wfull_bar + 6;                               // 6    (per CTA)
    uint64_t* tfull_bar = wempty_bar + 6;                               // 2    (per CTA)
    uint64_t* tempty_bar = tfull_bar + 2;                               // 2    (leader)
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    volatile uint32_t* epi_done = reinterpret_cast<volatile uint32_t*>(tmem_ptr_s + 4);  // kEpiWarps per-warp tile counters

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const TowerSched<NETS> sched(prm, nets);
    const int n_boards = sched.n_boards(prm);
    const int n_tiles = sched.n_tiles(prm, n_boards);
    const int tile_step = sched.tile_step();
    const int n_ranges = n_tiles > sched.tile_lo(prm) ? (n_tiles - sched.tile_lo(prm) + sched.range_tiles(prm) - 1) / sched.range_tiles(prm) : 0;
    // Per range r every role derives the same numbers: the pair's first tile, its tile count T (ranges without tiles for
    // this pair are skipped by all roles alike), and three running counters -- u0 / u1 = how often the weight groups of
    // channel half 0 / 1 have been loaded so far (barrier parities), cum = tiles this pair finished in earlier ranges.
#define TOWER_RANGE_BEGIN()                                                                                      \
    const int range_lo = sched.tile_lo(prm) + rg * sched.range_tiles(prm);                                        \
    const int range_hi = min(n_tiles, range_lo + sched.range_tiles(prm));                                        \
    const int first_tile = range_lo + sched.pair();                                                              \
    const int T = first_tile < range_hi ? (range_hi - first_tile + tile_step - 1) / tile_step : 0;               \
    if (T == 0) continue;
    const int stem = prm.stem;
    const int NL = prm.n_layers + stem;  // loop index L; tower layer = L - stem (-1 is the input convolution: one channel half)

    if (threadIdx.x == 0) {
        for (int i = 0; i < NS; i++) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 6; i++) { mbar_init(&wfull_bar[i], 1); mbar_init(&wempty_bar[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * kEpiWarps); }
        fence_barrier_init();
    }
    if (threadIdx.x < kEpiWarps) epi_done[threadIdx.x] = 0;
    float* bias_s = reinterpret_cast<float*>(misc + 512);  // [2][128]: bias of the current layer, double buffered by layer parity
    if (warp == 1) tmem2_alloc(tmem_ptr_s, kTmemCols2);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp == 0) {
        // ---------------------------------------------------------------- TMA producer (both CTAs)
        int stage = 0; uint32_t phase = 0;
        int u0 = 0, u1 = 0;
        uint32_t cum = 0;
        for (int rg = 0; rg < n_ranges; rg++) {
        TOWER_RANGE_BEGIN();
        for (int L = 0; L < NL; L++) {
            const int layer = L - stem;
            const int blk_second = layer >= 0 ? (layer & 1) : 0;
            const int in_buf = blk_second ? 1 : 0;   // block input in act[0], conv1 output in act[1], conv2 back into act[0]
            const CUtensorMap* in_map = layer >= 0 ? &sched.maps(prm)[(WIDE == 2 ? 28 : WIDE ? 25 : 0) + in_buf] : &sched.maps(prm)[23];
            const CUtensorMap* w_map = layer >= 0 ? &sched.maps(prm)[3 + layer] : &sched.maps(prm)[24];
            const int halves = layer >= 0 ? 2 : 1;
            for (int i = 0; i < T; i++) {
                const int t = first_tile + i * tile_step;
                if (L > 0) {  // this tile's input was written by this CTA's epilogue one layer ago
                    const uint32_t need = cum + (uint32_t)((L - 1) * T + i + 1);
                    long long t0 = clock64();
                    for (;;) {
                        bool ok = lane >= kEpiWarps || epi_done[lane & (kEpiWarps - 1)] >= need;
                        if (__all_sync(0xffffffffu, ok)) break;
                        if (clock64() - t0 > 4000000000LL) { if (lane == 0) printf(kTowerTimeoutMsg); __trap(); }
                    }
                    fence_proxy_async();
                }
                for (int half = 0; half < halves; half++)
                    for (int dxi = 0; dxi < 3; dxi++) {
                        const int grp = half * 3 + dxi;
                        if (i == 0) {  // (re)load this group's three weight tiles for the new layer
                            const int used = half == 0 ? u0 : u1;  // earlier layers (of any range) that went through this group
                            if (used > 0) mbar_wait(&wempty_bar[grp], (uint32_t)((used - 1) & 1), 21);
                            if (elect_one()) {
                                if (rank == 0) mbar_arrive_expect_tx(&wfull_bar[grp], 2 * kGroupBytes);
                                for (int dyi = 0; dyi < 3; dyi++)
                                    tma2_load_2d(w_sm + (grp * 3 + dyi) * kWTileBytes, w_map, &wfull_bar[grp], half * 64,
                                                 (dyi * 3 + dxi) * 128 + (int)rank * 64);
                            }
                            __syncwarp();
                        }
                        if (WIDE && dxi != 2) continue;   // one box per channel half, requested after its three weight groups
                        mbar_wait(&empty_bar[stage], phase ^ 1, 22);
                        if (elect_one()) {
                            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kStageBytes);
                            if (prm.l2_hint & 4) tma2_load_4d_hint(a_sm + stage * kStageBytes, in_map, &full_bar[stage], half * 64, WIDE ? -1 : dxi - 1, t * 4 + (int)rank * 2, -1, l2_policy_evict_last());
                            else tma2_load_4d(a_sm + stage * kStageBytes, in_map, &full_bar[stage], half * 64, WIDE ? -1 : dxi - 1, t * 4 + (int)rank * 2, -1);
                        }
                        __syncwarp();
                        if (++stage == NS) { stage = 0; phase ^= 1; }
                    }
            }
            u0++;
            if (halves == 2) u1++;
        }
        cum += (uint32_t)(NL * T);
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // ------------------------------------------------------------ MMA issuer (leader CTA)
            constexpr uint32_t idesc = umma_idesc_bf16(256, 128);
            const uint64_t dbase = umma_desc_base_sw128();
            const uint32_t w_lo = (smem_u32(w_sm) & 0x3FFFF) >> 4;
            int stage = 0; uint32_t phase = 0; int lt = 0;
            int u0 = 0, u1 = 0;
            for (int rg = 0; rg < n_ranges; rg++) {
            TOWER_RANGE_BEGIN();
            for (int L = 0; L < NL; L++) {
                const int layer = L - stem;
                const int halves = layer >= 0 ? 2 : 1;
                for (int i = 0; i < T; i++, lt++) {
                    const int acc = lt & 1; const uint32_t accphase = (lt >> 1) & 1;
                    mbar_wait(&tempty_bar[acc], accphase ^ 1, 23);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * 128;
                    for (int half = 0; half < halves; half++)
                        for (int dxi = 0; dxi < 3; dxi++) {
                            const int grp = half * 3 + dxi;
                            if (!WIDE || dxi == 0) mbar_wait(&full_bar[stage], phase, 24);
                            if (i == 0) mbar_wait(&wfull_bar[grp], (uint32_t)((half == 0 ? u0 : u1) & 1), 25);
                            tc_fence_after();
                            if (elect_one()) {
                                const uint32_t a_lo = (smem_u32(a_sm + stage * kStageBytes) & 0x3FFFF) >> 4;
                                const uint32_t b_lo = w_lo + (uint32_t)(grp * 3) * (kWTileBytes >> 4);
                                // WIDE: 8-row groups (one rank of one board) are 16 rows = 2048 bytes apart, a rank is 4096 bytes, and the
                                // horizontal tap is a window starting dxi rows into every group (the swizzle follows the address bits)
                                const uint64_t abase = WIDE ? (((uint64_t)1 << 16) | ((uint64_t)((S::kPitch * 128) >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61)) : dbase;
                                const uint32_t a_dy = (2 * S::kPitch * 128) >> 4, a_dx = WIDE ? (uint32_t)dxi * (128 >> 4) : 0u;
#pragma unroll
                                for (int dyi = 0; dyi < 3; dyi++) {
#pragma unroll
                                    for (int k = 0; k < 4; k++) {
                                        const uint64_t ad = abase | (uint64_t)(a_lo + dyi * a_dy + a_dx + k * 2);
                                        const uint64_t bd = dbase | (uint64_t)(b_lo + dyi * (kWTileBytes >> 4) + k * 2);
                                        umma2_bf16(d_tmem, ad, bd, idesc, (half | dxi | dyi | k) != 0 ? 1u : 0u);
                                    }
                                }
                                if (!WIDE || dxi == 2) umma2_commit_mc(&empty_bar[stage]);
                                if (i == T - 1) umma2_commit_mc(&wempty_bar[grp]);  // weights of this group are free for the next layer
                            }
                            __syncwarp();
                            if (!WIDE || dxi == 2) { if (++stage == NS) { stage = 0; phase ^= 1; } }
                        }
                    if (elect_one()) umma2_commit_mc(&tfull_bar[acc]);
                    __syncwarp();
                }
                u0++;
                if (halves == 2) u1++;
            }
            }
        }
    } else {
        // ------------------------------------------------ epilogue (TMEM lane quarter q, column group cg of kEpiCols columns)
        const int q = warp & 3;
        const int cg = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const int h = row >> 4, b = (row >> 3) & 1, w = row & 7;
        int lt = 0, g = 0;
        uint32_t done = 0;
        const uint64_t l2pol = l2_policy_evict_last();
        for (int rg = 0; rg < n_ranges; rg++) {
        TOWER_RANGE_BEGIN();
        // completion is published lazily (after the next accumulator wait) and only every 4th tile when the pair has
        // enough tiles in flight; the producer needs tile i of this layer only T tiles later (T >= 6: the published count lags by at most 3 tiles and the producer runs about 2 tiles ahead of the epilogue)
        const bool lazy = T >= 6;
        for (int L = 0; L < NL; L++, g++) {
            const int layer = L - stem;
            const int blk_second = layer >= 0 ? (layer & 1) : 0;
            const int out_buf = layer < 0 ? 0 : blk_second ? 0 : 1;
            __nv_bfloat16* out = prm.act[out_buf];
            // the residual of tile t is read (into registers, before the accumulator wait) by the same warp that then overwrites
            // tile t, and no other tile's convolution reads these boards: the block output can replace the block input in place,
            // which keeps the tower's footprint at two activation buffers (L2 residency)
            const __nv_bfloat16* residual = blk_second ? prm.act[0] : nullptr;
            // the epilogue warps switch layers together: whoever arrives refills the buffer last used two layers ago
            if (threadIdx.x - 64 < 128)
                bias_s[(g & 1) * 128 + threadIdx.x - 64] = sched.bias(prm)[(layer >= 0 ? layer : prm.n_layers) * 128 + threadIdx.x - 64];
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
            const float* bias = bias_s + (g & 1) * 128 + cg * kEpiCols;
            for (int i = 0; i < T; i++, lt++) {
                const int t = first_tile + i * tile_step;
                const int acc = lt & 1; const uint32_t accphase = (lt >> 1) & 1;
                const int board = t * 4 + (int)rank * 2 + b;
                const bool valid = board < n_boards;
                const size_t off = ((size_t)board * 64 + h * 8 + w) * 128 + cg * kEpiCols;
                const bool has_res = residual != nullptr && valid;
                uint32_t res[kEpiCols / 2];
                if (has_res) {
#pragma unroll
                    for (int k = 0; k < kEpiCols / 16; k++) {
                        if (prm.l2_hint & 2) ld_global_v8_hint(residual + off + k * 16, &res[k * 8], l2pol);
                        else ld_global_v8(residual + off + k * 16, &res[k * 8]);
                    }
                }
                mbar_wait(&tfull_bar[acc], accphase, 26);
                tc_fence_after();
                if (lazy && done > 0 && (done & 3) == 0) {  // earlier tiles' stores have had time to land
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) { __threadfence(); epi_done[warp - 2] = done; }
                }
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 128 + cg * kEpiCols;
#pragma unroll
                for (int chunk = 0; chunk < kEpiChunks; chunk++) {
                    uint32_t r[32];
                    tmem_ld32(taddr + chunk * 32, r);
                    tmem_ld_wait();
                    if (chunk == kEpiChunks - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { if (prm.release_arrive) mbar_arrive_cluster(&tempty_bar[acc], 0); else mbar_arrive_cluster_relaxed(&tempty_bar[acc], 0); }
                    }
                    if (valid) {
#pragma unroll
                        for (int v = 0; v < 2; v++) {
                            uint32_t packed[8];
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                const int c = v * 16 + j * 2;
                                const float2 bb = *reinterpret_cast<const float2*>(bias + chunk * 32 + c);
                                float x0 = __uint_as_float(r[c]) + bb.x;
                                float x1 = __uint_as_float(r[c + 1]) + bb.y;
                                if (has_res) {
                                    const uint32_t rr = res[chunk * 16 + v * 8 + j];
                                    x0 += __uint_as_float(rr << 16);
                                    x1 += __uint_as_float(rr & 0xFFFF0000u);
                                }
                                x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f);
                                __nv_bfloat162 pk = __floats2bfloat162_rn(x0, x1);
                                packed[j] = *reinterpret_cast<uint32_t*>(&pk);
                            }
                            if (prm.l2_hint & 1) st_global_v8_hint(out + off + chunk * 32 + v * 16, packed, l2pol);
                            else st_global_v8(out + off + chunk * 32 + v * 16, packed);
                        }
                    }
                }
                // Publish "this warp's part of tile i is in global memory and visible to the TMA (async proxy)".  The
                // fence waits for the stores to land, so with enough tiles in flight it is deferred until the next
                // accumulator is ready (the producer needs tile i only T tiles later); tiny batches publish eagerly.
                done++;
                if (!lazy) {
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) { __threadfence(); epi_done[warp - 2] = done; }
                }
            }
        }
        }
    }
#undef TOWER_RANGE_BEGIN
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) { tc_fence_after(); tmem2_dealloc(tmem_base, kTmemCols2); }
}

template <int WIDE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1)
conv_tower_kernel(const TowerParams prm) {
    conv_tower_body<WIDE, false>(prm, TowerNets{nullptr, 0, nullptr, nullptr});
}

// the tower of a multi-network batch: the CTA pairs are split between the two networks' weights (TowerSched<true>); the per-tile
// work is that of conv_tower_kernel, so a board's activations do not depend on the pair that computed them
template <int WIDE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1)
conv_tower_nets_kernel(const TowerParams prm, const TowerNets nets) {
    conv_tower_body<WIDE, true>(prm, nets);
}

int tc_tower_launch(cudaStream_t stream, const CUtensorMap* maps_dev, const float* bias, void* const* act, const int* n_boards_dev,
                    int n_boards_static, int n_layers, int stem, int grid, int tile_lo, int tile_hi, int range_tiles, int release_arrive,
                    int wide, int l2_hint) {
    static PerDeviceOnce once;
    if (once.first() &&
        (cudaFuncSetAttribute(conv_tower_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2>::kTotal) != cudaSuccess ||
         cudaFuncSetAttribute(conv_tower_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2, 128, 1>::kTotal) != cudaSuccess ||
         cudaFuncSetAttribute(conv_tower_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2, 128, 2>::kTotal) != cudaSuccess))
        return -2;
    if (wide && stem) return -5;   // the in-kernel input convolution exists for the narrow boxes only
    if (grid <= 0) grid = 148;
    grid &= ~1;
    TowerParams p;
    p.maps = maps_dev; p.bias = bias;
    for (int i = 0; i < 3; i++) p.act[i] = (__nv_bfloat16*)act[i];
    p.n_boards_ptr = n_boards_dev; p.n_boards_static = n_boards_static; p.n_layers = n_layers; p.stem = stem ? 1 : 0;
    p.tile_lo = tile_lo; p.tile_hi = tile_hi; p.range_tiles = range_tiles > 0 ? range_tiles : (1 << 30);
    p.release_arrive = release_arrive;
    p.l2_hint = l2_hint;
    if (wide == 2) conv_tower_kernel<2><<<grid, kThreads2, ConvSmem<2, 128, 2>::kTotal, stream>>>(p);
    else if (wide) conv_tower_kernel<1><<<grid, kThreads2, ConvSmem<2, 128, 1>::kTotal, stream>>>(p);
    else conv_tower_kernel<0><<<grid, kThreads2, ConvSmem<2>::kTotal, stream>>>(p);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

int tc_tower_nets_launch(cudaStream_t stream, const CUtensorMap* maps0_dev, const CUtensorMap* maps1_dev, const float* bias0,
                         const float* bias1, void* const* act, const int* counts_dev, int base1, int grid, int release_arrive, int l2_hint) {
    static PerDeviceOnce once;
    if (once.first() &&
        cudaFuncSetAttribute(conv_tower_nets_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2, 128, 2>::kTotal) != cudaSuccess)
        return -2;
    grid &= ~1;
    if (grid < 4) return -3;   // at least one pair per network
    TowerParams p;
    p.maps = maps0_dev; p.bias = bias0;
    for (int i = 0; i < 3; i++) p.act[i] = (__nv_bfloat16*)act[i];
    p.n_boards_ptr = nullptr; p.n_boards_static = 0; p.n_layers = 20; p.stem = 0;
    p.tile_lo = 0; p.tile_hi = 0x7FFFFFFF; p.range_tiles = 1;   // unused: the ranges follow from the device counts (TowerSched<true>)
    p.release_arrive = release_arrive;
    p.l2_hint = l2_hint;
    conv_tower_nets_kernel<2><<<grid, kThreads2, ConvSmem<2, 128, 2>::kTotal, stream>>>(p, TowerNets{counts_dev, base1, maps1_dev, bias1});
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

int tc_conv3x3_nets_launch(cudaStream_t stream, const CUtensorMap* in_map, const CUtensorMap* w_map0, const CUtensorMap* w_map1,
                           const float* bias0, const float* bias1, void* out, const int* counts_dev, int base1, int grid, int dbg) {
    static PerDeviceOnce once;
    if (once.first() &&
        cudaFuncSetAttribute(conv3x3_tc2_nets_kernel<1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<1, 64>::kTotal) != cudaSuccess)
        return -2;
    grid &= ~1;
    if (grid < 4) return -3;
    conv3x3_tc2_nets_kernel<1, 64><<<grid, kThreads2, ConvSmem<1, 64>::kTotal, stream>>>(*in_map, *w_map0, *w_map1, bias0, bias1,
                                                                                         (__nv_bfloat16*)out, counts_dev, base1, dbg);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) return nullptr;
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

int tc_make_act_map(CUtensorMap* map, const void* base, int channels, int max_boards, int wide) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return -1;
    // dims fastest-first: channel, file, board, rank  (SMEM box order becomes [rank][board][file][channel])
    cuuint64_t dims[4] = {(cuuint64_t)channels, 8, (cuuint64_t)max_boards, 8};
    cuuint64_t strides[3] = {(cuuint64_t)channels * 2, (cuuint64_t)channels * 2 * 64, (cuuint64_t)channels * 2 * 8};
    // 64 channels (128-byte rows, 128-byte swizzle) per box, or the whole row of the 32-channel plane layout (64-byte swizzle)
    // wide: files -1..14 (the files beyond the board are zero-filled), so that every (rank, board) group has a 16-row pitch
    cuuint32_t box[4] = {(cuuint32_t)(channels == 32 ? 32 : 64), (cuuint32_t)(wide == 1 ? 16 : wide == 2 ? 10 : 8), 2, 10};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, channels == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -(int)r - 1000;
}

int tc_make_rows_map(CUtensorMap* map, const void* base, int max_boards) {
    // the same NHWC activation buffer seen as a matrix [max_boards * 64 pixel rows][128 channels]: boxes of 128 rows x 64 channels
    PFN_encodeTiled enc = get_encode();
    if (!enc) return -1;
    cuuint64_t dims[2] = {128, (cuuint64_t)max_boards * 64};
    cuuint64_t strides[1] = {256};
    cuuint32_t box[2] = {64, 128};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -(int)r - 1000;
}

int tc_make_weight_map(CUtensorMap* map, const void* base, int cin) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return -1;
    cuuint64_t dims[2] = {(cuuint64_t)cin, 9 * 128};
    cuuint64_t strides[1] = {(cuuint64_t)cin * 2};
    cuuint32_t box[2] = {(cuuint32_t)(cin == 32 ? 32 : 64), 64};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, cin == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -(int)r - 1000;
}

int tc_conv3x3_launch(cudaStream_t stream, const CUtensorMap* in_map, const CUtensorMap* w_map, int cin, const float* bias,
                      const void* residual, void* out, const int* n_boards_dev, int n_boards_static, int relu, int grid, int dbg) {
    static PerDeviceOnce once;
    if (once.first()) {
        cudaError_t e1 = cudaFuncSetAttribute(conv3x3_tc2_kernel<1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<1>::kTotal);
        cudaError_t e2 = cudaFuncSetAttribute(conv3x3_tc2_kernel<2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2>::kTotal);
        cudaError_t e3 = cudaFuncSetAttribute(conv3x3_tc2_kernel<1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<1, 64>::kTotal);
        cudaError_t e4 = cudaFuncSetAttribute(conv3x3_tc2_kernel<2, 128, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2, 128, 1>::kTotal);
        cudaError_t e5 = cudaFuncSetAttribute(conv3x3_tc2_kernel<2, 128, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<2, 128, 2>::kTotal);
        cudaError_t e6 = cudaFuncSetAttribute(conv3x3_tc2_kernel<1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<1, 64, 2>::kTotal);
        cudaError_t e7 = cudaFuncSetAttribute(conv3x3_tc2_kernel<1, 64, 0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvSmem<1, 64>::kTotal);
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess || e5 != cudaSuccess || e6 != cudaSuccess || e7 != cudaSuccess) return -2;
    }
    if (grid <= 0) grid = 148;
    grid &= ~1;  // CTA pairs
    if (cin == 32 && (dbg & 256))   // 10-file boxes: in_map must have been made with wide = 2
        conv3x3_tc2_kernel<1, 64, 2><<<grid, kThreads2, ConvSmem<1, 64, 2>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                            (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 32 && (dbg & 1024))   // two epilogue sets on alternate tiles
        conv3x3_tc2_kernel<1, 64, 0, 2><<<grid, 64 + 2 * kEpiThreads, ConvSmem<1, 64>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                                  (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 32)
        conv3x3_tc2_kernel<1, 64><<<grid, kThreads2, ConvSmem<1, 64>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                       (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 64)
        conv3x3_tc2_kernel<1, 128><<<grid, kThreads2, ConvSmem<1>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                    (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 128 && (dbg & 256))  // 10-file boxes: in_map must have been made with wide = 2
        conv3x3_tc2_kernel<2, 128, 2><<<grid, kThreads2, ConvSmem<2, 128, 2>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                              (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 128 && (dbg & 64))   // 16-file boxes: in_map must have been made with wide = 1
        conv3x3_tc2_kernel<2, 128, 1><<<grid, kThreads2, ConvSmem<2, 128, 1>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                              (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else if (cin == 128)
        conv3x3_tc2_kernel<2, 128><<<grid, kThreads2, ConvSmem<2>::kTotal, stream>>>(*in_map, *w_map, bias, (const __nv_bfloat16*)residual,
                                                                                    (__nv_bfloat16*)out, n_boards_dev, n_boards_static, relu, dbg);
    else
        return -3;
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

}  // namespace azb
