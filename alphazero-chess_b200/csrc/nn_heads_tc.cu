// Policy and value heads of agent.rs:124-141 on tcgen05 (AZ_HEADS_TC=1, the default): the two 1x1 convolutions of the heads are
// GEMMs over pixel rows, so a tile of two boards (128 pixel rows = the 128 TMEM lanes) runs
//   stage 1  D1[128 px][48]  = X[128 px][128 ch] . W40^T      policy_conv_1 (32) | value_conv (8) | 8 zero columns
//   stage 2  D2[128 px][64]  = P1[128 px][32]    . W2^T       policy_conv_2, P1 = bf16(ReLU(D1 + b)) staged through shared memory
// as tcgen05.mma (cta_group::1, M128) with the accumulators in tensor memory.  Warp 0 streams the tower's output through a
// 3-stage TMA ring (32 KB per tile), warp 1 issues the MMAs, sixteen epilogue warps form two groups that alternate tiles.
// Inside a group warp (q, cg) owns TMEM lane quarter q (32 pixel rows) and column half cg, so a thread holds the 32 logits
// [co in its half][its square] of its board; the softmax of a board is a reduction over a team of four warps (named barrier
// of 128 threads) and the probabilities land as coalesced rows / a conflict-free [co][sq] tile in shared memory, from which
// thread e of the team writes the prior of legal move e into the search tree.  A group runs stage 1 of its next tile before
// the softmax of the current one, which hides the P1 -> stage 2 round trip.  The scatter's address chain (edge_off / n_edges ->
// edge_mv -> edge_P) is prefetched two tiles ahead.  The value head ([boards x 512] . [512 x 64] -> ReLU -> 64 -> 1 -> tanh)
// batches the boards of 16 tiles into two M = 16 mma.sync tiles; its fc1 weights are copied into the drained activation ring
// by cp.async.bulk while the last tiles are still in the epilogue.
// Against the warp-level kernel of nn_heads.cu (kept as AZ_HEADS_TC=0): the weights are read from shared memory by the tensor
// core once per 128 rows instead of once per 32 rows by every warp, the activations arrive asynchronously, and a board costs
// about a third fewer warp instructions.  49.0 -> 39.8 us per 4096 boards in the self-play loop (DESIGN.md section 5).
#include "nn.h"
#include "tc_conv.cuh"
#include "device_once.h"
#include <algorithm>

namespace azb {
namespace htc {
constexpr int kStages = 3;
constexpr int kStageBytes = 32768;                       // one tile: two K blocks of {128 pixel rows x 64 channels} bf16
constexpr int kOffA = 0;
constexpr int kW40Block = 48 * 128;                      // one K block of W40: 48 rows x 128 B (128-byte swizzle)
constexpr int kOffW40 = kOffA + kStages * kStageBytes;   //  98304
constexpr int kOffW2 = kOffW40 + 2 * kW40Block;          // 110592: 64 rows x 64 B (64-byte swizzle)
constexpr int kOffP1 = kOffW2 + 64 * 64;                 // 114688: per epilogue group 128 rows x 64 B (64-byte swizzle)
constexpr int kOffExp = kOffP1 + 2 * 8192;               // 131072: [2 groups][2 boards][64 co][64 sq] f32; value head: hidden sums
constexpr int kV1Pitch = 520;                            // 512 + 8 bf16: conflict-free fragment loads
constexpr int kOffV1 = kOffExp + 4 * 16384;              // 196608: [32 board rows][kV1Pitch] bf16
constexpr int kOffMisc = kOffV1 + 32 * kV1Pitch * 2;     // 229888
constexpr int kTotal = kOffMisc + 1024 + 1024;           // + alignment slack = 231936 <= 232448
constexpr int kGroupTiles = 16;                          // tiles per value-head batch (32 board rows)
constexpr int kEpiThreads = 512;
constexpr int kThreads = 64 + kEpiThreads;               // warp 0 TMA, warp 1 MMA / TMEM, warps 2-9 and 10-17 epilogue groups
constexpr int kTmemCols = 512;                           // per group: D1 at +0 (48 columns), D2 slots at +64 and +128
static_assert(kOffW40 % 1024 == 0 && kOffW2 % 1024 == 0 && kOffP1 % 1024 == 0 && kOffExp % 1024 == 0, "operand tiles must be 1024-byte aligned");
static_assert(kTotal <= 232448, "shared memory of one CTA");
static_assert(2 * kThreads >= 48 * 16, "two weight chunks per thread cover W40");
}  // namespace htc

// ---------------------------------------------------------------- cta_group::1 forms of the primitives in tc_conv.cuh
__device__ __forceinline__ void tmem1_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem1_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma1_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma1_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma1_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// plain (1-D) bulk copy global -> shared memory, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ float htc_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// generic -> async proxy fence for SHARED memory only: the unqualified form also orders global memory (MEMBAR.ALL.GPU in SASS) and
// would make an epilogue warp wait for the prior tile's outstanding scatter stores
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ uint32_t htc_pack_bf16(float lo, float hi) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ void htc_mma_16816(float* d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// -DAZ_HTC_TIMING (tools/htc_timing.sh): block 0 prints the clocks the first warp of each epilogue group, the MMA warp and the TMA warp spent per phase
#ifdef AZ_HTC_TIMING
#define HTC_T(i) do { const long long now_ = clock64(); tacc[i] += now_ - tlast; tlast = now_; } while (0)
#else
#define HTC_T(i) do { } while (0)
#endif

// Which tiles a CTA computes and with which weights.  HeadsSched<false> is the single-network launch (its expressions are those
// the kernel has always had, so its code is unchanged); HeadsSched<true> a multi-network batch (net_part in tc_conv.cuh): the
// CTAs are split between the networks, and a CTA stages and reads only its own network's weights.
struct HeadNets {
    const int* counts;   // device [2]: boards of each network
    int base1;           // first board of network 1
    const __nv_bfloat16 *w40, *wp2, *wl1t;   // network 1's weights (the parameters of k_heads_tc)
    const float *b40, *bp2, *bl1, *wl2, *bl2;
};
template <bool NETS> struct HeadsSched;
template <> struct HeadsSched<false> {
    __device__ __forceinline__ explicit HeadsSched(const HeadNets&) {}
    template <class T> __device__ __forceinline__ const T* pick(const T* w0, const T*) const { return w0; }
    __device__ __forceinline__ int n(const int* n_dev, int n_static) const { return n_dev ? *n_dev : n_static; }
    __device__ __forceinline__ int n_tiles(int n) const { return (n + 1) >> 1; }
    __device__ __forceinline__ int tile0() const { return 0; }
    __device__ __forceinline__ int cta() const { return (int)blockIdx.x; }
    __device__ __forceinline__ int ncta() const { return (int)gridDim.x; }
};
template <> struct HeadsSched<true> {
    NetPart np;
    __device__ __forceinline__ explicit HeadsSched(const HeadNets& h) : np(net_part(h.counts, h.base1, gridDim.x, blockIdx.x, 2)) {}
    template <class T> __device__ __forceinline__ const T* pick(const T* w0, const T* w1) const { return np.net ? w1 : w0; }
    __device__ __forceinline__ int n(const int*, int) const { return np.end_board; }
    __device__ __forceinline__ int n_tiles(int) const { return np.n_tiles; }
    __device__ __forceinline__ int tile0() const { return np.first_tile; }
    __device__ __forceinline__ int cta() const { return np.unit; }
    __device__ __forceinline__ int ncta() const { return np.units; }
};

template <bool NETS>
__device__ __forceinline__ void heads_tc_body(const CUtensorMap& act_map, const __nv_bfloat16* __restrict__ w40, const float* __restrict__ b40,
                                              const __nv_bfloat16* __restrict__ wp2, const float* __restrict__ bp2, const __nv_bfloat16* __restrict__ wl1t,
                                              const float* __restrict__ bl1, const float* __restrict__ wl2, const float* __restrict__ bl2,
                                              float* __restrict__ policy_out, float* __restrict__ value_out, const int* __restrict__ n_dev,
                                              int n_static, const HeadScatter& sc, const HeadNets& nets) {
    using namespace htc;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* misc = smem + kOffMisc;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(misc);   // [kStages]   TMA bytes landed
    uint64_t* a_empty = a_full + kStages;                   // [kStages]   stage 1 MMAs of the tile have read the stage
    uint64_t* d1_full = a_empty + kStages;                  // [2]         per epilogue group: D1 complete
    uint64_t* p1_ready = d1_full + 2;                       // [2]         D1 read out and P1 in shared memory (8 warp arrivals)
    uint64_t* d2_full = p1_ready + 2;                       // [2][2]      per group and D2 slot
    uint64_t* d2_free = d2_full + 4;                        // [2][2]      D2 slot read out (8 warp arrivals)
    uint64_t* wl1_full = d2_free + 4;                       // value head: fc1 weights staged into the (then idle) activation ring
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(wl1_full + 1);
    float* s_b40 = reinterpret_cast<float*>(misc + 160);    // [40]
    float* s_b2 = reinterpret_cast<float*>(misc + 320);     // [64]
    float* s_red = reinterpret_cast<float*>(misc + 576);    // [2 groups][2 boards][4 maxima, 4 sums]
    float* s_vsum = reinterpret_cast<float*>(misc + 704);   // [32 board rows][2]
    __nv_bfloat16* s_v1 = reinterpret_cast<__nv_bfloat16*>(smem + kOffV1);
    float* s_hid = reinterpret_cast<float*>(smem + kOffExp);   // [2 K halves][32][64], value head only (the exp tiles are dead by then)

#ifdef AZ_HTC_TIMING
    long long tacc[20] = {}, tlast = clock64();
    const long long tbegin = tlast;
#endif
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const HeadsSched<NETS> sched(nets);
    w40 = sched.pick(w40, nets.w40); b40 = sched.pick(b40, nets.b40); wp2 = sched.pick(wp2, nets.wp2); bp2 = sched.pick(bp2, nets.bp2);
    wl1t = sched.pick(wl1t, nets.wl1t); bl1 = sched.pick(bl1, nets.bl1); wl2 = sched.pick(wl2, nets.wl2); bl2 = sched.pick(bl2, nets.bl2);
    // The weight tiles are requested first and stored after everything that needs the board count: the count is a dependent
    // global load itself (the search kernel's batch counter), and the two round trips would otherwise add up in every thread
    uint4 wreg[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)}, w2reg = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int u = 0; u < 2; u++) {
        const int i = t + u * kThreads;
        if (i < 40 * 16) wreg[u] = __ldg(reinterpret_cast<const uint4*>(w40) + i);
    }
    if (t < 64 * 4) w2reg = __ldg(reinterpret_cast<const uint4*>(wp2) + t);
    float breg = 0.0f;
    if (t < 40) breg = b40[t];
    else if (t >= 64 && t < 128) breg = bp2[t - 64];
    const int n = sched.n(n_dev, n_static);
    const int n_tiles = sched.n_tiles(n);
    const int my_tiles = sched.cta() < n_tiles ? (n_tiles - sched.cta() + sched.ncta() - 1) / sched.ncta() : 0;

    // ---- epilogue thread coordinates (warps 2..17); computed here because the scatter metadata of the first two tiles is requested
    // before the set-up below, so that its (TLB-missing, ~3 us) latency overlaps the weight staging and the first TMA / MMA round trip
    const int et = t - 64;                 // 0..511
    const int ew = warp - 2;               // 0..15
    const int w = ew >> 3;                 // group: tiles k = w, w + 2, ...
    const int q = warp & 3;                // TMEM lane quarter of this warp
    const int cg = (ew & 7) >> 2;          // column half
    const int row = q * 32 + lane;         // pixel row of the tile
    const int bi = q >> 1, sq = row & 63;  // board of the tile, square
    const int ti = (q & 1) + 2 * cg;       // warp of the board's team
    const int tid128 = sq + 64 * cg;       // thread of the board's team
    const int nw = (my_tiles - w + 1) >> 1;
    // Scatter metadata two tiles ahead: (first edge, edge count) of the node waiting for this thread's board, and this thread's
    // move word one tile ahead -- the chain edge_off -> edge_mv -> edge_P would otherwise cost two dependent global round
    // trips per tile on the critical path of the group (ncu: the top stall of the first version)
    unsigned long long eo_cur = 0, eo_nxt = 0, eo_n2 = 0;
    int L_cur = 0, L_nxt = 0, L_n2 = 0;
    uint32_t mv_cur = 0, mv_nxt = 0;
    auto meta = [&](int j, unsigned long long& eo, int& L) {
        eo = 0; L = 0;
        if (sc.edge_P && j < nw) {
            const int b = (sched.tile0() + sched.cta() + (2 * j + w) * sched.ncta()) * 2 + bi;
            if (b < n) { eo = sc.edge_off[b]; L = sc.n_edges[b]; }
        }
    };
    if (warp >= 2) { meta(0, eo_cur, L_cur); meta(1, eo_nxt, L_nxt); }

    if (t == 0) {
        tma_prefetch_desc(&act_map);
        for (int i = 0; i < kStages; i++) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&d1_full[i], 1); mbar_init(&p1_ready[i], 8); }
        for (int i = 0; i < 4; i++) { mbar_init(&d2_full[i], 1); mbar_init(&d2_free[i], 8); }
        mbar_init(wl1_full, 1);
        fence_barrier_init();
        // the first tiles are requested before the weights are staged and the block synchronises: their latency hides behind the set-up
        for (int k = 0; k < kStages && k < my_tiles; k++) {
            const int tile = sched.tile0() + sched.cta() + k * sched.ncta();
            mbar_arrive_expect_tx(&a_full[k], kStageBytes);
            tma1_load_2d(smem + kOffA + k * kStageBytes, &act_map, &a_full[k], 0, tile * 128);
            tma1_load_2d(smem + kOffA + k * kStageBytes + 16384, &act_map, &a_full[k], 64, tile * 128);
        }
    }
    // weights into the swizzled K-major operand layouts the UMMA descriptors describe (16-byte chunks, chunk ^= row bits)
#pragma unroll
    for (int u = 0; u < 2; u++) {
        const int i = t + u * kThreads;   // rows 40..47 of W40 are zero (the MMA's N is a multiple of 16)
        if (i < 48 * 16) {
            const int r = i >> 4, ch = i & 15;
            *reinterpret_cast<uint4*>(smem + kOffW40 + (ch >> 3) * kW40Block + (r >> 3) * 1024 + (r & 7) * 128 + (((ch & 7) ^ (r & 7)) << 4)) = wreg[u];
        }
    }
    if (t < 64 * 4) {
        const int r = t >> 2, c = t & 3;
        *reinterpret_cast<uint4*>(smem + kOffW2 + (r >> 3) * 512 + (r & 7) * 64 + ((c ^ ((r >> 1) & 3)) << 4)) = w2reg;
    }
    if (t < 40) s_b40[t] = breg;
    if (t >= 64 && t < 128) s_b2[t - 64] = breg;
    fence_proxy_async_smem();   // the tensor core reads these tiles through the async proxy
    if (warp == 1) tmem1_alloc(tmem_ptr_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;
    HTC_T(0);

    if (warp == 0) {
        // ---------------------------------------------------------------- TMA producer
        int stage = 0; uint32_t phase = 1;   // the first kStages tiles were requested during the set-up
        for (int k = kStages; k < my_tiles; k++) {
            const int tile = sched.tile0() + sched.cta() + k * sched.ncta();
            mbar_wait(&a_empty[stage], phase ^ 1, 21);
            HTC_T(1);
            if (elect_one()) {
                mbar_arrive_expect_tx(&a_full[stage], kStageBytes);
                tma1_load_2d(smem + kOffA + stage * kStageBytes, &act_map, &a_full[stage], 0, tile * 128);
                tma1_load_2d(smem + kOffA + stage * kStageBytes + 16384, &act_map, &a_full[stage], 64, tile * 128);
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        // One value-head batch per CTA (the normal case): once stage 1 of the last tiles has drained the ring, the 64 KB of fc1
        // weights are copied into it, rows padded to the pitch of s_v1 (conflict-free fragment loads), while the epilogue groups
        // still work on their last tiles.  Otherwise every CTA would fetch them from the L2 at the same moment, after the barrier.
        if (my_tiles > 0 && my_tiles <= kGroupTiles) {
            for (int i = 0; i < kStages && i < my_tiles; i++) {
                mbar_wait(&a_empty[stage], phase ^ 1, 28);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            if (elect_one()) {
                mbar_arrive_expect_tx(wl1_full, 64 * 1024);
                for (int r = 0; r < 64; r++) bulk_load_1d(smem + kOffA + r * (kV1Pitch * 2), wl1t + (size_t)r * 512, 1024, wl1_full);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ---------------------------------------------------------------- MMA issuer
        constexpr uint32_t idesc1 = umma_idesc_bf16(128, 48), idesc2 = umma_idesc_bf16(128, 64);
        const uint64_t d128 = umma_desc_base_sw128(), d64 = umma_desc_base_sw64();
        const uint32_t w40_lo = (smem_u32(smem + kOffW40) & 0x3FFFF) >> 4, w2_lo = (smem_u32(smem + kOffW2) & 0x3FFFF) >> 4;
        int stage = 0; uint32_t phase = 0;
        auto stage1 = [&](int k) {
            const int w = k & 1;
            HTC_T(4);
            mbar_wait(&a_full[stage], phase, 22);
            HTC_T(1);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_lo = (smem_u32(smem + kOffA + stage * kStageBytes) & 0x3FFFF) >> 4;
                const uint32_t d = tmem_base + w * 192;
#pragma unroll
                for (int ks = 0; ks < 8; ks++) {
                    const uint64_t ad = d128 | (uint64_t)(a_lo + (ks >> 2) * (16384 >> 4) + (ks & 3) * 2);
                    const uint64_t bd = d128 | (uint64_t)(w40_lo + (ks >> 2) * (kW40Block >> 4) + (ks & 3) * 2);
                    umma1_bf16(d, ad, bd, idesc1, ks != 0 ? 1u : 0u);
                }
                umma1_commit(&a_empty[stage]);
                umma1_commit(&d1_full[w]);
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
        };
        if (my_tiles > 0) stage1(0);
        if (my_tiles > 1) stage1(1);
        for (int k = 0; k < my_tiles; k++) {
            const int w = k & 1, j = k >> 1, slot = j & 1;
            HTC_T(4);
            mbar_wait(&p1_ready[w], j & 1, 23);
            HTC_T(2);
            if (j >= 2) mbar_wait(&d2_free[w * 2 + slot], ((j >> 1) - 1) & 1, 24);
            HTC_T(3);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t p_lo = (smem_u32(smem + kOffP1 + w * 8192) & 0x3FFFF) >> 4;
                const uint32_t d = tmem_base + w * 192 + 64 + slot * 64;
#pragma unroll
                for (int ks = 0; ks < 2; ks++)
                    umma1_bf16(d, d64 | (uint64_t)(p_lo + ks * 2), d64 | (uint64_t)(w2_lo + ks * 2), idesc2, ks != 0 ? 1u : 0u);
                umma1_commit(&d2_full[w * 2 + slot]);
            }
            __syncwarp();
            if (k + 2 < my_tiles) stage1(k + 2);   // D1 of this group is free: p1_ready said so
        }
    } else {
        // ---------------------------------------------------------------- epilogue groups
        // group w (8 warps) takes the tiles k = w, w + 2, ...; inside a group warp (q, cg) owns TMEM lane quarter q (32 pixel rows)
        // and column half cg (16 of the 32 policy channels of D1, 32 of the 64 output channels of D2), so a board is a team of
        // four warps and every scheduler has four epilogue warps to switch between
        const uint32_t t_d1 = tmem_base + ((uint32_t)(q * 32) << 16) + w * 192;
        float* se = reinterpret_cast<float*>(smem + kOffExp) + (w * 2 + bi) * 4096;
        float* red = s_red + (w * 2 + bi) * 8;   // [max of the 4 warps][sum of the 4 warps]
        const int team_bar = 2 + w * 2 + bi;

        if (tid128 < L_cur) mv_cur = sc.edge_mv[eo_cur + tid128];   // the first move word (edge_off / n_edges were requested at kernel entry)

        // stage 1 of the group's tile j: D1 -> bias, ReLU -> P1 (bf16, shared memory) + the value head's input row
        auto epi1 = [&](int j) {
            const int k = 2 * j + w;
            HTC_T(15);
            mbar_wait(&d1_full[w], j & 1, 25);
            HTC_T(1);
            tc_fence_after();
            uint32_t v[16], u[4];
            tmem_ld16(t_d1 + cg * 16, v);
            tmem_ld4(t_d1 + 32 + cg * 4, u);
            tmem_ld_wait();
            uint32_t pk[8];
#pragma unroll
            for (int i = 0; i < 8; i++)
                pk[i] = htc_pack_bf16(fmaxf(__uint_as_float(v[2 * i]) + s_b40[cg * 16 + 2 * i], 0.0f),
                                      fmaxf(__uint_as_float(v[2 * i + 1]) + s_b40[cg * 16 + 2 * i + 1], 0.0f));
            __nv_bfloat16* vr = s_v1 + ((k & (kGroupTiles - 1)) * 2 + bi) * kV1Pitch + cg * 4 * 64 + sq;
#pragma unroll
            for (int c = 0; c < 4; c++) vr[c * 64] = __float2bfloat16_rn(fmaxf(__uint_as_float(u[c]) + s_b40[32 + cg * 4 + c], 0.0f));
            // stage 2 of the previous tile must have read P1 before it is overwritten
            HTC_T(2);
            if (j > 0) mbar_wait(&d2_full[w * 2 + ((j - 1) & 1)], ((j - 1) >> 1) & 1, 26);
            HTC_T(3);
            uint8_t* prow = smem + kOffP1 + w * 8192 + (row >> 3) * 512 + (row & 7) * 64;
            const int x = (row >> 1) & 3;
#pragma unroll
            for (int c = 0; c < 2; c++)
                *reinterpret_cast<uint4*>(prow + (((2 * cg + c) ^ x) << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p1_ready[w]);
            HTC_T(4);
        };
        // stage 2 of tile j: D2 -> bias -> softmax over the board (a team of four warps) -> priors / dense policy row
        auto epi2 = [&](int j) {
            const int k = 2 * j + w, slot = j & 1;
            const int b = (sched.tile0() + sched.cta() + k * sched.ncta()) * 2 + bi;
            const bool active = b < n;
            // rotate the prefetched metadata HERE, a whole tile after the loads were issued (rotating at the end of the previous
            // stage 2 made the register moves wait for loads issued a few thousand clocks earlier)
            if (j > 0) { eo_cur = eo_nxt; L_cur = L_nxt; mv_cur = mv_nxt; eo_nxt = eo_n2; L_nxt = L_n2; }
            const unsigned long long eo = eo_cur; const int L = L_cur; const uint32_t mv0 = mv_cur;
            mv_nxt = 0;
            if (tid128 < L_nxt) mv_nxt = sc.edge_mv[eo_nxt + tid128];   // consumed by the next tile of this group
            meta(j + 2, eo_n2, L_n2);
            HTC_T(5);
            mbar_wait(&d2_full[w * 2 + slot], (j >> 1) & 1, 27);
            HTC_T(6);
            tc_fence_after();
            uint32_t v[32];
            tmem_ld32(t_d1 + 64 + slot * 64 + cg * 32, v);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d2_free[w * 2 + slot]);
            // four independent chains for the maximum and the sum (a single chain of 32 dependent operations would leave the
            // scheduler waiting on every one of them)
            float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
            for (int i = 0; i < 32; i++) {
                const float x = __uint_as_float(v[i]) + s_b2[cg * 32 + i];
                v[i] = __float_as_uint(x);
                m4[i & 3] = fmaxf(m4[i & 3], x);
            }
            float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
            for (int d = 16; d; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
            if (lane == 0) red[ti] = mx;
            HTC_T(7);
            named_bar_sync(team_bar, 128);
            HTC_T(8);
            mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
            const float kLog2e = 1.4426950408889634f;
            const float off = -mx * kLog2e;
            float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int i = 0; i < 32; i++) {
                const float ev = htc_ex2(fmaf(__uint_as_float(v[i]), kLog2e, off));   // exp(x - max)
                v[i] = __float_as_uint(ev);
                s4[i & 3] += ev;
            }
            float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
            HTC_T(16);
            for (int d = 16; d; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
            if (lane == 0) red[4 + ti] = sum;
            HTC_T(17);
            if (sc.edge_P) {
#pragma unroll
                for (int i = 0; i < 32; i++) se[(cg * 32 + i) * 64 + sq] = __uint_as_float(v[i]);
            }
            HTC_T(9);
            named_bar_sync(team_bar, 128);
            HTC_T(10);
            const float inv = __fdividef(1.0f, (red[4] + red[5]) + (red[6] + red[7]));
            if (sc.edge_P) {   // priors of the legal moves only, written into the tree (tree.rs:84-104 reads nothing else)
                if (tid128 < L) sc.edge_P[eo + tid128] = se[mv0 >> 16] * inv;
                for (int e2 = tid128 + 128; e2 < L; e2 += 128) {   // more than 128 legal moves: rare
                    const uint32_t idx = sc.edge_mv[eo + e2] >> 16;
                    sc.edge_P[eo + e2] = se[idx] * inv;
                }
            }
            HTC_T(11);
            if (policy_out && active) {
                float* po = policy_out + (size_t)b * 4096 + cg * 32 * 64 + sq;
#pragma unroll
                for (int i = 0; i < 32; i++) po[i * 64] = __uint_as_float(v[i]) * inv;
            }
            HTC_T(5);
        };

        for (int g0 = 0; g0 < my_tiles; g0 += kGroupTiles) {
            const int jb = g0 >> 1, je = min(nw, jb + kGroupTiles / 2);
            if (jb < je) epi1(jb);
            for (int j = jb; j < je; j++) {
                if (j + 1 < je) epi1(j + 1);
                epi2(j);
            }
            HTC_T(15);
            // ---------------- value head of the group's 32 board rows (row = 2 * (k - g0) + board of the tile): warp ew sums K half
            // (ew >> 3) of hidden[row][8 (ew & 7) .. + 7]
            {
                const int hw = ew & 7, kh = ew >> 3, g = lane >> 2, tig = lane & 3;
                float acc[2][4] = {{0.0f, 0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f, 0.0f}};
                const bool staged = my_tiles <= kGroupTiles;   // fc1 weights in the activation ring (see the TMA warp)
                const uint32_t* W = staged ? reinterpret_cast<const uint32_t*>(smem + kOffA + (hw * 8 + g) * (kV1Pitch * 2)) + kh * 128
                                           : reinterpret_cast<const uint32_t*>(wl1t + (size_t)(hw * 8 + g) * 512) + kh * 128;
                if (staged) mbar_wait(wl1_full, 0, 29);
                uint32_t wf[16][2];
#pragma unroll
                for (int ks = 0; ks < 16; ks++) { wf[ks][0] = W[ks * 8 + tig]; wf[ks][1] = W[ks * 8 + tig + 4]; }
                HTC_T(12);
                named_bar_sync(1, kEpiThreads);
                HTC_T(13);
#pragma unroll
                for (int m = 0; m < 2; m++) {
                    const uint32_t* V0 = reinterpret_cast<const uint32_t*>(s_v1 + (16 * m + g) * kV1Pitch) + kh * 128;
                    const uint32_t* V1 = reinterpret_cast<const uint32_t*>(s_v1 + (16 * m + g + 8) * kV1Pitch) + kh * 128;
#pragma unroll
                    for (int ks = 0; ks < 16; ks++)
                        htc_mma_16816(acc[m], V0[ks * 8 + tig], V1[ks * 8 + tig], V0[ks * 8 + tig + 4], V1[ks * 8 + tig + 4], wf[ks][0], wf[ks][1]);
                    const int hn = hw * 8 + tig * 2;
                    float* hid = s_hid + kh * 2048;
                    hid[(16 * m + g) * 64 + hn] = acc[m][0];
                    hid[(16 * m + g) * 64 + hn + 1] = acc[m][1];
                    hid[(16 * m + g + 8) * 64 + hn] = acc[m][2];
                    hid[(16 * m + g + 8) * 64 + hn + 1] = acc[m][3];
                }
            }
            HTC_T(14);
            named_bar_sync(1, kEpiThreads);
            HTC_T(13);
            {   // 32 rows x 64 hidden units on 512 threads: ReLU(sum of the two K halves + bias) * w2, reduced per row
                const int hn = et & 63;
                const float b1 = bl1[hn], w2 = wl2[hn];
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const int vrow = r * 8 + (et >> 6);
                    float part = fmaxf(s_hid[vrow * 64 + hn] + s_hid[2048 + vrow * 64 + hn] + b1, 0.0f) * w2;
                    for (int d = 16; d; d >>= 1) part += __shfl_xor_sync(0xffffffffu, part, d);
                    if (lane == 0) s_vsum[vrow * 2 + ((et >> 5) & 1)] = part;
                }
            }
            named_bar_sync(1, kEpiThreads);
            if (et < 32) {
                const int k = g0 + (et >> 1);
                const int b = (sched.tile0() + sched.cta() + k * sched.ncta()) * 2 + (et & 1);
                if (k < my_tiles && b < n) value_out[b] = tanhf(bl2[0] + s_vsum[et * 2] + s_vsum[et * 2 + 1]);
            }
            HTC_T(14);
        }
    }
#ifdef AZ_HTC_TIMING
    if (blockIdx.x == 0 && lane == 0 && (warp <= 2 || warp == 10)) {
        const long long tot = clock64() - tbegin;
        printf("htc warp %d total %lld | setup %lld | p1 %lld p2 %lld p3 %lld p4 %lld p5 %lld p6 %lld p7 %lld p8 %lld p9 %lld p10 %lld p11 %lld p12 %lld p13 %lld p14 %lld p15 %lld | exp %lld shfl %lld\n", warp, tot,
               tacc[0], tacc[1], tacc[2], tacc[3], tacc[4], tacc[5], tacc[6], tacc[7], tacc[8], tacc[9], tacc[10], tacc[11], tacc[12], tacc[13], tacc[14], tacc[15], tacc[16], tacc[17]);
    }
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem1_dealloc(tmem_base, kTmemCols); }
}

__global__ void __launch_bounds__(htc::kThreads, 1)
k_heads_tc(const __grid_constant__ CUtensorMap act_map, const __nv_bfloat16* __restrict__ w40, const float* __restrict__ b40,
           const __nv_bfloat16* __restrict__ wp2, const float* __restrict__ bp2, const __nv_bfloat16* __restrict__ wl1t,
           const float* __restrict__ bl1, const float* __restrict__ wl2, const float* __restrict__ bl2, float* __restrict__ policy_out,
           float* __restrict__ value_out, const int* __restrict__ n_dev, int n_static, HeadScatter sc) {
    heads_tc_body<false>(act_map, w40, b40, wp2, bp2, wl1t, bl1, wl2, bl2, policy_out, value_out, n_dev, n_static, sc, HeadNets{});
}

// the heads of a multi-network batch (the weight parameters are network 0's, `nets` holds network 1's and the board ranges)
__global__ void __launch_bounds__(htc::kThreads, 1)
k_heads_tc_nets(const __grid_constant__ CUtensorMap act_map, const __nv_bfloat16* __restrict__ w40, const float* __restrict__ b40,
                const __nv_bfloat16* __restrict__ wp2, const float* __restrict__ bp2, const __nv_bfloat16* __restrict__ wl1t,
                const float* __restrict__ bl1, const float* __restrict__ wl2, const float* __restrict__ bl2, float* __restrict__ policy_out,
                float* __restrict__ value_out, HeadScatter sc, const HeadNets nets) {
    heads_tc_body<true>(act_map, w40, b40, wp2, bp2, wl1t, bl1, wl2, bl2, policy_out, value_out, nullptr, 0, sc, nets);
}

int launch_heads_tc(az_engine* e, const CUtensorMap* act_map, const int* n_dev, int n_static, float* policy_out, float* value_out,
                    const HeadScatter* scatter) {
    NetWeights* w = e->net;
    const int n_max = n_dev ? w->max_boards : n_static;
    if (n_max <= 0) return 0;
    const int grid = std::min((n_max + 1) / 2, e->sm_count);
    static PerDeviceOnce once;
    if (once.first()) cudaFuncSetAttribute(k_heads_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, htc::kTotal);
    HeadScatter sc{nullptr, nullptr, nullptr, nullptr};
    if (scatter) sc = *scatter;
    k_heads_tc<<<grid, htc::kThreads, htc::kTotal, e->stream>>>(*act_map, w->h_w40, w->f_b40, w->h_wp2, w->f_bp2, w->h_wl1t, w->f_bl1, w->f_wl2,
                                                               w->f_bl2, policy_out, value_out, n_dev, n_static, sc);
    return check_cuda(e, cudaGetLastError(), "k_heads_tc");
}

int launch_heads_tc_nets(az_engine* e, const NetWeights* w, const NetWeights* w1, const CUtensorMap* act_map, const int* counts_dev, int base1,
                         int n_max, float* policy_out, float* value_out, const HeadScatter* scatter) {
    if (n_max <= 0) return 0;
    const int grid = std::max(2, std::min((n_max + 1) / 2, e->sm_count));   // one CTA per network at least
    static PerDeviceOnce once;
    if (once.first()) cudaFuncSetAttribute(k_heads_tc_nets, cudaFuncAttributeMaxDynamicSharedMemorySize, htc::kTotal);
    HeadScatter sc{nullptr, nullptr, nullptr, nullptr};
    if (scatter) sc = *scatter;
    const HeadNets hn{counts_dev, base1, w1->h_w40, w1->h_wp2, w1->h_wl1t, w1->f_b40, w1->f_bp2, w1->f_bl1, w1->f_wl2, w1->f_bl2};
    k_heads_tc_nets<<<grid, htc::kThreads, htc::kTotal, e->stream>>>(*act_map, w->h_w40, w->f_b40, w->h_wp2, w->f_bp2, w->h_wl1t, w->f_bl1,
                                                                    w->f_wl2, w->f_bl2, policy_out, value_out, sc, hn);
    return check_cuda(e, cudaGetLastError(), "k_heads_tc_nets");
}

}  // namespace azb
