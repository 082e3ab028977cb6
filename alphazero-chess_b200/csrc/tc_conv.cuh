// Blackwell (sm_100a) primitives used by the tensor-core convolutions: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld) in CTA-pair form (cta_group::2) and the UMMA shared-memory + instruction
// descriptors.  Hand-written inline PTX; nothing here is a library call.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

namespace azb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the same-offset barrier of CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// Same without the release fence.  Used to hand a TMEM accumulator back to the MMA warp: the reads of TMEM are already
// complete (tcgen05.wait::ld) and ordered by tcgen05.fence::before_thread_sync; a release here would additionally make the
// warp wait for its outstanding global stores of the tile (MEMBAR + ERRBAR, about a microsecond per tile).
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint64_t* bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (and reports) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("azb: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, blockIdx.x, threadIdx.x, parity);
            __trap();
        }
    }
}

// ---------------------------------------------------------------- warp / cluster helpers
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ---------------------------------------------------------------- TMA (both CTAs of a pair signal the leader's barrier)
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// mbarrier address of the even CTA of the pair (peer bit cleared)
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma2_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
        : "memory");
}

// ---------------------------------------------------------------- tcgen05, CTA pair
__device__ __forceinline__ void tmem2_alloc(uint32_t* smem_dst, uint32_t ncols) {  // one warp in EACH CTA of the pair
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem2_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate.  M = 256 (128 rows per CTA), N split across the pair;
// issued by one thread of the leader CTA.
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the barrier at this SMEM offset in both CTAs once all prior MMAs of this thread completed
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (warp w may only touch lanes 32*(w%4)..+31)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows are 128 B apart, 8-row groups are 1024 B apart (densely packed).
// sm_100 UMMA shared-memory descriptor: start>>4 | LBO>>4 <<16 | SBO>>4 <<32 | version 1 <<46 | SWIZZLE_128B (2) <<61.
// The address field (low 14 bits, units of 16 B) is OR-ed in / advanced by the caller.
__device__ __forceinline__ uint64_t umma_desc_base_sw128() {
    return ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// The same for 64-byte rows (32 bf16 channels): SWIZZLE_64B (layout type 4), 8-row groups 512 B apart.
__device__ __forceinline__ uint64_t umma_desc_base_sw64() {
    return ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
// instruction descriptor: bf16 x bf16 -> fp32, both operands K-major
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---------------------------------------------------------------- 256-bit global accesses (one 32-byte sector per lane)
__device__ __forceinline__ void ld_global_v8(const void* p, uint32_t* r) {
    asm volatile("ld.global.L1::no_allocate.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t* r) {
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// ---------------------------------------------------------------- L2 eviction-priority hints (AZ_TOWER_L2HINT)
// The tower's activations are rewritten in place layer after layer; lines that stay in the L2 until they are overwritten never
// reach HBM.  evict_last asks the L2 to keep them in preference to everything else that streams through.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void ld_global_v8_hint(const void* p, uint32_t* r, uint64_t pol) {
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8], %9;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p), "l"(pol));
}
__device__ __forceinline__ void st_global_v8_hint(void* p, const uint32_t* r, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8}, %9;"
                 ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void tma2_load_4d_hint(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3), "l"(pol)
        : "memory");
}

// ---------------------------------------------------------------- multi-network batches (az_forward_networks, az_search_networks)
// Network s owns boards [base_s, base_s + count_s): base_0 = 0, base_1 a multiple of 4, the counts in device memory.  The
// persistent grid's `units` (CTA pairs of the convolutions, CTAs of the heads) are split between the networks in proportion to
// their tiles of `tile_boards` boards, with at least one unit for each network that has boards.  Every CTA derives the same
// split, so a unit only ever streams the weights of its own network and walks that network's tiles.
struct NetPart {
    int net;          // network of this unit
    int unit, units;  // this unit's index among the network's units, and their number
    int first_tile;   // the network's first tile (base_s / tile_boards)
    int n_tiles;      // the network's tiles
    int end_board;    // base_s + count_s
};
__device__ __forceinline__ NetPart net_part(const int* counts, int base1, int units, int unit, int tile_boards) {
    const int c0 = counts[0], c1 = counts[1];
    const int t0 = (c0 + tile_boards - 1) / tile_boards, t1 = (c1 + tile_boards - 1) / tile_boards;
    int u0 = t1 == 0 ? units : t0 == 0 ? 0 : (int)(((long long)units * t0 + (t0 + t1) / 2) / (t0 + t1));
    if (t0 > 0 && t1 > 0) u0 = min(max(u0, 1), units - 1);
    NetPart p;
    p.net = unit >= u0 ? 1 : 0;
    p.unit = p.net ? unit - u0 : unit;
    p.units = p.net ? units - u0 : u0;
    const int base = p.net ? base1 : 0;
    p.first_tile = base / tile_boards;
    p.n_tiles = p.net ? t1 : t0;
    p.end_board = base + (p.net ? c1 : c0);
    return p;
}

}  // namespace azb
