// Device-resident PUCT search and self-play: one warp per game, struct-of-arrays tree pools in HBM.
//
// Restates tree.rs (MCTree::new / simulation / expand / traverse_new / apply_dirichlet_noise / max_subtree_depth)
// and training.rs run_episode with exactly the reference's arithmetic: one simulation in flight per game
// (tree.rs:170-172), PUCT = q + ((c*P)*sqrt(total))/(1+N) evaluated left to right in f32 with strict '>' and
// first-max-in-move-order ties (tree.rs:184-195), W += v ; N += 1 on the way back with a sign flip per level
// (tree.rs:197-206), terminal children never stored (tree.rs:233-234), no tree reuse between moves (tree.rs:239-256).
// This translation unit is compiled with -fmad=false and uses explicit _rn intrinsics so no FMA contraction can
// change a bit.  A "wave" lets every game run until it needs a network evaluation; the evaluations of all games form
// one batch (the reference's recv_many batch, training.rs:369).
#include "mcts.h"
#include "nn.h"
#include "det_math.cuh"
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <cmath>

namespace azb {

constexpr int WARPS = 4;

struct WarpShared {
    double gam[AZ_MAX_MOVES];
    float fval[AZ_MAX_MOVES];
    uint16_t moves[AZ_MAX_MOVES];
    uint16_t sidx[AZ_MAX_MOVES];
    DPos child;
    DPos key;       // cache key of `child` (pseudo-legal ep, counters; no repetition bits)
    int n_moves;
    int term;       // 0 ongoing, 1 draw, 2 decisive (side to move in the child is mated)
    int has_ep;
    int pad;
};

// ------------------------------------------------------------------------------------------- deterministic RNG
// Counter-based generator + IEEE-exact log/exp, bit-identical to oracle/mcts.cpp (spec in DESIGN.md).
__device__ __forceinline__ u64 rng_u64(u64 seed, u64 game, u64 ply, u64 stream, u64 counter) {
    u64 h = splitmix64(seed);
    h = splitmix64(h ^ game);
    h = splitmix64(h ^ ply);
    h = splitmix64(h ^ stream);
    h = splitmix64(h ^ counter);
    return h;
}
__device__ __forceinline__ double rng_uniform(u64 seed, u64 game, u64 ply, u64 stream, u64 counter) {
    u64 h = rng_u64(seed, game, ply, stream, counter);
    return ((double)(h >> 12) + 0.5) * (1.0 / 4503599627370496.0);
}
// Gamma(alpha, 1), Marsaglia-Tsang with the alpha < 1 boost (the scheme of rand_distr 0.4.3)
__device__ double gamma_sample(u64 seed, u64 game, u64 ply, u64 stream, double alpha) {
    u64 ctr = 0;
    double a = alpha < 1.0 ? alpha + 1.0 : alpha;
    double d = a - 1.0 / 3.0;
    double c = 1.0 / sqrt(9.0 * d);
    double v, x;
    for (;;) {
        double u1, u2, s;
        do {
            u1 = 2.0 * rng_uniform(seed, game, ply, stream, ctr++) - 1.0;
            u2 = 2.0 * rng_uniform(seed, game, ply, stream, ctr++) - 1.0;
            s = u1 * u1 + u2 * u2;
        } while (s >= 1.0 || s == 0.0);
        x = u1 * sqrt(-2.0 * det_log(s) / s);
        v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        double u = rng_uniform(seed, game, ply, stream, ctr++);
        if (det_log(u) < 0.5 * x * x + d - d * v + d * det_log(v)) break;
    }
    double g = d * v;
    if (alpha < 1.0) { double u = rng_uniform(seed, game, ply, stream, ctr++); g = g * det_exp(det_log(u) / alpha); }
    return g;
}

// ------------------------------------------------------------------------------------------- synthetic evaluator
__device__ __forceinline__ u64 stub_position_hash(u64 seed, const DPos& p) {
    const u64 occ = occupied(p);
    u64 h = splitmix64(seed);
    h = splitmix64(h ^ p.pawn); h = splitmix64(h ^ p.knight); h = splitmix64(h ^ p.bishop);
    h = splitmix64(h ^ p.rook); h = splitmix64(h ^ p.queen); h = splitmix64(h ^ p.king);
    h = splitmix64(h ^ p.white); h = splitmix64(h ^ (occ ^ p.white));
    const int ep = pseudo_legal_ep(p);
    u64 meta = (u64)meta_turn(p.meta) | ((u64)meta_castling(p.meta) << 8) | ((u64)(ep + 1) << 16) | ((u64)meta_halfmoves(p.meta) << 32) |
               ((u64)meta_fullmoves(p.meta) << 48);
    return splitmix64(h ^ meta);
}
// one warp per request: policy [4096] normalised integers, value in [-1, 1)
__global__ void k_stub_eval(const DPos* __restrict__ req_pos, const int* __restrict__ n_dev, int n_static, u64 seed,
                            float* __restrict__ policy, float* __restrict__ value) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n = n_dev ? *n_dev : n_static;
    if (warp >= n) return;
    const DPos p = req_pos[warp];
    const u64 h = stub_position_hash(seed, p);
    u64 total = 0;
    float* po = policy + (size_t)warp * AZ_ACTION_SPACE;
    for (int i = lane; i < AZ_ACTION_SPACE; i += 32) {
        u64 r = ((splitmix64(h + (u64)i) >> 52) << 12) + (u64)i + 1;
        total += r;
        po[i] = (float)r;
    }
    for (int d = 16; d; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    const float tf = (float)total;
    __syncwarp();
    for (int i = lane; i < AZ_ACTION_SPACE; i += 32) po[i] = __fdiv_rn(po[i], tf);
    if (lane == 0) {
        u64 v = splitmix64(h ^ 0xA5A5A5A5A5A5A5A5ULL) >> 40;
        value[warp] = __fsub_rn(__fmul_rn((float)v, 1.0f / 8388608.0f), 1.0f);
    }
}

// ------------------------------------------------------------------------------------------- per-game helpers
struct Ctx {
    const SearchParams& prm;
    const SearchPtrs& ptr;
    WarpShared* sh;
    int g, lane;
    size_t nbase, ebase;   // first node / edge of this game
    GameCtl c;
    // statistics accumulated by lane 0
    unsigned int st_sims, st_pos, st_evals, st_term, st_games, st_depth, st_edges, st_hits, st_evict;
    unsigned int st_sdepth;        // sum of EpisodeStep::search_depth over the steps recorded (avg_search_depth, training.rs:91-97)
    unsigned long long new_link;   // edge_link value of the node create_node made last
};
// the initial position (az_position_start)
__device__ __forceinline__ DPos start_dpos() {
    az_position sp;
    sp.roles[0] = 0x00FF00000000FF00ULL; sp.roles[1] = 0x4200000000000042ULL; sp.roles[2] = 0x2400000000000024ULL;
    sp.roles[3] = 0x8100000000000081ULL; sp.roles[4] = 0x0800000000000008ULL; sp.roles[5] = 0x1000000000000010ULL;
    sp.colors[0] = 0xFFFFULL; sp.colors[1] = 0xFFFF000000000000ULL;
    sp.turn = 0; sp.castling = 15; sp.ep_square = -1; sp.reserved = 0; sp.halfmoves = 0; sp.fullmoves = 1;
    return dpos_from_wire(sp);
}

// the legal-move priors of the L edges from `off`, out of the dense policy row of request `slot` (when the heads did not
// scatter them into edge_P)
__device__ __forceinline__ void copy_priors(const SearchPtrs& ptr, size_t off, int L, int slot, int lane) {
    const float* pol = ptr.res_policy + (size_t)slot * AZ_ACTION_SPACE;
    for (int e = lane; e < L; e += 32) ptr.edge_P[off + e] = pol[ptr.edge_mv[off + e] >> 16];
}

__device__ __forceinline__ Ctx make_ctx(const SearchParams& prm, const SearchPtrs& ptr, WarpShared* sh, int g, const GameCtl& c) {
    return Ctx{prm, ptr, sh, g, (int)(threadIdx.x & 31), (size_t)g * prm.node_cap, (size_t)g * prm.edge_cap, c, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
}

// Expands `mv` from `parent` on lane 0: child position, its legal moves (into shared memory), mate / stalemate /
// insufficient material.  Repetition and move-count draws are decided afterwards by the whole warp.
__device__ __forceinline__ void lane0_make_child(Ctx& x, const DPos& parent, uint16_t mv) {
    // every lane builds the child (cheap, uniform), then the warp generates its legal moves cooperatively
    DPos child = make_move(parent, mv);
    int n = 0;
    const GenInfo gi = warp_gen_legal(child, x.sh->moves, x.lane, n);
    int term = 0;
    if (n == 0) term = gi.checkers ? 2 : 1;
    else if (insufficient_material(child)) term = 1;
    set_key_bits(child, gi.has_legal_ep);
    if (x.lane == 0) {
        x.sh->child = child;
        x.sh->n_moves = n;
        x.sh->term = term;
    }
    __syncwarp();
}

// chess.rs:52-60: pos_count[child] (this occurrence included) reaches REPETITIONS, or a move counter hits its limit.
// Candidates are the positions with the same side to move since the last irreversible move: they live on the
// search path (depth >= 1) or in the game history.  `depth_child` = edges from the root to the child, `path` = the
// descent that reached it (entries as in SearchPtrs::path).
__device__ __forceinline__ bool draw_by_rules(Ctx& x, const uint2* path, const DPos& child, int depth_child) {
    const int hm = meta_halfmoves(child.meta);
    if (hm >= x.prm.num_halfmoves || meta_fullmoves(child.meta) >= x.prm.num_fullmoves) return true;
    const int root_v = (int)x.c.hist_len - 1;          // virtual index of the root
    const int v = root_v + depth_child;
    int matches = 0;
    const int n_cand = hm >> 1;
    for (int k0 = 0; k0 < n_cand; k0 += 32) {
        const int k = k0 + x.lane + 1;
        bool eq = false;
        const int j = v - 2 * k;
        if (k <= n_cand && j >= 0) {
            const DPos* q;
            if (j > root_v) q = &x.ptr.node_pos[x.nbase + (path[j - root_v].x & 0xFFFF)];
            else q = &x.ptr.hist[(size_t)x.g * HIST_CAP + j];
            eq = same_position_key(*q, child);
        }
        matches += __popc(__ballot_sync(0xffffffffu, eq));
    }
    return matches + 1 >= x.prm.repetitions;
}

// tree.rs:272-289 on the edge list.  The reference draws one component per legal move INCLUDING the three
// under-promotion duplicates that share a policy index with the queen promotion; edges keep one entry per index,
// so a queen-promotion edge receives four consecutive components.
__device__ void apply_noise(Ctx& x, int node, u64 game_id, u64 ply) {
    const size_t off = x.ebase + x.ptr.node_edge_off[x.nbase + node];
    const int L = x.ptr.node_nedges[x.nbase + node], n = x.ptr.node_nmoves[x.nbase + node];
    if (n < 2) return;
    for (int i = x.lane; i < n; i += 32) x.sh->gam[i] = gamma_sample(x.prm.seed, game_id, ply, 1000 + (u64)i, (double)x.prm.alpha);
    __syncwarp();
    double sum = 0.0;
    if (x.lane == 0) for (int i = 0; i < n; i++) sum = sum + x.sh->gam[i];
    sum = __shfl_sync(0xffffffffu, sum, 0);
    for (int i = x.lane; i < n; i += 32) x.sh->fval[i] = (float)(x.sh->gam[i] / sum);
    // component offset of every edge
    if (x.lane == 0) {
        int comp = 0;
        for (int e = 0; e < L; e++) {
            x.sh->sidx[e] = (uint16_t)comp;
            comp += (((x.ptr.edge_mv[off + e] >> 12) & 7) == 4) ? 4 : 1;
        }
    }
    __syncwarp();
    const float keep = __fsub_rn(1.0f, x.prm.eps);
    for (int e = x.lane; e < L; e += 32) {
        float p = __fmul_rn(x.ptr.edge_P[off + e], keep);
        const int c0 = x.sh->sidx[e];
        const int reps = (((x.ptr.edge_mv[off + e] >> 12) & 7) == 4) ? 4 : 1;
        for (int r = 0; r < reps; r++) p = __fadd_rn(p, __fmul_rn(x.prm.eps, x.sh->fval[c0 + r]));
        x.ptr.edge_P[off + e] = p;
    }
    __syncwarp();
}

// Creates a tree node from sh->child / sh->moves (MCTree::new, tree.rs:84-104) without priors.
// Returns the node id or -1 on pool exhaustion.
__device__ __forceinline__ int create_node(Ctx& x, int depth) {
    const int n = x.sh->n_moves;
    int L = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + x.lane;
        bool keep = false;
        if (i < n) { int pr = (x.sh->moves[i] >> 12) & 7; keep = pr == 0 || pr == 4; }
        L += __popc(__ballot_sync(0xffffffffu, keep));
    }
    if ((int)x.c.n_nodes >= x.prm.node_cap || (int)x.c.n_edges + L > x.prm.edge_cap) return -1;
    const int node = (int)x.c.n_nodes;
    const uint32_t eoff = x.c.n_edges;
    const int turn = meta_turn(x.sh->child.meta);
    int written = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + x.lane;
        bool keep = false;
        uint16_t mv = 0;
        if (i < n) { mv = x.sh->moves[i]; int pr = (mv >> 12) & 7; keep = pr == 0 || pr == 4; }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const size_t e = x.ebase + eoff + written + __popc(bal & ((1u << x.lane) - 1));
            x.ptr.edge_mv[e] = (uint32_t)mv | ((uint32_t)move_to_index(mv, turn) << 16);
            x.ptr.edge_N[e] = 0.0f;
            x.ptr.edge_W[e] = 0.0f;
            x.ptr.edge_P[e] = 0.0f;
            x.ptr.edge_link[e] = EDGE_NO_CHILD;
        }
        written += __popc(bal);
    }
    if (x.lane == 0) {
        const size_t ni = x.nbase + node;
        x.ptr.node_pos[ni] = x.sh->child;
        x.ptr.node_edge_off[ni] = eoff;
        x.ptr.node_nedges[ni] = (uint16_t)L;
        x.ptr.node_nmoves[ni] = (uint16_t)n;
        x.ptr.node_depth[ni] = (uint16_t)depth;
    }
    x.c.n_nodes++;
    x.c.n_edges += L;
    x.new_link = (unsigned long long)node | ((unsigned long long)L << 16) | ((unsigned long long)eoff << 24);
    __syncwarp();
    return node;
}

// Request routing of az_search_networks: game g's requests go to the range of network net[g] (network 0 from slot 0, network 1
// from slot base1), each range with its own counter
struct NetRoute {
    const uint8_t* net;   // [G]
    int* counts;          // [AZ_MAX_NETWORKS]
    int base1;
};

// Queues the position in sh->child (the node create_node made last: its edge range is in x.new_link) for evaluation;
// returns the batch slot.  ROUTE: the slot is taken in the range of the game's network (rt).
template <bool ROUTE = false>
__device__ __forceinline__ int submit_request(Ctx& x, int node, const NetRoute* rt = nullptr) {
    int slot = 0;
    if (x.lane == 0) {
        if constexpr (ROUTE) {
            const int s = rt->net[x.g];
            slot = (s ? rt->base1 : 0) + atomicAdd(rt->counts + s, 1);
        } else {
            slot = atomicAdd(x.ptr.batch_count, 1);
        }
    }
    slot = __shfl_sync(0xffffffffu, slot, 0);
    const DPos child = x.sh->child;
    if (x.lane == 0) {
        x.ptr.req_pos[slot] = child;
        (void)node;
        x.ptr.req_edge_off[slot] = (unsigned long long)(x.ebase + (size_t)(x.new_link >> 24));
        x.ptr.req_nedges[slot] = (int)((x.new_link >> 16) & 0xFF);
    }
    if (x.prm.fp32_planes) {
        const u64 occ = occupied(child);
        const u64 ours = meta_turn(child.meta) == 0 ? child.white : occ ^ child.white;
        const int pep = pseudo_legal_ep(child);
        float* out = x.ptr.req_f32 + (size_t)slot * (AZ_NUM_PLANES * 64);
        for (int e = x.lane; e < AZ_NUM_PLANES * 64; e += 32) out[e] = plane_value(child, e >> 6, e & 63, pep, ours, occ ^ ours);
    } else {
        encode_bf16_warp(child, x.ptr.req_bf16 + (size_t)slot * 64 * x.prm.plane_ch, x.lane, x.prm.plane_ch);
    }
    if (x.lane == 0) x.st_evals++;
    return slot;
}

// W[a] += v ; N[a] += 1 along the stored path, leaf parent first (tree.rs:197-206).  `leaf_value` is what
// expand() returned (the child's point of view).  `spec` (nullable): this lane's path entry requested before the control block
// was known (levels 0..31), which takes one dependent load out of the chain ctl -> path -> edge.
__device__ __forceinline__ void backup(Ctx& x, float leaf_value, int path_len, const uint2* spec = nullptr) {
    for (int i0 = 0; i0 < path_len; i0 += 32) {
        const int i = i0 + x.lane;
        if (i < path_len) {
            const uint2 pe = (spec && i0 == 0) ? *spec : x.ptr.path[(size_t)x.g * x.prm.node_cap + i];
            const size_t e = x.ebase + pe.y;
            // levels above the leaf's parent: the sign flips once per level
            const int up = path_len - 1 - i;
            const float v = (up & 1) ? leaf_value : -leaf_value;
            x.ptr.edge_W[e] = __fadd_rn(x.ptr.edge_W[e], v);
            x.ptr.edge_N[e] = __fadd_rn(x.ptr.edge_N[e], 1.0f);
        }
    }
    __syncwarp();
}

// One PUCT descent from the root (tree.rs:180-202).  Fills the path and returns the leaf: its parent's node id, position and
// depth, and the chosen edge (pool index, wire move).
// The walk costs ONE dependent memory round trip per level: an edge carries its child's id together with the child's edge
// range (edge_link), the root's range is in the control block, and the chosen edge's move and every visited node's position
// (the leaf's parent needs it) are requested in the same batch of loads.
// total_visits (tree.rs:184: the sum of the node's visit counts) needs no loads at all: every simulation that passes through
// a node increments exactly one of its edges, and the simulations passing through a node are the visits of the edge leading
// into it minus the one that created it -- so total_visits + 1 is exactly that edge's N (at the root: simulations done + 1),
// the same integer in f32 the reference obtains by summing.
__device__ __forceinline__ void select_leaf(Ctx& x, int& leaf_node, size_t& leaf_pe, uint32_t& leaf_mv, int& depth, DPos& parent) {
    int node = 0;
    depth = 0;
    uint32_t eoff = 0;
    int L = (int)((x.c.flags >> 8) & 0xFF);
    float total = __fadd_rn((float)x.c.sims_done, 1.0f);
    for (;;) {
        const size_t off = x.ebase + eoff;
        u64 here = 0;   // lanes 0..7: the eight words of this node's position
        if (x.lane < 8) here = reinterpret_cast<const u64*>(&x.ptr.node_pos[x.nbase + node])[x.lane];
        const float sq = __fsqrt_rn(total);
        float best = -INFINITY;
        int best_e = 0x7FFFFFFF;
        // this lane's candidate: link, move and visit count of its best edge (lane 0 starts with edge 0 for the NaN fallback)
        u64 my_k = EDGE_NO_CHILD;
        uint32_t my_m = 0;
        float my_n = 0.0f;
        for (int e = x.lane; e < L; e += 32) {
            const float P = x.ptr.edge_P[off + e], N = x.ptr.edge_N[off + e], W = x.ptr.edge_W[off + e];
            const u64 K = x.ptr.edge_link[off + e];
            const uint32_t M = x.ptr.edge_mv[off + e];
            const float u = __fdiv_rn(__fmul_rn(__fmul_rn(x.prm.c_puct, P), sq), __fadd_rn(1.0f, N));
            const float q = N > 0.0f ? __fdiv_rn(W, N) : 0.0f;
            const float v = __fadd_rn(q, u);
            if (v > best) { best = v; best_e = e; my_k = K; my_m = M; my_n = N; }
            else if (e == x.lane) { my_k = K; my_m = M; my_n = N; }   // seed: lane 0 must hold edge 0 for the NaN fallback
        }
        // warp argmax over (score, edge): larger value wins, ties go to the earlier move (strict '>' in list order)
        for (int d = 16; d; d >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, d);
            const int oe = __shfl_xor_sync(0xffffffffu, best_e, d);
            if (ov > best || (ov == best && oe < best_e)) { best = ov; best_e = oe; }
        }
        if (best_e == 0x7FFFFFFF) best_e = 0;  // every score was NaN / -inf: the reference keeps max_index = 0 (first move)
        // the winning edge belongs to lane best_e % 32, whose candidate it is
        const int owner = best_e & 31;
        const u64 best_k = shfl_u64(my_k, owner);
        const uint32_t best_m = __shfl_sync(0xffffffffu, my_m, owner);
        const float best_n = __shfl_sync(0xffffffffu, my_n, owner);
        if (x.lane == 0) {
            x.ptr.path[(size_t)x.g * x.prm.node_cap + depth] =
                make_uint2((uint32_t)node | ((uint32_t)best_e << 16), eoff + (uint32_t)best_e);
            x.st_edges += L;
        }
        if (best_k == EDGE_NO_CHILD) {
            leaf_node = node; leaf_pe = off + best_e; leaf_mv = best_m;
            parent.pawn = shfl_u64(here, 0); parent.knight = shfl_u64(here, 1); parent.bishop = shfl_u64(here, 2);
            parent.rook = shfl_u64(here, 3); parent.queen = shfl_u64(here, 4); parent.king = shfl_u64(here, 5);
            parent.white = shfl_u64(here, 6); parent.meta = shfl_u64(here, 7);
            __syncwarp();
            return;
        }
        node = (int)(best_k & 0xFFFF);
        L = (int)((best_k >> 16) & 0xFF);
        eoff = (uint32_t)(best_k >> 24);
        total = best_n;   // = (visits through this child) + 1
        depth++;
    }
}


// ------------------------------------------------------------------------------------------- evaluation cache
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// entries are reused after eviction, so their contents are read from L2 (ld.cg), never from a possibly stale L1 line
__device__ __forceinline__ bool cache_key_equal(const CacheEntry* e, const DPos* key, int lane) {
    bool eq = true;
    if (lane < 8) eq = __ldcg(reinterpret_cast<const u64*>(&e->key) + lane) == reinterpret_cast<const u64*>(key)[lane];
    return __all_sync(0xffffffffu, eq);
}
constexpr int CACHE_PROBES = 8;
__device__ __forceinline__ uint32_t cache_tag(u64 h) { return (uint32_t)(h >> 46); }   // 18 bits
// whole warp; the key is in sh->key.  Returns the slot holding it (and the state word observed) or -1.
__device__ __forceinline__ int cache_lookup(Ctx& x, u64 h, uint32_t& seen) {
    const uint32_t tag = cache_tag(h);
    for (int probe = 0; probe < CACHE_PROBES; probe++) {
        const uint32_t slot = (uint32_t)(h + probe) & x.prm.cache_mask;
        const uint32_t s = ld_acquire_u32(&x.ptr.cache_state[slot]);
        if (s == 0) return -1;   // slots are replaced, never emptied: an empty slot ends every probe sequence
        if ((s & 3) == 2 && (s >> 14) == tag && cache_key_equal(&x.ptr.cache_entry[slot], &x.sh->key, x.lane)) { seen = s; return (int)slot; }
    }
    return -1;
}
// whole warp, after the entry's contents were copied: true if the slot still holds what cache_lookup saw
__device__ __forceinline__ bool cache_validate(Ctx& x, int slot, uint32_t seen) {
    __threadfence();   // the copies above are ordered before the second look at the state word
    __syncwarp();
    const uint32_t s2 = *reinterpret_cast<volatile uint32_t*>(&x.ptr.cache_state[slot]);
    const bool ok = __all_sync(0xffffffffu, ((s2 ^ seen) & ~CACHE_EPOCH_MASK) == 0);
    if (ok && x.lane == 0 && ((seen >> 2) & 63) != x.prm.cache_epoch)   // a hit keeps the entry young (failure is harmless)
        atomicCAS(&x.ptr.cache_state[slot], seen, (seen & ~CACHE_EPOCH_MASK) | (x.prm.cache_epoch << 2));
    return ok;
}
// whole warp: publishes (sh->key -> priors of `node`, value) unless it is already there; a full neighbourhood gives up
// its stalest entry (not inserted or hit for CACHE_MIN_AGE epochs or more)
__device__ __forceinline__ void cache_insert(Ctx& x, u64 h, int node, float value) {
    const uint32_t tag = cache_tag(h);
    const size_t off = x.ebase + x.ptr.node_edge_off[x.nbase + node];
    const int L = x.ptr.node_nedges[x.nbase + node];
    int target = -1, victim = -1, victim_age = CACHE_MIN_AGE - 1;
    uint32_t target_seq = 0, victim_s = 0;
    for (int probe = 0; probe < CACHE_PROBES && target < 0; probe++) {
        const uint32_t slot = (uint32_t)(h + probe) & x.prm.cache_mask;
        const uint32_t s = ld_acquire_u32(&x.ptr.cache_state[slot]);
        if ((s & 3) == 2 && (s >> 14) == tag && cache_key_equal(&x.ptr.cache_entry[slot], &x.sh->key, x.lane)) return;
        if (s == 0) {
            uint32_t old = 1;
            if (x.lane == 0) old = atomicCAS(&x.ptr.cache_state[slot], 0u, 1u);
            old = __shfl_sync(0xffffffffu, old, 0);
            if (old == 0) target = (int)slot;
        } else if ((s & 3) == 2) {
            const int age = (int)((x.prm.cache_epoch - (s >> 2)) & 63);
            if (age > victim_age) { victim = (int)slot; victim_age = age; victim_s = s; }
        }
    }
    if (target < 0) {
        if (victim < 0) return;
        uint32_t old = ~victim_s;
        if (x.lane == 0) old = atomicCAS(&x.ptr.cache_state[victim], victim_s, (victim_s & ~3u) | 1u);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old != victim_s) return;   // somebody else hit or replaced it meanwhile
        target = victim;
        target_seq = ((victim_s >> 8) + 1) & 63;
        if (x.lane == 0) x.st_evict++;
    }
    CacheEntry* e = &x.ptr.cache_entry[target];
    if (x.lane < 4) reinterpret_cast<uint4*>(&e->key)[x.lane] = reinterpret_cast<const uint4*>(&x.sh->key)[x.lane];
    if (x.lane == 4) { e->value = value; e->n_priors = (uint32_t)L; }
    for (int i = x.lane; i < L; i += 32) e->prior[i] = x.ptr.edge_P[off + i];
    __threadfence();
    __syncwarp();
    if (x.lane == 0) atomicExch(&x.ptr.cache_state[target], (tag << 14) | (target_seq << 8) | (x.prm.cache_epoch << 2) | 2u);
}

__device__ __forceinline__ void setup_root_from_shared(Ctx& x) {
    // fresh tree whose root is sh->child / sh->moves (priors are written by the caller)
    x.c.n_nodes = 0; x.c.n_edges = 0; x.c.sims_done = 0; x.c.max_depth = 0; x.c.pending_node = -1;
    create_node(x, 0);
    x.c.flags = (x.c.flags & 0xFFFF00FFu) | ((uint32_t)((x.new_link >> 16) & 0xFF) << 8);   // the root's edge count (its offset is 0)
}

// Start position, shared start-position priors, fresh noise (training.rs:352-361) -- or, when the generation's budget of
// games is used up (az_selfplay_begin_n), the slot goes idle.
__device__ void start_new_game(Ctx& x) {
    unsigned long long gid = 0;
    if (x.lane == 0) gid = atomicAdd(&x.ptr.counters->next_game_id, 1ULL);
    gid = __shfl_sync(0xffffffffu, gid, 0);
    if (x.prm.last_game_id != 0 && gid >= x.prm.last_game_id) { x.c.status = 1; x.c.n_samples = 0; return; }
    x.c.game_id = gid; x.c.ply = 0; x.c.n_samples = 0; x.c.hist_len = 1;
    if (x.lane == 0) {
        DPos s = start_dpos();
        ListSink sink{x.sh->moves, 0};
        GenInfo gi = gen_legal(s, sink);
        set_key_bits(s, gi.has_legal_ep);
        x.sh->child = s; x.sh->n_moves = sink.n; x.sh->term = 0;
        x.ptr.hist[(size_t)x.g * HIST_CAP] = s;
    }
    __syncwarp();
    setup_root_from_shared(x);
    const int L0 = x.ptr.node_nedges[x.nbase];
    for (int e = x.lane; e < L0; e += 32) x.ptr.edge_P[x.ebase + e] = x.ptr.start_prior[e];
    __syncwarp();
    apply_noise(x, 0, x.c.game_id, 0);
}

// The game in this slot is over and `scale` = result x decay (training.rs:332-335).  Its staged EpisodeSteps move to the
// sample queue only if ALL of them fit (the counter never covers unwritten slots); otherwise the game parks (status 4)
// with its samples staged and tries again in the next wave, after the host has drained.  Nothing is ever dropped.
__device__ void finish_game(Ctx& x, float scale) {
    const int ns = (int)x.c.n_samples;
    unsigned long long base = 0;
    int ok = 0;
    if (x.lane == 0) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&x.ptr.counters->samples_out);
        for (;;) {
            if (cur + (unsigned long long)ns > (unsigned long long)x.prm.sample_cap) break;
            const unsigned long long prev = atomicCAS(&x.ptr.counters->samples_out, cur, cur + (unsigned long long)ns);
            if (prev == cur) { base = cur; ok = 1; break; }
            cur = prev;
        }
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (!ok) {
        x.c.status = 4;
        x.c.park_scale = __float_as_uint(scale);
        return;
    }
    x.c.status = 0;
    az_sample* src = x.ptr.game_samples + (size_t)x.g * MAX_SAMPLE_PLIES;
    for (int i = x.lane; i < ns; i += 32) src[i].final_value = __fmul_rn(src[i].final_value, scale);
    __syncwarp();
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(x.ptr.out_samples + base);
    const int n16 = ns * (int)(sizeof(az_sample) / 16);
    for (int i = x.lane; i < n16; i += 32) d4[i] = s4[i];
    if (x.lane == 0) x.st_games++;
    start_new_game(x);
}

// training.rs:303-335 for one finished search: record the EpisodeStep, pick the move, advance or finish the game.
__device__ void move_step(Ctx& x) {
    const size_t ni = x.nbase;  // root
    const size_t off = x.ebase + x.ptr.node_edge_off[ni];
    const int L = x.ptr.node_nedges[ni];
    const DPos root = x.ptr.node_pos[ni];
    const int turn = meta_turn(root.meta);
    // ---- sort the visited edges by policy index (the reference works on the dense 4096-vector)
    int nv = 0;
    for (int e0 = 0; e0 < L; e0 += 32) {
        const int e = e0 + x.lane;
        int rank = -1;
        if (e < L && x.ptr.edge_N[off + e] > 0.0f) {
            const uint32_t my = x.ptr.edge_mv[off + e] >> 16;
            rank = 0;
            for (int o = 0; o < L; o++)
                if (x.ptr.edge_N[off + o] > 0.0f && (x.ptr.edge_mv[off + o] >> 16) < my) rank++;
            x.sh->sidx[rank] = (uint16_t)e;
        }
        nv += __popc(__ballot_sync(0xffffffffu, rank >= 0));
    }
    __syncwarp();
    // ---- EpisodeStep
    const uint32_t sidx_slot = x.c.n_samples;
    az_sample* smp = nullptr;
    if (sidx_slot < MAX_SAMPLE_PLIES) {
        smp = x.ptr.game_samples + (size_t)x.g * MAX_SAMPLE_PLIES + sidx_slot;
        for (int i = x.lane; i < AZ_MAX_MOVES; i += 32) {  // unused tail entries are zero (deterministic records)
            uint16_t si = 0, sc = 0;
            if (i < nv) {
                const size_t e = off + x.sh->sidx[i];
                si = (uint16_t)(x.ptr.edge_mv[e] >> 16);
                sc = (uint16_t)x.ptr.edge_N[e];
            }
            smp->index[i] = si;
            smp->count[i] = sc;
        }
    }
    // ---- improved policy weights (tree.rs:173-175): w = visits^(1/T) per visited index, summed in index order (the zeros of
    // the reference's dense vector add nothing); T = 1 gives w = visits and the sum = S exactly
    for (int i = x.lane; i < nv; i += 32) x.sh->fval[i] = pow_inv_temperature(x.ptr.edge_N[off + x.sh->sidx[i]], x.prm.inv_temperature);
    __syncwarp();
    // ---- action (training.rs:310-321)
    int action_edge = 0;
    if (x.lane == 0) {
        float S = 0.0f;  // weights_sum
        for (int i = 0; i < nv; i++) S = __fadd_rn(S, x.sh->fval[i]);
        if ((uint32_t)meta_fullmoves(root.meta) >= x.prm.anneal) {
            float best = -1.0f;  // Iterator::max_by keeps the LAST maximum in index order
            for (int i = 0; i < nv; i++) {
                const float w = __fdiv_rn(x.sh->fval[i], S);
                if (w >= best) { best = w; action_edge = x.sh->sidx[i]; }
            }
        } else {
            float total = 0.0f;  // WeightedIndex: cumulative f32 weights in index order
            for (int i = 0; i < nv; i++) total = __fadd_rn(total, __fdiv_rn(x.sh->fval[i], S));
            const u64 h = rng_u64(x.prm.seed, x.c.game_id, x.c.ply, 1, 0);
            const float u = __fmul_rn((float)(h >> 40), 1.0f / 16777216.0f);
            const float chosen = __fmul_rn(u, total);
            float cum = 0.0f;
            action_edge = nv > 0 ? x.sh->sidx[nv - 1] : 0;
            for (int i = 0; i < nv; i++) {
                cum = __fadd_rn(cum, __fdiv_rn(x.sh->fval[i], S));
                if (cum > chosen) { action_edge = x.sh->sidx[i]; break; }
            }
        }
    }
    action_edge = __shfl_sync(0xffffffffu, action_edge, 0);
    const uint32_t amv = x.ptr.edge_mv[off + action_edge];
    if (smp && x.lane == 0) {
        smp->position = dpos_to_wire(root);
        smp->final_value = turn == 0 ? 1.0f : -1.0f;
        smp->search_depth = (int32_t)x.c.max_depth;
        smp->game_id = x.c.game_id;
        smp->ply = x.c.ply;
        smp->action = (uint16_t)(amv >> 16);
        smp->n_visits = (uint16_t)nv;
        x.st_pos++;
        x.st_sdepth += x.c.max_depth;
    }
    x.c.n_samples = min(x.c.n_samples + 1, (uint32_t)MAX_SAMPLE_PLIES);
    // ---- play it (chess.rs:36-63)
    const unsigned long long child_link = x.ptr.edge_link[off + action_edge];
    const int child_node = child_link == EDGE_NO_CHILD ? -1 : (int)(child_link & 0xFFFF);
    lane0_make_child(x, root, (uint16_t)(amv & 0xFFFF));
    int term = x.sh->term;
    if (term == 0 && draw_by_rules(x, x.ptr.path + (size_t)x.g * x.prm.node_cap, x.sh->child, 1)) term = 1;
    if (term == 0) {
        // traverse_new (tree.rs:239-256): keep the child's priors, drop everything else, fresh noise
        float keepP[7];
        int Lc = 0;
        if (child_node >= 0) {
            const size_t coff = x.ebase + x.ptr.node_edge_off[x.nbase + child_node];
            Lc = x.ptr.node_nedges[x.nbase + child_node];
#pragma unroll
            for (int k = 0; k < 7; k++) { int e = x.lane + 32 * k; keepP[k] = e < Lc ? x.ptr.edge_P[coff + e] : 0.0f; }
        } else {
            x.c.status = 3;  // a move with visits but no stored child must be terminal
        }
        __syncwarp();
        if (x.lane == 0 && x.c.hist_len < HIST_CAP) x.ptr.hist[(size_t)x.g * HIST_CAP + x.c.hist_len] = x.sh->child;
        x.c.hist_len = min(x.c.hist_len + 1, (uint32_t)HIST_CAP);
        x.c.ply++;
        setup_root_from_shared(x);
#pragma unroll
        for (int k = 0; k < 7; k++) { int e = x.lane + 32 * k; if (e < Lc) x.ptr.edge_P[x.ebase + e] = keepP[k]; }
        __syncwarp();
        apply_noise(x, 0, x.c.game_id, x.c.ply);
        return;
    }
    // ---- game over: back-fill final_value (training.rs:332-335), publish the samples, start a new game
    const float mover = turn == 0 ? 1.0f : -1.0f;
    const float result = term == 1 ? 0.0f : mover;
    const float decay = __fsub_rn(1.0f, __fdiv_rn((float)meta_fullmoves(x.sh->child.meta), __fmul_rn(2.0f, (float)x.prm.num_fullmoves)));
    finish_game(x, __fmul_rn(result, decay));
}

// ------------------------------------------------------------------------------------------- cold paths of the wave kernel
// A finished search (once per S waves and game), a parked game and root noise are rare; compiled inline they sit in the middle
// of the hot instruction stream of a 20,000-instruction kernel whose warps stall on instruction fetch (ncu: "no instructions"
// is the second stall reason, profiles/r2_advance_v1_full.md).  They are real calls instead.  The game's control block goes in
// and out BY VALUE so that the hot path's copy stays in registers (a reference would pin it in local memory).
struct ColdOut {
    GameCtl c;
    unsigned int st_pos, st_games, st_sdepth;
};
__device__ __forceinline__ void absorb(Ctx& x, const ColdOut& o) {
    x.c = o.c; x.st_pos += o.st_pos; x.st_games += o.st_games; x.st_sdepth += o.st_sdepth;
}
__device__ __noinline__ ColdOut move_step_cold(const SearchParams* prm, const SearchPtrs* ptr, WarpShared* sh, int g, GameCtl c) {
    Ctx x = make_ctx(*prm, *ptr, sh, g, c);
    move_step(x);
    return ColdOut{x.c, x.st_pos, x.st_games, x.st_sdepth};
}
__device__ __noinline__ ColdOut finish_game_cold(const SearchParams* prm, const SearchPtrs* ptr, WarpShared* sh, int g, GameCtl c) {
    Ctx x = make_ctx(*prm, *ptr, sh, g, c);
    finish_game(x, __uint_as_float(c.park_scale));
    return ColdOut{x.c, x.st_pos, x.st_games, x.st_sdepth};
}
__device__ __noinline__ void root_noise_cold(const SearchParams* prm, const SearchPtrs* ptr, WarpShared* sh, int g, GameCtl c) {
    Ctx x = make_ctx(*prm, *ptr, sh, g, c);
    apply_noise(x, 0, c.game_id, c.noise_ply);
}

// ------------------------------------------------------------------------------------------- the wave kernel
#ifdef AZ_ADV_TIMING
#define ADV_T0() long long t_prev = clock64(), t_start = t_prev; unsigned long long t_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define ADV_T(k) do { const long long t_now = clock64(); t_acc[k] += (unsigned long long)(t_now - t_prev); t_prev = t_now; } while (0)
#else
#define ADV_T0() do { } while (0)
#define ADV_T(k) do { } while (0)
#endif
// MINB = resident groups of four warps per SM the register allocation is bounded for: the kernel is a chain of dependent global loads
// per game, so resident warps (latency hiding) are worth more than registers (AZ_ADV_MINB selects, see launch below)
template <int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB * 4 / WARPS) k_advance(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= prm.n_games) return;
    // the path of the pending simulation is requested together with the control block (its address needs only g)
    const uint2 path_spec = ptr.path[(size_t)g * prm.node_cap + min((int)(threadIdx.x & 31), prm.node_cap - 1)];
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, ptr.ctl[g]);
    if (g == 0 && x.lane == 0 && ptr.batch_zero) *ptr.batch_zero = 0;   // the other wave parity's request counter (see run_wave)
    if (x.c.status != 0 && x.c.status != 4) return;
    if (!prm.consume && x.c.pending_node >= 0) return;   // extra pass: this game already waits for the network

    ADV_T0();
    // ---- 0. game over, samples staged: publish now if the host has drained the queue, else stay parked
    if (x.c.status == 4) absorb(x, finish_game_cold(&prm, &ptr, x.sh, g, x.c));
    const bool runnable = x.c.status == 0;
    // ---- 1. the evaluation requested in the previous wave has arrived
    if (runnable && x.c.pending_node >= 0) {
        const int node = x.c.pending_node, slot = x.c.pending_slot;
        const size_t off = x.ebase + ptr.node_edge_off[x.nbase + node];
        const int L = ptr.node_nedges[x.nbase + node];
        if (!prm.priors_scattered) {
            const float* pol = ptr.res_policy + (size_t)slot * AZ_ACTION_SPACE;
            for (int e = x.lane; e < L; e += 32) ptr.edge_P[off + e] = pol[ptr.edge_mv[off + e] >> 16];
        }
        __syncwarp();
        if (prm.cache_mask && prm.mode == 1) {  // cache.insert (training.rs:413)
            if (x.lane == 0) x.sh->key = fen_key_of(ptr.node_pos[x.nbase + node]);
            __syncwarp();
            cache_insert(x, fen_key_hash(x.sh->key), node, ptr.res_value[slot]);
        }
        if (node == 0) {  // MCTree::init (tree.rs:37-64): root priors, optional noise, no backup
            if (x.c.flags & 1) root_noise_cold(&prm, &ptr, x.sh, g, x.c);
        } else {
            backup(x, ptr.res_value[slot], (int)x.c.path_len, &path_spec);
            x.c.sims_done++;
            if (x.lane == 0) x.st_sims++;
        }
        x.c.pending_node = -1;
    }

    ADV_T(0);
    // ---- 2. run until the network is needed again
    for (int iter = 0; runnable && iter < prm.max_iters; iter++) {
        if ((int)x.c.sims_done >= prm.S) {
            if (prm.mode == 0) { x.c.status = 1; break; }
            absorb(x, move_step_cold(&prm, &ptr, x.sh, g, x.c));
            ADV_T(6);
            if (x.c.status != 0) break;   // idle (generation complete), parked (sample queue full) or an error
            continue;
        }
        int node, depth;
        size_t pe;
        uint32_t leaf_mv;
        DPos parent;
        select_leaf(x, node, pe, leaf_mv, depth, parent);
        ADV_T(1);
        lane0_make_child(x, parent, (uint16_t)(leaf_mv & 0xFFFF));
        int term = x.sh->term;
        ADV_T(2);
        if (term == 0 && draw_by_rules(x, ptr.path + (size_t)g * prm.node_cap, x.sh->child, depth + 1)) term = 1;
        ADV_T(3);
        if (x.lane == 0) x.st_depth += depth + 1;
        if (term != 0) {
            // Draw -> 0.0, decisive -> -1.0 from the child's side (tree.rs:233-234); nothing is stored
            backup(x, term == 1 ? 0.0f : -1.0f, depth + 1);
            x.c.sims_done++;
            if (x.lane == 0) { x.st_sims++; x.st_term++; }
            continue;
        }
        const int child = create_node(x, depth + 1);
        ADV_T(4);
        if (child < 0) { x.c.status = 2; if (x.lane == 0) atomicAdd(&ptr.counters->errors, 1ULL); break; }
        if (x.lane == 0) ptr.edge_link[pe] = x.new_link;
        x.c.max_depth = max(x.c.max_depth, (uint32_t)(depth + 1));
        if (prm.cache_mask && prm.mode == 1) {  // cache.get (tree.rs:214-218): a hit needs no network evaluation
            if (x.lane == 0) x.sh->key = fen_key_of(x.sh->child);
            __syncwarp();
            uint32_t seen = 0;
            const int slot = cache_lookup(x, fen_key_hash(x.sh->key), seen);
            if (slot >= 0) {
                const CacheEntry* ce = &ptr.cache_entry[slot];
                const size_t coff = x.ebase + ptr.node_edge_off[x.nbase + child];
                const int Lc = ptr.node_nedges[x.nbase + child];
                for (int e = x.lane; e < Lc; e += 32) ptr.edge_P[coff + e] = __ldcg(&ce->prior[e]);
                const float cv = __ldcg(&ce->value);
                if (cache_validate(x, slot, seen)) {   // else: the entry was being replaced; evaluate as a miss (edge_P is overwritten)
                    backup(x, cv, depth + 1);
                    x.c.sims_done++;
                    if (x.lane == 0) { x.st_sims++; x.st_hits++; }
                    continue;
                }
            }
        }
        x.c.pending_node = child;
        x.c.pending_slot = submit_request(x, child);
        x.c.path_len = depth + 1;
        ADV_T(5);
        break;
    }

    if (x.lane == 0) {
        ptr.ctl[g] = x.c;
        // statistics: same field order as Counters; 64 stripes keep 4096 warps from queueing on eight addresses
        unsigned long long* ct = ptr.stats + (size_t)(blockIdx.x & (STAT_STRIPES - 1)) * STAT_WIDTH;
        if (x.st_sims) atomicAdd(&ct[0], (unsigned long long)x.st_sims);
        if (x.st_pos) atomicAdd(&ct[1], (unsigned long long)x.st_pos);
        if (x.st_evals) atomicAdd(&ct[2], (unsigned long long)x.st_evals);
        if (x.st_hits) atomicAdd(&ct[3], (unsigned long long)x.st_hits);
        if (x.st_term) atomicAdd(&ct[4], (unsigned long long)x.st_term);
        if (x.st_games) atomicAdd(&ct[5], (unsigned long long)x.st_games);
        if (x.st_depth) atomicAdd(&ct[6], (unsigned long long)x.st_depth);
        if (x.st_edges) atomicAdd(&ct[7], (unsigned long long)x.st_edges);
        if (x.st_evict) atomicAdd(&ct[16], (unsigned long long)x.st_evict);
        if (x.st_sdepth) atomicAdd(&ct[17], (unsigned long long)x.st_sdepth);
#ifdef AZ_ADV_TIMING
        t_acc[7] = (unsigned long long)(clock64() - t_start);
        for (int k = 0; k < 8; k++) atomicAdd(&ct[8 + k], t_acc[k]);
        atomicAdd(&ct[24 + min(15, (int)(t_acc[7] >> 12))], 1ULL);
#endif
    }
}

// Root set-up for az_search (MCTree::init): node 0 from the given position, evaluation pending.
template <bool ROUTE>
__device__ __forceinline__ void init_search_body(const SearchParams& prm, const SearchPtrs& ptr, const az_position* __restrict__ roots,
                                                 const az_position* __restrict__ hist, const uint32_t* __restrict__ hist_off,
                                                 const unsigned long long* __restrict__ noise_ids, const uint32_t* __restrict__ noise_plies,
                                                 const NetRoute& rt) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= prm.n_games) return;
    GameCtl c;
    memset(&c, 0, sizeof c);
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, c);
    x.c.game_id = noise_ids ? noise_ids[g] : 0;
    x.c.noise_ply = noise_plies ? noise_plies[g] : 0;
    x.c.flags = noise_ids ? 1 : 0;
    // history (positions already counted, current root last); key bits need the legal ep square of each entry
    int hl = 1;
    if (hist) {
        const uint32_t h0 = hist_off[g], h1 = hist_off[g + 1];
        int n = (int)(h1 - h0);
        const uint32_t skip = n > HIST_CAP ? n - HIST_CAP : 0;
        n -= skip;
        for (int i = x.lane; i < n; i += 32) {
            DPos q = dpos_from_wire(hist[h0 + skip + i]);
            bool q_ep = false;
            if (meta_ep(q.meta) >= 0) { CountSink t{0}; q_ep = gen_legal(q, t).has_legal_ep; }
            set_key_bits(q, q_ep);
            ptr.hist[(size_t)g * HIST_CAP + i] = q;
        }
        hl = max(n, 1);
    }
    __syncwarp();
    if (x.lane == 0) {
        DPos r = dpos_from_wire(roots[g]);
        ListSink sink{x.sh->moves, 0};
        GenInfo gi = gen_legal(r, sink);
        set_key_bits(r, gi.has_legal_ep);
        x.sh->child = r; x.sh->n_moves = sink.n; x.sh->term = 0;
        if (!hist || hist_off[g + 1] == hist_off[g]) ptr.hist[(size_t)g * HIST_CAP] = r;
    }
    __syncwarp();
    x.c.hist_len = hl;
    setup_root_from_shared(x);
    x.c.pending_node = 0;
    x.c.pending_slot = submit_request<ROUTE>(x, 0, &rt);
    if (x.sh->n_moves == 0) x.c.status = 1;  // nothing to search in a terminal position
    if (x.lane == 0) ptr.ctl[g] = x.c;
}
__global__ void __launch_bounds__(WARPS * 32) k_init_search(SearchParams prm, SearchPtrs ptr, const az_position* __restrict__ roots,
                                                            const az_position* __restrict__ hist, const uint32_t* __restrict__ hist_off,
                                                            const unsigned long long* __restrict__ noise_ids,
                                                            const uint32_t* __restrict__ noise_plies) {
    init_search_body<false>(prm, ptr, roots, hist, hist_off, noise_ids, noise_plies, NetRoute{nullptr, nullptr, 0});
}
// the same with the root's request in the range of its network (az_search_networks)
__global__ void __launch_bounds__(WARPS * 32) k_init_search_nets(SearchParams prm, SearchPtrs ptr, const az_position* __restrict__ roots,
                                                                 const az_position* __restrict__ hist, const uint32_t* __restrict__ hist_off,
                                                                 const unsigned long long* __restrict__ noise_ids,
                                                                 const uint32_t* __restrict__ noise_plies, const NetRoute rt) {
    init_search_body<true>(prm, ptr, roots, hist, hist_off, noise_ids, noise_plies, rt);
}

// Game set-up for self-play (training.rs:352-361): start position, shared priors, Dirichlet noise.
__global__ void __launch_bounds__(WARPS * 32) k_init_selfplay(SearchParams prm, SearchPtrs ptr, unsigned long long first_game_id) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= prm.n_games) return;
    GameCtl c;
    memset(&c, 0, sizeof c);
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, c);
    x.c.game_id = first_game_id + g;
    x.c.hist_len = 1;
    if (x.lane == 0) {
        DPos s = start_dpos();
        ListSink sink{x.sh->moves, 0};
        GenInfo gi = gen_legal(s, sink);
        set_key_bits(s, gi.has_legal_ep);
        x.sh->child = s; x.sh->n_moves = sink.n; x.sh->term = 0;
        ptr.hist[(size_t)g * HIST_CAP] = s;
    }
    __syncwarp();
    setup_root_from_shared(x);
    const int L0 = ptr.node_nedges[x.nbase];
    for (int e = x.lane; e < L0; e += 32) ptr.edge_P[x.ebase + e] = ptr.start_prior[e];
    __syncwarp();
    apply_noise(x, 0, x.c.game_id, 0);
    if (x.lane == 0) ptr.ctl[g] = x.c;
}

// start-position priors from a policy row (the single shared forward of training.rs:344-350)
__global__ void k_start_prior(const float* __restrict__ policy_row, float* __restrict__ start_prior) {
    if (threadIdx.x == 0) {
        DPos s = start_dpos();
        uint16_t mv[AZ_MAX_MOVES];
        ListSink sink{mv, 0};
        gen_legal(s, sink);
        for (int i = 0; i < sink.n && i < 32; i++) start_prior[i] = policy_row[move_to_index(mv[i], 0)];
    }
}

// dense export of the root statistics (Box<[f32; 4096]> visits / scores)
__global__ void k_export_root(SearchParams prm, SearchPtrs ptr, float* __restrict__ visits, float* __restrict__ scores,
                              int32_t* __restrict__ depth) {
    const int g = blockIdx.x;
    float* vo = visits + (size_t)g * AZ_ACTION_SPACE;
    float* so = scores ? scores + (size_t)g * AZ_ACTION_SPACE : nullptr;
    for (int i = threadIdx.x; i < AZ_ACTION_SPACE; i += blockDim.x) { vo[i] = 0.0f; if (so) so[i] = 0.0f; }
    __syncthreads();
    const size_t nb = (size_t)g * prm.node_cap, eb = (size_t)g * prm.edge_cap + ptr.node_edge_off[nb];
    const int L = ptr.node_nedges[nb];
    for (int e = threadIdx.x; e < L; e += blockDim.x) {
        const int idx = ptr.edge_mv[eb + e] >> 16;
        vo[idx] = ptr.edge_N[eb + e];
        if (so) so[idx] = ptr.edge_W[eb + e];
    }
    if (threadIdx.x == 0 && depth) depth[g] = (int32_t)ptr.ctl[g].max_depth;
}

__global__ void k_count_active(SearchParams prm, SearchPtrs ptr, int* out) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < prm.n_games) {
        const uint32_t s = ptr.ctl[g].status;
        if (s == 0) atomicAdd(&out[0], 1);
        if (s == 2 || s == 3) atomicAdd(&out[1], 1);
        if (s == 4) atomicAdd(&out[2], 1);
    }
}

// ------------------------------------------------------------------------------------------- leaf-parallel search (az_search_vl)
// Not in the reference: each root gathers up to K leaves per network round, steering later descents away from the paths
// already taken with a virtual loss (semantics in DESIGN.md section 5).  A wave is k_vl_gather (one warp per root: back up the
// previous batch in leaf order, then descend K times), k_vl_expand (one warp per leaf) and the network.  With K = 1 every
// in-flight count is 0 at every selection and the results are those of az_search.
struct VLPtrs {
    uint32_t* V;          // [G * edge_cap] descents of the current batch through each edge (0 between batches)
    uint2* path;          // [max_batch][node_cap] the descent of leaf g * K + k, entries as in SearchPtrs::path
    int* len;             // [max_batch] edges on that descent
    int* slot;            // [max_batch] request slot of the leaf's evaluation, or -1: terminal, its value is in `value`
    float* value;         // [max_batch]
    int* count;           // [G] leaves of the root's current batch
    unsigned long long* stats;  // [4] leaves gathered, terminal leaves, collisions
    int K;
    float lambda;
};

// lane 0 at the end of a leaf-parallel wave: the leaves of the slot's new batch (what the next wave backs up) and its statistics
__device__ __forceinline__ void vl_publish(const VLPtrs& vl, int g, int n_leaf, int collided) {
    vl.count[g] = n_leaf;
    if (n_leaf) atomicAdd(&vl.stats[0], (unsigned long long)n_leaf);
    if (collided) atomicAdd(&vl.stats[2], 1ULL);
}

// One descent of the gather: PUCT on N' = N + V and W' = W - lambda * V.  `total` is the root's N' (sims done + leaves
// gathered so far + 1).  Writes path[0..depth] and returns the depth of the leaf edge, or -1 when the chosen edge has no child
// but another descent of this batch already ends there (a collision).
__device__ __forceinline__ int vl_descend(Ctx& x, const VLPtrs& vl, uint2* path, float total) {
    int node = 0, depth = 0;
    uint32_t eoff = 0;
    int L = (int)((x.c.flags >> 8) & 0xFF);
    for (;;) {
        const size_t off = x.ebase + eoff;
        const float sq = __fsqrt_rn(total);
        float best = -INFINITY;
        int best_e = 0x7FFFFFFF;
        u64 my_k = EDGE_NO_CHILD;
        float my_n = 0.0f;
        uint32_t my_v = 0;
        for (int e = x.lane; e < L; e += 32) {
            const float P = x.ptr.edge_P[off + e], N = x.ptr.edge_N[off + e], W = x.ptr.edge_W[off + e];
            const u64 K = x.ptr.edge_link[off + e];
            const uint32_t V = vl.V[off + e];
            const float fv = __uint2float_rn(V);
            const float n = __fadd_rn(N, fv);
            const float w = __fsub_rn(W, __fmul_rn(vl.lambda, fv));
            const float u = __fdiv_rn(__fmul_rn(__fmul_rn(x.prm.c_puct, P), sq), __fadd_rn(1.0f, n));
            const float q = n > 0.0f ? __fdiv_rn(w, n) : 0.0f;
            const float v = __fadd_rn(q, u);
            if (v > best) { best = v; best_e = e; my_k = K; my_n = n; my_v = V; }
            else if (e == x.lane) { my_k = K; my_n = n; my_v = V; }   // lane 0 holds edge 0 for the NaN fallback
        }
        for (int d = 16; d; d >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, d);
            const int oe = __shfl_xor_sync(0xffffffffu, best_e, d);
            if (ov > best || (ov == best && oe < best_e)) { best = ov; best_e = oe; }
        }
        if (best_e == 0x7FFFFFFF) best_e = 0;
        const int owner = best_e & 31;
        const u64 best_k = shfl_u64(my_k, owner);
        const float best_n = __shfl_sync(0xffffffffu, my_n, owner);
        const uint32_t best_v = __shfl_sync(0xffffffffu, my_v, owner);
        if (x.lane == 0) path[depth] = make_uint2((uint32_t)node | ((uint32_t)best_e << 16), eoff + (uint32_t)best_e);
        if (best_k == EDGE_NO_CHILD) {
            __syncwarp();
            return best_v > 0 ? -1 : depth;
        }
        node = (int)(best_k & 0xFFFF);
        L = (int)((best_k >> 16) & 0xFF);
        eoff = (uint32_t)(best_k >> 24);
        total = best_n;
        depth++;
    }
}

// Backs up the root's previous batch (vl.count[g] leaves) in leaf order, so that the f32 additions on a shared edge happen in a
// fixed order, and returns the number of leaves.  Without fused heads the evaluated leaves' priors are copied here first.
__device__ __forceinline__ int vl_backup_batch(Ctx& x, const SearchParams& prm, const SearchPtrs& ptr, const VLPtrs& vl) {
    const int nl = vl.count[x.g];
    for (int k = 0; k < nl; k++) {
        const int leaf = x.g * vl.K + k;
        const int s = vl.slot[leaf];
        float value;
        if (s >= 0) {
            if (!prm.priors_scattered) copy_priors(ptr, ptr.req_edge_off[s], ptr.req_nedges[s], s, x.lane);
            value = ptr.res_value[s];
        } else {
            value = vl.value[leaf];
        }
        const int len = vl.len[leaf];
        const uint2* path = vl.path + (size_t)leaf * prm.node_cap;
        for (int i = x.lane; i < len; i += 32) {
            const size_t e = x.ebase + path[i].y;
            const float v = ((len - 1 - i) & 1) ? value : -value;
            ptr.edge_W[e] = __fadd_rn(ptr.edge_W[e], v);
            ptr.edge_N[e] = __fadd_rn(ptr.edge_N[e], 1.0f);
            vl.V[e] -= 1;
        }
        __syncwarp();
    }
    return nl;
}

// Gathers the root's next batch: up to min(K, S - sims_done) descents, ended early by a collision (collided = 1).  Returns the
// number of leaves; depth_sum grows by the edges on their descents.
__device__ __forceinline__ int vl_gather_batch(Ctx& x, const SearchParams& prm, const VLPtrs& vl, int& collided, unsigned int& depth_sum) {
    int n_leaf = 0;
    const int kb = min(vl.K, prm.S - (int)x.c.sims_done);
    for (int k = 0; k < kb; k++) {
        const int leaf = x.g * vl.K + k;
        uint2* path = vl.path + (size_t)leaf * prm.node_cap;
        const int depth = vl_descend(x, vl, path, __fadd_rn((float)(x.c.sims_done + k), 1.0f));
        if (depth < 0) { collided = 1; break; }
        for (int i = x.lane; i <= depth; i += 32) vl.V[x.ebase + path[i].y] += 1;
        if (x.lane == 0) vl.len[leaf] = depth + 1;
        __syncwarp();
        depth_sum += depth + 1;
        n_leaf++;
    }
    return n_leaf;
}

// one warp per root: consume the previous batch (the root's own evaluation on the first wave), then gather the next one
__global__ void __launch_bounds__(WARPS * 32) k_vl_gather(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr,
                                                          const __grid_constant__ VLPtrs vl) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g == 0 && (threadIdx.x & 31) == 0) *ptr.batch_count = 0;   // requests of this wave are counted by k_vl_expand, which runs next
    if (g >= prm.n_games) return;
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, ptr.ctl[g]);
    if (x.c.status != 0) return;
    // ---- 1. the evaluations of the previous wave have arrived
    if (x.c.pending_node == 0) {   // MCTree::init: root priors, optional noise
        const int L = ptr.node_nedges[x.nbase];
        if (!prm.priors_scattered) copy_priors(ptr, x.ebase, L, x.c.pending_slot, x.lane);
        for (int e = x.lane; e < L; e += 32) vl.V[x.ebase + e] = 0;
        __syncwarp();
        if (x.c.flags & 1) apply_noise(x, 0, x.c.game_id, x.c.noise_ply);
        x.c.pending_node = -1;
    } else {
        x.c.sims_done += vl_backup_batch(x, prm, ptr, vl);
    }
    // ---- 2. gather the next batch
    int n_leaf = 0, collided = 0;
    if ((int)x.c.sims_done >= prm.S) {
        x.c.status = 1;
    } else {
        unsigned int depth_sum = 0;
        n_leaf = vl_gather_batch(x, prm, vl, collided, depth_sum);
    }
    if (x.lane == 0) {
        vl_publish(vl, g, n_leaf, collided);
        ptr.ctl[g] = x.c;
    }
}

// one warp per gathered leaf (g * K + k): tree.rs expand; the new node is linked to the leaf edge and queued for evaluation
template <bool ROUTE>
__device__ __forceinline__ void vl_expand_body(const SearchParams& prm, const SearchPtrs& ptr, const VLPtrs& vl, const NetRoute& rt) {
    __shared__ WarpShared shared[WARPS];
    const int leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int g = leaf / vl.K;
    if (g >= prm.n_games || leaf - g * vl.K >= vl.count[g] || ptr.ctl[g].status != 0) return;
    GameCtl c;
    memset(&c, 0, sizeof c);
    c.hist_len = ptr.ctl[g].hist_len;
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, c);
    const uint2* path = vl.path + (size_t)leaf * prm.node_cap;
    const int len = vl.len[leaf];
    const uint2 last = path[len - 1];
    const size_t pe = x.ebase + last.y;
    const DPos parent = ptr.node_pos[x.nbase + (last.x & 0xFFFF)];
    lane0_make_child(x, parent, (uint16_t)(ptr.edge_mv[pe] & 0xFFFF));
    int term = x.sh->term;
    if (term == 0 && draw_by_rules(x, path, x.sh->child, len)) term = 1;
    if (term != 0) {   // draw -> 0, decisive -> -1 from the child's side (tree.rs:233-234); nothing is stored
        if (x.lane == 0) {
            vl.slot[leaf] = -1;
            vl.value[leaf] = term == 1 ? 0.0f : -1.0f;
            atomicAdd(&vl.stats[1], 1ULL);
        }
        return;
    }
    // the node id and the edge range come from the game's counters, shared by the expansions of this wave
    const int n = x.sh->n_moves;
    int L = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + x.lane;
        bool keep = false;
        if (i < n) { const int pr = (x.sh->moves[i] >> 12) & 7; keep = pr == 0 || pr == 4; }
        L += __popc(__ballot_sync(0xffffffffu, keep));
    }
    uint32_t node = 0, eoff = 0;
    if (x.lane == 0) { node = atomicAdd(&ptr.ctl[g].n_nodes, 1u); eoff = atomicAdd(&ptr.ctl[g].n_edges, (uint32_t)L); }
    node = __shfl_sync(0xffffffffu, node, 0);
    eoff = __shfl_sync(0xffffffffu, eoff, 0);
    x.c.n_nodes = node;
    x.c.n_edges = eoff;
    const int child = create_node(x, len);
    if (child < 0) {
        if (x.lane == 0) { ptr.ctl[g].status = 2; atomicAdd(&ptr.counters->errors, 1ULL); }
        return;
    }
    for (int e = x.lane; e < L; e += 32) vl.V[x.ebase + eoff + e] = 0;
    if (x.lane == 0) {
        ptr.edge_link[pe] = x.new_link;
        atomicMax(&ptr.ctl[g].max_depth, (uint32_t)len);
    }
    const int slot = submit_request<ROUTE>(x, child, &rt);
    if (x.lane == 0) vl.slot[leaf] = slot;
}
__global__ void __launch_bounds__(WARPS * 32) k_vl_expand(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr,
                                                          const __grid_constant__ VLPtrs vl) {
    vl_expand_body<false>(prm, ptr, vl, NetRoute{nullptr, nullptr, 0});
}
// the same with the leaf's request in the range of its root's network (az_search_networks)
__global__ void __launch_bounds__(WARPS * 32) k_vl_expand_nets(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr,
                                                               const __grid_constant__ VLPtrs vl, const __grid_constant__ NetRoute rt) {
    vl_expand_body<true>(prm, ptr, vl, rt);
}

// Self-play with leaf-parallel search (az_selfplay_begin_vl), one warp per game slot: publish a parked game, back up the previous
// batch, play the move once the search has its S simulations (move_step: record, choose, traverse_new or finish / restart), then
// gather the next batch -- of the next ply when a move was just played, so no wave is spent between plies.  k_vl_expand and the
// network follow.  Root priors come from the start-position forward or from traverse_new, as in k_advance.
__global__ void __launch_bounds__(WARPS * 32) k_vl_selfplay(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr,
                                                            const __grid_constant__ VLPtrs vl) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g == 0 && (threadIdx.x & 31) == 0) *ptr.batch_count = 0;   // requests of this wave are counted by k_vl_expand, which runs next
    if (g >= prm.n_games) return;
    Ctx x = make_ctx(prm, ptr, &shared[threadIdx.x >> 5], g, ptr.ctl[g]);
    if (x.c.status != 0 && x.c.status != 4) return;   // idle slot or error: vl.count[g] is already 0
    if (x.c.status == 4)   // game over, samples staged: publish now if the host has drained the queue, else stay parked
        absorb(x, finish_game_cold(&prm, &ptr, x.sh, g, x.c));
    int n_leaf = 0, collided = 0;
    if (x.c.status == 0) {
        const int nl = vl_backup_batch(x, prm, ptr, vl);   // 0 for a game that has just started
        x.c.sims_done += nl;
        if (x.lane == 0) x.st_sims += nl;
        if ((int)x.c.sims_done >= prm.S) absorb(x, move_step_cold(&prm, &ptr, x.sh, g, x.c));
        if (x.c.status == 0) {
            if (x.c.sims_done == 0) {   // a fresh root (game start or traverse_new): no descent is in flight through its edges
                const int L = (int)((x.c.flags >> 8) & 0xFF);
                for (int e = x.lane; e < L; e += 32) vl.V[x.ebase + e] = 0;
                __syncwarp();
            }
            n_leaf = vl_gather_batch(x, prm, vl, collided, x.st_depth);
        }
    }
    if (x.lane == 0) {
        vl_publish(vl, g, n_leaf, collided);   // 0 when the slot parked, went idle or failed: the next wave backs up nothing
        ptr.ctl[g] = x.c;
        // the statistics of az_selfplay_step, striped as in k_advance; evaluations and terminal leaves come from vl.stats
        unsigned long long* ct = ptr.stats + (size_t)(blockIdx.x & (STAT_STRIPES - 1)) * STAT_WIDTH;
        if (x.st_sims) atomicAdd(&ct[0], (unsigned long long)x.st_sims);
        if (x.st_pos) atomicAdd(&ct[1], (unsigned long long)x.st_pos);
        if (x.st_games) atomicAdd(&ct[5], (unsigned long long)x.st_games);
        if (x.st_depth) atomicAdd(&ct[6], (unsigned long long)x.st_depth);
        if (x.st_sdepth) atomicAdd(&ct[17], (unsigned long long)x.st_sdepth);
    }
}

// ------------------------------------------------------------------------------------------- evaluation matches (az_match_*)
// evaluate (validation.rs:155-282) as alphazero-chess_b200/evaluation.py plays it on one engine, resident: one warp per slot
// searches a fresh root per ply with az_search_networks' semantics (or takes the priors, for BaseModel players), chooses the move
// with evaluation.py's rules, plays it through the rules path of move_step and records it.  Semantics in DESIGN.md section 5.
struct MatchParams {
    az_position startpos;               // the initial position
    unsigned long long seed;
    unsigned long long first_game, end_game;   // the match's game indices [first_game, end_game)
    unsigned long long* next_game;      // the next game index to start
    unsigned long long* stats;          // [4] evaluations of network 0, of network 1, plies played, games ended
    uint8_t* net;                       // [slots] the network of each slot's mover (what NetRoute::net reads)
    int8_t* result;                     // [games] from White's side
    uint16_t* plies;                    // [games]
    uint8_t* finished;                  // [games] 1: ended by the rules
    uint16_t* moves;                    // [games][row] policy indices played
    uint32_t row, max_plies, n_stochastic;
    int base_model;                     // 1: BaseModel players: the move comes from the root's priors, no search
    int first_wave;                     // 1: every slot starts a game
    uint8_t network[2];                 // network slot of player 1 and of player 2
};

// _uniform(seed, game, ply) of evaluation.py (its _mix, not rng_u64), rounded to f32 as _weighted_index does
__device__ __forceinline__ float match_uniform(u64 seed, u64 game, u64 ply) {
    u64 h = 0x9E3779B97F4A7C15ULL;
    h = (h ^ seed) * 0xBF58476D1CE4E5B9ULL; h ^= h >> 29;
    h = (h ^ game) * 0xBF58476D1CE4E5B9ULL; h ^= h >> 29;
    h = (h ^ ply) * 0xBF58476D1CE4E5B9ULL; h ^= h >> 29;
    return __double2float_rn(__dmul_rn((double)(h >> 11), 1.0 / 9007199254740992.0));
}

// the mover's network: player 1 is White in even games (validation.rs:196-200), so player 1 moves when game + ply is even
__device__ __forceinline__ int match_network(const MatchParams& mp, u64 game, uint32_t ply) { return mp.network[(game + ply) & 1]; }

// The root of the slot's next ply from sh->child / sh->moves, its evaluation queued in the range of the mover's network
__device__ __forceinline__ void match_root(Ctx& x, const MatchParams& mp, const NetRoute& rt, unsigned int* evals) {
    setup_root_from_shared(x);
    const int s = match_network(mp, x.c.game_id, x.c.ply);
    if (x.lane == 0) mp.net[x.g] = (uint8_t)s;
    x.c.pending_node = 0;
    x.c.pending_slot = submit_request<true>(x, 0, &rt);
    evals[s]++;
}

// The next unplayed game starts in this slot (its root queued for evaluation), or the slot goes idle
__device__ __forceinline__ void match_start_game(Ctx& x, const MatchParams& mp, const NetRoute& rt, unsigned int* evals) {
    unsigned long long gid = 0;
    if (x.lane == 0) gid = atomicAdd(mp.next_game, 1ULL);
    gid = __shfl_sync(0xffffffffu, gid, 0);
    if (gid >= mp.end_game) { x.c.status = 1; return; }
    x.c.game_id = gid; x.c.ply = 0; x.c.hist_len = 1;
    if (x.lane == 0) {
        DPos s = dpos_from_wire(mp.startpos);
        ListSink sink{x.sh->moves, 0};
        const GenInfo gi = gen_legal(s, sink);
        set_key_bits(s, gi.has_legal_ep);
        x.sh->child = s; x.sh->n_moves = sink.n; x.sh->term = 0;
        x.ptr.hist[(size_t)x.g * HIST_CAP] = s;
    }
    __syncwarp();
    match_root(x, mp, rt, evals);
}

// evaluation.py's move choice at the root: the weights are the visit counts over their f32 sum (_choose_from_visits) or the priors
// of the legal moves (_choose_from_policy), in policy-index order.  While fullmoves <= num_stochastic_moves: _weighted_index (f32
// cumulative sums, the first one > f32(u) x total, else the last positive weight); after: _last_argmax.  Zero weights change no
// cumulative sum and win no maximum, so only the positive ones are ranked.  Returns the chosen root edge.
__device__ __forceinline__ int match_choose(Ctx& x, const MatchParams& mp, const DPos& root) {
    const size_t off = x.ebase;   // the root's edges start at 0
    const int L = (int)((x.c.flags >> 8) & 0xFF);
    const float* w = mp.base_model ? x.ptr.edge_P + off : x.ptr.edge_N + off;
    float sum = 0.0f;   // visit counts are integers below 2^24: the f32 sum is exact in any order
    for (int e = x.lane; e < L; e += 32) sum = __fadd_rn(sum, w[e]);
    for (int d = 16; d; d >>= 1) sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, d));
    int nv = 0;
    for (int e0 = 0; e0 < L; e0 += 32) {
        const int e = e0 + x.lane;
        int rank = -1;
        if (e < L && w[e] > 0.0f) {
            const uint32_t my = x.ptr.edge_mv[off + e] >> 16;
            rank = 0;
            for (int o = 0; o < L; o++)
                if (w[o] > 0.0f && (x.ptr.edge_mv[off + o] >> 16) < my) rank++;
            x.sh->sidx[rank] = (uint16_t)e;
        }
        nv += __popc(__ballot_sync(0xffffffffu, rank >= 0));
    }
    __syncwarp();
    for (int i = x.lane; i < nv; i += 32) {
        const float v = w[x.sh->sidx[i]];
        x.sh->fval[i] = mp.base_model ? v : __fdiv_rn(v, sum);
    }
    __syncwarp();
    int edge = 0;
    if (x.lane == 0 && nv > 0) {
        edge = x.sh->sidx[nv - 1];
        if ((uint32_t)meta_fullmoves(root.meta) <= mp.n_stochastic) {
            float total = 0.0f;
            for (int i = 0; i < nv; i++) total = __fadd_rn(total, x.sh->fval[i]);
            const float chosen = __fmul_rn(match_uniform(mp.seed, x.c.game_id, x.c.ply), total);
            float cum = 0.0f;
            for (int i = 0; i < nv; i++) {
                cum = __fadd_rn(cum, x.sh->fval[i]);
                if (cum > chosen) { edge = x.sh->sidx[i]; break; }
            }
        } else {
            float best = -1.0f;
            for (int i = 0; i < nv; i++)
                if (x.sh->fval[i] >= best) { best = x.sh->fval[i]; edge = x.sh->sidx[i]; }
        }
    }
    return __shfl_sync(0xffffffffu, edge, 0);
}

// One wave of a match, one warp per slot: consume the root's evaluation or back up the previous batch in leaf order; once the
// root has S visits (BaseModel: at once) choose and play the move, then either queue the next ply's root in the new mover's
// network range or record the game and start the next unplayed one; otherwise gather the next batch.  k_vl_expand_nets (leaves
// routed by mp.net) and the multi-network forward follow.
__global__ void __launch_bounds__(WARPS * 32) k_match(const __grid_constant__ SearchParams prm, const __grid_constant__ SearchPtrs ptr,
                                                      const __grid_constant__ VLPtrs vl, const __grid_constant__ NetRoute rt,
                                                      const __grid_constant__ MatchParams mp) {
    __shared__ WarpShared shared[WARPS];
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= prm.n_games) return;
    GameCtl c;
    if (mp.first_wave) memset(&c, 0, sizeof c);
    else c = ptr.ctl[g];
    // not make_ctx: built from this conditionally initialised c, it orders the prologue's zero-initialisations differently
    Ctx x{prm, ptr, &shared[threadIdx.x >> 5], g, (int)(threadIdx.x & 31), (size_t)g * prm.node_cap, (size_t)g * prm.edge_cap, c,
          0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (!mp.first_wave && x.c.status != 0) return;   // idle slot or pool overflow: vl.count[g] is already 0
    unsigned int evals[AZ_MAX_NETWORKS] = {0, 0}, plies = 0, games = 0;
    int n_leaf = 0, collided = 0;
    bool move = false;
    if (mp.first_wave) {
        match_start_game(x, mp, rt, evals);
    } else if (x.c.pending_node == 0) {   // MCTree::init: the root's priors (no noise), no descent in flight
        const int L = (int)((x.c.flags >> 8) & 0xFF);
        if (!prm.priors_scattered) copy_priors(ptr, x.ebase, L, x.c.pending_slot, x.lane);
        for (int e = x.lane; e < L; e += 32) vl.V[x.ebase + e] = 0;
        __syncwarp();
        x.c.pending_node = -1;
        move = mp.base_model != 0;
    } else {
        const int nl = vl.count[g];
        int evaluated = 0;   // leaves that went to the network (the others were terminal)
        for (int k0 = 0; k0 < nl; k0 += 32) {
            const int k = k0 + x.lane;
            evaluated += __popc(__ballot_sync(0xffffffffu, k < nl && vl.slot[g * vl.K + k] >= 0));
        }
        evals[match_network(mp, x.c.game_id, x.c.ply)] += evaluated;
        x.c.sims_done += vl_backup_batch(x, prm, ptr, vl);
        move = (int)x.c.sims_done >= prm.S;
    }
    if (move) {
        const DPos root = ptr.node_pos[x.nbase];
        const int e = match_choose(x, mp, root);
        const uint32_t amv = ptr.edge_mv[x.ebase + e];
        lane0_make_child(x, root, (uint16_t)(amv & 0xFFFF));
        int term = x.sh->term;
        if (term == 0 && draw_by_rules(x, ptr.path + (size_t)g * prm.node_cap, x.sh->child, 1)) term = 1;
        const size_t gi = (size_t)(x.c.game_id - mp.first_game);
        if (x.lane == 0 && x.c.ply < mp.row) mp.moves[gi * mp.row + x.c.ply] = (uint16_t)(amv >> 16);
        plies++;
        if (term != 0 || x.c.ply + 1 >= mp.max_plies) {
            if (x.lane == 0) {   // term 2: the side to move in the child is mated, the mover won
                mp.result[gi] = term == 2 ? (meta_turn(root.meta) == 0 ? 1 : -1) : 0;
                mp.plies[gi] = (uint16_t)(x.c.ply + 1);
                mp.finished[gi] = term != 0 ? 1 : 0;
            }
            games++;
            match_start_game(x, mp, rt, evals);
        } else {
            if (x.lane == 0 && x.c.hist_len < HIST_CAP) ptr.hist[(size_t)g * HIST_CAP + x.c.hist_len] = x.sh->child;
            x.c.hist_len = min(x.c.hist_len + 1, (uint32_t)HIST_CAP);
            x.c.ply++;
            match_root(x, mp, rt, evals);
        }
    } else if (x.c.status == 0 && x.c.pending_node < 0) {
        unsigned int depth_sum = 0;
        n_leaf = vl_gather_batch(x, prm, vl, collided, depth_sum);
    }
    if (x.lane == 0) {
        vl_publish(vl, g, n_leaf, collided);   // 0 when the slot moved, went idle or waits for its root: the next wave backs up nothing
        if (evals[0]) atomicAdd(&mp.stats[0], (unsigned long long)evals[0]);
        if (evals[1]) atomicAdd(&mp.stats[1], (unsigned long long)evals[1]);
        if (plies) atomicAdd(&mp.stats[2], (unsigned long long)plies);
        if (games) atomicAdd(&mp.stats[3], (unsigned long long)games);
        ptr.ctl[g] = x.c;
    }
}

// ------------------------------------------------------------------------------------------- host side
template <class T>
static int salloc(az_engine* e, SearchState* st, T** p, size_t n) {
    cudaError_t r = cudaMalloc(p, n * sizeof(T));
    if (r != cudaSuccess) return check_cuda(e, r, "cudaMalloc(search)");
    st->allocs.push_back(*p);
    return 0;
}

int search_create(az_engine* e) {
    SearchState* st = new SearchState;
    e->search = st;
    const az_config& c = e->cfg;
    const int G = c.max_games;
    st->G = G;
    SearchParams& p = st->prm;
    p.n_games = G; p.S = c.num_simulations; p.c_puct = c.c_puct; p.alpha = c.dirichlet_alpha; p.eps = c.dirichlet_epsilon;
    p.anneal = c.temperature_annealing; p.num_halfmoves = (int)c.num_halfmoves; p.num_fullmoves = (int)c.num_fullmoves;
    p.repetitions = (int)c.repetitions; p.seed = c.seed;
    p.node_cap = c.num_simulations + 2;
    if (p.node_cap > 65535) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "num_simulations must be < 65534");
    // a game ends by the fullmove limit, so its history and its sample staging hold < 2 * num_fullmoves positions
    if (2 * (int)c.num_fullmoves > std::min(HIST_CAP, MAX_SAMPLE_PLIES) || c.num_fullmoves == 0 || c.num_halfmoves == 0 || c.repetitions == 0)
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "num_fullmoves must be in 1..256, num_halfmoves and repetitions positive");
    if (!(c.c_puct > 0.0f) || !(c.dirichlet_alpha > 0.0f) || c.dirichlet_epsilon < 0.0f || c.dirichlet_epsilon > 1.0f)
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "c_puct and dirichlet_alpha must be positive, dirichlet_epsilon in [0, 1]");
    const int per_node = c.edge_capacity_per_node > 0 ? c.edge_capacity_per_node : 96;
    p.edge_cap = std::max(p.node_cap * std::min(per_node, 218), 256);
    // A game whose leaf was terminal could go on selecting within the same wave, but those few warps (about 8 of 4096) then
    // run two or three times longer than the rest and set the kernel's duration; they continue in the next wave instead
    // (measured per wave: 8 -> 73.6 us, 2 -> 66.4 us, 1 -> 64.2 us; results do not depend on the schedule).
    // With the evaluation cache a hit completes a simulation without the network, so games may go further per wave.
    p.mode = 0; p.max_iters = c.cache_log2 > 0 ? 4 : 2;
    if (const char* v = getenv("AZ_ADV_MAX_ITERS")) p.max_iters = std::max(1, atoi(v));
    p.last_game_id = 0; p.cache_epoch = 0; p.consume = 1;
    if (const char* v = getenv("AZ_ADV_PASSES")) st->adv_passes = std::max(1, std::min(4, atoi(v)));
    if (!(c.temperature > 0.0f)) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "temperature must be positive");
    p.inv_temperature = 1.0f / c.temperature;
    p.fp32_planes = c.precision == 1 ? 1 : 0;
    p.plane_ch = e->net->in_ch;
    // finished games' samples wait here for az_selfplay_drain / az_replay_add_pending; a game that does not fit parks until
    // the host has drained (finish_game), so the only hard requirement is room for one whole game
    p.sample_cap = std::max(G * 128, 1 << 16);
    if (const char* v = getenv("AZ_SAMPLE_CAP")) p.sample_cap = std::max(MAX_SAMPLE_PLIES, atoi(v));   // tests: force parking
    SearchPtrs& q = st->ptr;
    const size_t NN = (size_t)G * p.node_cap, NE = (size_t)G * p.edge_cap;
    int r = 0;
    r |= salloc(e, st, &q.node_pos, NN); r |= salloc(e, st, &q.node_edge_off, NN); r |= salloc(e, st, &q.node_nedges, NN);
    r |= salloc(e, st, &q.node_nmoves, NN); r |= salloc(e, st, &q.node_depth, NN);
    r |= salloc(e, st, &q.edge_P, NE); r |= salloc(e, st, &q.edge_N, NE); r |= salloc(e, st, &q.edge_W, NE);
    r |= salloc(e, st, &q.edge_link, NE); r |= salloc(e, st, &q.edge_mv, NE);
    r |= salloc(e, st, &q.ctl, (size_t)G); r |= salloc(e, st, &q.path, NN); r |= salloc(e, st, &q.hist, (size_t)G * HIST_CAP);
    r |= salloc(e, st, &q.batch_count, 8); r |= salloc(e, st, &q.req_pos, (size_t)e->max_batch);
    r |= salloc(e, st, &q.req_f32, (size_t)e->max_batch * AZ_NUM_PLANES * 64);
    r |= salloc(e, st, &q.req_edge_off, (size_t)e->max_batch); r |= salloc(e, st, &q.req_nedges, (size_t)e->max_batch);
    r |= salloc(e, st, &q.start_prior, 32); r |= salloc(e, st, &q.counters, 1);
    r |= salloc(e, st, &q.stats, (size_t)STAT_STRIPES * STAT_WIDTH);
    r |= salloc(e, st, &st->d_noise_ids, (size_t)G); r |= salloc(e, st, &st->d_noise_plies, (size_t)G);
    if (r) return AZ_ERR_OUT_OF_MEMORY;
    p.cache_mask = 0; q.cache_state = nullptr; q.cache_entry = nullptr;
    if (c.cache_log2 > 0) {
        if (c.cache_log2 > 26) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "cache_log2 must be <= 26");
        const size_t slots = (size_t)1 << c.cache_log2;
        if (salloc(e, st, &q.cache_state, slots) || salloc(e, st, &q.cache_entry, slots)) return AZ_ERR_OUT_OF_MEMORY;
        cudaMemset(q.cache_state, 0, slots * sizeof(uint32_t));
        p.cache_mask = (uint32_t)(slots - 1);
    }
    q.req_bf16 = e->net->a_in;
    q.res_policy = e->d_policy;
    q.res_value = e->d_value;
    q.game_samples = nullptr;
    q.out_samples = nullptr;
    cudaMemset(q.counters, 0, sizeof(Counters));
    cudaMemset(q.stats, 0, (size_t)STAT_STRIPES * STAT_WIDTH * sizeof(unsigned long long));
    cudaMemset(q.batch_count, 0, 32);
    st->batch_base = q.batch_count;
    q.batch_zero = nullptr;
    return 0;
}

void search_destroy(az_engine* e) {
    SearchState* st = e->search;
    if (!st) return;
    for (void* p : st->allocs) cudaFree(p);
    const MatchState& m = st->match;
    for (void* p : {(void*)m.result.p, (void*)m.plies.p, (void*)m.finished.p, (void*)m.moves.p}) cudaFree(p);
    delete st;
    e->search = nullptr;
}

// the bf16 network's heads write the legal-move priors straight into edge_P (HeadScatter)
static bool fused_heads(const az_engine* e) { return e->stub_kind == 0 && e->cfg.precision != 1; }

static bool selfplay_on(const SearchState* st) { return st->session == Session::selfplay || st->session == Session::selfplay_vl; }

// evaluates the queued requests: the network (bf16 or fp32) or the synthetic evaluator.  nb: a multi-network batch (requests
// routed by NetRoute); under the synthetic evaluator network s evaluates with seed stub_seed + s
static int evaluate_batch(az_engine* e, SearchState* st, const NetBatch* nb = nullptr) {
    const SearchPtrs& q = st->ptr;
    if (nb) {
        if (e->stub_kind == 1) {
            const int warps = e->max_batch;
            for (int s = 0; s < AZ_MAX_NETWORKS; s++) {
                const size_t base = s ? (size_t)nb->base1 : 0;
                e->n_launches++;
                k_stub_eval<<<(warps + 3) / 4, 128, 0, e->stream>>>(q.req_pos + base, nb->counts_dev + s, 0, e->stub_seed + (uint64_t)s,
                                                                    e->d_policy + base * AZ_ACTION_SPACE, e->d_value + base);
                AZ_CUDA(e, cudaGetLastError());
            }
            return AZ_OK;
        }
        if (e->cfg.precision == 1) return net_forward_networks(e, *nb, q.req_f32, e->d_policy, e->d_value);
        HeadScatter sc{q.req_edge_off, q.req_nedges, q.edge_mv, q.edge_P};
        return net_forward_networks(e, *nb, nullptr, nullptr, e->d_value, &sc);
    }
    if (e->stub_kind == 1) {
        const int warps = e->max_batch;
        e->n_launches++;
        k_stub_eval<<<(warps + 3) / 4, 128, 0, e->stream>>>(q.req_pos, q.batch_count, 0, e->stub_seed, e->d_policy, e->d_value);
        return check_cuda(e, cudaGetLastError(), "k_stub_eval");
    }
    if (e->cfg.precision == 1) return net_forward_fp32(e, q.req_f32, q.batch_count, 0, e->d_policy, e->d_value);
    HeadScatter sc{q.req_edge_off, q.req_nedges, q.edge_mv, q.edge_P};
    return net_forward_bf16(e, q.batch_count, 0, nullptr, e->d_value, &sc);
}

int search_pending_samples(az_engine* e, const az_sample** d_samples, int* n) {
    SearchState* st = e->search;
    if (!selfplay_on(st)) return set_err(e, AZ_ERR_STATE, "az_selfplay_begin has not been called");
    unsigned long long out;
    AZ_CUDA(e, cudaMemcpyAsync(&out, &st->ptr.counters->samples_out, sizeof out, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    *d_samples = st->ptr.out_samples;
    *n = (int)std::min<unsigned long long>(out, st->prm.sample_cap);
    return 0;
}
int search_clear_pending(az_engine* e) {
    SearchState* st = e->search;
    AZ_CUDA(e, cudaMemsetAsync(&st->ptr.counters->samples_out, 0, sizeof(unsigned long long), e->stream));
    return 0;
}

// az_profile: when the coming forward will be sampled, the search kernels launched from here on are timed up to its start
static void prof_mark_search(az_engine* e) {
    if (e->prof_every > 0 && fused_heads(e) && (e->prof_counter % (uint64_t)e->prof_every) == 0 &&
        !e->prof_adv_event) {
        cudaEventCreate(&e->prof_adv_event);
        cudaEventRecord(e->prof_adv_event, e->stream);
    }
}

static int run_wave(az_engine* e, SearchState* st) {
    const int blocks = (st->prm.n_games + WARPS - 1) / WARPS;
    st->prm.priors_scattered = fused_heads(e) ? 1 : 0;
    if (st->prm.mode == 1) st->prm.cache_epoch = (uint32_t)((st->wave_counter++ / (unsigned long long)std::max(st->prm.S, 1)) & 63);
    // Two request counters alternate between waves: this wave's k_advance counts into one and clears the other, which the
    // previous wave's network kernels (complete by stream order) were the last to read -- no memset launch per wave.
    st->batch_parity ^= 1;
    st->ptr.batch_count = st->batch_base + st->batch_parity;
    st->ptr.batch_zero = st->batch_base + (st->batch_parity ^ 1);
    prof_mark_search(e);
    // AZ_ADV_PASSES > 1 (experiment, default 1): extra k_advance passes per wave in which only the games that completed their
    // max_iters network-free simulations without needing the network go on.  Measured at 14 % / 45 % / 63 % cache hits
    // (profiles/r2_passes_raw.jsonl): always slower -- the fuller batch costs tower time in proportion, and more simulations
    // per wave mean more games evaluating the same position in the same wave before anybody's result reaches the cache.
    const int passes = st->prm.mode == 1 && st->prm.cache_mask ? st->adv_passes : 1;
    for (int pass = 0; pass < passes; pass++) {
    st->prm.consume = pass == 0 ? 1 : 0;
    e->n_launches++;
    const int minb = e->knobs.adv_minb;
    // groups of four warps per SM (register bound): 3 -> 162 registers, 4 -> 128, 5 -> 96, 6 -> 80, 7 -> 72 with 216 bytes of
    // spills.  With 7, all 4096 games of a wave are resident at once (148 SMs x 28 warps) and the kernel is one round of
    // latency chains instead of two: measured per wave 4 -> 67.6 us, 5 -> 68.5, 6 -> 69.6, 7 -> 54.7.
    switch (minb) {
        case 4: k_advance<4><<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr); break;
        case 5: k_advance<5><<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr); break;
        case 6: k_advance<6><<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr); break;
        case 7: k_advance<7><<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr); break;
        default: k_advance<3><<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr); break;
    }
    }
    st->prm.consume = 1;
    AZ_CUDA(e, cudaGetLastError());
    return evaluate_batch(e, st);
}

// Input staging of az_search and az_search_vl (MCTree::init for n roots): validates the arguments, copies roots, history and
// noise keys to the device, creates every root (k_init_search) and evaluates the roots.  `run` becomes the call's copy of the
// search state.  Returns AZ_OK, an error, or 1 when there is nothing to do (n == 0).
static int search_begin(az_engine* e, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                        int num_simulations, const uint64_t* noise_game_ids, const uint32_t* noise_plies, const float* visits_out,
                        SearchState& run, const NetRoute* route = nullptr, const NetBatch* nb = nullptr) {
    SearchState* st = e->search;
    if (n < 0 || n > st->G) return set_err(e, AZ_ERR_CAPACITY, "more roots than az_config.max_games");
    if (n == 0) return 1;
    if (!roots || !visits_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    if (num_simulations <= 0 || num_simulations + 2 > st->prm.node_cap)
        return set_err(e, AZ_ERR_CAPACITY, "num_simulations exceeds az_config.num_simulations (pool size)");
    if (e->stub_kind == 0 && !route && !e->net->loaded) return set_err(e, AZ_ERR_NO_WEIGHTS, "az_load_weights has not been called");
    cudaSetDevice(e->cfg.device);
    st->session = Session::none;
    SearchParams prm = st->prm;
    prm.n_games = n; prm.S = num_simulations; prm.mode = 0;
    run = *st;
    run.prm = prm;
    // stage inputs
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, roots, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    const az_position* d_hist = nullptr;
    if (history && hist_offsets) {
        // GameState::pos_count already holds the current position (chess.rs:23,52-53): the last history entry IS the root
        for (int g = 0; g < n; g++) {
            if (hist_offsets[g + 1] < hist_offsets[g]) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "hist_offsets must be non-decreasing");
            if (hist_offsets[g + 1] == hist_offsets[g]) continue;
            const az_position& last = history[hist_offsets[g + 1] - 1];
            const az_position& r0 = roots[g];
            if (std::memcmp(last.roles, r0.roles, sizeof last.roles) || std::memcmp(last.colors, r0.colors, sizeof last.colors) ||
                last.turn != r0.turn || last.castling != r0.castling || last.ep_square != r0.ep_square)
                return set_err(e, AZ_ERR_INVALID_ARGUMENT, "the last history entry of a game must be its root position");
        }
        size_t total = hist_offsets[n];
        if (total > e->hist_cap) {
            cudaFree(e->d_hist); e->d_hist = nullptr; e->hist_cap = 0;
            AZ_CUDA(e, cudaMalloc(&e->d_hist, std::max<size_t>(total, 1024) * sizeof(az_position)));
            e->hist_cap = std::max<size_t>(total, 1024);
        }
        if (total) AZ_CUDA(e, cudaMemcpyAsync(e->d_hist, history, total * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
        AZ_CUDA(e, cudaMemcpyAsync(e->d_hist_off, hist_offsets, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, e->stream));
        d_hist = e->d_hist ? e->d_hist : (const az_position*)e->d_wire;
    }
    unsigned long long* d_ids = nullptr;
    uint32_t* d_plies = nullptr;
    if (noise_game_ids) {
        d_ids = st->d_noise_ids;   // persistent staging: no allocation (= no implicit device synchronisation) per call
        d_plies = st->d_noise_plies;
        AZ_CUDA(e, cudaMemcpyAsync(d_ids, noise_game_ids, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
        if (noise_plies) AZ_CUDA(e, cudaMemcpyAsync(d_plies, noise_plies, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
        else AZ_CUDA(e, cudaMemsetAsync(d_plies, 0, (size_t)n * 4, e->stream));
    }
    const int blocks = (n + WARPS - 1) / WARPS;
    run.batch_parity = 0;
    run.ptr.batch_count = run.batch_base;
    run.ptr.batch_zero = nullptr;
    AZ_CUDA(e, cudaMemsetAsync(run.batch_base, 0, 16, e->stream));
    e->n_launches++;
    if (route) k_init_search_nets<<<blocks, WARPS * 32, 0, e->stream>>>(run.prm, run.ptr, e->d_wire, d_hist, e->d_hist_off, d_ids, d_plies, *route);
    else k_init_search<<<blocks, WARPS * 32, 0, e->stream>>>(run.prm, run.ptr, e->d_wire, d_hist, e->d_hist_off, d_ids, d_plies);
    AZ_CUDA(e, cudaGetLastError());
    return evaluate_batch(e, &run, nb);
}

// dense export of the roots' statistics (Box<[f32; 4096]> visits / scores, max_subtree_depth) to the caller's buffers
static int search_export(az_engine* e, const SearchState& run, int n, float* visits_out, float* scores_out, int32_t* depth_out) {
    float* d_vis = e->d_policy;  // reuse the result buffers for the dense export
    float* d_sc = nullptr;
    if (scores_out) {
        if (!e->d_scores) AZ_CUDA(e, cudaMalloc(&e->d_scores, (size_t)e->max_batch * AZ_ACTION_SPACE * 4));
        d_sc = e->d_scores;
    }
    k_export_root<<<n, 256, 0, e->stream>>>(run.prm, run.ptr, d_vis, d_sc, e->d_count);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(visits_out, d_vis, (size_t)n * AZ_ACTION_SPACE * 4, cudaMemcpyDeviceToHost, e->stream));
    if (scores_out) AZ_CUDA(e, cudaMemcpyAsync(scores_out, d_sc, (size_t)n * AZ_ACTION_SPACE * 4, cudaMemcpyDeviceToHost, e->stream));
    if (depth_out) AZ_CUDA(e, cudaMemcpyAsync(depth_out, e->d_count, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

// enqueues k_count_active over the first n slots and the copy of its flags to the host, where they are valid after the
// caller's next stream synchronise: flags[0] active, flags[1] failed (pool overflow or illegal state), flags[2] parked
static int enqueue_poll(az_engine* e, const SearchState& run, int n, int flags[4]) {
    int* d_flags = run.batch_base + 4;
    AZ_CUDA(e, cudaMemsetAsync(d_flags, 0, 16, e->stream));
    k_count_active<<<(n + 127) / 128, 128, 0, e->stream>>>(run.prm, run.ptr, d_flags);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(flags, d_flags, 16, cudaMemcpyDeviceToHost, e->stream));
    return AZ_OK;
}

static int search_poll(az_engine* e, const SearchState& run, int n, int flags[4]) {
    const int r = enqueue_poll(e, run, n, flags);
    if (r) return r;
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

// the in-flight counts and the per-leaf records of az_search_vl and az_selfplay_begin_vl, allocated by the first such call
static int vl_alloc(az_engine* e, SearchState* st) {
    if (st->vl_V) return AZ_OK;
    cudaSetDevice(e->cfg.device);
    const size_t NE = (size_t)st->G * st->prm.edge_cap, B = (size_t)e->max_batch;
    int a = salloc(e, st, &st->vl_V, NE);
    a |= salloc(e, st, &st->vl_path, B * st->prm.node_cap);
    a |= salloc(e, st, &st->vl_len, B); a |= salloc(e, st, &st->vl_slot, B); a |= salloc(e, st, &st->vl_value, B);
    a |= salloc(e, st, &st->vl_count, (size_t)st->G); a |= salloc(e, st, &st->vl_stats, 4);
    return a ? AZ_ERR_OUT_OF_MEMORY : AZ_OK;
}

static VLPtrs vl_ptrs(const SearchState* st, int K, float lambda) {
    return VLPtrs{st->vl_V, st->vl_path, st->vl_len, st->vl_slot, st->vl_value, st->vl_count, st->vl_stats, K, lambda};
}

// the leaves per root (`what`: leaves_per_root or leaves_per_game) and the virtual loss of a leaf-parallel call
static int check_vl_args(az_engine* e, int K, float virtual_loss, const char* what) {
    if (K < 1) return set_err(e, AZ_ERR_INVALID_ARGUMENT, (std::string(what) + " must be >= 1").c_str());
    if (!(virtual_loss >= 0.0f) || !std::isfinite(virtual_loss))
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "virtual_loss must be finite and >= 0");
    return AZ_OK;
}

// the board ranges of a multi-network batch with n0 / n1 roots (or slots) of K leaves each: network 0 from board 0, network 1
// from base1 = round4(n0 x K), so no tile of the network kernels mixes networks; `end` is the end of network 1's range rounded to 4
struct NetLayout { long long base1, end; };
static NetLayout net_layout(long long n0, long long n1, int K) {
    const long long base1 = (n0 * K + 3) & ~3LL;
    return NetLayout{base1, base1 + ((n1 * K + 3) & ~3LL)};
}

// no batch in flight for the first n roots or slots, no leaf-parallel statistics yet
static int vl_clear(az_engine* e, const SearchState* st, int n) {
    if (n) AZ_CUDA(e, cudaMemsetAsync(st->vl_count, 0, (size_t)n * sizeof(int), e->stream));
    AZ_CUDA(e, cudaMemsetAsync(st->vl_stats, 0, 4 * sizeof(unsigned long long), e->stream));
    return AZ_OK;
}

// vl_stats (leaves gathered, terminal leaves, collisions) as az_search_stats: every gathered leaf that was not terminal was evaluated
static az_search_stats vl_search_stats(const unsigned long long s[4], uint64_t waves) {
    return az_search_stats{waves, s[0] - s[1], s[1], s[2]};
}

// the tail of a leaf-parallel wave after its gather kernel: k_vl_expand (k_vl_expand_nets into the networks' ranges when rt is
// given) over n roots or slots, then the evaluation of the batch (a multi-network one when nb is given)
static int vl_expand_evaluate(az_engine* e, SearchState* run, const VLPtrs& vl, int n, const NetRoute* rt = nullptr,
                              const NetBatch* nb = nullptr) {
    const int blocks = (n * vl.K + WARPS - 1) / WARPS;
    if (rt) k_vl_expand_nets<<<blocks, WARPS * 32, 0, e->stream>>>(run->prm, run->ptr, vl, *rt);
    else k_vl_expand<<<blocks, WARPS * 32, 0, e->stream>>>(run->prm, run->ptr, vl);
    AZ_CUDA(e, cudaGetLastError());
    return evaluate_batch(e, run, nb);
}

// az_search_vl, and az_search_networks when `network` (one id per root) is given: the requests of each root then go to the
// range of its network (k_init_search_nets, k_vl_expand_nets) and every wave evaluates both ranges in one multi-network forward
static int search_vl_run(az_engine* e, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                         int num_simulations, int leaves_per_root, float virtual_loss, const uint8_t* network,
                         const uint64_t* noise_game_ids, const uint32_t* noise_plies, float* visits_out, float* scores_out,
                         int32_t* depth_out, az_search_stats* stats_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (stats_out) std::memset(stats_out, 0, sizeof *stats_out);
    const int K = leaves_per_root;
    int r = check_vl_args(e, K, virtual_loss, "leaves_per_root");
    if (r) return r;
    if (n > 0 && (long long)n * K > (long long)e->max_batch)
        return set_err(e, AZ_ERR_CAPACITY, "roots x leaves_per_root exceeds az_config.max_batch");
    SearchState* st = e->search;
    int count[AZ_MAX_NETWORKS] = {0, 0};
    int base1 = 0;
    if (network && n > 0 && n <= st->G) {
        for (int g = 0; g < n; g++) {
            if (network[g] >= AZ_MAX_NETWORKS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "network id must be < AZ_MAX_NETWORKS");
            count[network[g]]++;
        }
        for (int s = 0; s < AZ_MAX_NETWORKS; s++) {
            const NetWeights* w = net_slot(e, s);
            if (count[s] && e->stub_kind == 0 && (!w || !w->loaded))
                return set_err(e, AZ_ERR_NO_WEIGHTS, "a root names a network that has not been loaded");
        }
        const NetLayout lay = net_layout(count[0], count[1], K);
        if (lay.end > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "network ranges (roots x leaves_per_root each) exceed az_config.max_batch");
        base1 = (int)lay.base1;
    }
    if (n >= 0 && n <= st->G) {
        const int a = vl_alloc(e, st);
        if (a) return a;
    }
    NetRoute route{nullptr, st->batch_base, base1};
    NetBatch nb{st->batch_base, base1, base1 + count[1] * K};
    if (network && n > 0 && n <= st->G) {
        if (!st->d_net) {
            cudaSetDevice(e->cfg.device);
            if (salloc(e, st, &st->d_net, (size_t)st->G)) return AZ_ERR_OUT_OF_MEMORY;
        }
        AZ_CUDA(e, cudaMemcpyAsync(st->d_net, network, (size_t)n, cudaMemcpyHostToDevice, e->stream));
        route.net = st->d_net;
    }
    const NetRoute* rt = route.net ? &route : nullptr;
    const NetBatch* nbp = route.net ? &nb : nullptr;
    SearchState run;
    r = search_begin(e, n, roots, history, hist_offsets, num_simulations, noise_game_ids, noise_plies, visits_out, run, rt, nbp);
    if (r) return r == 1 ? AZ_OK : r;
    const VLPtrs vl = vl_ptrs(st, K, virtual_loss);
    r = vl_clear(e, st, n);
    if (r) return r;
    run.prm.priors_scattered = fused_heads(e) ? 1 : 0;
    uint64_t waves = 1;   // the roots' evaluation
    // a batch adds at least one leaf per active root, so every root is done after at most S batches; the first poll comes
    // after the earliest wave at which the last batch can have been consumed
    const int first_poll = (num_simulations + K - 1) / K;
    int rc = AZ_OK;
    for (int wave = 0;; wave++) {
        prof_mark_search(e);
        e->n_launches += 2;
        k_vl_gather<<<(n + WARPS - 1) / WARPS, WARPS * 32, 0, e->stream>>>(run.prm, run.ptr, vl);
        AZ_CUDA(e, cudaGetLastError());
        if (wave >= first_poll) {
            int flags[4] = {0, 0, 0, 0};
            r = search_poll(e, run, n, flags);
            if (r) return r;
            if (flags[1]) { rc = set_err(e, AZ_ERR_CAPACITY, "a per-game node/edge pool overflowed (raise edge_capacity_per_node)"); break; }
            if (flags[0] == 0) break;
            if (wave > num_simulations + 16) { rc = set_err(e, AZ_ERR_STATE, "search did not converge"); break; }
        }
        if (rt)   // both request counters start the wave at 0 (k_vl_gather clears only the first)
            AZ_CUDA(e, cudaMemsetAsync(run.batch_base, 0, AZ_MAX_NETWORKS * sizeof(int), e->stream));
        r = vl_expand_evaluate(e, &run, vl, n, rt, nbp);
        if (r) return r;
        waves++;
    }
    if (e->prof_adv_event) {   // the last gather is followed by no forward: its mark must not time the next call's kernels
        cudaEventDestroy(e->prof_adv_event);
        e->prof_adv_event = nullptr;
    }
    if (rc == AZ_OK) rc = search_export(e, run, n, visits_out, scores_out, depth_out);
    if (rc == AZ_OK && stats_out) {
        unsigned long long s[4];
        AZ_CUDA(e, cudaMemcpyAsync(s, vl.stats, sizeof s, cudaMemcpyDeviceToHost, e->stream));
        AZ_CUDA(e, cudaStreamSynchronize(e->stream));
        *stats_out = vl_search_stats(s, waves);
        stats_out->evaluations += (uint64_t)n;   // and the roots
    }
    return rc;
}

// az_selfplay_begin_n (K = 0: k_advance waves) and az_selfplay_begin_vl (K >= 1: k_vl_selfplay waves with K leaves per game)
static int selfplay_begin(az_engine* e, int n_games, uint64_t first_game_id, uint64_t total_games, int K, float virtual_loss) {
    SearchState* st = e->search;
    if (total_games != 0 && (uint64_t)n_games > total_games) n_games = (int)total_games;   // never more slots than games to play
    if (n_games <= 0 || n_games > st->G) return set_err(e, AZ_ERR_CAPACITY, "more games than az_config.max_games");
    if (K > 0 && (long long)n_games * K > (long long)e->max_batch)
        return set_err(e, AZ_ERR_CAPACITY, "games x leaves_per_game exceeds az_config.max_batch");
    if (K > 0 && st->prm.cache_mask)
        return set_err(e, AZ_ERR_STATE, "az_selfplay_begin_vl does not support the evaluation cache (cache_log2 > 0)");
    if (e->stub_kind == 0 && !e->net->loaded) return set_err(e, AZ_ERR_NO_WEIGHTS, "az_load_weights has not been called");
    cudaSetDevice(e->cfg.device);
    if (K > 0) {
        const int a = vl_alloc(e, st);
        if (a) return a;
    }
    SearchPtrs& q = st->ptr;
    if (!q.game_samples) {
        int r = salloc(e, st, &q.game_samples, (size_t)st->G * MAX_SAMPLE_PLIES);
        r |= salloc(e, st, &q.out_samples, (size_t)st->prm.sample_cap);
        if (r) return AZ_ERR_OUT_OF_MEMORY;
    }
    st->prm.n_games = n_games; st->prm.mode = 1; st->prm.S = e->cfg.num_simulations;
    st->prm.last_game_id = total_games ? first_game_id + total_games : 0;
    st->wave_counter = 0; st->prm.cache_epoch = 0;
    if (st->prm.cache_mask)  // a new cache per generation (training.rs:342)
        AZ_CUDA(e, cudaMemsetAsync(q.cache_state, 0, ((size_t)st->prm.cache_mask + 1) * sizeof(uint32_t), e->stream));
    Counters zero;
    std::memset(&zero, 0, sizeof zero);
    zero.next_game_id = first_game_id + n_games;
    AZ_CUDA(e, cudaMemcpyAsync(q.counters, &zero, sizeof zero, cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemsetAsync(q.stats, 0, (size_t)STAT_STRIPES * STAT_WIDTH * sizeof(unsigned long long), e->stream));
    // the one shared forward of the start position (training.rs:344-350)
    az_position sp;
    az_position_start(&sp);
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, &sp, sizeof sp, cudaMemcpyHostToDevice, e->stream));
    int r;
    if (e->stub_kind == 1) {
        DPos d = dpos_from_wire(sp);
        AZ_CUDA(e, cudaMemcpyAsync(q.req_pos, &d, sizeof d, cudaMemcpyHostToDevice, e->stream));
        k_stub_eval<<<1, 128, 0, e->stream>>>(q.req_pos, nullptr, 1, e->stub_seed, e->d_policy, e->d_value);
        r = check_cuda(e, cudaGetLastError(), "k_stub_eval");
    } else if (e->cfg.precision == 1) {
        launch_encode_f32(e->stream, e->d_wire, e->d_planes, 1);
        r = net_forward_fp32(e, e->d_planes, nullptr, 1, e->d_policy, e->d_value);
    } else {
        launch_encode_bf16_wire(e->stream, e->d_wire, e->net->a_in, 1, e->net->in_ch);
        r = net_forward_bf16(e, nullptr, 1, e->d_policy, e->d_value);
    }
    if (r) return r;
    st->batch_parity = 0;
    q.batch_count = st->batch_base;
    q.batch_zero = nullptr;
    AZ_CUDA(e, cudaMemsetAsync(st->batch_base, 0, 8, e->stream));   // both request counters (run_wave alternates them)
    k_start_prior<<<1, 32, 0, e->stream>>>(e->d_policy, q.start_prior);
    const int blocks = (n_games + WARPS - 1) / WARPS;
    e->n_launches += 2;
    k_init_selfplay<<<blocks, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr, first_game_id);
    AZ_CUDA(e, cudaGetLastError());
    if (K > 0 && (r = vl_clear(e, st, n_games))) return r;
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    st->sp_vl = SelfplayVL{K, virtual_loss, 0};
    st->session = K > 0 ? Session::selfplay_vl : Session::selfplay;
    return AZ_OK;
}

// one wave of az_selfplay_begin_vl's self-play: k_vl_selfplay, k_vl_expand, the network
static int run_wave_vl(az_engine* e, SearchState* st) {
    const int n = st->prm.n_games;
    st->prm.priors_scattered = fused_heads(e) ? 1 : 0;
    const VLPtrs vl = vl_ptrs(st, st->sp_vl.K, st->sp_vl.lambda);
    prof_mark_search(e);
    e->n_launches += 2;
    k_vl_selfplay<<<(n + WARPS - 1) / WARPS, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr, vl);
    AZ_CUDA(e, cudaGetLastError());
    st->sp_vl.waves++;
    return vl_expand_evaluate(e, st, vl, n);
}

#ifdef AZ_ADV_TIMING
// AZ_ADV_TIMING: k_advance's phase clocks and warp-time histogram (stripe fields 8..15 and 24..39) of the waves since the last
// report, per game and wave
static void adv_timing_report(const unsigned long long* stripes, int n_games, int waves) {
    unsigned long long tc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < STAT_STRIPES * STAT_WIDTH; i++) if (i % STAT_WIDTH >= 8 && i % STAT_WIDTH < 16) tc[i % STAT_WIDTH - 8] += stripes[i];
    unsigned long long hist[16] = {0};
    for (int i = 0; i < STAT_STRIPES * STAT_WIDTH; i++) if (i % STAT_WIDTH >= 24) hist[i % STAT_WIDTH - 24] += stripes[i];
    {   // the device counters are cumulative since az_selfplay_begin: report this call's share
        static unsigned long long prev_tc[8], prev_hist[16];
        for (int k = 0; k < 8; k++) { const unsigned long long c = tc[k]; tc[k] = c >= prev_tc[k] ? c - prev_tc[k] : c; prev_tc[k] = c; }
        for (int k = 0; k < 16; k++) { const unsigned long long c = hist[k]; hist[k] = c >= prev_hist[k] ? c - prev_hist[k] : c; prev_hist[k] = c; }
    }
    if (waves <= 0) return;
    fprintf(stderr, "azb: k_advance warp-time histogram (buckets of 4096 clocks):");
    for (int k = 0; k < 16; k++) fprintf(stderr, " %llu", hist[k]);
    fprintf(stderr, "\n");
    const double per = (double)n_games * waves;
    fprintf(stderr, "azb: k_advance phase clocks per warp-wave: consume %.0f select %.0f child %.0f rules %.0f create %.0f submit %.0f move %.0f total %.0f\n",
            (double)tc[0] / per, (double)tc[1] / per, (double)tc[2] / per, (double)tc[3] / per, (double)tc[4] / per, (double)tc[5] / per,
            (double)tc[6] / per, (double)tc[7] / per);
}
#endif

// az_selfplay_drain (kind: device to host) and az_selfplay_drain_dev (device to device), ordered on the engine's stream after
// the self-play waves and any az_replay_add_pending before it
static int selfplay_drain(az_engine* e, az_sample* out, int max_samples, int* n_out, cudaMemcpyKind kind) {
    if (!e || !n_out) return AZ_ERR_INVALID_ARGUMENT;
    cudaSetDevice(e->cfg.device);
    const az_sample* d_samples = nullptr;
    int n = 0;
    int r = search_pending_samples(e, &d_samples, &n);
    if (r) return r;
    if ((unsigned long long)n > (unsigned long long)max_samples) return set_err(e, AZ_ERR_CAPACITY, "drain buffer smaller than the pending sample count");
    if (n && out) AZ_CUDA(e, cudaMemcpyAsync(out, d_samples, (size_t)n * sizeof(az_sample), kind, e->stream));
    if ((r = search_clear_pending(e))) return r;
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    *n_out = n;
    return AZ_OK;
}

template <class T>
static int grow(az_engine* e, GrowBuf<T>& b, size_t n) {
    if (n <= b.cap) return AZ_OK;
    cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
    AZ_CUDA(e, cudaMalloc(&b.p, n * sizeof(T)));
    b.cap = n;
    return AZ_OK;
}

// the match's per-game results, reallocated when a match needs more room than the last one (freed by search_destroy)
static int match_alloc(az_engine* e, SearchState* st, size_t games, size_t row) {
    MatchState& m = st->match;
    if (!m.next && (salloc(e, st, &m.next, 1) || salloc(e, st, &m.stats, 4))) return AZ_ERR_OUT_OF_MEMORY;
    int r = grow(e, m.result, games);
    if (!r) r = grow(e, m.plies, games);
    if (!r) r = grow(e, m.finished, games);
    if (!r) r = grow(e, m.moves, games * row);
    return r;
}

static MatchParams match_params(const SearchState* st) {
    const MatchState& m = st->match;
    const az_match_config& c = m.cfg;
    MatchParams mp;
    mp.startpos = m.startpos;
    mp.seed = c.seed;
    mp.first_game = m.first;
    mp.end_game = m.first + m.games;
    mp.next_game = m.next;
    mp.stats = m.stats;
    mp.net = st->d_net;
    mp.result = m.result.p; mp.plies = m.plies.p; mp.finished = m.finished.p; mp.moves = m.moves.p;
    mp.row = m.row; mp.max_plies = c.max_plies; mp.n_stochastic = c.num_stochastic_moves;
    mp.base_model = c.player_kind == 1 ? 1 : 0;
    mp.first_wave = m.first_wave;
    mp.network[0] = c.network[0]; mp.network[1] = c.network[1];
    return mp;
}

}  // namespace azb

using namespace azb;

extern "C" {

int az_set_evaluator_stub(az_engine* e, int kind, uint64_t seed) {
    if (!e || kind < 0 || kind > 1) return AZ_ERR_INVALID_ARGUMENT;
    e->stub_kind = kind;
    e->stub_seed = seed;
    return AZ_OK;
}

int az_search(az_engine* e, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
              int num_simulations, const uint64_t* noise_game_ids, const uint32_t* noise_plies, float* visits_out, float* scores_out,
              int32_t* depth_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    SearchState run;
    int r = search_begin(e, n, roots, history, hist_offsets, num_simulations, noise_game_ids, noise_plies, visits_out, run);
    if (r) return r == 1 ? AZ_OK : r;
    // every wave completes at least one simulation per active game
    int rc = AZ_OK;
    for (int wave = 0;; wave++) {
        r = run_wave(e, &run);
        if (r) { rc = r; break; }
        if (wave + 1 >= num_simulations && (wave + 1 - num_simulations) % 4 == 0) {
            int flags[4] = {0, 0, 0, 0};
            r = search_poll(e, run, n, flags);
            if (r) return r;
            if (flags[1]) { rc = set_err(e, AZ_ERR_CAPACITY, "a per-game node/edge pool overflowed (raise edge_capacity_per_node)"); break; }
            if (flags[0] == 0) break;
            if (wave > 4 * num_simulations + 16) { rc = set_err(e, AZ_ERR_STATE, "search did not converge"); break; }
        }
    }
    if (rc == AZ_OK) rc = search_export(e, run, n, visits_out, scores_out, depth_out);
    return rc;
}

int az_search_vl(az_engine* e, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                 int num_simulations, int leaves_per_root, float virtual_loss, const uint64_t* noise_game_ids, const uint32_t* noise_plies,
                 float* visits_out, float* scores_out, int32_t* depth_out, az_search_stats* stats_out) {
    return search_vl_run(e, n, roots, history, hist_offsets, num_simulations, leaves_per_root, virtual_loss, nullptr, noise_game_ids,
                         noise_plies, visits_out, scores_out, depth_out, stats_out);
}

int az_search_networks(az_engine* e, int n, const az_position* roots, const az_position* history, const uint32_t* hist_offsets,
                       int num_simulations, int leaves_per_root, float virtual_loss, const uint8_t* network, const uint64_t* noise_game_ids,
                       const uint32_t* noise_plies, float* visits_out, float* scores_out, int32_t* depth_out, az_search_stats* stats_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (n > 0 && !network) {
        if (stats_out) std::memset(stats_out, 0, sizeof *stats_out);
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null network buffer");
    }
    return search_vl_run(e, n, roots, history, hist_offsets, num_simulations, leaves_per_root, virtual_loss, network, noise_game_ids,
                         noise_plies, visits_out, scores_out, depth_out, stats_out);
}

int az_selfplay_begin(az_engine* e, int n_games, uint64_t first_game_id) { return az_selfplay_begin_n(e, n_games, first_game_id, 0); }

int az_selfplay_begin_n(az_engine* e, int n_games, uint64_t first_game_id, uint64_t total_games) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    return selfplay_begin(e, n_games, first_game_id, total_games, 0, 0.0f);
}

int az_selfplay_begin_vl(az_engine* e, int n_concurrent, uint64_t first_game_id, uint64_t total_games, int leaves_per_game,
                         float virtual_loss) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    const int r = check_vl_args(e, leaves_per_game, virtual_loss, "leaves_per_game");
    if (r) return r;
    return selfplay_begin(e, n_concurrent, first_game_id, total_games, leaves_per_game, virtual_loss);
}

int az_selfplay_vl_stats(az_engine* e, az_search_stats* out) {
    if (!e || !out) return AZ_ERR_INVALID_ARGUMENT;
    std::memset(out, 0, sizeof *out);
    SearchState* st = e->search;
    if (st->session != Session::selfplay_vl) return set_err(e, AZ_ERR_STATE, "az_selfplay_begin_vl has not been called");
    cudaSetDevice(e->cfg.device);
    unsigned long long s[4];
    AZ_CUDA(e, cudaMemcpyAsync(s, st->vl_stats, sizeof s, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    *out = vl_search_stats(s, st->sp_vl.waves);
    return AZ_OK;
}

int az_selfplay_step(az_engine* e, int waves, az_selfplay_stats* out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    SearchState* st = e->search;
    if (!selfplay_on(st)) return set_err(e, AZ_ERR_STATE, "az_selfplay_begin has not been called");
    cudaSetDevice(e->cfg.device);
    const bool vl = st->session == Session::selfplay_vl;
    for (int w = 0; w < waves; w++) {
        int r = vl ? run_wave_vl(e, st) : run_wave(e, st);
        if (r) return r;
    }
    Counters c;
    unsigned long long stripes[STAT_STRIPES * STAT_WIDTH];
    int flags[4] = {0, 0, 0, 0};
    const int r = enqueue_poll(e, *st, st->prm.n_games, flags);
    if (r) return r;
    AZ_CUDA(e, cudaMemcpyAsync(&c, st->ptr.counters, sizeof c, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(stripes, st->ptr.stats, sizeof stripes, cudaMemcpyDeviceToHost, e->stream));
    unsigned long long vls[4] = {0, 0, 0, 0};
    if (vl) AZ_CUDA(e, cudaMemcpyAsync(vls, st->vl_stats, sizeof vls, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    {
        unsigned long long sum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        unsigned long long evictions = 0, sdepth = 0;
        for (int i = 0; i < STAT_STRIPES * STAT_WIDTH; i++) {
            const int f = i % STAT_WIDTH;
            if (f < 8) sum[f] += stripes[i];
            if (f == 16) evictions += stripes[i];
            if (f == 17) sdepth += stripes[i];
        }
        st->cache_evictions = evictions;
        st->sum_search_depth = sdepth;
#ifdef AZ_ADV_TIMING
        adv_timing_report(stripes, st->prm.n_games, waves);
#endif
        c.simulations = sum[0]; c.positions = sum[1]; c.evaluations = sum[2]; c.cache_hits = sum[3];
        c.terminal_leaves = sum[4]; c.games_finished = sum[5]; c.sum_leaf_depth = sum[6]; c.sum_edges = sum[7];
        if (vl) {   // k_vl_expand counts the terminal leaves
            const az_search_stats v = vl_search_stats(vls, 0);
            c.evaluations = v.evaluations; c.terminal_leaves = v.terminal_leaves;
        }
    }
    if (out) {
        out->simulations = c.simulations; out->positions = c.positions; out->evaluations = c.evaluations; out->cache_hits = c.cache_hits;
        out->terminal_leaves = c.terminal_leaves; out->games_finished = c.games_finished; out->sum_leaf_depth = c.sum_leaf_depth;
        out->sum_edges = c.sum_edges; out->waves = (uint64_t)waves; out->pending_samples = std::min<unsigned long long>(c.samples_out, st->prm.sample_cap);
        out->active_games = (uint64_t)(flags[0] + flags[2]); out->parked_games = (uint64_t)flags[2]; out->cache_evictions = st->cache_evictions;
        out->sum_search_depth = st->sum_search_depth;
    }
    if (c.errors || flags[1]) return set_err(e, AZ_ERR_CAPACITY, "a per-game node/edge pool overflowed during self-play (raise edge_capacity_per_node)");
    return AZ_OK;
}

int az_selfplay_drain(az_engine* e, az_sample* out, int max_samples, int* n_out) {
    return selfplay_drain(e, out, max_samples, n_out, cudaMemcpyDeviceToHost);
}

int az_selfplay_drain_dev(az_engine* e, az_sample* out_dev, int max_samples, int* n_out) {
    return selfplay_drain(e, out_dev, max_samples, n_out, cudaMemcpyDeviceToDevice);
}

/* test hook: the EpisodeSteps the game in slot `slot` has staged so far (they are published when the game ends) */
int az_dbg_selfplay_staged(az_engine* e, int slot, az_sample* out, int max_samples, int* n_out) {
    if (!e || !out || !n_out) return AZ_ERR_INVALID_ARGUMENT;
    SearchState* st = e->search;
    if (!selfplay_on(st)) return set_err(e, AZ_ERR_STATE, "az_selfplay_begin has not been called");
    if (slot < 0 || slot >= st->prm.n_games) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "slot out of range");
    cudaSetDevice(e->cfg.device);
    GameCtl c;
    AZ_CUDA(e, cudaMemcpyAsync(&c, st->ptr.ctl + slot, sizeof c, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    const int n = std::min<int>((int)c.n_samples, max_samples);
    if (n) {
        AZ_CUDA(e, cudaMemcpyAsync(out, st->ptr.game_samples + (size_t)slot * MAX_SAMPLE_PLIES, (size_t)n * sizeof(az_sample),
                                   cudaMemcpyDeviceToHost, e->stream));
        AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    }
    *n_out = n;
    return AZ_OK;
}

int az_match_begin(az_engine* e, int n_concurrent, uint32_t first_game, uint32_t n_games, const az_match_config* cfg) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (!cfg) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null config");
    SearchState* st = e->search;
    const bool mcts = cfg->player_kind == 0;
    if (cfg->player_kind != 0 && cfg->player_kind != 1) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "player_kind must be 0 (MCTS) or 1 (BaseModel)");
    if (cfg->network[0] >= AZ_MAX_NETWORKS || cfg->network[1] >= AZ_MAX_NETWORKS)
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "network id must be < AZ_MAX_NETWORKS");
    const int S = cfg->num_simulations ? cfg->num_simulations : e->cfg.num_simulations;
    if (mcts) {
        const int r = check_vl_args(e, cfg->leaves_per_root, cfg->virtual_loss, "leaves_per_root");
        if (r) return r;
        if (S < 1 || S > e->cfg.num_simulations)
            return set_err(e, AZ_ERR_INVALID_ARGUMENT, "num_simulations must be in 1 .. az_config.num_simulations");
    }
    if (n_concurrent < 1 || n_games == 0 || cfg->max_plies == 0)
        return set_err(e, AZ_ERR_INVALID_ARGUMENT, "n_concurrent, n_games and max_plies must be positive");
    const int K = mcts ? cfg->leaves_per_root : 1;
    if (n_concurrent > st->G) return set_err(e, AZ_ERR_CAPACITY, "more slots than az_config.max_games");
    const int n = (int)std::min<uint64_t>((uint64_t)n_concurrent, n_games);
    if (net_layout(n, n, K).end > (long long)e->max_batch)   // at worst every slot's mover is on the same network
        return set_err(e, AZ_ERR_CAPACITY, "network ranges (2 x round4(slots x leaves_per_root)) exceed az_config.max_batch");
    if (e->stub_kind == 0) {
        for (int p = 0; p < 2; p++) {
            const NetWeights* w = net_slot(e, cfg->network[p]);
            if (!w || !w->loaded) return set_err(e, AZ_ERR_NO_WEIGHTS, "a player names a network that has not been loaded");
        }
        const int r = net_networks_supported(e);
        if (r) return r;
    }
    cudaSetDevice(e->cfg.device);
    int r = vl_alloc(e, st);
    if (r) return r;
    if (!st->d_net && salloc(e, st, &st->d_net, (size_t)st->G)) return AZ_ERR_OUT_OF_MEMORY;
    const uint32_t row = std::min<uint32_t>(cfg->max_plies, HIST_CAP);   // a game ends by the fullmove rule before HIST_CAP plies
    r = match_alloc(e, st, n_games, row);
    if (r) return r;
    st->session = Session::none;
    MatchState& m = st->match;
    m.cfg = *cfg;
    m.cfg.num_simulations = S;
    m.first = first_game;
    m.games = n_games;
    m.K = K;
    m.row = row;
    m.first_wave = 1;
    m.waves = 0;
    az_position_start(&m.startpos);
    st->prm.n_games = n; st->prm.S = S; st->prm.mode = 0;
    st->prm.priors_scattered = fused_heads(e) ? 1 : 0;
    st->ptr.batch_count = st->batch_base;
    st->ptr.batch_zero = nullptr;
    const unsigned long long next = first_game;
    AZ_CUDA(e, cudaMemcpyAsync(m.next, &next, sizeof next, cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemsetAsync(m.stats, 0, 4 * sizeof(unsigned long long), e->stream));
    if ((r = vl_clear(e, st, 0))) return r;   // k_match sets every slot's leaf count in the first wave
    AZ_CUDA(e, cudaMemsetAsync(m.result.p, 0, n_games, e->stream));
    AZ_CUDA(e, cudaMemsetAsync(m.plies.p, 0, (size_t)n_games * sizeof(uint16_t), e->stream));
    AZ_CUDA(e, cudaMemsetAsync(m.finished.p, 0, n_games, e->stream));
    AZ_CUDA(e, cudaMemsetAsync(m.moves.p, 0xFF, (size_t)n_games * row * sizeof(uint16_t), e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    st->session = Session::match;
    return AZ_OK;
}

int az_match_step(az_engine* e, int waves, az_match_stats* out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (out) std::memset(out, 0, sizeof *out);
    SearchState* st = e->search;
    if (st->session != Session::match) return set_err(e, AZ_ERR_STATE, "no match in progress (az_match_begin)");
    cudaSetDevice(e->cfg.device);
    MatchState& m = st->match;
    // a slot queues at most K boards per wave (its batch or its next root), all in its mover's range
    const int n = st->prm.n_games, base1 = (int)net_layout(n, n, m.K).base1;
    const VLPtrs vl = vl_ptrs(st, m.K, m.cfg.virtual_loss);
    const NetRoute route{st->d_net, st->batch_base, base1};
    const NetBatch nb{st->batch_base, base1, base1 + n * m.K};
    for (int w = 0; w < waves; w++) {
        const MatchParams mp = match_params(st);
        AZ_CUDA(e, cudaMemsetAsync(st->batch_base, 0, AZ_MAX_NETWORKS * sizeof(int), e->stream));   // both ranges start empty
        prof_mark_search(e);
        e->n_launches += 2;
        k_match<<<(n + WARPS - 1) / WARPS, WARPS * 32, 0, e->stream>>>(st->prm, st->ptr, vl, route, mp);
        AZ_CUDA(e, cudaGetLastError());
        const int r = vl_expand_evaluate(e, st, vl, n, &route, &nb);
        if (r) return r;
        m.first_wave = 0;
        m.waves++;
    }
    int flags[4] = {0, 0, 0, 0};
    unsigned long long ms[4], vs[4];
    const int r = enqueue_poll(e, *st, n, flags);
    if (r) return r;
    AZ_CUDA(e, cudaMemcpyAsync(ms, m.stats, sizeof ms, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(vs, st->vl_stats, sizeof vs, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    if (out) {
        out->waves = m.waves;
        out->evaluations[0] = ms[0]; out->evaluations[1] = ms[1];
        out->leaves = vs[0]; out->terminal_leaves = vs[1]; out->collisions = vs[2];
        out->plies = ms[2]; out->games_finished = ms[3];
        out->active_games = m.first_wave ? std::min<uint64_t>((uint64_t)n, m.games) : (uint64_t)flags[0];
    }
    if (flags[1]) return set_err(e, AZ_ERR_CAPACITY, "a per-game node/edge pool overflowed during the match (raise edge_capacity_per_node)");
    return AZ_OK;
}

int az_match_results(az_engine* e, int8_t* result_out, uint16_t* plies_out, uint8_t* finished_out, uint16_t* moves_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    const MatchState& m = e->search->match;
    if (!m.games) return set_err(e, AZ_ERR_STATE, "az_match_begin has not been called");
    if (!result_out || !plies_out || !finished_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    cudaSetDevice(e->cfg.device);
    const size_t n = m.games;
    AZ_CUDA(e, cudaMemcpyAsync(result_out, m.result.p, n, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(plies_out, m.plies.p, n * sizeof(uint16_t), cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(finished_out, m.finished.p, n, cudaMemcpyDeviceToHost, e->stream));
    if (moves_out) {   // [n][max_plies]: the device keeps row <= max_plies moves per game, the rest is AZ_MOVE_NONE
        const size_t mp = m.cfg.max_plies, row = m.row;
        if (row < mp) std::memset(moves_out, 0xFF, n * mp * sizeof(uint16_t));
        AZ_CUDA(e, cudaMemcpy2DAsync(moves_out, mp * sizeof(uint16_t), m.moves.p, row * sizeof(uint16_t), row * sizeof(uint16_t), n,
                                     cudaMemcpyDeviceToHost, e->stream));
    }
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

}  // extern "C"
