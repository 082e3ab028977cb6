// C ABI: engine lifetime and the batched chess.rs entry points (host staging + kernel launches).
#include "engine.h"
#include "nn.h"
#include "mcts.h"
#include <cstring>
#include <cstdio>
#include <cctype>
#include <cstdlib>
#include <algorithm>

namespace azb {

int set_err(az_engine* e, int code, const char* what) {
    if (e) e->err = what;
    return code;
}
int check_cuda(az_engine* e, cudaError_t r, const char* what) {
    if (r == cudaSuccess) return 0;
    if (e) e->err = std::string(what) + ": " + cudaGetErrorString(r);
    return r == cudaErrorMemoryAllocation ? AZ_ERR_OUT_OF_MEMORY : AZ_ERR_CUDA;
}

}  // namespace azb

using namespace azb;

extern "C" {

const char* az_version(void) { return "az_b200 0.1 (sm_100a)"; }

void az_config_default(az_config* c) {
    std::memset(c, 0, sizeof *c);
    c->device = 0;
    c->max_games = 4096;
    c->max_batch = 0;
    c->num_simulations = 256;       // parameters.rs:32
    c->c_puct = 3.0f;               // parameters.rs:34
    c->dirichlet_alpha = 0.3f;      // parameters.rs:28
    c->dirichlet_epsilon = 0.25f;   // parameters.rs:29
    c->temperature_annealing = 15;  // parameters.rs:31
    c->num_halfmoves = 100;         // chess.rs:9
    c->num_fullmoves = 200;         // chess.rs:10
    c->repetitions = 3;             // chess.rs:11
    c->seed = 42;                   // parameters.rs:6
    c->precision = 0;
    c->cache_log2 = 0;
    c->edge_capacity_per_node = 0;
    c->temperature = 1.0f;          // parameters.rs:33
}

const char* az_last_error(const az_engine* e) { return e ? e->err.c_str() : "null engine"; }

void az_position_start(az_position* out) {
    az_position_from_fen("rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1", out);
}

int az_position_from_fen(const char* fen, az_position* out) {
    if (!fen || !out) return AZ_ERR_INVALID_ARGUMENT;
    az_position p;
    std::memset(&p, 0, sizeof p);
    p.ep_square = -1; p.fullmoves = 1;
    int r = 7, f = 0;
    const char* c = fen;
    for (; *c && *c != ' '; c++) {
        if (*c == '/') { r--; f = 0; continue; }
        if (isdigit((unsigned char)*c)) { f += *c - '0'; continue; }
        int role;
        switch (tolower((unsigned char)*c)) {
            case 'p': role = 0; break; case 'n': role = 1; break; case 'b': role = 2; break;
            case 'r': role = 3; break; case 'q': role = 4; break; case 'k': role = 5; break;
            default: return AZ_ERR_INVALID_ARGUMENT;
        }
        if (r < 0 || f > 7) return AZ_ERR_INVALID_ARGUMENT;
        uint64_t b = 1ULL << (r * 8 + f);
        p.roles[role] |= b;
        p.colors[isupper((unsigned char)*c) ? 0 : 1] |= b;
        f++;
    }
    if (*c != ' ') return AZ_ERR_INVALID_ARGUMENT;
    c++;
    p.turn = *c == 'b' ? 1 : 0;
    if (*c) c++;
    if (*c == ' ') c++;
    for (; *c && *c != ' '; c++) {
        if (*c == 'K') p.castling |= 1; else if (*c == 'Q') p.castling |= 2;
        else if (*c == 'k') p.castling |= 4; else if (*c == 'q') p.castling |= 8;
    }
    if (*c == ' ') c++;
    if (*c && *c != '-') { p.ep_square = (int8_t)((c[1] - '1') * 8 + (c[0] - 'a')); c += 2; } else if (*c) c++;
    char* endp;
    if (*c == ' ') { p.halfmoves = (uint16_t)strtol(c + 1, &endp, 10); c = endp; }
    if (*c == ' ') { p.fullmoves = (uint16_t)strtol(c + 1, &endp, 10); c = endp; }
    *out = p;
    return AZ_OK;
}

int az_engine_create(const az_config* cfg, az_engine** out) {
    if (!cfg || !out) return AZ_ERR_INVALID_ARGUMENT;
    if (cfg->max_games <= 0 || cfg->num_simulations <= 0) return AZ_ERR_INVALID_ARGUMENT;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return AZ_ERR_NO_DEVICE;
    if (cfg->device < 0 || cfg->device >= ndev) return AZ_ERR_INVALID_ARGUMENT;
    az_engine* e = new az_engine;
    e->cfg = *cfg;
    e->max_batch = cfg->max_batch > 0 ? cfg->max_batch : cfg->max_games;
    if (e->max_batch < cfg->max_games) e->max_batch = cfg->max_games;
    *out = e;
    AZ_CUDA(e, cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    AZ_CUDA(e, cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) { e->err = "this library contains sm_100a code only (Blackwell B200 required)"; return AZ_ERR_NO_DEVICE; }
    e->sm_count = prop.multiProcessorCount;
    AZ_CUDA(e, cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    {
        auto env_int = [](const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; };
        e->knobs.tower_fused = env_int("AZ_TOWER_FUSED", 1);
        e->knobs.tower_split = std::max(0, env_int("AZ_TOWER_SPLIT", 0));
        e->knobs.tower_inkernel = env_int("AZ_TOWER_INKERNEL", 1);
        e->knobs.tc_release_arrive = env_int("AZ_TC_RELEASE_ARRIVE", 0);
        e->knobs.tower_grid = std::max(0, env_int("AZ_TOWER_GRID", 0));
        e->knobs.tower_wide = std::min(2, std::max(0, env_int("AZ_TOWER_WIDE", 2)));
        e->knobs.tower_l2hint = env_int("AZ_TOWER_L2HINT", 1) & 15;
        e->knobs.input_epi2 = env_int("AZ_INPUT_EPI2", 0) ? 1 : 0;
        e->knobs.heads_tc = env_int("AZ_HEADS_TC", 1) ? 1 : 0;
        e->knobs.input_k32 = env_int("AZ_INPUT_K32", 1) ? 1 : 0;
    }
    const size_t nb = (size_t)e->max_batch;
    AZ_CUDA(e, cudaMalloc(&e->d_wire, nb * sizeof(az_position)));
    AZ_CUDA(e, cudaMalloc(&e->d_hist_off, (nb + 1) * sizeof(uint32_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_moves, nb * AZ_MAX_MOVES * sizeof(uint16_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_index, nb * AZ_MAX_MOVES * sizeof(uint16_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_count, nb * sizeof(int32_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_u16a, nb * sizeof(uint16_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_u16b, nb * sizeof(uint16_t)));
    AZ_CUDA(e, cudaMalloc(&e->d_planes, nb * AZ_NUM_PLANES * 64 * sizeof(float)));
    AZ_CUDA(e, cudaMalloc(&e->d_policy, nb * AZ_ACTION_SPACE * sizeof(float)));
    AZ_CUDA(e, cudaMalloc(&e->d_value, nb * sizeof(float)));
    AZ_CUDA(e, cudaMalloc(&e->d_perft_count, sizeof(unsigned long long)));
    int r = net_create(e);
    if (r) return r;
    r = search_create(e);
    if (r) return r;
    return AZ_OK;
}

void az_engine_destroy(az_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    search_destroy(e);
    net_destroy(e);
    cudaFree(e->d_wire); cudaFree(e->d_hist); cudaFree(e->d_hist_off); cudaFree(e->d_moves); cudaFree(e->d_index);
    cudaFree(e->d_count); cudaFree(e->d_u16a); cudaFree(e->d_u16b); cudaFree(e->d_planes); cudaFree(e->d_policy);
    cudaFree(e->d_value); cudaFree(e->d_scores); cudaFree(e->d_perft_count); cudaFree(e->d_perft_nodes);
    for (auto p : e->perft_pos) cudaFree(p);
    for (auto p : e->perft_root) cudaFree(p);
    for (auto p : e->mm_score) cudaFree(p);
    cudaFree(e->d_mm_first); cudaFree(e->d_mm_nchild); cudaFree(e->d_mm_out); cudaFree(e->d_mm_count);
    for (auto& ps : e->prof_pending) { if (ps.adv) cudaEventDestroy(ps.adv); cudaEventDestroy(ps.in0); cudaEventDestroy(ps.a); cudaEventDestroy(ps.b); cudaEventDestroy(ps.h1); }
    if (e->prof_counts_host) cudaFreeHost(e->prof_counts_host);
    if (e->timer0) { cudaEventDestroy(e->timer0); cudaEventDestroy(e->timer1); }
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

static int check_batch(az_engine* e, int n) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (n < 0) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "negative batch");
    if (n > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "batch larger than az_config.max_batch");
    cudaSetDevice(e->cfg.device);
    return 0;
}

int az_timer_start(az_engine* e) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    cudaSetDevice(e->cfg.device);
    if (!e->timer0) { AZ_CUDA(e, cudaEventCreate(&e->timer0)); AZ_CUDA(e, cudaEventCreate(&e->timer1)); }
    AZ_CUDA(e, cudaEventRecord(e->timer0, e->stream));
    return AZ_OK;
}
int az_timer_stop(az_engine* e, float* ms_out) {
    if (!e || !ms_out || !e->timer0) return AZ_ERR_INVALID_ARGUMENT;
    cudaSetDevice(e->cfg.device);
    AZ_CUDA(e, cudaEventRecord(e->timer1, e->stream));
    AZ_CUDA(e, cudaEventSynchronize(e->timer1));
    AZ_CUDA(e, cudaEventElapsedTime(ms_out, e->timer0, e->timer1));
    return AZ_OK;
}
int az_profile_enable(az_engine* e, int every) {
    if (!e || every < 0) return AZ_ERR_INVALID_ARGUMENT;
    cudaSetDevice(e->cfg.device);
    if (every > 0 && !e->prof_counts_host) AZ_CUDA(e, cudaMallocHost(&e->prof_counts_host, 4096 * sizeof(int)));
    e->prof_every = every;
    e->prof_counter = 0;
    return AZ_OK;
}
int az_profile_read(az_engine* e, az_profile* out) {
    if (!e || !out) return AZ_ERR_INVALID_ARGUMENT;
    cudaSetDevice(e->cfg.device);
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    for (auto& ps : e->prof_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ps.a, ps.b) == cudaSuccess) {
            e->prof_ms += ms; e->prof_samples++; e->prof_boards += (uint64_t)e->prof_counts_host[ps.slot];
            if (cudaEventElapsedTime(&ms, ps.in0, ps.a) == cudaSuccess) e->prof_input_ms += ms;
            if (cudaEventElapsedTime(&ms, ps.b, ps.h1) == cudaSuccess) e->prof_heads_ms += ms;
            if (ps.adv && cudaEventElapsedTime(&ms, ps.adv, ps.in0) == cudaSuccess) e->prof_adv_ms += ms;
        }
        if (ps.adv) cudaEventDestroy(ps.adv);
        cudaEventDestroy(ps.in0); cudaEventDestroy(ps.a); cudaEventDestroy(ps.b); cudaEventDestroy(ps.h1);
    }
    e->prof_pending.clear();
    out->tower_ms = e->prof_ms; out->tower_samples = e->prof_samples; out->tower_boards = e->prof_boards;
    out->tower_launches = e->prof_launches;
    out->input_ms = e->prof_input_ms; out->heads_ms = e->prof_heads_ms; out->advance_ms = e->prof_adv_ms;
    e->prof_ms = 0; e->prof_samples = 0; e->prof_boards = 0; e->prof_launches = 0; e->prof_input_ms = 0; e->prof_heads_ms = 0; e->prof_adv_ms = 0;
    return AZ_OK;
}
uint64_t az_launch_count(const az_engine* e) { return e ? e->n_launches : 0; }

int az_movegen(az_engine* e, int n, const az_position* pos, az_move* moves_out, uint16_t* index_out, int32_t* count_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !moves_out || !count_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    e->n_launches++;
    launch_movegen(e->stream, e->d_wire, n, e->d_moves, index_out ? e->d_index : nullptr, e->d_count);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(moves_out, e->d_moves, (size_t)n * AZ_MAX_MOVES * 2, cudaMemcpyDeviceToHost, e->stream));
    if (index_out) AZ_CUDA(e, cudaMemcpyAsync(index_out, e->d_index, (size_t)n * AZ_MAX_MOVES * 2, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(count_out, e->d_count, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_dbg_movegen_warp(az_engine* e, int n, const az_position* pos, az_move* moves_out, int32_t* count_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !moves_out || !count_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    e->n_launches++;
    launch_movegen_warp(e->stream, e->d_wire, n, e->d_moves, e->d_count);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(moves_out, e->d_moves, (size_t)n * AZ_MAX_MOVES * 2, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(count_out, e->d_count, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_play_move(az_engine* e, int n, az_position* pos_inout, const az_position* history, const uint32_t* hist_offsets,
                 const uint16_t* action_index, int32_t* result_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos_inout || !action_index || !result_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    const az_position* d_hist = nullptr;
    if (history && hist_offsets) {
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
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos_inout, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_u16a, action_index, (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
    RuleParams rp{(int)e->cfg.num_halfmoves, (int)e->cfg.num_fullmoves, (int)e->cfg.repetitions};
    e->n_launches++;
    launch_play_move(e->stream, e->d_wire, d_hist, e->d_hist_off, e->d_u16a, e->d_count, n, rp);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(pos_inout, e->d_wire, (size_t)n * sizeof(az_position), cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(result_out, e->d_count, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_move_to_index(az_engine* e, int n, const az_position* pos, const az_move* moves, uint16_t* index_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !moves || !index_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_u16a, moves, (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
    e->n_launches++;
    launch_move_to_index(e->stream, e->d_wire, e->d_u16a, e->d_u16b, n);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(index_out, e->d_u16b, (size_t)n * 2, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_index_to_move(az_engine* e, int n, const az_position* pos, const uint16_t* index, az_move* moves_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !index || !moves_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_u16a, index, (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
    e->n_launches++;
    launch_index_to_move(e->stream, e->d_wire, e->d_u16a, e->d_u16b, n);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(moves_out, e->d_u16b, (size_t)n * 2, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_encode(az_engine* e, int n, const az_position* pos, float* planes_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !planes_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    e->n_launches++;
    launch_encode_f32(e->stream, e->d_wire, e->d_planes, n);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(planes_out, e->d_planes, (size_t)n * AZ_NUM_PLANES * 64 * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

// ------------------------------------------------------------------------------------------------- perft
// Breadth-first over device-resident level buffers.  A chunk of parents is sized so that even 218 children each fit the
// next level's buffer; the last ply is bulk-counted without materialising positions.
static int perft_buffers(az_engine* e, int level) {  // level buffers shared by az_perft and az_minimax
    if (e->perft_cap == 0) {
        e->perft_cap = std::max<size_t>((size_t)1 << 24, (size_t)e->max_batch);
        AZ_CUDA(e, cudaMalloc(&e->d_perft_nodes, (size_t)e->max_batch * sizeof(unsigned long long)));
    }
    while ((int)e->perft_pos.size() <= level) {
        DPos* p = nullptr; uint32_t* q = nullptr;
        AZ_CUDA(e, cudaMalloc(&p, e->perft_cap * sizeof(DPos)));
        e->perft_pos.push_back(p);
        AZ_CUDA(e, cudaMalloc(&q, e->perft_cap * sizeof(uint32_t)));
        e->perft_root.push_back(q);
    }
    return 0;
}

static int perft_level(az_engine* e, int level, size_t n, int depth_remaining) {
    if (depth_remaining == 1) {
        const size_t step = 1u << 24;
        for (size_t s = 0; s < n; s += step)
            e->n_launches++, launch_perft_count(e->stream, e->perft_pos[level] + s, e->perft_root[level] + s, (int)std::min(step, n - s), e->d_perft_nodes);
        AZ_CUDA(e, cudaGetLastError());
        return 0;
    }
    if (int rb = perft_buffers(e, level + 1)) return rb;
    const size_t chunk = e->perft_cap / 218;
    for (size_t s = 0; s < n; s += chunk) {
        size_t m = std::min(chunk, n - s);
        AZ_CUDA(e, cudaMemsetAsync(e->d_perft_count, 0, sizeof(unsigned long long), e->stream));
        e->n_launches++;
        launch_perft_expand(e->stream, e->perft_pos[level] + s, e->perft_root[level] + s, (int)m, e->perft_pos[level + 1],
                            e->perft_root[level + 1], e->d_perft_count);
        AZ_CUDA(e, cudaGetLastError());
        unsigned long long produced = 0;
        AZ_CUDA(e, cudaMemcpyAsync(&produced, e->d_perft_count, sizeof produced, cudaMemcpyDeviceToHost, e->stream));
        AZ_CUDA(e, cudaStreamSynchronize(e->stream));
        if (produced > e->perft_cap) return set_err(e, AZ_ERR_CAPACITY, "perft level buffer overflow");
        int r = perft_level(e, level + 1, (size_t)produced, depth_remaining - 1);
        if (r) return r;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------- minimax
// negamax(node, d) for the n nodes of `level` into mm_score[level]; chunks are sized like perft's.
static int mm_level(az_engine* e, int level, size_t n, int d, int* scores_out_dev, int* count_out_dev) {
    while ((int)e->mm_score.size() <= level + 1) {
        int* p = nullptr;
        AZ_CUDA(e, cudaMalloc(&p, e->perft_cap * sizeof(int)));
        e->mm_score.push_back(p);
    }
    if (d == 0) {
        e->n_launches++;
        launch_mm_leaf(e->stream, e->perft_pos[level], (int)n, e->mm_score[level]);
        AZ_CUDA(e, cudaGetLastError());
        return 0;
    }
    int r = perft_buffers(e, level + 1);
    if (r) return r;
    const bool root = level == 0;
    const size_t chunk = e->perft_cap / 218;
    for (size_t s = 0; s < n; s += chunk) {
        const size_t m = std::min(chunk, n - s);
        AZ_CUDA(e, cudaMemsetAsync(e->d_perft_count, 0, sizeof(unsigned long long), e->stream));
        e->n_launches++;
        launch_mm_expand(e->stream, e->perft_pos[level] + s, (int)m, d, root ? 1 : 0, e->perft_pos[level + 1], e->perft_root[level + 1],
                         e->d_perft_count, e->mm_score[level] + s, root ? e->d_mm_first + s : nullptr, root ? e->d_mm_nchild + s : nullptr);
        AZ_CUDA(e, cudaGetLastError());
        unsigned long long produced = 0;
        AZ_CUDA(e, cudaMemcpyAsync(&produced, e->d_perft_count, sizeof produced, cudaMemcpyDeviceToHost, e->stream));
        AZ_CUDA(e, cudaStreamSynchronize(e->stream));
        if (produced > e->perft_cap) return set_err(e, AZ_ERR_CAPACITY, "minimax level buffer overflow");
        r = mm_level(e, level + 1, (size_t)produced, d - 1, nullptr, nullptr);
        if (r) return r;
        e->n_launches++;
        if (root)
            launch_mm_root(e->stream, e->d_mm_first + s, e->d_mm_nchild + s, e->mm_score[level + 1], (int)m,
                           scores_out_dev + s * AZ_MAX_MOVES, count_out_dev + s);
        else
            launch_mm_backup(e->stream, e->mm_score[level + 1], e->perft_root[level + 1], (int)produced, e->mm_score[level] + s);
        AZ_CUDA(e, cudaGetLastError());
    }
    return 0;
}

int az_minimax(az_engine* e, int n, const az_position* pos, int depth, int32_t* scores_out, int32_t* count_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !scores_out || !count_out || depth < 1 || depth > 8) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "bad minimax arguments");
    r = perft_buffers(e, 0);
    if (r) return r;
    if (!e->d_mm_out) {
        AZ_CUDA(e, cudaMalloc(&e->d_mm_first, (size_t)e->max_batch * sizeof(unsigned int)));
        AZ_CUDA(e, cudaMalloc(&e->d_mm_nchild, (size_t)e->max_batch * sizeof(int)));
        AZ_CUDA(e, cudaMalloc(&e->d_mm_count, (size_t)e->max_batch * sizeof(int)));
        AZ_CUDA(e, cudaMalloc(&e->d_mm_out, (size_t)e->max_batch * AZ_MAX_MOVES * sizeof(int)));
    }
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    launch_wire_to_dpos(e->stream, e->d_wire, e->perft_pos[0], e->perft_root[0], n);
    r = mm_level(e, 0, (size_t)n, depth, e->d_mm_out, e->d_mm_count);
    if (r) return r;
    AZ_CUDA(e, cudaMemcpyAsync(scores_out, e->d_mm_out, (size_t)n * AZ_MAX_MOVES * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(count_out, e->d_mm_count, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_perft(az_engine* e, int n, const az_position* pos, int depth, uint64_t* nodes_out) {
    int r = check_batch(e, n);
    if (r || n == 0) return r;
    if (!pos || !nodes_out || depth < 0 || depth > 12) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "bad perft arguments");
    if (depth == 0) { for (int i = 0; i < n; i++) nodes_out[i] = 1; return AZ_OK; }
    r = perft_buffers(e, 0);
    if (r) return r;
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemsetAsync(e->d_perft_nodes, 0, (size_t)n * sizeof(unsigned long long), e->stream));
    launch_wire_to_dpos(e->stream, e->d_wire, e->perft_pos[0], e->perft_root[0], n);
    r = perft_level(e, 0, (size_t)n, depth);
    if (r) return r;
    AZ_CUDA(e, cudaMemcpyAsync(nodes_out, e->d_perft_nodes, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

}  // extern "C"
