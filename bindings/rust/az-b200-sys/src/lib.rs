//! Raw bindings to `libaz_b200.so` (include/az_b200.h), 1:1 with the header.
//!
//! SOURCE ONLY: the image this project is built in has no Rust toolchain, so this crate has never been compiled; it is
//! kept in sync with the header by `tests/test_abi_cpu.py::test_rust_bindings_list_every_header_function`, which checks
//! that every function the header declares has an `extern "C"` declaration here.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)] #[derive(Clone, Copy)]
pub struct az_position { pub roles: [u64; 6], pub colors: [u64; 2], pub turn: u8, pub castling: u8,
                         pub ep_square: i8, pub reserved: u8, pub halfmoves: u16, pub fullmoves: u16 }   // 72 bytes
#[repr(C)] #[derive(Clone, Copy)]
pub struct az_config { pub device: i32, pub max_games: i32, pub max_batch: i32, pub num_simulations: i32,
                       pub c_puct: f32, pub dirichlet_alpha: f32, pub dirichlet_epsilon: f32,
                       pub temperature_annealing: u32, pub num_halfmoves: u32, pub num_fullmoves: u32,
                       pub repetitions: u32, pub seed: u64, pub precision: i32, pub cache_log2: i32,
                       pub edge_capacity_per_node: i32, pub temperature: f32 }
#[repr(C)] pub struct az_sample { pub position: az_position, pub final_value: f32, pub search_depth: i32,
                                  pub game_id: u64, pub ply: u32, pub action: u16, pub n_visits: u16,
                                  pub index: [u16; 256], pub count: [u16; 256] }                          // 1120 bytes
#[repr(C)] #[derive(Default)] pub struct az_selfplay_stats { pub simulations: u64, pub positions: u64, pub evaluations: u64,
    pub cache_hits: u64, pub terminal_leaves: u64, pub games_finished: u64, pub sum_leaf_depth: u64, pub sum_edges: u64,
    pub waves: u64, pub pending_samples: u64, pub active_games: u64, pub parked_games: u64, pub cache_evictions: u64,
    pub sum_search_depth: u64 }
#[repr(C)] #[derive(Default)] pub struct az_search_stats { pub waves: u64, pub evaluations: u64, pub terminal_leaves: u64,
    pub collisions: u64 }                                                                       // not in the reference
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct az_match_config { pub player_kind: i32, pub network: [u8; 2],
    pub num_simulations: i32, pub leaves_per_root: i32, pub virtual_loss: f32, pub num_stochastic_moves: u32, pub max_plies: u32,
    pub seed: u64 }
#[repr(C)] #[derive(Default)] pub struct az_match_stats { pub waves: u64, pub evaluations: [u64; 2], pub leaves: u64,
    pub terminal_leaves: u64, pub collisions: u64, pub plies: u64, pub games_finished: u64, pub active_games: u64 }
pub enum az_engine {}

extern "C" {
    pub fn az_config_default(cfg: *mut az_config);
    pub fn az_engine_create(cfg: *const az_config, out: *mut *mut az_engine) -> c_int;
    pub fn az_engine_destroy(eng: *mut az_engine);
    pub fn az_last_error(eng: *const az_engine) -> *const c_char;
    pub fn az_position_start(out: *mut az_position);
    pub fn az_load_weights(eng: *mut az_engine, arrays: *const *const f32, n_arrays: c_int) -> c_int;
    pub fn az_forward_planes(eng: *mut az_engine, n: c_int, planes: *const f32, policy: *mut f32, value: *mut f32) -> c_int;
    pub fn az_forward(eng: *mut az_engine, n: c_int, pos: *const az_position, policy: *mut f32, value: *mut f32) -> c_int;
    pub fn az_load_network(eng: *mut az_engine, network: c_int, arrays: *const *const f32, n_arrays: c_int) -> c_int;
    pub fn az_forward_networks(eng: *mut az_engine, n: c_int, pos: *const az_position, network: *const u8, policy: *mut f32,
                               value: *mut f32) -> c_int;
    pub fn az_movegen(eng: *mut az_engine, n: c_int, pos: *const az_position, moves: *mut u16, index: *mut u16, count: *mut i32) -> c_int;
    pub fn az_perft(eng: *mut az_engine, n: c_int, pos: *const az_position, depth: c_int, nodes: *mut u64) -> c_int;
    pub fn az_play_move(eng: *mut az_engine, n: c_int, pos: *mut az_position, history: *const az_position,
                        hist_offsets: *const u32, action_index: *const u16, result: *mut i32) -> c_int;
    pub fn az_move_to_index(eng: *mut az_engine, n: c_int, pos: *const az_position, moves: *const u16, index: *mut u16) -> c_int;
    pub fn az_index_to_move(eng: *mut az_engine, n: c_int, pos: *const az_position, index: *const u16, moves: *mut u16) -> c_int;
    pub fn az_encode(eng: *mut az_engine, n: c_int, pos: *const az_position, planes: *mut f32) -> c_int;
    pub fn az_search(eng: *mut az_engine, n: c_int, roots: *const az_position, history: *const az_position,
                     hist_offsets: *const u32, num_simulations: c_int, noise_game_ids: *const u64, noise_plies: *const u32,
                     visits: *mut f32, scores: *mut f32, depth: *mut i32) -> c_int;
    pub fn az_search_vl(eng: *mut az_engine, n: c_int, roots: *const az_position, history: *const az_position,
                        hist_offsets: *const u32, num_simulations: c_int, leaves_per_root: c_int, virtual_loss: f32,
                        noise_game_ids: *const u64, noise_plies: *const u32, visits: *mut f32, scores: *mut f32, depth: *mut i32,
                        stats: *mut az_search_stats) -> c_int;
    pub fn az_search_networks(eng: *mut az_engine, n: c_int, roots: *const az_position, history: *const az_position,
                              hist_offsets: *const u32, num_simulations: c_int, leaves_per_root: c_int, virtual_loss: f32,
                              network: *const u8, noise_game_ids: *const u64, noise_plies: *const u32, visits: *mut f32,
                              scores: *mut f32, depth: *mut i32, stats: *mut az_search_stats) -> c_int;
    pub fn az_selfplay_begin(eng: *mut az_engine, n_games: c_int, first_game_id: u64) -> c_int;
    pub fn az_selfplay_begin_n(eng: *mut az_engine, n_concurrent: c_int, first_game_id: u64, total_games: u64) -> c_int;
    pub fn az_selfplay_begin_vl(eng: *mut az_engine, n_concurrent: c_int, first_game_id: u64, total_games: u64,
                                leaves_per_game: c_int, virtual_loss: f32) -> c_int;                 // not in the reference
    pub fn az_selfplay_vl_stats(eng: *mut az_engine, stats: *mut az_search_stats) -> c_int;
    pub fn az_selfplay_step(eng: *mut az_engine, waves: c_int, stats: *mut az_selfplay_stats) -> c_int;
    pub fn az_match_begin(eng: *mut az_engine, n_concurrent: c_int, first_game: u32, n_games: u32, config: *const az_match_config) -> c_int;
    pub fn az_match_step(eng: *mut az_engine, waves: c_int, stats: *mut az_match_stats) -> c_int;
    pub fn az_match_results(eng: *mut az_engine, result: *mut i8, plies: *mut u16, finished: *mut u8, moves: *mut u16) -> c_int;
    pub fn az_selfplay_drain(eng: *mut az_engine, out: *mut az_sample, max_samples: c_int, n_out: *mut c_int) -> c_int;
    pub fn az_selfplay_drain_dev(eng: *mut az_engine, out_dev: *mut az_sample, max_samples: c_int, n_out: *mut c_int) -> c_int;
    // callers beyond self-play (section 3)
    pub fn az_version() -> *const c_char;
    pub fn az_position_from_fen(fen: *const c_char, out: *mut az_position) -> c_int;
    pub fn az_weight_name(i: c_int) -> *const c_char;
    pub fn az_weight_size(i: c_int) -> i64;
    pub fn az_load_weights_dev(eng: *mut az_engine, arrays_dev: *const *const f32, n_arrays: c_int) -> c_int;
    pub fn az_set_evaluator_stub(eng: *mut az_engine, kind: c_int, seed: u64) -> c_int;
    pub fn az_minimax(eng: *mut az_engine, n: c_int, pos: *const az_position, depth: c_int, scores: *mut i32, count: *mut i32) -> c_int;
    pub fn az_replay_create(eng: *mut az_engine, capacity: c_int, max_batch: c_int, out: *mut *mut az_replay) -> c_int;
    pub fn az_replay_destroy(rp: *mut az_replay);
    pub fn az_replay_add(rp: *mut az_replay, samples: *const az_sample, n: c_int, new_unique: *mut c_int) -> c_int;
    pub fn az_replay_add_pending(rp: *mut az_replay, n_added: *mut c_int, new_unique: *mut c_int) -> c_int;
    pub fn az_replay_add_dev(rp: *mut az_replay, samples_dev: *const az_sample, n: c_int, new_unique: *mut c_int) -> c_int;
    pub fn az_replay_len(rp: *mut az_replay, len: *mut c_int) -> c_int;
    pub fn az_replay_sample(rp: *mut az_replay, batch: c_int, seed: u64, planes: *mut f32, policy: *mut f32, value: *mut f32, n_out: *mut c_int) -> c_int;
    pub fn az_replay_sample_dev(rp: *mut az_replay, batch: c_int, seed: u64, planes_dev: *mut f32, policy_dev: *mut f32, value_dev: *mut f32, n_out: *mut c_int) -> c_int;
    pub fn az_replay_export(rp: *mut az_replay, first: c_int, n: c_int, pos: *mut az_position, policy: *mut f32, value: *mut f32,
                            visits: *mut u32, n_out: *mut c_int) -> c_int;
    pub fn az_replay_import(rp: *mut az_replay, n: c_int, pos: *const az_position, policy: *const f32, value: *const f32, visits: *const u32) -> c_int;
    pub fn az_replay_get(rp: *mut az_replay, pos: *const az_position, policy: *mut f32, value: *mut f32, visits: *mut u32) -> c_int;
    // measurement hooks used by bench.py (az_profile mirrors the C struct) and two kernel-test entry points
    pub fn az_timer_start(eng: *mut az_engine) -> c_int;
    pub fn az_timer_stop(eng: *mut az_engine, ms: *mut f32) -> c_int;
    pub fn az_profile_enable(eng: *mut az_engine, every_n_forwards: c_int) -> c_int;
    pub fn az_profile_read(eng: *mut az_engine, out: *mut az_profile) -> c_int;
    pub fn az_launch_count(eng: *const az_engine) -> u64;
}
pub enum az_replay {}
#[repr(C)] pub struct az_profile { pub tower_ms: f64, pub tower_samples: u64, pub tower_boards: u64, pub input_ms: f64,
                                   pub heads_ms: f64, pub advance_ms: f64, pub tower_launches: u64 }
