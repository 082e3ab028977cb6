//! Safe wrapper over `az-b200-sys` for the reference crate (agent.rs / training.rs / memory.rs / validation.rs).
//!
//! SOURCE ONLY: never compiled in the image this project is built in (no Rust toolchain); the C ABI underneath is what
//! the test-suite exercises (through the Python and C++ mirrors).  The types here are the ABI's own (`az_position`,
//! `az_sample`); converting `shakmaty::Chess` to and from `az_position` is a field copy that belongs in the reference
//! crate (INTEGRATION.md section 2), so this crate has no dependency on shakmaty.
use az_b200_sys as sys;
use std::ffi::CStr;
use std::ptr;

pub const ACTION_SPACE: usize = 4096; // parameters.rs:3
pub const MAX_MOVES: usize = 256;

#[derive(Debug)]
pub struct Error { pub code: i32, pub message: String }
pub type Result<T> = std::result::Result<T, Error>;

/// One engine per GPU; calls are serialised by the owner (the reference's single inference-loop thread).
pub struct Engine { raw: *mut sys::az_engine, cfg: sys::az_config }
unsafe impl Send for Engine {}

impl Engine {
    pub fn default_config() -> sys::az_config {
        let mut c = std::mem::MaybeUninit::<sys::az_config>::uninit();
        unsafe { sys::az_config_default(c.as_mut_ptr()); c.assume_init() }
    }
    pub fn new(cfg: sys::az_config) -> Result<Engine> {
        let mut raw: *mut sys::az_engine = ptr::null_mut();
        let rc = unsafe { sys::az_engine_create(&cfg, &mut raw) };
        let e = Engine { raw, cfg };
        if rc != 0 { return Err(e.error(rc)); }
        Ok(e)
    }
    fn error(&self, code: i32) -> Error {
        let message = if self.raw.is_null() { String::from("az_engine_create failed") } else {
            unsafe { CStr::from_ptr(sys::az_last_error(self.raw)) }.to_string_lossy().into_owned()
        };
        Error { code, message }
    }
    fn check(&self, rc: i32) -> Result<()> { if rc == 0 { Ok(()) } else { Err(self.error(rc)) } }
    pub fn config(&self) -> &sys::az_config { &self.cfg }

    /// load_model (main.rs:109-116): the 144 tensors of the burn record in `az_weight_name` order.
    pub fn load_weights(&mut self, arrays: &[&[f32]]) -> Result<()> {
        let ptrs: Vec<*const f32> = arrays.iter().map(|a| a.as_ptr()).collect();
        self.check(unsafe { sys::az_load_weights(self.raw, ptrs.as_ptr(), ptrs.len() as i32) })
    }

    /// process_batch (training.rs:380-422) without the channel plumbing: N positions in, N (policy, value) out.
    pub fn forward(&mut self, positions: &[sys::az_position]) -> Result<(Vec<f32>, Vec<f32>)> {
        let n = positions.len();
        let mut policy = vec![0f32; n * ACTION_SPACE];
        let mut value = vec![0f32; n];
        self.check(unsafe { sys::az_forward(self.raw, n as i32, positions.as_ptr(), policy.as_mut_ptr(), value.as_mut_ptr()) })?;
        Ok((policy, value))
    }

    /// Chess::legal_moves() for a batch: (wire moves, policy indices, counts).
    pub fn legal_moves(&mut self, positions: &[sys::az_position]) -> Result<(Vec<u16>, Vec<u16>, Vec<i32>)> {
        let n = positions.len();
        let (mut moves, mut index, mut count) = (vec![0u16; n * MAX_MOVES], vec![0u16; n * MAX_MOVES], vec![0i32; n]);
        self.check(unsafe { sys::az_movegen(self.raw, n as i32, positions.as_ptr(), moves.as_mut_ptr(), index.as_mut_ptr(), count.as_mut_ptr()) })?;
        Ok((moves, index, count))
    }

    /// MCTree::init(model, state, noise) + monte_carlo_tree_search (validation.rs:39-40): `history[i]` holds every position
    /// already counted in that game's `pos_count` (including the root).  Returns visits [n][4096] and max_subtree_depth [n];
    /// `visits / sims` is the improved policy (tree.rs:173-175 with TEMPERATURE = 1).
    pub fn search(&mut self, roots: &[sys::az_position], history: &[Vec<sys::az_position>], sims: i32,
                  noise: Option<(&[u64], &[u32])>) -> Result<(Vec<f32>, Vec<i32>)> {
        let n = roots.len();
        let mut flat = Vec::new();
        let mut offs = vec![0u32; n + 1];
        for (i, h) in history.iter().enumerate() { flat.extend_from_slice(h); offs[i + 1] = flat.len() as u32; }
        let (ids, plies) = match noise { Some((g, p)) => (g.as_ptr(), p.as_ptr()), None => (ptr::null(), ptr::null()) };
        let mut visits = vec![0f32; n * ACTION_SPACE];
        let mut depth = vec![0i32; n];
        self.check(unsafe { sys::az_search(self.raw, n as i32, roots.as_ptr(), flat.as_ptr(), offs.as_ptr(), sims, ids, plies,
                                           visits.as_mut_ptr(), ptr::null_mut(), depth.as_mut_ptr()) })?;
        Ok((visits, depth))
    }

    /// Not in the reference: `search` with up to `leaves_per_root` leaves per root in each network round, steered apart by
    /// `virtual_loss` (az_search_vl); `leaves_per_root = 1` gives `search`'s results.  Returns visits, depths and the stats.
    pub fn search_vl(&mut self, roots: &[sys::az_position], history: &[Vec<sys::az_position>], sims: i32, leaves_per_root: i32,
                     virtual_loss: f32, noise: Option<(&[u64], &[u32])>) -> Result<(Vec<f32>, Vec<i32>, sys::az_search_stats)> {
        let n = roots.len();
        let mut flat = Vec::new();
        let mut offs = vec![0u32; n + 1];
        for (i, h) in history.iter().enumerate() { flat.extend_from_slice(h); offs[i + 1] = flat.len() as u32; }
        let (ids, plies) = match noise { Some((g, p)) => (g.as_ptr(), p.as_ptr()), None => (ptr::null(), ptr::null()) };
        let mut visits = vec![0f32; n * ACTION_SPACE];
        let mut depth = vec![0i32; n];
        let mut stats = sys::az_search_stats::default();
        self.check(unsafe { sys::az_search_vl(self.raw, n as i32, roots.as_ptr(), flat.as_ptr(), offs.as_ptr(), sims, leaves_per_root,
                                              virtual_loss, ids, plies, visits.as_mut_ptr(), ptr::null_mut(), depth.as_mut_ptr(),
                                              &mut stats) })?;
        Ok((visits, depth, stats))
    }

    /// Loads a network (144 f32 arrays in az_weight_name order) into slot `network` (az_load_network): slot 0 is what every
    /// single-network call uses, slot 1 the second network of `search_networks`.
    pub fn load_network(&mut self, network: i32, arrays: &[&[f32]]) -> Result<()> {
        let ptrs: Vec<*const f32> = arrays.iter().map(|a| a.as_ptr()).collect();
        self.check(unsafe { sys::az_load_network(self.raw, network, ptrs.as_ptr(), ptrs.len() as i32) })
    }

    /// `search_vl` with a network slot per root (az_search_networks): the roots of both networks share every network round,
    /// the two players of a match in one call.  Returns visits, depths and the stats.
    pub fn search_networks(&mut self, roots: &[sys::az_position], history: &[Vec<sys::az_position>], network: &[u8], sims: i32,
                           leaves_per_root: i32, virtual_loss: f32, noise: Option<(&[u64], &[u32])>)
                           -> Result<(Vec<f32>, Vec<i32>, sys::az_search_stats)> {
        let n = roots.len();
        assert_eq!(network.len(), n, "one network id per root");
        let mut flat = Vec::new();
        let mut offs = vec![0u32; n + 1];
        for (i, h) in history.iter().enumerate() { flat.extend_from_slice(h); offs[i + 1] = flat.len() as u32; }
        let (ids, plies) = match noise { Some((g, p)) => (g.as_ptr(), p.as_ptr()), None => (ptr::null(), ptr::null()) };
        let mut visits = vec![0f32; n * ACTION_SPACE];
        let mut depth = vec![0i32; n];
        let mut stats = sys::az_search_stats::default();
        self.check(unsafe { sys::az_search_networks(self.raw, n as i32, roots.as_ptr(), flat.as_ptr(), offs.as_ptr(), sims,
                                                    leaves_per_root, virtual_loss, network.as_ptr(), ids, plies, visits.as_mut_ptr(),
                                                    ptr::null_mut(), depth.as_mut_ptr(), &mut stats) })?;
        Ok((visits, depth, stats))
    }

    /// evaluate (validation.rs:155-282) resident on the device (az_match_*): `n_games` games between network slot `network_1`
    /// (player 1, White in even games) and `network_2`, both searching with `sims` simulations (0: the config's) at
    /// `leaves_per_root` (1: az_search semantics; more is not in the reference), or both playing the raw policy when `base_model`.
    /// Moves are sampled while fullmoves <= `num_stochastic_moves`, keyed by (seed, game, ply); games still on after `max_plies`
    /// count as draws.  As many games run at once as max_games and the two network ranges (2 x round4(slots x K) <= max_batch)
    /// allow.  Returns (winrate, drawrate, lossrate) from player 1's side.
    pub fn evaluate(&mut self, network_1: u8, network_2: u8, n_games: u32, num_stochastic_moves: u32, seed: u64, max_plies: u32, sims: i32,
                    leaves_per_root: i32, virtual_loss: f32, base_model: bool) -> Result<(f32, f32, f32)> {
        let cfg = sys::az_match_config { player_kind: base_model as i32, network: [network_1, network_2], num_simulations: sims,
                                         leaves_per_root, virtual_loss, num_stochastic_moves, max_plies, seed };
        let k = if base_model { 1 } else { leaves_per_root.max(1) };
        let max_batch = self.config().max_batch.max(self.config().max_games);
        let slots = (n_games as i64).min(self.config().max_games as i64).min(((max_batch / 2) / 4 * 4 / k) as i64) as i32;
        self.check(unsafe { sys::az_match_begin(self.raw, slots, 0, n_games, &cfg) })?;
        let mut stats = sys::az_match_stats::default();
        loop {
            self.check(unsafe { sys::az_match_step(self.raw, 256, &mut stats) })?;
            if stats.active_games == 0 { break; }
        }
        let n = n_games as usize;
        let (mut white, mut plies, mut finished) = (vec![0i8; n], vec![0u16; n], vec![0u8; n]);
        self.check(unsafe { sys::az_match_results(self.raw, white.as_mut_ptr(), plies.as_mut_ptr(), finished.as_mut_ptr(), ptr::null_mut()) })?;
        let (mut wins, mut draws) = (0f32, 0f32);
        for (g, w) in white.iter().enumerate() {
            let p1 = if g % 2 == 0 { *w } else { -*w };   // validation.rs:196-200
            if p1 == 1 { wins += 1.0 } else if p1 == 0 { draws += 1.0 }
        }
        let total = n_games as f32;
        Ok(((wins + draws / 2.0) / total, draws / total, (total - wins - draws) / total))
    }

    /// run_all_episodes (training.rs:340-378): EXACTLY `n_games` self-play games (ids first_game_id ..), each played to
    /// completion; the callback receives the finished games' steps (values already back-filled) as they become available.
    /// Returns the average batch size (= evaluations per wave).
    pub fn run_all_episodes<F: FnMut(&[sys::az_sample])>(&mut self, n_games: i32, first_game_id: u64, sink: F) -> Result<f32> {
        self.check(unsafe { sys::az_selfplay_begin_n(self.raw, n_games, first_game_id, n_games as u64) })?;
        self.collect_episodes(n_games, sink)
    }

    /// Not in the reference: `run_all_episodes` with every ply searched leaf-parallel, up to `leaves_per_game` leaves per game
    /// and network round under `virtual_loss` (az_selfplay_begin_vl); `leaves_per_game = 1` plays the same games record for
    /// record.  Needs `n_games * leaves_per_game <= max_batch`.
    pub fn run_all_episodes_vl<F: FnMut(&[sys::az_sample])>(&mut self, n_games: i32, first_game_id: u64, leaves_per_game: i32,
                                                            virtual_loss: f32, sink: F) -> Result<f32> {
        self.check(unsafe { sys::az_selfplay_begin_vl(self.raw, n_games, first_game_id, n_games as u64, leaves_per_game, virtual_loss) })?;
        self.collect_episodes(n_games, sink)
    }

    // steps the self-play just begun until every game has ended, handing the finished games' steps to `sink`
    fn collect_episodes<F: FnMut(&[sys::az_sample])>(&mut self, n_games: i32, mut sink: F) -> Result<f32> {
        let mut buf: Vec<sys::az_sample> = Vec::with_capacity((n_games as usize * 128).max(1 << 16));
        let mut stats = sys::az_selfplay_stats::default();
        let mut waves = 0u64;
        loop {
            self.check(unsafe { sys::az_selfplay_step(self.raw, 64, &mut stats) })?;
            waves += 64;
            if stats.pending_samples > 0 {
                let mut n = 0i32;
                self.check(unsafe { sys::az_selfplay_drain(self.raw, buf.as_mut_ptr(), buf.capacity() as i32, &mut n) })?;
                unsafe { buf.set_len(n as usize) };
                sink(&buf);
            }
            if stats.active_games == 0 && stats.pending_samples == 0 { break; }   // every game of the generation has ended
        }
        Ok(stats.evaluations as f32 / waves as f32)
    }

    /// get_best_move up to its random tie-break (chess.rs:295-318): negamax score of every legal move of `pos`.
    pub fn minimax_scores(&mut self, pos: &sys::az_position, depth: i32) -> Result<Vec<i32>> {
        let mut scores = vec![0i32; MAX_MOVES];
        let mut count = 0i32;
        self.check(unsafe { sys::az_minimax(self.raw, 1, pos, depth, scores.as_mut_ptr(), &mut count) })?;
        scores.truncate(count as usize);
        Ok(scores)
    }
}

impl Drop for Engine {
    fn drop(&mut self) { if !self.raw.is_null() { unsafe { sys::az_engine_destroy(self.raw) } } }
}

/// improved_policy of one EpisodeStep (training.rs:303-308) from the sparse record the engine emits.
pub fn improved_policy(sample: &sys::az_sample, sims: u32) -> Box<[f32; ACTION_SPACE]> {
    let mut policy = Box::new([0f32; ACTION_SPACE]);
    for k in 0..sample.n_visits as usize { policy[sample.index[k] as usize] = sample.count[k] as f32 / sims as f32; }
    policy
}

/// ReplayBuffer (memory.rs:26-118), device resident.  The buffer must not outlive its engine.
pub struct ReplayBuffer { raw: *mut sys::az_replay }

impl ReplayBuffer {
    pub fn new(engine: &mut Engine, capacity: i32, max_batch: i32) -> Result<ReplayBuffer> {
        let mut raw: *mut sys::az_replay = ptr::null_mut();
        let rc = unsafe { sys::az_replay_create(engine.raw, capacity, max_batch, &mut raw) };
        if rc != 0 { return Err(engine.error(rc)); }
        Ok(ReplayBuffer { raw })
    }
    /// add() for every finished self-play step still in device memory; returns (steps, new unique positions).
    pub fn add_pending(&mut self) -> (i32, i32) {
        let (mut n, mut nu) = (0i32, 0i32);
        unsafe { sys::az_replay_add_pending(self.raw, &mut n, &mut nu) };
        (n, nu)
    }
    pub fn len(&self) -> usize {
        let mut n = 0i32;
        unsafe { sys::az_replay_len(self.raw, &mut n) };
        n as usize
    }
    /// sample(batch_size) (memory.rs:78-97): stacked planes [n,19,8,8], policies [n,4096] and values [n].
    pub fn sample(&mut self, batch_size: usize, seed: u64) -> (usize, Vec<f32>, Vec<f32>, Vec<f32>) {
        let (mut planes, mut policy, mut value) = (vec![0f32; batch_size * 19 * 64], vec![0f32; batch_size * ACTION_SPACE], vec![0f32; batch_size]);
        let mut n = 0i32;
        unsafe { sys::az_replay_sample(self.raw, batch_size as i32, seed, planes.as_mut_ptr(), policy.as_mut_ptr(), value.as_mut_ptr(), &mut n) };
        let n = n as usize;
        planes.truncate(n * 19 * 64); policy.truncate(n * ACTION_SPACE); value.truncate(n);
        (n, planes, policy, value)
    }
}

impl Drop for ReplayBuffer {
    fn drop(&mut self) { if !self.raw.is_null() { unsafe { sys::az_replay_destroy(self.raw) } } }
}
