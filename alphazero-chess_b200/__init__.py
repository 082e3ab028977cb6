"""alphazero-chess_b200: B200-native batched self-play engine.

Host-side Python mirror of the reference's interface for the self-play hot path (chess.rs / tree.rs / agent.rs /
training.rs of AlexandreGac/alphazero-chess) over the C ABI in include/az_b200.h.  All compute happens in the
sm_100a CUDA library next to this file; there is no CPU fallback: a missing library or a missing GPU is an error.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libaz_b200.so")
_lib = None

ACTION_SPACE = 4096
MAX_MOVES = 256
NUM_PLANES = 19
NUM_WEIGHT_ARRAYS = 144
MOVE_NONE = 0xFFFF
ONGOING, DRAW, WHITE_WINS, BLACK_WINS, ILLEGAL = 0, 1, 2, 3, -1

POSITION_DTYPE = np.dtype(
    [("roles", "<u8", 6), ("colors", "<u8", 2), ("turn", "u1"), ("castling", "u1"), ("ep_square", "i1"), ("reserved", "u1"),
     ("halfmoves", "<u2"), ("fullmoves", "<u2")]
)
assert POSITION_DTYPE.itemsize == 72

SAMPLE_DTYPE = np.dtype(
    [("position", POSITION_DTYPE), ("final_value", "<f4"), ("search_depth", "<i4"), ("game_id", "<u8"), ("ply", "<u4"),
     ("action", "<u2"), ("n_visits", "<u2"), ("index", "<u2", MAX_MOVES), ("count", "<u2", MAX_MOVES)]
)
assert SAMPLE_DTYPE.itemsize == 1120


class Config(ctypes.Structure):
    """az_config: parameters.rs as runtime configuration."""

    _fields_ = [
        ("device", ctypes.c_int32), ("max_games", ctypes.c_int32), ("max_batch", ctypes.c_int32), ("num_simulations", ctypes.c_int32),
        ("c_puct", ctypes.c_float), ("dirichlet_alpha", ctypes.c_float), ("dirichlet_epsilon", ctypes.c_float),
        ("temperature_annealing", ctypes.c_uint32), ("num_halfmoves", ctypes.c_uint32), ("num_fullmoves", ctypes.c_uint32),
        ("repetitions", ctypes.c_uint32), ("seed", ctypes.c_uint64), ("precision", ctypes.c_int32), ("cache_log2", ctypes.c_int32),
        ("edge_capacity_per_node", ctypes.c_int32), ("temperature", ctypes.c_float),
    ]


class SelfplayStats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in ("simulations", "positions", "evaluations", "cache_hits", "terminal_leaves",
                                               "games_finished", "sum_leaf_depth", "sum_edges", "waves", "pending_samples",
                                               "active_games", "parked_games", "cache_evictions", "sum_search_depth")]


class SearchStats(ctypes.Structure):
    """az_search_stats of az_search_vl."""

    _fields_ = [(n, ctypes.c_uint64) for n in ("waves", "evaluations", "terminal_leaves", "collisions")]


class MatchConfig(ctypes.Structure):
    """az_match_config."""

    _fields_ = [("player_kind", ctypes.c_int32), ("network", ctypes.c_uint8 * 2), ("num_simulations", ctypes.c_int32),
                ("leaves_per_root", ctypes.c_int32), ("virtual_loss", ctypes.c_float), ("num_stochastic_moves", ctypes.c_uint32),
                ("max_plies", ctypes.c_uint32), ("seed", ctypes.c_uint64)]


class MatchStats(ctypes.Structure):
    """az_match_stats: totals since az_match_begin."""

    _fields_ = [("waves", ctypes.c_uint64), ("evaluations", ctypes.c_uint64 * 2)] + [
        (n, ctypes.c_uint64) for n in ("leaves", "terminal_leaves", "collisions", "plies", "games_finished", "active_games")]


MATCH_MCTS, MATCH_BASE_MODEL = 0, 1


class EngineError(RuntimeError):
    pass


def lib():
    """Loads the CUDA extension; a missing library is an error (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a) first")
        L = ctypes.CDLL(LIB_PATH)
        L.az_last_error.restype = ctypes.c_char_p
        L.az_version.restype = ctypes.c_char_p
        L.az_weight_name.restype = ctypes.c_char_p
        L.az_weight_size.restype = ctypes.c_int64
        L.az_engine_destroy.restype = None
        L.az_config_default.restype = None
        L.az_position_start.restype = None
        _lib = L
    return _lib


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else ctypes.c_void_p(0)


def default_config(**overrides):
    c = Config()
    lib().az_config_default(ctypes.byref(c))
    for k, v in overrides.items():
        setattr(c, k, v)
    return c


def start_position():
    p = np.zeros(1, POSITION_DTYPE)
    lib().az_position_start(_ptr(p))
    return p[0]


def position_from_fen(fen):
    p = np.zeros(1, POSITION_DTYPE)
    rc = lib().az_position_from_fen(fen.encode(), _ptr(p))
    if rc:
        raise ValueError(f"bad FEN: {fen}")
    return p[0]


def weight_names():
    L = lib()
    return [L.az_weight_name(i).decode() for i in range(NUM_WEIGHT_ARRAYS)]


def weight_sizes():
    L = lib()
    return [int(L.az_weight_size(i)) for i in range(NUM_WEIGHT_ARRAYS)]


_FAN_IN = {"input_conv": 19 * 9, "conv1": 128 * 9, "conv2": 128 * 9, "policy_conv_1": 128, "policy_conv_2": 32, "value_conv": 128,
           "value_linear_1": 512, "value_linear_2": 64}


def random_weights(seed=42, randomize_bn=False, sizes=None, names=None):
    """Random-init 10x128 network in burn's layout (AlphaZero::new, agent.rs:69-110): conv/linear U(-k, k) with
    k = 1/sqrt(fan_in); BatchNorm gamma 1, beta 0, mean 0, var 1 (optionally randomised for tests)."""
    names = names or weight_names()
    sizes = sizes or weight_sizes()
    rng = np.random.default_rng(seed)
    out = []
    for name, size in zip(names, sizes):
        parts = name.split(".")
        layer, field = parts[-2], parts[-1]
        if field in ("weight", "bias"):
            k = 1.0 / np.sqrt(_FAN_IN[layer])
            a = rng.uniform(-k, k, size).astype(np.float32)
        elif field == "gamma":
            a = rng.uniform(0.5, 1.5, size).astype(np.float32) if randomize_bn else np.ones(size, np.float32)
        elif field == "running_var":
            a = rng.uniform(0.5, 1.5, size).astype(np.float32) if randomize_bn else np.ones(size, np.float32)
        else:
            a = rng.uniform(-0.2, 0.2, size).astype(np.float32) if randomize_bn else np.zeros(size, np.float32)
        out.append(a)
    return out


class Engine:
    """One engine per GPU (az_engine).  Methods mirror the reference items named in include/az_b200.h."""

    def __init__(self, config=None, **overrides):
        self._L = lib()
        self.config = config if config is not None else default_config(**overrides)
        self._h = ctypes.c_void_p(0)
        rc = self._L.az_engine_create(ctypes.byref(self.config), ctypes.byref(self._h))
        if rc:
            msg = self._L.az_last_error(self._h).decode() if self._h else "az_engine_create failed"
            if self._h:
                self._L.az_engine_destroy(self._h)
                self._h = ctypes.c_void_p(0)
            raise EngineError(f"az_engine_create: {rc}: {msg}")

    def close(self):
        if self._h:
            self._L.az_engine_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc:
            raise EngineError(f"{what}: {rc}: {self._L.az_last_error(self._h).decode()}")

    @staticmethod
    def _positions(pos):
        a = np.ascontiguousarray(np.atleast_1d(pos), dtype=POSITION_DTYPE)
        return a

    # ---- agent.rs ---------------------------------------------------------------------------------------------
    def load_weights(self, arrays, network=0):
        """load_model (main.rs:109-116): 144 f32 arrays in az_weight_name order, into network slot `network`
        (0 = what every single-network call uses; 1 = the second network of forward_networks / search_networks)."""
        arrs = [np.ascontiguousarray(a, np.float32).ravel() for a in arrays]
        sizes = weight_sizes()
        if len(arrs) != NUM_WEIGHT_ARRAYS or any(a.size != s for a, s in zip(arrs, sizes)):
            raise ValueError("expected 144 arrays with the sizes of az_weight_size")
        ptrs = (ctypes.c_void_p * NUM_WEIGHT_ARRAYS)(*[a.ctypes.data for a in arrs])
        if network == 0:
            self._check(self._L.az_load_weights(self._h, ptrs, NUM_WEIGHT_ARRAYS), "az_load_weights")
        else:
            self._check(self._L.az_load_network(self._h, int(network), ptrs, NUM_WEIGHT_ARRAYS), "az_load_network")

    def load_mpk(self, path):
        """load_model (main.rs:109-116) from a burn `.mpk` checkpoint (see mpk.py)."""
        from . import mpk
        self.load_weights(mpk.load_mpk(path))

    def load_weights_dev(self, device_ptrs):
        ptrs = (ctypes.c_void_p * NUM_WEIGHT_ARRAYS)(*device_ptrs)
        self._check(self._L.az_load_weights_dev(self._h, ptrs, NUM_WEIGHT_ARRAYS), "az_load_weights_dev")

    def forward_planes(self, planes):
        """AlphaZero::forward (agent.rs:112-144): [n,19,8,8] -> (policy [n,4096], value [n])."""
        x = np.ascontiguousarray(planes, np.float32).reshape(-1, NUM_PLANES, 8, 8)
        n = x.shape[0]
        policy = np.empty((n, ACTION_SPACE), np.float32)
        value = np.empty(n, np.float32)
        self._check(self._L.az_forward_planes(self._h, n, _ptr(x), _ptr(policy), _ptr(value)), "az_forward_planes")
        return policy, value

    def forward(self, pos):
        p = self._positions(pos)
        n = p.shape[0]
        policy = np.empty((n, ACTION_SPACE), np.float32)
        value = np.empty(n, np.float32)
        self._check(self._L.az_forward(self._h, n, _ptr(p), _ptr(policy), _ptr(value)), "az_forward")
        return policy, value

    @staticmethod
    def _networks(network, n):
        net = np.ascontiguousarray(np.broadcast_to(np.asarray(network), (n,)), np.uint8)
        if np.any(np.asarray(network) < 0):
            raise ValueError("network ids must be >= 0")
        return net

    def forward_networks(self, pos, network):
        """forward() with a network slot per board (an int or [n] ids): both networks run in the same launches."""
        p = self._positions(pos)
        n = p.shape[0]
        net = self._networks(network, n)
        policy = np.empty((n, ACTION_SPACE), np.float32)
        value = np.empty(n, np.float32)
        self._check(self._L.az_forward_networks(self._h, n, _ptr(p), _ptr(net), _ptr(policy), _ptr(value)), "az_forward_networks")
        return policy, value

    # ---- chess.rs ---------------------------------------------------------------------------------------------
    def movegen(self, pos):
        """Chess::legal_moves + move_to_index: (moves [n,256], indices [n,256], counts [n])."""
        p = self._positions(pos)
        n = p.shape[0]
        moves = np.empty((n, MAX_MOVES), np.uint16)
        index = np.empty((n, MAX_MOVES), np.uint16)
        count = np.empty(n, np.int32)
        self._check(self._L.az_movegen(self._h, n, _ptr(p), _ptr(moves), _ptr(index), _ptr(count)), "az_movegen")
        return moves, index, count

    def perft(self, pos, depth):
        p = self._positions(pos)
        n = p.shape[0]
        nodes = np.zeros(n, np.uint64)
        self._check(self._L.az_perft(self._h, n, _ptr(p), int(depth), _ptr(nodes)), "az_perft")
        return nodes

    def minimax(self, pos, depth):
        """get_best_move without its random tie-break (chess.rs:295-318): (scores [n][256], count [n]); scores[i, k] is
        -negamax(child k, depth - 1) for legal move k of position i in movegen order."""
        p = self._positions(pos)
        n = p.shape[0]
        scores = np.zeros((n, MAX_MOVES), np.int32)
        count = np.zeros(n, np.int32)
        self._check(self._L.az_minimax(self._h, n, _ptr(p), int(depth), _ptr(scores), _ptr(count)), "az_minimax")
        return scores, count

    def play_move(self, pos, action_index, history=None, hist_offsets=None):
        """play_move (chess.rs:36-63) through a policy index; returns (new positions, GameResult codes)."""
        p = self._positions(pos).copy()
        n = p.shape[0]
        act = np.ascontiguousarray(np.atleast_1d(action_index), np.uint16)
        res = np.empty(n, np.int32)
        h = self._positions(history) if history is not None else None
        ho = np.ascontiguousarray(hist_offsets, np.uint32) if hist_offsets is not None else None
        self._check(self._L.az_play_move(self._h, n, _ptr(p), _ptr(h), _ptr(ho), _ptr(act), _ptr(res)), "az_play_move")
        return p, res

    def move_to_index(self, pos, moves):
        p = self._positions(pos)
        m = np.ascontiguousarray(np.atleast_1d(moves), np.uint16)
        out = np.empty(p.shape[0], np.uint16)
        self._check(self._L.az_move_to_index(self._h, p.shape[0], _ptr(p), _ptr(m), _ptr(out)), "az_move_to_index")
        return out

    def index_to_move(self, pos, index):
        p = self._positions(pos)
        i = np.ascontiguousarray(np.atleast_1d(index), np.uint16)
        out = np.empty(p.shape[0], np.uint16)
        self._check(self._L.az_index_to_move(self._h, p.shape[0], _ptr(p), _ptr(i), _ptr(out)), "az_index_to_move")
        return out

    def encode(self, pos):
        """to_tensor (chess.rs:191-245): [n,19,8,8] f32."""
        p = self._positions(pos)
        out = np.empty((p.shape[0], NUM_PLANES, 8, 8), np.float32)
        self._check(self._L.az_encode(self._h, p.shape[0], _ptr(p), _ptr(out)), "az_encode")
        return out

    # ---- tree.rs ----------------------------------------------------------------------------------------------
    def set_evaluator_stub(self, kind, seed=0):
        self._check(self._L.az_set_evaluator_stub(self._h, int(kind), ctypes.c_uint64(seed)), "az_set_evaluator_stub")

    def _search_inputs(self, roots, history, hist_offsets, noise_game_ids, noise_plies, want_scores):
        """The arguments and output arrays of the az_search* calls: (roots, n, visits, scores or None, depth, history,
        hist_offsets, noise ids, noise plies), the optional inputs None when not given."""
        p = self._positions(roots)
        n = p.shape[0]
        visits = np.empty((n, ACTION_SPACE), np.float32)
        scores = np.empty((n, ACTION_SPACE), np.float32) if want_scores else None
        depth = np.empty(n, np.int32)
        h = self._positions(history) if history is not None else None
        ho = np.ascontiguousarray(hist_offsets, np.uint32) if hist_offsets is not None else None
        ids = np.ascontiguousarray(noise_game_ids, np.uint64) if noise_game_ids is not None else None
        pl = np.ascontiguousarray(noise_plies, np.uint32) if noise_plies is not None else None
        return p, n, visits, scores, depth, h, ho, ids, pl

    def search(self, roots, num_simulations=None, history=None, hist_offsets=None, noise_game_ids=None, noise_plies=None,
               want_scores=False):
        """MCTree::init + monte_carlo_tree_search for a batch of roots: (visits [n,4096], scores or None, depth [n])."""
        p, n, visits, scores, depth, h, ho, ids, pl = self._search_inputs(roots, history, hist_offsets, noise_game_ids, noise_plies,
                                                                          want_scores)
        sims = int(num_simulations or self.config.num_simulations)
        self._check(self._L.az_search(self._h, n, _ptr(p), _ptr(h), _ptr(ho), sims, _ptr(ids), _ptr(pl), _ptr(visits), _ptr(scores),
                                      _ptr(depth)), "az_search")
        return visits, scores, depth

    def search_vl(self, roots, num_simulations, leaves_per_root, virtual_loss=1.0, history=None, hist_offsets=None,
                  noise_game_ids=None, noise_plies=None, want_scores=False):
        """Leaf-parallel search with virtual loss (az_search_vl; not in the reference, identical to search() at
        leaves_per_root = 1): up to leaves_per_root leaves per root share one network round.
        Returns (visits [n,4096], scores or None, depth [n], SearchStats)."""
        p, n, visits, scores, depth, h, ho, ids, pl = self._search_inputs(roots, history, hist_offsets, noise_game_ids, noise_plies,
                                                                          want_scores)
        st = SearchStats()
        self._check(self._L.az_search_vl(self._h, n, _ptr(p), _ptr(h), _ptr(ho), int(num_simulations), int(leaves_per_root),
                                         ctypes.c_float(virtual_loss), _ptr(ids), _ptr(pl), _ptr(visits), _ptr(scores), _ptr(depth),
                                         ctypes.byref(st)), "az_search_vl")
        return visits, scores, depth, st

    def search_networks(self, roots, network, num_simulations, leaves_per_root=1, virtual_loss=1.0, history=None, hist_offsets=None,
                        noise_game_ids=None, noise_plies=None, want_scores=False):
        """search_vl() with a network slot per root (an int or [n] ids): the roots of both networks share every network round.
        Returns (visits [n,4096], scores or None, depth [n], SearchStats)."""
        p, n, visits, scores, depth, h, ho, ids, pl = self._search_inputs(roots, history, hist_offsets, noise_game_ids, noise_plies,
                                                                          want_scores)
        net = self._networks(network, n)
        st = SearchStats()
        self._check(self._L.az_search_networks(self._h, n, _ptr(p), _ptr(h), _ptr(ho), int(num_simulations), int(leaves_per_root),
                                               ctypes.c_float(virtual_loss), _ptr(net), _ptr(ids), _ptr(pl), _ptr(visits), _ptr(scores),
                                               _ptr(depth), ctypes.byref(st)), "az_search_networks")
        return visits, scores, depth, st

    # ---- validation.rs ----------------------------------------------------------------------------------------
    def match_begin(self, n_concurrent, n_games, player_kind, networks=(0, 1), num_simulations=None, leaves_per_root=1,
                    virtual_loss=1.0, num_stochastic_moves=15, max_plies=450, seed=0, first_game=0):
        """evaluate (validation.rs:155-282) resident on the device (az_match_begin): games first_game .. first_game + n_games - 1
        on n_concurrent slots, player 1 on network slot networks[0] and White in even games, player 2 on networks[1].
        player_kind: MATCH_MCTS (both search, num_simulations None = the config's) or MATCH_BASE_MODEL (both play the policy)."""
        c = MatchConfig()
        c.player_kind = int(player_kind)
        if any(int(s) < 0 for s in networks):
            raise ValueError("network ids must be >= 0")
        c.network[0], c.network[1] = (min(int(s), 255) for s in networks)
        c.num_simulations = int(num_simulations or 0)
        c.leaves_per_root, c.virtual_loss = int(leaves_per_root), float(virtual_loss)
        c.num_stochastic_moves, c.max_plies, c.seed = int(num_stochastic_moves), int(max_plies), int(seed)
        self._check(self._L.az_match_begin(self._h, int(n_concurrent), ctypes.c_uint32(first_game), ctypes.c_uint32(n_games),
                                           ctypes.byref(c)), "az_match_begin")
        self._match_shape = (int(n_games), int(max_plies))

    def match_step(self, waves):
        """Advances the match by `waves` network rounds; returns MatchStats (active_games == 0: complete)."""
        st = MatchStats()
        self._check(self._L.az_match_step(self._h, int(waves), ctypes.byref(st)), "az_match_step")
        return st

    def match_results(self):
        """Per game of the last match begun: (result from White's side [n] int8, plies [n] uint16, finished by the rules [n]
        bool, moves [n, max_plies] uint16 policy indices, MOVE_NONE after the last)."""
        n, max_plies = getattr(self, "_match_shape", (0, 0))
        result, plies = np.empty(n, np.int8), np.empty(n, np.uint16)
        finished, moves = np.empty(n, np.uint8), np.empty((n, max_plies), np.uint16)
        self._check(self._L.az_match_results(self._h, _ptr(result), _ptr(plies), _ptr(finished), _ptr(moves)), "az_match_results")
        return result, plies, finished.astype(bool), moves

    # ---- training.rs ------------------------------------------------------------------------------------------
    def selfplay_begin(self, n_games, first_game_id=0, total_games=0, leaves_per_game=None, virtual_loss=1.0):
        """run_all_episodes set-up.  total_games = 0: every finished game restarts with a fresh id (throughput runs);
        total_games = N: exactly the games first_game_id .. first_game_id + N - 1 are played to completion on n_games
        concurrent slots (training.rs:352-361,376-377) and stats.active_games reaches 0 when the last one has ended.
        leaves_per_game = K (any int, 1 included) searches every ply leaf-parallel with virtual loss (az_selfplay_begin_vl; not in
        the reference, records identical to the default path at K = 1): up to K leaves per game share each network round."""
        if leaves_per_game is None:
            self._check(self._L.az_selfplay_begin_n(self._h, int(n_games), ctypes.c_uint64(first_game_id), ctypes.c_uint64(total_games)),
                        "az_selfplay_begin_n")
        else:
            self._check(self._L.az_selfplay_begin_vl(self._h, int(n_games), ctypes.c_uint64(first_game_id), ctypes.c_uint64(total_games),
                                                     int(leaves_per_game), ctypes.c_float(virtual_loss)), "az_selfplay_begin_vl")

    def selfplay_vl_stats(self):
        """SearchStats of the az_selfplay_begin_vl self-play since its begin call: waves, leaf evaluations, terminal leaves,
        collisions."""
        st = SearchStats()
        self._check(self._L.az_selfplay_vl_stats(self._h, ctypes.byref(st)), "az_selfplay_vl_stats")
        return st

    def selfplay_step(self, waves):
        st = SelfplayStats()
        self._check(self._L.az_selfplay_step(self._h, int(waves), ctypes.byref(st)), "az_selfplay_step")
        return st

    def selfplay_drain(self, max_samples=None):
        cap = int(max_samples or max(self.config.max_games * 128, 1 << 16))
        out = np.empty(cap, SAMPLE_DTYPE)
        n = ctypes.c_int(0)
        self._check(self._L.az_selfplay_drain(self._h, _ptr(out), cap, ctypes.byref(n)), "az_selfplay_drain")
        return out[: n.value]


    def selfplay_drain_dev(self, device_ptr, max_samples):
        """az_selfplay_drain into device memory (device_ptr: room for max_samples az_sample records); returns the count."""
        n = ctypes.c_int(0)
        self._check(self._L.az_selfplay_drain_dev(self._h, ctypes.c_void_p(int(device_ptr)), int(max_samples), ctypes.byref(n)),
                    "az_selfplay_drain_dev")
        return n.value

    def selfplay_staged(self, slot, max_samples=512):
        """Test hook: the EpisodeSteps the unfinished game in `slot` has recorded so far."""
        out = np.empty(max_samples, SAMPLE_DTYPE)
        n = ctypes.c_int(0)
        self._check(self._L.az_dbg_selfplay_staged(self._h, int(slot), _ptr(out), int(max_samples), ctypes.byref(n)), "az_dbg_selfplay_staged")
        return out[: n.value]


class ReplayBuffer:
    """memory.rs ReplayBuffer, device resident (az_replay_*)."""

    def __init__(self, engine, capacity=100_000, max_batch=512):
        self._e = engine
        self._L = engine._L
        self._h = ctypes.c_void_p(0)
        self._max_batch = int(max_batch)
        engine._check(self._L.az_replay_create(engine._h, int(capacity), int(max_batch), ctypes.byref(self._h)), "az_replay_create")
        self._L.az_replay_destroy.restype = None

    def close(self):
        if self._h:
            self._L.az_replay_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add(self, samples):
        """ReplayBuffer::add for drained az_sample records, in order; returns the number of new unique positions."""
        s = np.ascontiguousarray(samples, SAMPLE_DTYPE)
        nu = ctypes.c_int(0)
        self._e._check(self._L.az_replay_add(self._h, _ptr(s), int(s.shape[0]), ctypes.byref(nu)), "az_replay_add")
        return nu.value

    def add_dev(self, device_ptr, n):
        """ReplayBuffer::add for n az_sample records already in device memory (e.g. delivered by an NCCL gather)."""
        nu = ctypes.c_int(0)
        self._e._check(self._L.az_replay_add_dev(self._h, ctypes.c_void_p(int(device_ptr)), int(n), ctypes.byref(nu)), "az_replay_add_dev")
        return nu.value

    def add_pending(self):
        """Consumes the finished-game samples still in device memory; returns (steps added, new unique positions)."""
        n, nu = ctypes.c_int(0), ctypes.c_int(0)
        self._e._check(self._L.az_replay_add_pending(self._h, ctypes.byref(n), ctypes.byref(nu)), "az_replay_add_pending")
        return n.value, nu.value

    def __len__(self):
        n = ctypes.c_int(0)
        self._e._check(self._L.az_replay_len(self._h, ctypes.byref(n)), "az_replay_len")
        return n.value

    def sample(self, batch_size, seed=0):
        """ReplayBuffer::sample: (planes [n,19,8,8], policy [n,4096], value [n]) with n = min(batch_size, len)."""
        planes = np.empty((batch_size, NUM_PLANES, 8, 8), np.float32)
        policy = np.empty((batch_size, ACTION_SPACE), np.float32)
        value = np.empty(batch_size, np.float32)
        n = ctypes.c_int(0)
        self._e._check(self._L.az_replay_sample(self._h, int(batch_size), ctypes.c_uint64(seed), _ptr(planes), _ptr(policy), _ptr(value),
                                                ctypes.byref(n)), "az_replay_sample")
        return planes[: n.value], policy[: n.value], value[: n.value]

    def sample_torch(self, batch_size, seed=0):
        """ReplayBuffer::sample straight into CUDA tensors on the engine's device (az_replay_sample_dev): the same batch as
        sample(batch_size, seed), without the device -> host -> device round trip of the numpy path."""
        import torch

        dev = torch.device("cuda", int(self._e.config.device))
        # The engine fills the tensors on ITS stream.  torch's caching allocator may hand out a block that kernels still queued on
        # torch's stream (the previous step's backward / optimizer) are using under another name -- it only orders reuse within one
        # stream -- so torch's stream is drained first; the engine call returns after synchronising its own stream.
        torch.cuda.current_stream(dev).synchronize()
        planes = torch.empty((batch_size, NUM_PLANES, 8, 8), dtype=torch.float32, device=dev)
        policy = torch.empty((batch_size, ACTION_SPACE), dtype=torch.float32, device=dev)
        value = torch.empty(batch_size, dtype=torch.float32, device=dev)
        n = ctypes.c_int(0)
        self._e._check(self._L.az_replay_sample_dev(self._h, int(batch_size), ctypes.c_uint64(seed), ctypes.c_void_p(planes.data_ptr()),
                                                    ctypes.c_void_p(policy.data_ptr()), ctypes.c_void_p(value.data_ptr()), ctypes.byref(n)),
                       "az_replay_sample_dev")
        return planes[: n.value], policy[: n.value], value[: n.value]

    def export(self, first, n):
        """Entries [first, first + n) in FIFO order (oldest first): (positions, policy [k,4096], value [k], visit_count [k])."""
        pos = np.zeros(n, POSITION_DTYPE)
        policy = np.empty((n, ACTION_SPACE), np.float32)
        value = np.empty(n, np.float32)
        visits = np.empty(n, np.uint32)
        k = ctypes.c_int(0)
        self._e._check(self._L.az_replay_export(self._h, int(first), int(n), _ptr(pos), _ptr(policy), _ptr(value), _ptr(visits),
                                                ctypes.byref(k)), "az_replay_export")
        return pos[: k.value], policy[: k.value], value[: k.value], visits[: k.value]

    def import_entries(self, pos, policy, value, visits):
        """Appends stored entries (running means and visit counts as given) as the newest ones, in order."""
        pos = np.ascontiguousarray(pos, POSITION_DTYPE)
        policy = np.ascontiguousarray(policy, np.float32)
        value = np.ascontiguousarray(value, np.float32)
        visits = np.ascontiguousarray(visits, np.uint32)
        self._e._check(self._L.az_replay_import(self._h, int(pos.shape[0]), _ptr(pos), _ptr(policy), _ptr(value), _ptr(visits)),
                       "az_replay_import")

    def save(self, path, page=512):
        """ReplayBuffer::save (memory.rs:100-104): the reference's bincode file (see replay_io.py)."""
        from . import replay_io
        n, page = len(self), min(page, self._max_batch)
        replay_io.write_file(path, (self.export(first, page) for first in range(0, n, page)), n)

    def load(self, path, page=512):
        """ReplayBuffer::load (memory.rs:107-114) into this (normally empty) buffer."""
        from . import replay_io
        pos, policy, value, visits = replay_io.read_file(path)
        page = min(page, self._max_batch)
        for first in range(0, len(pos), page):
            sl = slice(first, first + page)
            self.import_entries(pos[sl], policy[sl], value[sl], visits[sl])
        return len(pos)

    def get(self, pos):
        p = np.ascontiguousarray(np.atleast_1d(pos), POSITION_DTYPE)
        policy = np.empty(ACTION_SPACE, np.float32)
        value = ctypes.c_float(0)
        visits = ctypes.c_uint32(0)
        self._e._check(self._L.az_replay_get(self._h, _ptr(p), _ptr(policy), ctypes.byref(value), ctypes.byref(visits)), "az_replay_get")
        return policy, value.value, visits.value


class Profile(ctypes.Structure):
    _fields_ = [("tower_ms", ctypes.c_double), ("tower_samples", ctypes.c_uint64), ("tower_boards", ctypes.c_uint64),
                ("input_ms", ctypes.c_double), ("heads_ms", ctypes.c_double), ("advance_ms", ctypes.c_double),
                ("tower_launches", ctypes.c_uint64)]


def _engine_measurement_methods():
    def timer_start(self):
        self._check(self._L.az_timer_start(self._h), "az_timer_start")

    def timer_stop(self):
        ms = ctypes.c_float(0)
        self._check(self._L.az_timer_stop(self._h, ctypes.byref(ms)), "az_timer_stop")
        return ms.value

    def profile_enable(self, every):
        self._check(self._L.az_profile_enable(self._h, int(every)), "az_profile_enable")

    def profile_read(self):
        p = Profile()
        self._check(self._L.az_profile_read(self._h, ctypes.byref(p)), "az_profile_read")
        return p

    def launch_count(self):
        self._L.az_launch_count.restype = ctypes.c_uint64
        return int(self._L.az_launch_count(self._h))

    for f in (timer_start, timer_stop, profile_enable, profile_read, launch_count):
        setattr(Engine, f.__name__, f)


_engine_measurement_methods()

# algorithmic FLOPs of one network evaluation (2 x MAC, direct convolution; SURVEY.md 8(d))
FLOPS_PER_EVAL = 381_272_192
FLOPS_PER_TOWER_CONV = 2 * 64 * 128 * 1152  # one 3x3 128->128 convolution on one board
FLOPS_PER_INPUT_CONV = 2 * 64 * 128 * 19 * 9  # the 3x3 19->128 input convolution on one board


def improved_policy(sample, num_simulations=None):
    """Dense EpisodeStep::improved_policy (Box<[f32; 4096]>) of a drained sample at T = 1: visits / sum(visits)
    (tree.rs:173-177); the sum is the search's simulation count, which `num_simulations` may state explicitly."""
    dense = np.zeros(ACTION_SPACE, np.float32)
    k = int(sample["n_visits"])
    counts = sample["count"][:k].astype(np.float32)
    total = np.float32(num_simulations) if num_simulations else np.float32(counts.sum(dtype=np.float64))
    dense[sample["index"][:k]] = counts / total
    return dense
