"""Match play and Elo (SURVEY section 8(f) #3; validation.rs:155-384, ratings.rs:5-144) on top of the engine.

A match advances all its games in lockstep: per ply the positions whose side to move belongs to a player are handed to
that player as ONE batch (az_search / az_forward / az_movegen), then az_play_move applies all chosen moves.  The
reference runs 256 async games against two inference servers; batching by player is the same schedule without the
channel hops.  The Human player (terminal input) is out of scope.
Randomness (move sampling in the opening, the random player) uses the engine's counter-based generator convention,
keyed by (seed, game, ply); the reference draws from an unseeded thread_rng.
"""
import numpy as np

from . import ACTION_SPACE, DRAW, ILLEGAL, ONGOING, POSITION_DTYPE, WHITE_WINS, start_position

EVALUATION_GAMES = 256          # parameters.rs:37
TEMPERATURE_ANNEALING = 15      # parameters.rs:31


def _mix(*vals):
    h = np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        for v in vals:
            h = (h ^ np.uint64(v)) * np.uint64(0xBF58476D1CE4E5B9)
            h ^= h >> np.uint64(29)
    return int(h)


def _uniform(seed, game, ply):
    return (_mix(seed, game, ply) >> 11) * (1.0 / (1 << 53))


def _last_argmax(weights):
    """Iterator::max_by keeps the LAST maximum (validation.rs:301-305)."""
    m = weights.max()
    return int(np.flatnonzero(weights == m).max())


def _weighted_index(weights, u):
    """rand::WeightedIndex restated: cumulative f32 weights in index order, first cumulative > u * total."""
    cum = np.cumsum(weights, dtype=np.float32)
    idx = int(np.searchsorted(cum, np.float32(u) * cum[-1], side="right"))
    return idx if idx < len(weights) else int(np.flatnonzero(weights > 0).max())


def _stack_histories(histories):
    hist = np.concatenate(histories)
    offs = np.zeros(len(histories) + 1, np.uint32)
    offs[1:] = np.cumsum([len(h) for h in histories])
    return hist, offs


def _choose_from_visits(visits, stochastic, seed, game_ids, plies):
    out = []
    for k in range(len(visits)):
        w = visits[k] / visits[k].sum()
        out.append(_weighted_index(w, _uniform(seed, game_ids[k], plies[k])) if stochastic[k] else _last_argmax(w))
    return out


def _choose_from_policy(policy, index, count, stochastic, seed, game_ids, plies):
    out = []
    for k in range(len(policy)):
        masked = np.zeros(ACTION_SPACE, np.float32)
        legal = index[k, : count[k]]
        masked[legal] = policy[k, legal]
        out.append(_weighted_index(masked, _uniform(seed, game_ids[k], plies[k])) if stochastic[k] else _last_argmax(masked))
    return out


class MctsPlayer:
    """Player::MctsModel: MCTree::init(model, state, false) + search, then argmax or sampling (validation.rs:293-308).
    leaves_per_root > 1 searches with virtual loss (Engine.search_vl, not in the reference): up to that many leaves per
    root share one network round, which cuts the latency of searches over few roots.  `network` names the engine's network
    slot (Engine.load_weights(..., network)); a non-zero slot searches through Engine.search_networks."""

    def __init__(self, engine, num_simulations=None, leaves_per_root=1, virtual_loss=1.0, network=0):
        self.engine, self.sims = engine, num_simulations
        self.leaves_per_root, self.virtual_loss = int(leaves_per_root), float(virtual_loss)
        self.network = int(network)

    def _num_simulations(self):
        return int(self.sims or self.engine.config.num_simulations)

    def choose(self, positions, histories, fullmoves, stochastic, seed, game_ids, plies):
        hist, offs = _stack_histories(histories)
        if self.network != 0:
            visits, _, _, _ = self.engine.search_networks(positions, self.network, self._num_simulations(), self.leaves_per_root,
                                                          self.virtual_loss, history=hist, hist_offsets=offs)
        elif self.leaves_per_root > 1:
            visits, _, _, _ = self.engine.search_vl(positions, self._num_simulations(), self.leaves_per_root, self.virtual_loss,
                                                    history=hist, hist_offsets=offs)
        else:
            visits, _, _ = self.engine.search(positions, num_simulations=self.sims, history=hist, hist_offsets=offs)
        return _choose_from_visits(visits, stochastic, seed, game_ids, plies)


class BasePlayer:
    """Player::BaseModel: the raw policy masked to the legal moves, no search (validation.rs:310-350).  `network` names the
    engine's network slot; a non-zero slot evaluates through Engine.forward_networks."""

    def __init__(self, engine, network=0):
        self.engine, self.network = engine, int(network)

    def choose(self, positions, histories, fullmoves, stochastic, seed, game_ids, plies):
        if self.network != 0:
            policy, _ = self.engine.forward_networks(positions, self.network)
        else:
            policy, _ = self.engine.forward(positions)
        _, index, count = self.engine.movegen(positions)
        return _choose_from_policy(policy, index, count, stochastic, seed, game_ids, plies)


def _joint_choose(player_1, player_2):
    """When both players search (or evaluate) on the same engine with the same search settings, one ply of all games is one
    search_networks (forward_networks) call with a network slot per game, so both players share every network round.
    Returns choose(positions, histories, movers, stochastic, seed, game_ids, plies) or None; movers[k] is 0 for player 1."""
    if player_1.engine is not player_2.engine or type(player_1) is not type(player_2):
        return None
    eng = player_1.engine
    if type(player_1) is MctsPlayer:
        settings = [(p._num_simulations(), p.leaves_per_root, p.virtual_loss) for p in (player_1, player_2)]
        if settings[0] != settings[1]:
            return None
        sims, k, vl = settings[0]

        def choose(positions, histories, movers, stochastic, seed, game_ids, plies):
            hist, offs = _stack_histories(histories)
            nets = np.where(movers == 0, player_1.network, player_2.network)
            visits, _, _, _ = eng.search_networks(positions, nets, sims, k, vl, history=hist, hist_offsets=offs)
            return _choose_from_visits(visits, stochastic, seed, game_ids, plies)
        return choose
    if type(player_1) is BasePlayer:
        def choose(positions, histories, movers, stochastic, seed, game_ids, plies):
            policy, _ = eng.forward_networks(positions, np.where(movers == 0, player_1.network, player_2.network))
            _, index, count = eng.movegen(positions)
            return _choose_from_policy(policy, index, count, stochastic, seed, game_ids, plies)
        return choose
    return None


class RandomPlayer:
    """Player::Random: a uniformly random legal move (validation.rs:359-365); needs an engine only for movegen."""

    def __init__(self, engine):
        self.engine = engine

    def choose(self, positions, histories, fullmoves, stochastic, seed, game_ids, plies):
        _, index, count = self.engine.movegen(positions)
        return [int(index[k, int(_uniform(seed ^ 0x5151, game_ids[k], plies[k]) * count[k])]) for k in range(len(positions))]


class MiniMaxPlayer:
    """Player::MiniMax(depth) (validation.rs:113-120, 352-358; chess.rs:247-318): full-width negamax over material, a
    random choice among the best-scoring moves.  The whole batch of positions is searched by az_minimax in one call; the
    reference default is depth 4 (main.rs:103, training.rs:254)."""

    def __init__(self, engine, depth=4):
        self.engine, self.depth = engine, depth

    def choose(self, positions, histories, fullmoves, stochastic, seed, game_ids, plies):
        scores, count = self.engine.minimax(positions, self.depth)
        _, index, _ = self.engine.movegen(positions)
        out = []
        for k in range(len(positions)):
            sc = scores[k, : count[k]]
            best = np.flatnonzero(sc == sc.max())
            out.append(int(index[k, best[int(_uniform(seed ^ 0x3A3A, game_ids[k], plies[k]) * len(best))]]))
        return out


def evaluate(player_1, player_2, rules_engine, n_games=EVALUATION_GAMES, num_stochastic_moves=TEMPERATURE_ANNEALING, seed=0,
             max_plies=450):
    """evaluate (validation.rs:155-282): n_games games, colours alternate by game parity, result from player 1's side.
    Returns dict(winrate, p1_winrate, drawrate, p2_winrate, results)."""
    pos = np.repeat(np.array([start_position()], POSITION_DTYPE), n_games)
    hist = [[pos[g].copy()] for g in range(n_games)]
    result = np.zeros(n_games, np.float32)       # white's point of view: 1, 0, -1
    active = np.ones(n_games, bool)
    players = (player_1, player_2)
    joint = _joint_choose(player_1, player_2)
    for ply in range(max_plies):
        if not active.any():
            break
        white_to_move = ply % 2 == 0
        chosen = np.zeros(n_games, np.int64)
        if joint is not None:
            # every active game has one mover: player 1 in game g when (g even) == (White to move)
            ids = np.flatnonzero(active)
            movers = np.array([0 if (g % 2 == 0) == white_to_move else 1 for g in ids])
            fm = pos["fullmoves"][ids]
            chosen[ids] = joint(pos[ids], [np.array(hist[g], POSITION_DTYPE) for g in ids], movers, fm <= num_stochastic_moves, seed,
                                ids, np.full(len(ids), ply))
        for which in (0, 1) if joint is None else ():
            # game g: player_1 is White when g is even (validation.rs:196-200)
            owns = np.array([active[g] and ((g % 2 == 0) == (which == 0)) == white_to_move for g in range(n_games)])
            ids = np.flatnonzero(owns)
            if len(ids) == 0:
                continue
            fm = pos["fullmoves"][ids]
            acts = players[which].choose(pos[ids], [np.array(hist[g], POSITION_DTYPE) for g in ids], fm, fm <= num_stochastic_moves, seed,
                                         ids, np.full(len(ids), ply))
            chosen[ids] = acts
        ids = np.flatnonzero(active)
        h = np.concatenate([np.array(hist[g], POSITION_DTYPE) for g in ids])
        offs = np.zeros(len(ids) + 1, np.uint32)
        offs[1:] = np.cumsum([len(hist[g]) for g in ids])
        new_pos, res = rules_engine.play_move(pos[ids], chosen[ids].astype(np.uint16), h, offs)
        for k, g in enumerate(ids):
            if res[k] == ILLEGAL:
                raise RuntimeError(f"game {g}: an illegal move was played (policy index {chosen[g]})")  # the reference panics
            pos[g] = new_pos[k]
            hist[g].append(new_pos[k].copy())
            if res[k] != ONGOING:
                active[g] = False
                result[g] = 0.0 if res[k] == DRAW else (1.0 if res[k] == WHITE_WINS else -1.0)
    p1 = np.where(np.arange(n_games) % 2 == 0, result, -result)   # validation.rs:196-200
    wins, draws = float((p1 == 1).sum()), float((p1 == 0).sum())
    return {"winrate": (wins + draws / 2.0) / n_games, "p1_winrate": wins / n_games, "drawrate": draws / n_games,
            "p2_winrate": (n_games - wins - draws) / n_games, "results": p1, "unfinished": int(active.sum())}


def evaluate_on_device(player_1, player_2, n_games=EVALUATION_GAMES, num_stochastic_moves=TEMPERATURE_ANNEALING, seed=0, max_plies=450,
                       concurrent=None, waves_per_step=256):
    """evaluate() played resident on the device (Engine.match_begin / match_step / match_results): the same games, bit for bit,
    for the pairs whose plies evaluate() runs as one joint call -- two MctsPlayers with equal (num_simulations, leaves_per_root,
    virtual_loss) or two BasePlayers, on one engine -- without a host round trip per ply.  `concurrent` games run at once (None:
    as many as max_games and the two network ranges allow, 2 x round4(slots x leaves_per_root) <= max_batch).  All n_games run
    at once, as evaluate() searches them, only when max_games >= n_games and max_batch >= 2 x round4(n_games x leaves_per_root);
    with fewer slots the games are the same but the match takes more network rounds, so size the engine accordingly.  Returns
    evaluate()'s dict plus `moves` [n_games, max_plies] (the policy indices played, MOVE_NONE after the last), `plies` [n_games]
    and `stats` (MatchStats: waves, evaluations per network, ...).
    Raises ValueError for other pairs."""
    from . import MATCH_BASE_MODEL, MATCH_MCTS

    kinds = (type(player_1), type(player_2))
    if kinds[0] is not kinds[1] or kinds[0] not in (MctsPlayer, BasePlayer):
        raise ValueError("evaluate_on_device plays two MctsPlayers or two BasePlayers; use evaluate() for other pairs")
    if player_1.engine is not player_2.engine:
        raise ValueError("evaluate_on_device needs both players on one engine (network slots 0 and 1)")
    eng = player_1.engine
    if max_plies < 1:
        raise ValueError("max_plies must be >= 1")
    kw = {}
    if kinds[0] is MctsPlayer:
        settings = [(p._num_simulations(), p.leaves_per_root, p.virtual_loss) for p in (player_1, player_2)]
        if settings[0] != settings[1]:
            raise ValueError("evaluate_on_device needs equal (num_simulations, leaves_per_root, virtual_loss) for both players")
        kw = dict(num_simulations=settings[0][0], leaves_per_root=settings[0][1], virtual_loss=settings[0][2])
    k = kw.get("leaves_per_root", 1)
    if concurrent is None:   # all games at once, as far as max_games and the two network ranges (2 x round4(slots x K)) allow
        max_batch = max(int(eng.config.max_batch), int(eng.config.max_games))
        concurrent = min(n_games, int(eng.config.max_games), (max_batch // 2) // 4 * 4 // k)
    slots = min(int(concurrent), n_games)
    eng.match_begin(slots, n_games, MATCH_MCTS if kinds[0] is MctsPlayer else MATCH_BASE_MODEL, (player_1.network, player_2.network),
                    num_stochastic_moves=num_stochastic_moves, max_plies=max_plies, seed=seed, **kw)
    stats = eng.match_step(waves_per_step)
    while stats.active_games:
        stats = eng.match_step(waves_per_step)
    white, plies, finished, moves = eng.match_results()
    result = white.astype(np.float32)
    p1 = np.where(np.arange(n_games) % 2 == 0, result, -result)   # validation.rs:196-200
    wins, draws = float((p1 == 1).sum()), float((p1 == 0).sum())
    return {"winrate": (wins + draws / 2.0) / n_games, "p1_winrate": wins / n_games, "drawrate": draws / n_games,
            "p2_winrate": (n_games - wins - draws) / n_games, "results": p1, "unfinished": int((~finished).sum()),
            "moves": moves, "plies": plies, "stats": stats}


def compute_elos(winrate_matrix, base_elo):
    """ratings.rs:113-144 in f32: player 0 is the anchor, 1000 synchronous updates with step 8."""
    w = np.asarray(winrate_matrix, np.float32)
    n = w.shape[0]
    elos = np.full(n, base_elo, np.float32)
    lr = np.float32(8.0)
    for _ in range(1000):
        prev = elos.copy()
        for i in range(1, n):
            actual = np.float32(0.0)
            expected = np.float32(0.0)
            for j in range(n):
                if i == j:
                    continue
                actual = np.float32(actual + w[i, j])
                diff = np.float32(prev[j] - prev[i])
                expected = np.float32(expected + np.float32(1.0) / (np.float32(1.0) + np.power(np.float32(10.0), np.float32(diff / np.float32(400.0)))))
            elos[i] = np.float32(elos[i] + lr * np.float32(actual - expected))
    return elos


def compute_elo_rankings(players, base_elo, rules_engine, n_games=EVALUATION_GAMES, seed=0):
    """ratings.rs:5-111 without the pretty printer: round robin (i vs j for j < i), then the Elo fit."""
    n = len(players)
    matrix = np.full((n, n), 0.5, np.float32)
    for i in range(n):
        for j in range(i):
            wr = evaluate(players[i], players[j], rules_engine, n_games=n_games, seed=seed + 1000 * i + j)["winrate"]
            matrix[i, j] = wr
            matrix[j, i] = 1.0 - wr
    return compute_elos(matrix, base_elo), matrix
