"""The restatement of a match between two independent players (tests/match_players_oracle.py) and the host side of
Engine.match_begin_players / evaluation.evaluate_on_device, without a device: for two equal players the restatement is
tests/match_oracle.py, a Random ply is evaluation.RandomPlayer's choice, and the arguments are checked before the library is
called."""
import numpy as np
import pytest

import alphazero_chess_b200 as az
import match_oracle as mo
import match_players_oracle as mpo
from alphazero_chess_b200 import evaluation as ev
from helpers import orc

STUB_SEED = 17


@pytest.mark.parametrize("game,networks", [(0, (0, 1)), (3, (1, 0)), (6, (0, 0))])
@pytest.mark.parametrize("kind,k", [("mcts", 1), ("mcts", 4), ("base", 1)])
def test_equal_players_are_the_match_restatement(kind, k, game, networks):
    kw = dict(num_stochastic_moves=3, max_plies=14, seed=11)
    players = [mpo.player(kind, s, num_simulations=16, leaves_per_root=k, virtual_loss=0.5) for s in networks]
    got = mpo.match_game(game, players, STUB_SEED, **kw)
    want = mo.match_game(game, kind, networks, STUB_SEED, num_simulations=16, leaves_per_root=k, virtual_loss=0.5, **kw)
    for key in ("result", "plies", "finished", "moves"):
        assert got[key] == want[key], key


class _Batch:
    """What evaluation.RandomPlayer needs of an engine: az_movegen restated by the oracle (policy indices in its move order)."""

    def movegen(self, positions):
        index = np.full((len(positions), az.MAX_MOVES), 0xFFFF, np.uint16)
        count = np.zeros(len(positions), np.int32)
        for k, p in enumerate(positions):
            _, ix = orc.legal_moves(p)
            index[k, : len(ix)], count[k] = ix, len(ix)
        return None, index, count


def test_random_ply_is_random_player_choice():
    # positions from random games, promotions among them: the restatement's choice is RandomPlayer.choose's
    rp = ev.RandomPlayer(_Batch())
    seen_under = 0
    for game in range(6):
        pos, hist = orc.startpos(), [orc.startpos()]
        for ply in range(300):
            action, under = mpo.random_choice(pos, 5, game, ply)
            seen_under += under
            assert rp.choose(np.array([pos], orc.POSITION_DTYPE), None, None, None, 5, [game], [ply]) == [action]
            pos, res = orc.play_move(pos, action, np.array(hist, orc.POSITION_DTYPE))
            hist.append(pos)
            if res != 0:
                break
    assert seen_under > 0


def test_random_ignores_the_stochastic_opening_and_the_network():
    players = [mpo.player("random", 1), mpo.player("random", 0)]
    a = mpo.match_game(4, players, STUB_SEED, num_stochastic_moves=0, max_plies=30, seed=3)
    b = mpo.match_game(4, [mpo.player("random")] * 2, STUB_SEED + 1, num_stochastic_moves=1000, max_plies=30, seed=3)
    assert a == b and a["evaluations"] == [0, 0]


def test_mixed_game_counts_the_evaluations_of_each_network():
    players = [mpo.player("mcts", 1, num_simulations=8, leaves_per_root=2), mpo.player("base", 0)]
    out = mpo.match_game(1, players, STUB_SEED, max_plies=10)
    # game 1: player 2 (BaseModel, network 0) moves at even plies, one evaluation each; the MCTS plies evaluate on network 1
    assert out["evaluations"][0] == 5 and out["evaluations"][1] >= 5


# ---- host side, no device -------------------------------------------------------------------------------------------
def test_match_player_descriptions():
    p = az.match_player(az.PLAYER_MCTS, 1, 64, 8, 0.5)
    assert (p.kind, p.network, p.num_simulations, p.leaves_per_root, p.virtual_loss) == (0, 1, 64, 8, 0.5)
    b = az.match_player(az.PLAYER_BASE_MODEL, 1, 64, 8, 0.5)
    assert (b.kind, b.network, b.num_simulations, b.leaves_per_root) == (1, 1, 0, 1)
    r = az.match_player(az.PLAYER_RANDOM, 1)
    assert (r.kind, r.network) == (2, 0)
    for bad in (3, -1):
        with pytest.raises(ValueError):
            az.match_player(bad)
    with pytest.raises(ValueError):
        az.match_player(az.PLAYER_MCTS, -1)
    assert az.match_player(az.PLAYER_MCTS, 300).network == 255   # left for the library to refuse


def test_match_begin_players_checks_its_players_before_the_library():
    eng = az.Engine.__new__(az.Engine)   # no device: the checks must fail before self._L is touched
    ok = az.match_player(az.PLAYER_RANDOM)
    for bad in (dict(kind=7), dict(kind=az.PLAYER_MCTS, network=-2), "random", None):
        with pytest.raises((ValueError, TypeError)):
            eng.match_begin_players(2, 2, bad, ok)
        with pytest.raises((ValueError, TypeError)):
            eng.match_begin_players(2, 2, ok, bad)


class _Config:
    def __init__(self, max_games, max_batch):
        self.max_games, self.max_batch, self.num_simulations = max_games, max_batch, 16


class _FakeEngine:
    """Records the match evaluate_on_device begins and ends it at once."""

    def __init__(self, max_games=64, max_batch=128):
        self.config, self.begun = _Config(max_games, max_batch), None

    def match_begin_players(self, slots, n_games, p1, p2, **kw):
        self.begun = (slots, n_games, p1, p2, kw)
        self.n = n_games

    def match_step(self, waves):
        return az.MatchStats()

    def match_results(self):
        n = self.n
        return np.zeros(n, np.int8), np.ones(n, np.uint16), np.ones(n, np.uint8), np.zeros((n, 1), np.uint16)


def test_evaluate_on_device_pairings_and_engines():
    e, other = _FakeEngine(), _FakeEngine()
    with pytest.raises(ValueError):
        ev.evaluate_on_device(ev.MctsPlayer(e, 16), ev.MiniMaxPlayer(e))
    with pytest.raises(ValueError):
        ev.evaluate_on_device(ev.MiniMaxPlayer(e), ev.RandomPlayer(e))
    with pytest.raises(ValueError):
        ev.evaluate_on_device(ev.MctsPlayer(e, 16), ev.BasePlayer(other))
    with pytest.raises(ValueError):
        ev.evaluate_on_device(ev.MctsPlayer(e, 16), ev.RandomPlayer(e), max_plies=0)
    # a RandomPlayer's engine is not used
    out = ev.evaluate_on_device(ev.RandomPlayer(None), ev.MctsPlayer(e, 16, leaves_per_root=2, network=1), n_games=8)
    assert e.begun is not None and out["drawrate"] == 1.0
    slots, n, p1, p2, kw = e.begun
    assert (p1.kind, p2.kind, p2.network, p2.num_simulations, p2.leaves_per_root) == (az.PLAYER_RANDOM, az.PLAYER_MCTS, 1, 16, 2)
    out = ev.evaluate_on_device(ev.BasePlayer(other), ev.RandomPlayer(e), n_games=4)
    assert other.begun[2].kind == az.PLAYER_BASE_MODEL and other.begun[3].kind == az.PLAYER_RANDOM
    # two RandomPlayers: player 1's engine
    a, b = _FakeEngine(), _FakeEngine()
    ev.evaluate_on_device(ev.RandomPlayer(a), ev.RandomPlayer(b), n_games=5)
    assert a.begun is not None and b.begun is None and a.begun[0] == 5


@pytest.mark.parametrize("pair,max_games,max_batch,want", [
    (("mcts8_0", "mcts1_1"), 64, 128, 14),   # round4(14 x 8) + round4(14) = 112 + 16 = 128
    (("mcts8_0", "mcts2_0"), 64, 128, 16),   # one network: round4(16 x 8) = 128
    (("base_0", "random"), 64, 32, 64),      # max_batch is at least max_games: round4(64 x 1) = 64
    (("random", "random"), 40, 8, 40),       # no network: max_games
    (("mcts4_0", "base_1"), 64, 96, 19),     # round4(19 x 4) + round4(19) = 76 + 20 = 96
])
def test_default_concurrency_follows_the_capacity_rule(pair, max_games, max_batch, want):
    e = _FakeEngine(max_games, max_batch)

    def make(d):
        if d == "random":
            return ev.RandomPlayer(e)
        kind, net = d.split("_")
        if kind == "base":
            return ev.BasePlayer(e, network=int(net))
        return ev.MctsPlayer(e, 16, leaves_per_root=int(kind[4:]), network=int(net))

    ev.evaluate_on_device(make(pair[0]), make(pair[1]), n_games=64)
    slots = e.begun[0]
    k = [0, 0]
    for d in pair:
        if d != "random":
            kind, net = d.split("_")
            k[int(net)] = max(k[int(net)], 1 if kind == "base" else int(kind[4:]))
    need = lambda s: sum((s * kk + 3) // 4 * 4 for kk in k)
    assert need(slots) <= max(max_batch, max_games) and (slots == min(64, max_games) or need(slots + 1) > max(max_batch, max_games))
    assert slots == want
