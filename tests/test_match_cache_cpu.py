"""The host side of a match's evaluation cache without a device: the ctypes layouts carry cache_log2 and cache_hits where the C
header has them, Engine.match_begin_players writes cache_log2 into the config, and evaluation.evaluate_on_device passes it through
(0 when not given)."""
import ctypes

import numpy as np

import alphazero_chess_b200 as az
from alphazero_chess_b200 import evaluation as ev


def test_layouts_follow_the_header():
    # az_match_players_config: two 20-byte players, two u32, the u64 seed at 48, cache_log2 at 56, padded to 64
    assert az.MatchPlayersConfig.cache_log2.offset == 56 and ctypes.sizeof(az.MatchPlayersConfig) == 64
    # az_match_stats: waves, evaluations[2], six counters, then cache_hits[2]
    assert az.MatchStats.cache_hits.offset == 8 * 9 and ctypes.sizeof(az.MatchStats) == 8 * 11
    assert az.MatchPlayersConfig().cache_log2 == 0   # a zero-initialised config plays without the cache


class _Lib:
    def __init__(self):
        self.config = None

    def az_match_begin_players(self, h, slots, first, n_games, cfg):
        self.config = ctypes.cast(cfg, ctypes.POINTER(az.MatchPlayersConfig)).contents
        return 0


def test_match_begin_players_writes_cache_log2():
    eng = az.Engine.__new__(az.Engine)   # no device: the library is a recorder
    eng._L, eng._h, eng._check = _Lib(), None, lambda r, what: None
    p = az.match_player(az.PLAYER_RANDOM)
    eng.match_begin_players(2, 2, p, p)
    assert eng._L.config.cache_log2 == 0
    eng.match_begin_players(2, 2, p, p, cache_log2=20)
    assert eng._L.config.cache_log2 == 20


class _Config:
    max_games, max_batch, num_simulations = 64, 128, 16


class _FakeEngine:
    """Records the match evaluate_on_device begins and ends it at once."""

    config = _Config()

    def match_begin_players(self, slots, n_games, p1, p2, **kw):
        self.kw, self.n = kw, n_games

    def match_step(self, waves):
        return az.MatchStats()

    def match_results(self):
        n = self.n
        return np.zeros(n, np.int8), np.ones(n, np.uint16), np.ones(n, np.uint8), np.zeros((n, 1), np.uint16)


def test_evaluate_on_device_passes_cache_log2_through():
    e = _FakeEngine()
    ev.evaluate_on_device(ev.MctsPlayer(e, 16), ev.BasePlayer(e, network=1), n_games=4)
    assert e.kw["cache_log2"] == 0
    ev.evaluate_on_device(ev.MctsPlayer(e, 16), ev.RandomPlayer(e), n_games=4, cache_log2=12)
    assert e.kw["cache_log2"] == 12
