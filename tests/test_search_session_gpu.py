"""The session an engine is in (none, self-play, leaf-parallel self-play, match) decides which session-bound calls succeed:
the status every such call returns in each state, the launches one call of each kind counts (az_launch_count, reported by
bench.py as gpu_launches), and the order of the pending-sample counter's updates between az_replay_add_pending and a drain."""
import ctypes

import numpy as np
import pytest

import alphazero_chess_b200 as az
from helpers import KIWIPETE, orc

pytestmark = pytest.mark.gpu

OK, STATE = 0, -8
SLOTS = 4


def _engine(**kw):
    e = az.Engine(max_games=8, max_batch=64, num_simulations=16, **kw)
    e.set_evaluator_stub(1, 5)
    return e


def _roots(n=4):
    fens = ["rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1", KIWIPETE]
    return np.array([orc.from_fen(fens[i % 2]) for i in range(n)], az.POSITION_DTYPE)


def _statuses(e):
    """The status of every session-bound entry point, called so that none of them changes the session."""
    L, h = e._L, e._h
    n = ctypes.c_int(0)
    samples = np.empty(1 << 16, az.SAMPLE_DTYPE)
    result, plies, finished = np.empty(64, np.int8), np.empty(64, np.uint16), np.empty(64, np.uint8)
    rb = az.ReplayBuffer(e, capacity=1024, max_batch=64)
    try:
        out = {
            "selfplay_step": L.az_selfplay_step(h, 0, ctypes.byref(az.SelfplayStats())),
            "selfplay_vl_stats": L.az_selfplay_vl_stats(h, ctypes.byref(az.SearchStats())),
            "selfplay_drain": L.az_selfplay_drain(h, az._ptr(samples), samples.shape[0], ctypes.byref(n)),
            "selfplay_drain_dev": L.az_selfplay_drain_dev(h, ctypes.c_void_p(0), samples.shape[0], ctypes.byref(n)),
            "selfplay_staged": L.az_dbg_selfplay_staged(h, 0, az._ptr(samples), 512, ctypes.byref(n)),
            "replay_add_pending": L.az_replay_add_pending(rb._h, ctypes.byref(n), ctypes.byref(n)),
            "match_step": L.az_match_step(h, 0, ctypes.byref(az.MatchStats())),
            "match_results": L.az_match_results(h, az._ptr(result), az._ptr(plies), az._ptr(finished), None),
        }
    finally:
        rb.close()
    return out


NONE = dict.fromkeys(["selfplay_step", "selfplay_vl_stats", "selfplay_drain", "selfplay_drain_dev", "selfplay_staged",
                      "replay_add_pending", "match_step", "match_results"], STATE)
SELFPLAY = {**NONE, "selfplay_step": OK, "selfplay_drain": OK, "selfplay_drain_dev": OK, "selfplay_staged": OK,
            "replay_add_pending": OK}
SELFPLAY_VL = {**SELFPLAY, "selfplay_vl_stats": OK}
MATCH = {**NONE, "match_step": OK, "match_results": OK}
MATCH_ENDED = {**NONE, "match_results": OK}


def _begin_match(e):
    e.match_begin(SLOTS, 4, az.MATCH_MCTS, (0, 0), num_simulations=8, leaves_per_root=2, max_plies=8)


def _failed(call):
    with pytest.raises(az.EngineError):
        call()


STATES = {
    "fresh": ([], NONE),
    "selfplay": ([lambda e: e.selfplay_begin(SLOTS)], SELFPLAY),
    "selfplay_vl": ([lambda e: e.selfplay_begin(SLOTS, leaves_per_game=2)], SELFPLAY_VL),
    "match": ([_begin_match], MATCH),
    "search_after_match": ([_begin_match, lambda e: e.search(_roots(), 8)], MATCH_ENDED),
    "search_vl_after_selfplay_vl": ([lambda e: e.selfplay_begin(SLOTS, leaves_per_game=2), lambda e: e.search_vl(_roots(), 8, 2)],
                                    NONE),
    "search_after_selfplay": ([lambda e: e.selfplay_begin(SLOTS), lambda e: e.search(_roots(), 8)], NONE),
    "zero_root_search_after_selfplay": ([lambda e: e.selfplay_begin(SLOTS), lambda e: e.search(np.zeros(0, az.POSITION_DTYPE), 8)],
                                        SELFPLAY),
    "rejected_search_after_match": ([_begin_match, lambda e: _failed(lambda: e.search(_roots(), 64))], MATCH),
    "rejected_search_vl_after_selfplay_vl": ([lambda e: e.selfplay_begin(SLOTS, leaves_per_game=2),
                                              lambda e: _failed(lambda: e.search_vl(_roots(), 8, 0))], SELFPLAY_VL),
    "failed_begin_vl_after_selfplay": ([lambda e: e.selfplay_begin(SLOTS), lambda e: _failed(lambda: e.selfplay_begin(SLOTS, leaves_per_game=0))],
                                       SELFPLAY),
    "failed_match_begin_after_selfplay_vl": ([lambda e: e.selfplay_begin(SLOTS, leaves_per_game=2),
                                              lambda e: _failed(lambda: e.match_begin(SLOTS, 4, az.MATCH_MCTS, leaves_per_root=0))],
                                             SELFPLAY_VL),
    "failed_selfplay_begin_after_match": ([_begin_match, lambda e: _failed(lambda: e.selfplay_begin(100))], MATCH),
}


@pytest.mark.parametrize("state", list(STATES))
def test_session_status_matrix(state):
    calls, expected = STATES[state]
    with _engine() as e:
        for c in calls:
            c(e)
        assert _statuses(e) == expected


def _launches(e, call):
    before = e.launch_count()
    call()
    return e.launch_count() - before


def test_launch_counts_per_call():
    # under the synthetic evaluator one batch costs one k_stub_eval per network; k_count_active and k_export_root are not counted
    with _engine() as e:
        n = _launches(e, lambda: e.search(_roots(), 16))
        assert n >= 2 + 2 * 16 and n % 2 == 0   # k_init_search, the roots' evaluation, then k_advance + evaluation per wave
        out = []
        n = _launches(e, lambda: out.append(e.search_vl(_roots(), 16, 4)))
        # k_init_search and the roots' evaluation, k_vl_gather + k_vl_expand + evaluation per wave, and the last k_vl_gather,
        # counted with its k_vl_expand although the search ends before it
        assert n == 3 * out[-1][3].waves + 1
        n = _launches(e, lambda: out.append(e.search_networks(_roots(), [0, 1, 0, 1], 16, 2)))
        assert n == 4 * out[-1][3].waves + 1
        e.selfplay_begin(SLOTS)
        assert _launches(e, lambda: e.selfplay_step(5)) == 5 * 2   # k_advance + evaluation
        e.selfplay_begin(SLOTS, leaves_per_game=2)
        assert _launches(e, lambda: e.selfplay_step(5)) == 5 * 3   # k_vl_selfplay + k_vl_expand + evaluation
        _begin_match(e)
        assert _launches(e, lambda: e.match_step(5)) == 5 * 4      # k_match + k_vl_expand_nets + one evaluation per network


@pytest.mark.parametrize("leaves_per_game", [None, 2])
def test_drain_after_add_pending_returns_nothing(leaves_per_game):
    with _engine(num_fullmoves=4) as e:
        rb = az.ReplayBuffer(e, capacity=4096, max_batch=64)
        e.selfplay_begin(SLOTS, leaves_per_game=leaves_per_game)
        while e.selfplay_step(16).pending_samples == 0:
            pass
        added, _ = rb.add_pending()
        assert added > 0
        assert len(e.selfplay_drain()) == 0   # the samples just added are not handed out a second time
        while True:
            pending = e.selfplay_step(16).pending_samples
            if pending:
                break
        drained = e.selfplay_drain()
        assert len(drained) == pending
        assert e.selfplay_step(0).pending_samples == 0
        rb.close()
