"""Matches with their own evaluation cache (az_match_players_config.cache_log2): every pairing plays the games, plies and moves of
the same match without the cache and of evaluation.evaluate(), under the synthetic evaluator (network s uses seed + s, so a key
without the network slot would mix the networks' entries), on bf16 networks (waves across the tower's range split included) and
on the fp32 path; per network, evaluations + cache_hits equal the evaluations without the cache.  A small table evicts and still
plays the same games; every match starts with an empty table; the engine's self-play cache and az_search_networks are untouched;
out-of-range cache_log2 is refused and leaves the engine usable."""
import json
import os
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
from alphazero_chess_b200 import evaluation as ev
from helpers import ROOT

pytestmark = pytest.mark.gpu

STUB_SEED = 17
M, B, R = az.PLAYER_MCTS, az.PLAYER_BASE_MODEL, az.PLAYER_RANDOM

# name: (player 1, player 2), each (kind, network, S, K); S and K matter for MCTS only
PAIRINGS = {
    "mcts_mcts_01_k1": ((M, 0, 16, 1), (M, 1, 16, 1)),
    "mcts_mcts_00_k1": ((M, 0, 16, 1), (M, 0, 16, 1)),
    "mcts_mcts_01_k4": ((M, 0, 16, 4), (M, 1, 16, 4)),
    "mcts_mcts_00_k4": ((M, 0, 16, 4), (M, 0, 16, 4)),
    "mcts16_mcts4": ((M, 0, 16, 1), (M, 0, 4, 1)),
    "mcts_base_00": ((M, 0, 16, 2), (B, 0, 1, 1)),
    "mcts_base_01": ((M, 0, 16, 2), (B, 1, 1, 1)),
    "base_base": ((B, 0, 1, 1), (B, 1, 1, 1)),
    "mcts_random": ((M, 1, 16, 2), (R, 0, 1, 1)),
    "random_random": ((R, 0, 1, 1), (R, 0, 1, 1)),
}
# evaluate()'s BasePlayer reads forward / forward_networks, which have no synthetic evaluator
STUB_EVALUATE = [p for p in PAIRINGS if "base" not in p]


def _device(spec):
    kind, net, s, k = spec
    return az.match_player(kind, net, s, k, 0.5)


def _host(eng, spec):
    kind, net, s, k = spec
    if kind == M:
        return ev.MctsPlayer(eng, s, k, 0.5, network=net)
    return ev.BasePlayer(eng, network=net) if kind == B else ev.RandomPlayer(eng)


def _searches(pairing):
    """S >= 16 for an evaluating player: its later plies revisit what earlier ones expanded, so the cache must hit"""
    return any(kind == M and s >= 16 for kind, _, s, _ in PAIRINGS[pairing])


def _stub_engine(slots, sims=16, max_batch=None, **kw):
    e = az.Engine(max_games=slots, max_batch=max_batch or 16 * slots, num_simulations=sims, **kw)
    e.set_evaluator_stub(1, STUB_SEED)
    return e


def _net_engine(weights, **cfg):
    e = az.Engine(**cfg)
    e.load_weights(weights[0])
    e.load_weights(weights[1], network=1)
    return e


def _play(e, slots, n_games, p1, p2, cache_log2, waves=256, **kw):
    e.match_begin_players(slots, n_games, p1, p2, cache_log2=cache_log2, **kw)
    st = e.match_step(waves)
    while st.active_games:
        st = e.match_step(waves)
    assert st.games_finished == n_games
    return e.match_results(), st


def _same_games(a, b):
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _check_cached(off, on, pairing):
    """on: (results, stats) with the cache, off: without; the same games and, per network, evaluations + hits = evaluations off"""
    _same_games(off[0], on[0])
    st_off, st_on = off[1], on[1]
    assert list(st_off.cache_hits) == [0, 0]
    for s in range(2):
        assert st_on.evaluations[s] + st_on.cache_hits[s] == st_off.evaluations[s], s
    for f in ("leaves", "terminal_leaves", "collisions", "plies", "games_finished"):
        assert getattr(st_on, f) == getattr(st_off, f), f
    assert st_on.waves <= st_off.waves
    if _searches(pairing):
        assert sum(st_on.cache_hits) > 0
    if pairing == "random_random":
        assert list(st_on.cache_hits) == [0, 0] and list(st_on.evaluations) == [0, 0]


def _captured_evaluate(eng, p1, p2, **kw):
    """evaluate() with the moves of every ply captured by wrapping play_move."""
    played, orig = [], eng.play_move
    eng.play_move = lambda pos, act, *a, **k: (played.append(np.array(act)), orig(pos, act, *a, **k))[1]
    try:
        return ev.evaluate(p1, p2, eng, **kw), played
    finally:
        del eng.play_move


def _check_against_evaluate(ref, played, dev):
    assert np.array_equal(dev["results"], ref["results"]) and dev["unfinished"] == ref["unfinished"]
    moves, plies = dev["moves"], dev["plies"]
    assert len(played) == int(plies.max())
    for p, acts in enumerate(played):   # the games still on at ply p, in game order
        assert np.array_equal(moves[plies > p, p], acts), p


# ---- synthetic evaluator ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pairing", list(PAIRINGS))
def test_stub_full_length_games_equal_the_uncached_match(pairing):
    p1, p2 = (_device(s) for s in PAIRINGS[pairing])
    n = 24 if "random" in pairing else 8
    with _stub_engine(8) as e:
        off = _play(e, 8, n, p1, p2, 0, seed=3)
        for log2 in (12, 20):
            _check_cached(off, _play(e, 8, n, p1, p2, log2, seed=3), pairing)
    assert off[0][2].any()   # some games ended by the rules


@pytest.mark.parametrize("pairing", STUB_EVALUATE)
def test_stub_cached_match_equals_evaluate(pairing):
    with _stub_engine(16, max_batch=256) as e:
        p1, p2 = (_host(e, s) for s in PAIRINGS[pairing])
        ref, played = _captured_evaluate(e, p1, p2, n_games=12, max_plies=120, seed=9)
        off = ev.evaluate_on_device(p1, p2, n_games=12, max_plies=120, seed=9, concurrent=5)
        for log2 in (12, 20):
            dev = ev.evaluate_on_device(p1, p2, n_games=12, max_plies=120, seed=9, concurrent=5, cache_log2=log2)
            _check_against_evaluate(ref, played, dev)
            for s in range(2):
                assert dev["stats"].evaluations[s] + dev["stats"].cache_hits[s] == off["stats"].evaluations[s]


def test_stub_small_table_evicts_and_plays_the_same_games():
    p1, p2 = _device((M, 0, 16, 1)), _device((M, 1, 16, 1))
    with _stub_engine(16) as e:
        off = _play(e, 16, 16, p1, p2, 0, seed=5)
        small = _play(e, 16, 16, p1, p2, 4, seed=5)
        large = _play(e, 16, 16, p1, p2, 20, seed=5)
    _check_cached(off, small, "mcts_mcts_01_k1")
    _check_cached(off, large, "mcts_mcts_01_k1")
    assert sum(small[1].cache_hits) < sum(large[1].cache_hits)


def test_every_match_starts_with_an_empty_cache():
    # one slot: the schedule is sequential, so the hits of a match depend only on what the match itself inserted
    p1, p2 = _device((M, 0, 16, 1)), _device((M, 1, 16, 1))
    with _stub_engine(4) as e:
        a = _play(e, 1, 3, p1, p2, 14, seed=2, max_plies=120)
        b = _play(e, 1, 3, p1, p2, 14, seed=2, max_plies=120)
    _same_games(a[0], b[0])
    assert sum(a[1].cache_hits) > 0
    assert list(a[1].cache_hits) == list(b[1].cache_hits) and list(a[1].evaluations) == list(b[1].evaluations)


def _selfplay_records(e, n):
    e.selfplay_begin(n, first_game_id=0, total_games=n)
    out = []
    while True:
        st = e.selfplay_step(64)
        if st.pending_samples:
            out.append(e.selfplay_drain())
        if st.active_games == 0:
            break
    s = np.concatenate(out)
    return s[np.lexsort((s["ply"], s["game_id"]))]


def test_selfplay_cache_and_search_are_untouched_by_a_cached_match():
    # The search half compares state a match could leave behind (pools, leaf records, network ranges) with a fresh engine.  The
    # self-play half pins that self-play still runs with its own cache after a cached match; it cannot see stray writes into the
    # engine's table, which selfplay_begin empties and which never changes a record.  The other tests run their cached matches on
    # engines without a table of their own (az_config.cache_log2 = 0), so those matches can only have used theirs.
    roots = np.array([az.start_position()] * 4, az.POSITION_DTYPE)
    net = np.array([0, 1, 1, 0], np.uint8)
    kw = dict(sims=16, max_batch=128, cache_log2=12, seed=7)
    with _stub_engine(8, **kw) as fresh:
        want_sp = _selfplay_records(fresh, 8)
        want_v, want_s, want_d, _ = fresh.search_networks(roots, net, 16, leaves_per_root=2)
    with _stub_engine(8, **kw) as e:
        _, st = _play(e, 8, 8, _device((M, 0, 16, 2)), _device((M, 1, 16, 2)), 12, max_plies=60)
        assert sum(st.cache_hits) > 0
        got_sp = _selfplay_records(e, 8)
        _play(e, 8, 8, _device((M, 0, 16, 2)), _device((B, 1, 1, 1)), 12, max_plies=60)
        v, s, d, _ = e.search_networks(roots, net, 16, leaves_per_root=2)
    assert got_sp.tobytes() == want_sp.tobytes()
    assert np.array_equal(v, want_v) and np.array_equal(s, want_s) and np.array_equal(d, want_d)


def test_out_of_range_cache_log2_is_refused():
    pos = np.array([az.start_position()] * 2, az.POSITION_DTYPE)
    with _stub_engine(4) as e:
        for bad in (-1, 27):
            with pytest.raises(az.EngineError, match=": -1:"):
                e.match_begin_players(2, 2, _device((M, 0, 16, 1)), _device((R, 0, 1, 1)), cache_log2=bad, max_plies=4)
            v, _, _ = e.search(pos, num_simulations=8)
            assert np.all(v.sum(1) == 8)


# ---- real networks ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def weights():
    return az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)


@pytest.mark.parametrize("pairing", list(PAIRINGS))
def test_bf16_cached_match_equals_evaluate(weights, pairing):
    with _net_engine(weights, max_games=16, max_batch=256, num_simulations=16) as e:
        p1, p2 = (_host(e, s) for s in PAIRINGS[pairing])
        ref, played = _captured_evaluate(e, p1, p2, n_games=8, max_plies=60, seed=4)
        off = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=60, seed=4)
        for log2 in (12, 20):
            dev = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=60, seed=4, cache_log2=log2)
            _check_against_evaluate(ref, played, dev)
            for s in range(2):
                assert dev["stats"].evaluations[s] + dev["stats"].cache_hits[s] == off["stats"].evaluations[s]
            if _searches(pairing):
                assert sum(dev["stats"].cache_hits) > 0


@pytest.mark.parametrize("pairing", ["mcts_base", "mcts_mcts"])
def test_bf16_cached_waves_across_the_tower_range_split(weights, pairing):
    # 512 slots x 8 leaves on network 0: up to 4096 boards per wave in its range, more than one tower range (2072 boards)
    with _net_engine(weights, max_games=512, max_batch=8192, num_simulations=16) as e:
        p1 = ev.MctsPlayer(e, 16, leaves_per_root=8, network=0)
        p2 = ev.BasePlayer(e, network=1) if pairing == "mcts_base" else ev.MctsPlayer(e, 16, leaves_per_root=8, network=0)
        ref, played = _captured_evaluate(e, p1, p2, n_games=512, max_plies=6, seed=4)
        off = ev.evaluate_on_device(p1, p2, n_games=512, max_plies=6, seed=4)
        dev = ev.evaluate_on_device(p1, p2, n_games=512, max_plies=6, seed=4, cache_log2=20)
    _check_against_evaluate(ref, played, dev)
    for s in range(2):
        assert dev["stats"].evaluations[s] + dev["stats"].cache_hits[s] == off["stats"].evaluations[s]
    assert sum(dev["stats"].cache_hits) > 0


@pytest.mark.parametrize("pairing", ["mcts_base_01", "mcts_mcts_00_k4", "mcts_random"])
def test_fp32_cached_match_equals_evaluate(weights, pairing):
    with _net_engine(weights, max_games=16, max_batch=64, num_simulations=16, precision=1) as e:
        p1, p2 = (_host(e, s) for s in PAIRINGS[pairing])
        ref, played = _captured_evaluate(e, p1, p2, n_games=8, max_plies=24, seed=6)
        off = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=24, seed=6)
        dev = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=24, seed=6, cache_log2=12)
    _check_against_evaluate(ref, played, dev)
    for s in range(2):
        assert dev["stats"].evaluations[s] + dev["stats"].cache_hits[s] == off["stats"].evaluations[s]
    assert sum(dev["stats"].cache_hits) > 0


def test_cpp_evaluate_players_with_cache(tmp_path):
    exe = str(tmp_path / "test_match_cache")
    lib_dir = os.path.dirname(az.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_match_cache.cpp"), "-o", exe, "-L", lib_dir, "-laz_b200",
                           f"-Wl,-rpath,{lib_dir}"])
    out = subprocess.run([exe, str(STUB_SEED)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    res = {d["pairing"]: d for d in (json.loads(l) for l in out.stdout.splitlines() if l.startswith("{"))}
    with _stub_engine(8, max_batch=64) as e:
        mcts, mcts8, rnd = ev.MctsPlayer(e, 16, leaves_per_root=2, network=0), ev.MctsPlayer(e, 8, network=1), ev.RandomPlayer(e)
        for name, (p1, p2) in {"mcts16_mcts8": (mcts, mcts8), "mcts_random": (mcts, rnd)}.items():
            ref = ev.evaluate(p1, p2, e, n_games=12, seed=4, max_plies=100)
            for key in ("winrate", "drawrate", "p2_winrate"):   # f32 in C++, f64 in Python
                assert abs(res[name][key] - ref[key]) < 1e-6, (name, key)
