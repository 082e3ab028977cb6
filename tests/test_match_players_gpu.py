"""Matches between two independent players resident on the device (az_match_begin_players): every game's moves and result equal
the test restatement (tests/match_players_oracle.py) under the synthetic evaluator and equal evaluation.evaluate() of the same
players on the same engine, whatever the slots, the engines and the network path; az_match_begin is the same match for two equal
players; errors leave the engine usable."""
import json
import os
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
import match_players_oracle as mpo
from alphazero_chess_b200 import evaluation as ev
from helpers import ROOT

pytestmark = pytest.mark.gpu

STUB_SEED = 17
MOVE_NONE = 0xFFFF

# (player 1, player 2) without their networks: kind, num_simulations, leaves_per_root, virtual_loss
PAIRINGS = {
    "mcts_base": (("mcts", 16, 4, 1.0), ("base",)),
    "base_mcts": (("base",), ("mcts", 16, 1, 1.0)),
    "mcts64_mcts16": (("mcts", 64, 1, 1.0), ("mcts", 16, 1, 1.0)),
    "mcts_k1_k8": (("mcts", 16, 1, 1.0), ("mcts", 16, 8, 0.5)),
    "mcts_random": (("mcts", 16, 2, 1.0), ("random",)),
    "base_random": (("base",), ("random",)),
    "random_random": (("random",), ("random",)),
}
NETWORKS = [(0, 1), (1, 0), (0, 0)]


def _oracle_players(pairing, networks):
    out = []
    for spec, net in zip(PAIRINGS[pairing], networks):
        if spec[0] == "mcts":
            out.append(mpo.player("mcts", net, spec[1], spec[2], spec[3]))
        else:
            out.append(mpo.player(spec[0], net))
    return out


def _device_players(pairing, networks):
    kinds = {"mcts": az.PLAYER_MCTS, "base": az.PLAYER_BASE_MODEL, "random": az.PLAYER_RANDOM}
    return [az.match_player(kinds[p["kind"]], p["network"], p["num_simulations"], p["leaves_per_root"], p["virtual_loss"])
            for p in _oracle_players(pairing, networks)]


def _eval_players(eng, pairing, networks):
    out = []
    for p in _oracle_players(pairing, networks):
        if p["kind"] == "mcts":
            out.append(ev.MctsPlayer(eng, p["num_simulations"], p["leaves_per_root"], p["virtual_loss"], network=p["network"]))
        elif p["kind"] == "base":
            out.append(ev.BasePlayer(eng, network=p["network"]))
        else:
            out.append(ev.RandomPlayer(eng))
    return out


def _stub_engine(slots, sims=64, max_batch=None, **kw):
    e = az.Engine(max_games=slots, max_batch=max_batch or 16 * slots, num_simulations=sims, **kw)
    e.set_evaluator_stub(1, STUB_SEED)
    return e


def _play(e, slots, n_games, players, first_game=0, waves=64, **kw):
    e.match_begin_players(slots, n_games, players[0], players[1], first_game=first_game, **kw)
    while True:
        st = e.match_step(waves)
        if st.active_games == 0:
            break
    assert st.games_finished == n_games
    return e.match_results(), st


def _check_restatement(res, st, first_game, players, nsm=15, max_plies=450, seed=0):
    white, plies, finished, moves = res
    evals, under = [0, 0], 0
    for i in range(len(white)):
        g = first_game + i
        ref = mpo.match_game(g, players, STUB_SEED, num_stochastic_moves=nsm, max_plies=max_plies, seed=seed)
        assert plies[i] == ref["plies"] and finished[i] == ref["finished"] and white[i] == ref["result"], g
        assert list(moves[i, : plies[i]]) == ref["moves"], g
        assert np.all(moves[i, plies[i]:] == MOVE_NONE), g
        evals = [a + b for a, b in zip(evals, ref["evaluations"])]
        under += ref["random_underpromotions"]
    # plies = their sum; evaluations[s] = the roots of the non-Random plies on s + the non-terminal leaves
    assert st.plies == int(plies.astype(int).sum())
    assert list(st.evaluations) == evals
    return under


@pytest.mark.parametrize("networks", NETWORKS)
@pytest.mark.parametrize("pairing", list(PAIRINGS))
def test_short_games_equal_the_restatement(pairing, networks):
    # fullmove <= 3 samples, later plies take the last maximum; 14 plies leave most games unfinished
    players = _oracle_players(pairing, networks)
    with _stub_engine(4, 64) as e:
        res, st = _play(e, 3, 5, _device_players(pairing, networks), first_game=5, num_stochastic_moves=3, max_plies=14, seed=11)
    _check_restatement(res, st, 5, players, nsm=3, max_plies=14, seed=11)


@pytest.mark.parametrize("pairing", list(PAIRINGS))
def test_full_length_games_equal_the_restatement(pairing):
    players = _oracle_players(pairing, (0, 1))
    n = 24 if pairing == "random_random" else 4
    with _stub_engine(8, 64) as e:
        res, st = _play(e, 4, n, _device_players(pairing, (0, 1)), seed=3)
    assert res[2].any()
    under = _check_restatement(res, st, 0, players, seed=3)
    if pairing == "random_random":
        # Random picks from az_movegen's list, under-promotions included: the root edges must follow that list's order
        assert under > 0
        assert st.evaluations[0] == st.evaluations[1] == 0 and st.leaves == 0


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
    for key in ("winrate", "p1_winrate", "drawrate", "p2_winrate"):
        assert dev[key] == ref[key], key
    moves, plies = dev["moves"], dev["plies"]
    assert len(played) == int(plies.max())
    for p, acts in enumerate(played):   # the games still on at ply p, in game order
        assert np.array_equal(moves[plies > p, p], acts), p


# evaluate()'s BasePlayer reads forward / forward_networks, which have no synthetic evaluator: the pairings with a BaseModel player
# are compared with evaluate() on real networks below
STUB_EVALUATE_PAIRINGS = [p for p in PAIRINGS if "base" not in p]
BASE_PAIRINGS = [p for p in PAIRINGS if "base" in p]


@pytest.mark.parametrize("networks", NETWORKS)
@pytest.mark.parametrize("pairing", STUB_EVALUATE_PAIRINGS)
def test_stub_match_equals_evaluate(pairing, networks):
    with _stub_engine(16, 64, max_batch=256) as e:
        p1, p2 = _eval_players(e, pairing, networks)
        ref, played = _captured_evaluate(e, p1, p2, n_games=12, max_plies=80, seed=9)
        dev = ev.evaluate_on_device(p1, p2, n_games=12, max_plies=80, seed=9, concurrent=5)
    _check_against_evaluate(ref, played, dev)


@pytest.mark.parametrize("pairing", ["mcts_k1_k8", "mcts_random", "base_mcts"])
def test_results_do_not_depend_on_slots_or_engines(pairing):
    players = _device_players(pairing, (1, 0))
    kw = dict(max_plies=60, seed=2)
    out = []
    with _stub_engine(16, 16, max_batch=512) as e:
        for slots in (1, 3, 16):
            out.append(_play(e, slots, 16, players, **kw)[0])
    with _stub_engine(8, 16, max_batch=128) as a, _stub_engine(8, 16, max_batch=128) as b:
        ra, _ = _play(a, 8, 9, players, **kw)
        rb, _ = _play(b, 8, 7, players, first_game=9, **kw)
    out.append(tuple(np.concatenate([x, y]) for x, y in zip(ra, rb)))
    for r in out[1:]:
        assert all(np.array_equal(x, y) for x, y in zip(r, out[0]))


def test_random_vs_random_needs_no_weights():
    with az.Engine(max_games=16, max_batch=16, num_simulations=16) as e:   # no network loaded, no synthetic evaluator
        p1, p2 = ev.RandomPlayer(e), ev.RandomPlayer(e)
        ref, played = _captured_evaluate(e, p1, p2, n_games=16, max_plies=450, seed=1)
        dev = ev.evaluate_on_device(p1, p2, n_games=16, max_plies=450, seed=1, concurrent=4)
    _check_against_evaluate(ref, played, dev)
    st = dev["stats"]
    assert list(st.evaluations) == [0, 0] and st.plies == int(dev["plies"].astype(int).sum())


# ---- real networks ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def weights():
    return az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)


def _net_engine(weights, **cfg):
    e = az.Engine(**cfg)
    e.load_weights(weights[0])
    e.load_weights(weights[1], network=1)
    return e


@pytest.mark.parametrize("pairing,networks,n_games,max_plies", [("mcts_base", (0, 1), 32, 80), ("base_mcts", (1, 1), 16, 450),
                                                                ("mcts_random", (1, 0), 32, 450), ("mcts64_mcts16", (0, 1), 16, 40)])
def test_bf16_match_equals_evaluate(weights, pairing, networks, n_games, max_plies):
    with _net_engine(weights, max_games=64, max_batch=512, num_simulations=64) as e:
        p1, p2 = _eval_players(e, pairing, networks)
        ref, played = _captured_evaluate(e, p1, p2, n_games=n_games, max_plies=max_plies, seed=4)
        dev = ev.evaluate_on_device(p1, p2, n_games=n_games, max_plies=max_plies, seed=4)
    _check_against_evaluate(ref, played, dev)


@pytest.mark.parametrize("pairing", ["mcts_base", "mcts_random"])
def test_bf16_waves_across_the_tower_range_split(weights, pairing):
    # 512 slots x 8 leaves on network 0: up to 4096 boards per wave in its range, more than one tower range (2072 boards)
    with _net_engine(weights, max_games=512, max_batch=8192, num_simulations=16) as e:
        p1 = ev.MctsPlayer(e, 16, leaves_per_root=8, network=0)
        p2 = ev.BasePlayer(e, network=1) if pairing == "mcts_base" else ev.RandomPlayer(e)
        ref, played = _captured_evaluate(e, p1, p2, n_games=512, max_plies=6, seed=4)
        dev = ev.evaluate_on_device(p1, p2, n_games=512, max_plies=6, seed=4)
    _check_against_evaluate(ref, played, dev)


@pytest.mark.parametrize("networks", NETWORKS)
@pytest.mark.parametrize("pairing", BASE_PAIRINGS)
def test_bf16_base_pairings_equal_evaluate(weights, pairing, networks):
    with _net_engine(weights, max_games=16, max_batch=256, num_simulations=16) as e:
        p1, p2 = _eval_players(e, pairing, networks)
        ref, played = _captured_evaluate(e, p1, p2, n_games=12, max_plies=80, seed=9)
        dev = ev.evaluate_on_device(p1, p2, n_games=12, max_plies=80, seed=9, concurrent=5)
    _check_against_evaluate(ref, played, dev)


def test_fp32_match_equals_evaluate(weights):
    with _net_engine(weights, max_games=16, max_batch=64, num_simulations=16, precision=1) as e:
        p1, p2 = _eval_players(e, "mcts_base", (1, 0))
        ref, played = _captured_evaluate(e, p1, p2, n_games=8, max_plies=24, seed=6)
        dev = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=24, seed=6)
    _check_against_evaluate(ref, played, dev)


@pytest.mark.parametrize("kind,k", [(az.MATCH_MCTS, 1), (az.MATCH_MCTS, 4), (az.MATCH_BASE_MODEL, 1)])
def test_match_begin_is_begin_players_with_two_equal_players(weights, kind, k):
    kw = dict(num_stochastic_moves=5, max_plies=60, seed=8)
    with _net_engine(weights, max_games=16, max_batch=256, num_simulations=16) as e:
        e.match_begin(8, 12, kind, (1, 0), num_simulations=16, leaves_per_root=k, virtual_loss=0.5, **kw)
        while e.match_step(64).active_games:
            pass
        st_a, res_a = e.match_step(0), e.match_results()
        pk = az.PLAYER_MCTS if kind == az.MATCH_MCTS else az.PLAYER_BASE_MODEL
        players = [az.match_player(pk, s, 16, k, 0.5) for s in (1, 0)]
        res_b, st_b = _play(e, 8, 12, players, **kw)
    assert all(np.array_equal(x, y) for x, y in zip(res_a, res_b))
    for f in ("evaluations", "leaves", "terminal_leaves", "collisions", "plies", "games_finished", "active_games"):
        assert np.array_equal(np.array(getattr(st_a, f)), np.array(getattr(st_b, f))), f


def test_errors_leave_the_engine_usable(weights, monkeypatch):
    ok = dict(max_plies=4)
    M, B, R = az.PLAYER_MCTS, az.PLAYER_BASE_MODEL, az.PLAYER_RANDOM
    pos = np.array([az.start_position()] * 2, az.POSITION_DTYPE)

    def usable(e):
        v, _, _ = e.search(pos, num_simulations=8)
        assert np.all(v.sum(1) == 8)

    with az.Engine(max_games=8, max_batch=16, num_simulations=16) as e:
        e.load_weights(weights[0])
        # slot 1 is never loaded: an error only when a non-Random player uses it
        with pytest.raises(az.EngineError, match=": -5:"):
            e.match_begin_players(2, 2, az.match_player(M, 1, 16), az.match_player(R), **ok)
        usable(e)
        with pytest.raises(az.EngineError, match=": -5:"):
            e.match_begin_players(2, 2, az.match_player(R), az.match_player(B, 1), **ok)
        usable(e)
        _play(e, 2, 2, [az.match_player(B, 0), az.match_player(R)], **ok)
        cases = [
            (-1, az.MatchPlayer(3, 0, 16, 1, 1.0), az.match_player(R)),                    # MiniMax
            (-1, az.match_player(R), az.MatchPlayer(-1, 0, 0, 1, 0.0)),
            (-1, az.match_player(M, 0, 16, 0), az.match_player(R)),                      # K < 1
            (-1, az.match_player(R), az.match_player(M, 0, 16, 1, -1.0)),               # lambda < 0
            (-1, az.match_player(M, 0, 16, 1, float("nan")), az.match_player(B, 0)),
            (-1, az.match_player(M, 0, 17), az.match_player(B, 0)),                      # S > num_simulations
            (-1, az.MatchPlayer(M, 0, -1, 1, 1.0), az.match_player(B, 0)),
            (-1, az.match_player(B, 2), az.match_player(R)),                             # network id
            (-6, az.match_player(M, 0, 16, 3), az.match_player(B, 0)),                   # 6 slots: round4(6 x 3) = 20 > 16
        ]
        for code, p1, p2 in cases:
            slots = 6 if code == -6 else 2
            with pytest.raises(az.EngineError, match=f": {code}:"):
                e.match_begin_players(slots, slots, p1, p2, **ok)
            usable(e)
        for slots, n, mp in ((2, 0, 4), (0, 2, 4), (2, 2, 0)):
            with pytest.raises(az.EngineError, match=": -1:"):
                e.match_begin_players(slots, n, az.match_player(R), az.match_player(R), max_plies=mp)
            usable(e)
        with pytest.raises(az.EngineError, match=": -6:"):   # more slots than max_games
            e.match_begin_players(9, 9, az.match_player(R), az.match_player(R), **ok)
        usable(e)
        # the capacity rule: one network used, round4(4 x 4) = 16 fits; round4(5 x 4) = 20 does not
        _play(e, 4, 4, [az.match_player(M, 0, 16, 4), az.match_player(B, 0)], **ok)
        with pytest.raises(az.EngineError, match=": -6:"):
            e.match_begin_players(5, 5, az.match_player(M, 0, 16, 4), az.match_player(R), **ok)
        usable(e)
        e.load_weights(weights[1], network=1)
        # two networks: round4(4 x 2) + round4(4) = 12 fits, round4(6 x 2) + round4(6) = 20 does not
        _play(e, 4, 4, [az.match_player(M, 0, 16, 2), az.match_player(B, 1)], **ok)
        with pytest.raises(az.EngineError, match=": -6:"):
            e.match_begin_players(6, 6, az.match_player(M, 0, 16, 2), az.match_player(B, 1), **ok)
        usable(e)
    monkeypatch.setenv("AZ_HEADS_TC", "0")
    with az.Engine(max_games=8, max_batch=16, num_simulations=16) as e:
        e.load_weights(weights[0])
        e.load_weights(weights[1], network=1)
        with pytest.raises(az.EngineError, match=": -8:"):
            e.match_begin_players(2, 2, az.match_player(M, 0, 16), az.match_player(R), **ok)
        usable(e)
        _play(e, 2, 2, [az.match_player(R), az.match_player(R)], **ok)   # no network: the knobs do not matter


def test_cpp_evaluate_players(tmp_path):
    exe = str(tmp_path / "test_match_players")
    lib_dir = os.path.dirname(az.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_match_players.cpp"), "-o", exe, "-L", lib_dir, "-laz_b200",
                           f"-Wl,-rpath,{lib_dir}"])
    out = subprocess.run([exe, str(STUB_SEED)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    res = {d["pairing"]: d for d in (json.loads(l) for l in out.stdout.splitlines() if l.startswith("{"))}
    with _stub_engine(8, 16, max_batch=64) as e:
        mcts, mcts8, rnd = ev.MctsPlayer(e, 16, leaves_per_root=2, network=0), ev.MctsPlayer(e, 8, network=1), ev.RandomPlayer(e)
        for name, (p1, p2) in {"mcts16_mcts8": (mcts, mcts8), "mcts_random": (mcts, rnd), "random_mcts": (rnd, mcts)}.items():
            ref = ev.evaluate(p1, p2, e, n_games=12, seed=4, max_plies=100)
            for key in ("winrate", "drawrate", "p2_winrate"):   # f32 in C++, f64 in Python
                assert abs(res[name][key] - ref[key]) < 1e-6, (name, key)
