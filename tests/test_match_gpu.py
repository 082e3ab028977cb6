"""Evaluation matches resident on the device (az_match_begin / az_match_step / az_match_results): every game's moves and result
equal the test restatement (tests/match_oracle.py) under the synthetic evaluator and equal evaluation.evaluate() of the same
players on the same engine, whatever the slots, the engines and the network path; errors leave the engine usable."""
import json
import os
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
import match_oracle as mo
from alphazero_chess_b200 import evaluation as ev
from helpers import ROOT, orc

pytestmark = pytest.mark.gpu

STUB_SEED = 17
MOVE_NONE = 0xFFFF


def _stub_engine(slots, sims=64, max_batch=None, **kw):
    e = az.Engine(max_games=slots, max_batch=max_batch or 2 * slots, num_simulations=sims, **kw)
    e.set_evaluator_stub(1, STUB_SEED)
    return e


def _play(e, slots, n_games, kind, networks=(0, 1), first_game=0, waves=64, **kw):
    e.match_begin(slots, n_games, kind, networks, first_game=first_game, **kw)
    while True:
        st = e.match_step(waves)
        if st.active_games == 0:
            break
    assert st.games_finished == n_games
    return e.match_results(), st


def _check_restatement(res, first_game, kind, networks, sims=16, k=1, lam=1.0, nsm=15, max_plies=450, seed=0):
    white, plies, finished, moves = res
    for i in range(len(white)):
        g = first_game + i
        ref = mo.match_game(g, kind, networks, STUB_SEED, num_simulations=sims, leaves_per_root=k, virtual_loss=lam,
                            num_stochastic_moves=nsm, max_plies=max_plies, seed=seed)
        assert plies[i] == ref["plies"] and finished[i] == ref["finished"] and white[i] == ref["result"], g
        assert list(moves[i, : plies[i]]) == ref["moves"], g
        assert np.all(moves[i, plies[i]:] == MOVE_NONE), g


@pytest.mark.parametrize("networks", [(0, 1), (1, 0), (0, 0)])
@pytest.mark.parametrize("sims", [16, 64])
@pytest.mark.parametrize("lam", [1.0, 0.25])
@pytest.mark.parametrize("k", [1, 4, 16])
def test_mcts_games_equal_the_restatement(k, lam, sims, networks):
    # fullmove <= 3 samples, later plies take the last maximum; 14 plies leave every game unfinished
    with _stub_engine(4, sims, max_batch=2 * 4 * 16) as e:
        res, st = _play(e, 2, 3, az.MATCH_MCTS, networks, first_game=5, num_simulations=sims, leaves_per_root=k, virtual_loss=lam,
                        num_stochastic_moves=3, max_plies=14, seed=11)
    _check_restatement(res, 5, "mcts", networks, sims, k, lam, nsm=3, max_plies=14, seed=11)
    assert st.plies == int(res[1].astype(int).sum()) and st.leaves == st.plies * sims
    assert sum(st.evaluations) == st.plies + st.leaves - st.terminal_leaves
    if networks == (0, 0):
        assert st.evaluations[1] == 0


@pytest.mark.parametrize("k", [1, 4])
def test_full_length_mcts_games_equal_the_restatement(k):
    with _stub_engine(4, 16, max_batch=64) as e:
        res, _ = _play(e, 4, 4, az.MATCH_MCTS, (0, 1), num_simulations=16, leaves_per_root=k, seed=3)
    assert res[2].all()   # every game ended by the rules
    _check_restatement(res, 0, "mcts", (0, 1), 16, k, seed=3)


def _end_reason(moves, n):
    pos, hist = orc.startpos(), [orc.startpos()]
    for a in moves[:n]:
        pos, r = orc.play_move(pos, int(a), np.array(hist, orc.POSITION_DTYPE))
        hist.append(pos)
    mv, _ = orc.legal_moves(pos)
    if len(mv) == 0:
        return "mate" if r != 1 else "stalemate"
    if int(pos["halfmoves"]) >= 100 or int(pos["fullmoves"]) >= 200:
        return "counters"
    return "repetition or material"


@pytest.mark.parametrize("nsm", [15, 1000])
def test_base_model_games_equal_the_restatement(nsm):
    # nsm = 1000: every move is sampled, which ends games in every way the rules know
    with _stub_engine(16) as e:
        res, _ = _play(e, 16, 48, az.MATCH_BASE_MODEL, (1, 0), num_stochastic_moves=nsm, seed=7)
        cut, _ = _play(e, 5, 6, az.MATCH_BASE_MODEL, (0, 1), num_stochastic_moves=nsm, max_plies=9, seed=7)
    _check_restatement(res, 0, "base", (1, 0), nsm=nsm, seed=7)
    _check_restatement(cut, 0, "base", (0, 1), nsm=nsm, max_plies=9, seed=7)
    assert not cut[2].any() and np.all(cut[1] == 9) and np.all(cut[0] == 0)
    if nsm == 1000:
        reasons = {_end_reason(res[3][i], res[1][i]) for i in range(48)}
        assert {"mate", "counters", "repetition or material"} <= reasons, reasons


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


def _players(eng, kind, k=1, sims=16):
    if kind == "base":
        return ev.BasePlayer(eng, network=0), ev.BasePlayer(eng, network=1)
    return (ev.MctsPlayer(eng, num_simulations=sims, leaves_per_root=k, network=0),
            ev.MctsPlayer(eng, num_simulations=sims, leaves_per_root=k, network=1))


@pytest.mark.parametrize("seed", [0, 9])
@pytest.mark.parametrize("k", [1, 4])
def test_stub_match_equals_evaluate(k, seed):
    with _stub_engine(32, 16, max_batch=256) as e:
        p1, p2 = _players(e, "mcts", k)
        ref, played = _captured_evaluate(e, p1, p2, n_games=24, max_plies=120, seed=seed)
        dev = ev.evaluate_on_device(p1, p2, n_games=24, max_plies=120, seed=seed, concurrent=10)
    _check_against_evaluate(ref, played, dev)


@pytest.fixture(scope="module")
def weights():
    return az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)


def _net_engine(weights, **cfg):
    e = az.Engine(**cfg)
    e.load_weights(weights[0])
    e.load_weights(weights[1], network=1)
    return e


@pytest.mark.parametrize("kind,k,seed,n_games", [("mcts", 1, 0, 16), ("mcts", 4, 1, 32), ("base", 1, 2, 64), ("mcts", 1, 3, 16)])
def test_bf16_match_equals_evaluate(weights, kind, k, seed, n_games):
    max_plies = 450 if seed == 3 else 80
    with _net_engine(weights, max_games=64, max_batch=512, num_simulations=32) as e:
        p1, p2 = _players(e, kind, k, sims=32)
        ref, played = _captured_evaluate(e, p1, p2, n_games=n_games, max_plies=max_plies, seed=seed)
        dev = ev.evaluate_on_device(p1, p2, n_games=n_games, max_plies=max_plies, seed=seed)
    _check_against_evaluate(ref, played, dev)


def test_bf16_waves_across_the_tower_range_split(weights):
    # 512 slots x 8 leaves: up to 4096 boards per network range and wave, more than one tower range (2072 boards)
    with _net_engine(weights, max_games=512, max_batch=8192, num_simulations=16) as e:
        p1, p2 = _players(e, "mcts", 8, sims=16)
        ref, played = _captured_evaluate(e, p1, p2, n_games=512, max_plies=6, seed=4)
        dev = ev.evaluate_on_device(p1, p2, n_games=512, max_plies=6, seed=4)
    _check_against_evaluate(ref, played, dev)


@pytest.mark.parametrize("kind", ["mcts", "base"])
def test_fp32_match_equals_evaluate(weights, kind):
    with _net_engine(weights, max_games=16, max_batch=64, num_simulations=16, precision=1) as e:
        p1, p2 = _players(e, kind, 1, sims=16)
        ref, played = _captured_evaluate(e, p1, p2, n_games=8, max_plies=24, seed=6)
        dev = ev.evaluate_on_device(p1, p2, n_games=8, max_plies=24, seed=6)
    _check_against_evaluate(ref, played, dev)


def test_results_do_not_depend_on_slots_or_engines():
    kw = dict(num_simulations=16, leaves_per_root=4, virtual_loss=0.5, max_plies=60, seed=2)
    out = []
    with _stub_engine(64, 16, max_batch=1024) as e:
        for slots in (1, 7, 64):
            out.append(_play(e, slots, 16, az.MATCH_MCTS, (1, 0), **kw)[0])
    with _stub_engine(8, 16, max_batch=64) as a, _stub_engine(8, 16, max_batch=64) as b:
        ra, _ = _play(a, 8, 9, az.MATCH_MCTS, (1, 0), **kw)
        rb, _ = _play(b, 8, 7, az.MATCH_MCTS, (1, 0), first_game=9, **kw)
    out.append(tuple(np.concatenate([x, y]) for x, y in zip(ra, rb)))
    for r in out[1:]:
        assert all(np.array_equal(x, y) for x, y in zip(r, out[0]))


def test_errors_leave_the_engine_usable(weights, monkeypatch):
    ok = dict(num_simulations=16, max_plies=4)
    with az.Engine(max_games=8, max_batch=16, num_simulations=16) as e:
        e.load_weights(weights[0])
        for call in (lambda: e.match_step(1), lambda: e.match_results()):
            with pytest.raises(az.EngineError, match=": -8:"):
                call()
        with pytest.raises(az.EngineError, match=": -5:"):   # slot 1 never loaded
            e.match_begin(2, 2, az.MATCH_MCTS, (0, 1), **ok)
        e.match_begin(2, 2, az.MATCH_MCTS, (0, 0), **ok)
        e.load_weights(weights[1], network=1)
        cases = [(-1, (2, 2, 7, (0, 1), dict(ok))), (-1, (2, 2, 0, (0, 2), dict(ok))), (-1, (2, 2, 0, (0, 1), dict(ok, leaves_per_root=0))),
                 (-1, (2, 2, 0, (0, 1), dict(ok, virtual_loss=-1.0))), (-1, (2, 2, 0, (0, 1), dict(ok, virtual_loss=float("nan")))),
                 (-1, (2, 2, 0, (0, 1), dict(ok, num_simulations=17))), (-1, (2, 0, 0, (0, 1), dict(ok))), (-1, (0, 2, 0, (0, 1), dict(ok))),
                 (-1, (2, 2, 0, (0, 1), dict(ok, max_plies=0))), (-6, (9, 9, 0, (0, 1), dict(ok))), (-6, (9, 2, 0, (0, 1), dict(ok))),
                 (-6, (5, 5, 0, (0, 1), dict(ok, leaves_per_root=2)))]   # 2 x round4(5 x 2) = 24 > max_batch
        for code, (slots, n, kind, nets, kw) in cases:
            with pytest.raises(az.EngineError, match=f": {code}:"):
                e.match_begin(slots, n, kind, nets, **kw)
            _play(e, 2, 2, az.MATCH_MCTS, (0, 1), **ok)
        # the results stay readable after a search ends the match, and the match cannot be stepped any more
        res = e.match_results()
        e.search(np.array([az.start_position()]), num_simulations=8)
        with pytest.raises(az.EngineError, match=": -8:"):
            e.match_step(1)
        assert all(np.array_equal(x, y) for x, y in zip(res, e.match_results()))
    monkeypatch.setenv("AZ_HEADS_TC", "0")
    with az.Engine(max_games=8, max_batch=16, num_simulations=16) as e:
        e.load_weights(weights[0])
        e.load_weights(weights[1], network=1)
        with pytest.raises(az.EngineError, match=": -8:"):
            e.match_begin(2, 2, az.MATCH_MCTS, (0, 1), **ok)


def test_search_and_selfplay_after_a_match_equal_a_fresh_engine():
    # the match runs fewer slots and simulations than what follows uses, so state it left behind would show
    pos = np.array([az.start_position()] * 6, az.POSITION_DTYPE)

    def run(e):
        v1, s1, d1 = e.search(pos, num_simulations=32, want_scores=True)
        v2, s2, d2, _ = e.search_networks(pos, [0, 1, 1, 0, 1, 0], 32, 4, 1.0, want_scores=True)
        e.selfplay_begin(6, first_game_id=0, total_games=6)
        while e.selfplay_step(64).active_games:
            pass
        recs = e.selfplay_drain()
        recs = recs[np.lexsort((recs["ply"], recs["game_id"]))]
        return [v1, s1, d1, v2, s2, d2, recs.tobytes()]

    with _stub_engine(8, 32, max_batch=64, seed=1) as fresh:
        want = run(fresh)
    with _stub_engine(8, 32, max_batch=64, seed=1) as used:
        _play(used, 3, 5, az.MATCH_MCTS, (0, 1), num_simulations=12, leaves_per_root=4, max_plies=30)
        got = run(used)
    for a, b in zip(want, got):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b


def test_cpp_evaluate(tmp_path):
    exe = str(tmp_path / "test_match")
    lib_dir = os.path.dirname(az.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_match.cpp"),
                           "-o", exe, "-L", lib_dir, "-laz_b200", f"-Wl,-rpath,{lib_dir}"])
    out = subprocess.run([exe, str(STUB_SEED)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    with _stub_engine(8, 16, max_batch=64) as e:
        p1, p2 = _players(e, "mcts", 2, sims=16)
        dev = ev.evaluate_on_device(p1, p2, n_games=12, max_plies=100, seed=4)
    for key in ("winrate", "drawrate", "p2_winrate"):   # f32 in C++, f64 in Python
        assert abs(res[key] - dev[key]) < 1e-6, key
