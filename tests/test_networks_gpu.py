"""Two networks in one engine (az_load_network, az_forward_networks, az_search_networks): every board or root is evaluated by the
network it names, bit for bit as on an engine that holds only that network, and a match between two networks on one engine
plays the same games as the match between two engines."""
import numpy as np
import pytest

import alphazero_chess_b200 as az
from alphazero_chess_b200 import evaluation as ev
import vl_oracle as vl
from helpers import orc, random_playouts

pytestmark = pytest.mark.gpu

SEED = 23


@pytest.fixture(scope="module")
def weights():
    return az.random_weights(seed=101, randomize_bn=True), az.random_weights(seed=202, randomize_bn=True)


@pytest.fixture(scope="module")
def engines(weights):
    """one engine holding both networks, and one engine per network"""
    cfg = dict(max_games=4200, max_batch=4200, num_simulations=64)
    both, e0, e1 = az.Engine(**cfg), az.Engine(**cfg), az.Engine(**cfg)
    both.load_weights(weights[0])
    both.load_weights(weights[1], network=1)
    e0.load_weights(weights[0])
    e1.load_weights(weights[1])
    yield both, e0, e1
    for e in (both, e0, e1):
        e.close()


def _positions(n, seed):
    positions, _ = random_playouts(n, seed=seed, max_plies=60)
    return positions[:n]


def _roots(n, seed):
    positions, histories = random_playouts(3 * n, seed=seed, max_plies=100)
    keep = [i for i in range(len(positions)) if orc.outcome(positions[i]) == 0][:n]
    return positions[keep], [histories[i] for i in keep]


def _flat(histories):
    offs = np.zeros(len(histories) + 1, np.uint32)
    offs[1:] = np.cumsum([len(h) for h in histories])
    return np.concatenate(histories), offs


def _splits(n, rng):
    yield "interleaved", (np.arange(n) % 2).astype(np.uint8)
    yield "random", rng.integers(0, 2, n).astype(np.uint8)
    one = np.zeros(n, np.uint8)
    one[n // 2] = 1
    yield "one on network 1", one
    yield "all on network 1", np.ones(n, np.uint8)
    yield "all on network 0", np.zeros(n, np.uint8)


@pytest.mark.parametrize("n", [1, 3, 64, 2072, 2073, 4096])
def test_forward_rows_are_those_of_the_single_network_engines(engines, n):
    both, e0, e1 = engines
    pos = np.resize(_positions(min(n, 600), 1000 + n), n)
    p0, v0 = e0.forward(pos)
    p1, v1 = e1.forward(pos)
    assert not np.array_equal(v0, v1)
    for name, net in _splits(n, np.random.default_rng(n)):
        policy, value = both.forward_networks(pos, net)
        on1 = net == 1
        assert np.array_equal(policy[~on1], p0[~on1]) and np.array_equal(value[~on1], v0[~on1]), name
        assert np.array_equal(policy[on1], p1[on1]) and np.array_equal(value[on1], v1[on1]), name
    # network 0 of the two-network engine is what forward() evaluates
    assert np.array_equal(both.forward(pos)[1], v0)


@pytest.mark.parametrize("k", [1, 8])
def test_stub_search_matches_the_restatement(k):
    with az.Engine(max_games=64, max_batch=1024, num_simulations=128) as eng:
        eng.set_evaluator_stub(1, SEED)
        roots, histories = _roots(40, 300 + k)
        hist, offs = _flat(histories)
        net = (np.arange(len(roots)) * 7 % 3 == 0).astype(np.uint8)
        ids = np.arange(len(roots), dtype=np.uint64) + 500
        plies = np.arange(len(roots), dtype=np.uint32) % 4
        noisy = np.arange(len(roots)) % 2 == 0
        sims = 96
        visits, scores, depth, st = eng.search_networks(roots, net, sims, k, 1.0, history=hist, hist_offsets=offs, noise_game_ids=ids,
                                                        noise_plies=plies, want_scores=True)
        tot = dict(evaluations=0, collisions=0, terminal_leaves=0)
        for i, r in enumerate(roots):
            o = vl.search_vl(r, vl.stub(SEED + int(net[i])), sims, k, 1.0, history=histories[i], noise_game=int(ids[i]),
                             noise_ply=int(plies[i]))
            assert np.array_equal(visits[i], o["visits"]) and np.array_equal(scores[i], o["scores"]) and depth[i] == o["depth"], i
            for f in tot:
                tot[f] += o[f]
        assert (st.evaluations, st.collisions, st.terminal_leaves) == (tot["evaluations"], tot["collisions"], tot["terminal_leaves"])
        assert noisy.any()


@pytest.mark.parametrize("n_roots,k", [(256, 1), (256, 8), (2100, 1)])
def test_bf16_search_equals_single_network_search(engines, n_roots, k):
    both, e0, e1 = engines
    roots, histories = _roots(min(n_roots, 300), 700 + k)
    idx = np.arange(n_roots) % len(roots)
    roots = roots[idx]
    histories = [histories[i] for i in idx]
    hist, offs = _flat(histories)
    net = (np.arange(n_roots) % 2).astype(np.uint8)
    sims = 32 if n_roots > 1000 else 64
    visits, scores, depth, _ = both.search_networks(roots, net, sims, k, 1.0, history=hist, hist_offsets=offs, want_scores=True)
    for s, e in ((0, e0), (1, e1)):
        sel = np.flatnonzero(net == s)
        h, o = _flat([histories[i] for i in sel])
        v, sc, d, _ = e.search_vl(roots[sel], sims, k, 1.0, history=h, hist_offsets=o, want_scores=True)
        assert np.array_equal(visits[sel], v) and np.array_equal(scores[sel], sc) and np.array_equal(depth[sel], d), s
        if k == 1:
            v2, sc2, d2 = e.search(roots[sel], num_simulations=sims, history=h, hist_offsets=o, want_scores=True)
            assert np.array_equal(visits[sel], v2) and np.array_equal(scores[sel], sc2) and np.array_equal(depth[sel], d2), s


def _count_calls(engine, names):
    calls = {n: 0 for n in names}
    for n in names:
        orig = getattr(engine, n)

        def wrapped(*a, _orig=orig, _n=n, **kw):
            calls[_n] += 1
            return _orig(*a, **kw)
        setattr(engine, n, wrapped)
    return calls


@pytest.mark.parametrize("kind", ["mcts1", "mcts4", "base"])
def test_match_on_one_engine_equals_the_two_engine_match(weights, kind):
    cfg = dict(max_games=64, max_batch=512, num_simulations=32)
    with az.Engine(**cfg) as both, az.Engine(**cfg) as e0, az.Engine(**cfg) as e1:
        both.load_weights(weights[0])
        both.load_weights(weights[1], network=1)
        e0.load_weights(weights[0])
        e1.load_weights(weights[1])
        if kind == "base":
            make = lambda e, s: ev.BasePlayer(e, network=s)
        else:
            k = 1 if kind == "mcts1" else 4
            make = lambda e, s: ev.MctsPlayer(e, num_simulations=32, leaves_per_root=k, network=s)
        moves = {}
        for name, e in (("joint", both), ("apart", e0)):   # the moves each match plays, ply by ply
            played, orig = moves.setdefault(name, []), e.play_move
            e.play_move = lambda pos, act, *a, _o=orig, _p=played, **kw: (_p.append(np.array(act)), _o(pos, act, *a, **kw))[1]
        calls = _count_calls(both, ["search", "search_vl", "search_networks", "forward", "forward_networks"])
        joint = ev.evaluate(make(both, 0), make(both, 1), both, n_games=16, max_plies=24, seed=5)
        apart = ev.evaluate(make(e0, 0), make(e1, 0), e0, n_games=16, max_plies=24, seed=5)
        assert np.array_equal(joint["results"], apart["results"])
        assert len(moves["joint"]) == len(moves["apart"]) > 0
        assert all(np.array_equal(a, b) for a, b in zip(moves["joint"], moves["apart"]))
        joint_call = "forward_networks" if kind == "base" else "search_networks"
        assert calls[joint_call] == len(moves["joint"]) and sum(v for c, v in calls.items() if c != joint_call) == 0, calls


def test_errors_leave_the_engine_usable(weights):
    pos = _positions(8, 9)
    with az.Engine(max_games=8, max_batch=8, num_simulations=32) as eng:
        eng.load_weights(weights[0])
        with pytest.raises(az.EngineError, match=": -1:"):
            eng.forward_networks(pos, np.full(8, 2, np.uint8))
        with pytest.raises(az.EngineError, match=": -5:"):
            eng.forward_networks(pos, np.ones(8, np.uint8))
        with pytest.raises(az.EngineError, match=": -5:"):
            eng.search_networks(pos[:2], [0, 1], 16)
        eng.load_weights(weights[1], network=1)
        with pytest.raises(az.EngineError, match=": -6:"):   # 5 -> 8 and 3 -> 4 boards: 12 > max_batch
            eng.forward_networks(pos, np.array([0, 0, 0, 0, 0, 1, 1, 1], np.uint8))
        with pytest.raises(az.EngineError, match=": -6:"):
            eng.search_networks(pos, [0, 0, 0, 0, 0, 1, 1, 1], 16)
        with pytest.raises(az.EngineError, match=": -1:"):
            eng.search_networks(pos[:2], [0, 3], 16)
        policy, value = eng.forward_networks(pos, np.array([0, 0, 0, 0, 1, 1, 1, 1], np.uint8))
        assert np.array_equal(value[:4], eng.forward(pos[:4])[1])
        visits, _, _, _ = eng.search_networks(pos[:2], [0, 1], 16)
        assert np.all(visits.sum(1) == 16)


def test_fp32_forward_networks_matches_single_network_engines(weights):
    pos = _positions(24, 11)
    net = (np.arange(24) % 3 == 1).astype(np.uint8)
    cfg = dict(max_games=16, max_batch=64, precision=1)
    with az.Engine(**cfg) as both, az.Engine(**cfg) as e0, az.Engine(**cfg) as e1:
        both.load_weights(weights[0])
        both.load_weights(weights[1], network=1)
        e0.load_weights(weights[0])
        e1.load_weights(weights[1])
        policy, value = both.forward_networks(pos, net)
        p0, v0 = e0.forward(pos)
        p1, v1 = e1.forward(pos)
        on1 = net == 1
        assert np.array_equal(policy[~on1], p0[~on1]) and np.array_equal(value[~on1], v0[~on1])
        assert np.array_equal(policy[on1], p1[on1]) and np.array_equal(value[on1], v1[on1])
