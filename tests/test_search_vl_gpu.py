"""az_search_vl (leaf-parallel search with virtual loss, not in the reference) on the GPU against the oracle's restatement of
its semantics (tests/vl_oracle.py): visits, accumulated scores, depths and the collision / terminal / evaluation counts are bit-exact, with the
shared synthetic evaluator and with the bf16 network's own outputs."""
import numpy as np
import pytest

import alphazero_chess_b200 as az
from alphazero_chess_b200 import evaluation as ev
import vl_oracle as vl
from helpers import SPECIAL_FENS, orc, random_playouts

pytestmark = pytest.mark.gpu

SEED = 17


@pytest.fixture(scope="module")
def eng():
    e = az.Engine(max_games=64, max_batch=2048, num_simulations=256)
    e.set_evaluator_stub(1, SEED)
    yield e
    e.close()


def _roots(n, seed):
    positions, histories = random_playouts(3 * n, seed=seed, max_plies=100)
    keep = [i for i in range(len(positions)) if orc.outcome(positions[i]) == 0][:n]
    return positions[keep], [histories[i] for i in keep]


def _flat(histories):
    offs = np.zeros(len(histories) + 1, np.uint32)
    offs[1:] = np.cumsum([len(h) for h in histories])
    return np.concatenate(histories), offs


def test_one_leaf_per_root_equals_az_search(eng):
    roots, histories = _roots(48, 5)
    hist, offs = _flat(histories)
    v1, s1, d1 = eng.search(roots, num_simulations=100, history=hist, hist_offsets=offs, want_scores=True)
    v2, s2, d2, st = eng.search_vl(roots, 100, 1, 1.0, history=hist, hist_offsets=offs, want_scores=True)
    assert np.array_equal(v1, v2) and np.array_equal(s1, s2) and np.array_equal(d1, d2)
    assert st.collisions == 0 and st.waves == 101
    prm = orc.make_params(num_simulations=100)
    evs = orc.make_evaluator("stub", stub_seed=SEED)
    for i in range(0, len(roots), 6):
        v, s, d, _ = orc.search(roots[i], prm, evs, history=histories[i])
        assert np.array_equal(v2[i], v) and np.array_equal(s2[i], s) and d2[i] == d, i


@pytest.mark.parametrize("lam", [1.0, 0.25])
@pytest.mark.parametrize("sims", [16, 100, 256])
@pytest.mark.parametrize("k", [2, 8, 32])
def test_bit_exact_vs_oracle(eng, k, sims, lam):
    roots, histories = _roots(40 if k < 32 else 24, 100 + 7 * k + sims)
    hist, offs = _flat(histories)
    visits, scores, depth, st = eng.search_vl(roots, sims, k, lam, history=hist, hist_offsets=offs, want_scores=True)
    assert np.all(visits.sum(1) == sims)
    tot = dict(evaluations=0, collisions=0, terminal_leaves=0)
    for i, r in enumerate(roots):
        o = vl.search_vl(r, vl.stub(SEED), sims, k, lam, history=histories[i])
        assert np.array_equal(visits[i], o["visits"]), i
        assert np.array_equal(scores[i], o["scores"]), i
        assert depth[i] == o["depth"], i
        for f in tot:
            tot[f] += o[f]
    assert (st.evaluations, st.collisions, st.terminal_leaves) == (tot["evaluations"], tot["collisions"], tot["terminal_leaves"])
    assert st.waves <= sims + 1


def test_special_positions_noise_and_repetitions(eng):
    roots = np.array([orc.from_fen(f) for f in SPECIAL_FENS if orc.outcome(orc.from_fen(f)) == 0], orc.POSITION_DTYPE)
    ids = np.arange(len(roots), dtype=np.uint64) + 2000
    plies = np.arange(len(roots), dtype=np.uint32) % 5
    visits, scores, depth, _ = eng.search_vl(roots, 96, 8, 1.0, noise_game_ids=ids, noise_plies=plies, want_scores=True)
    for i, r in enumerate(roots):
        o = vl.search_vl(r, vl.stub(SEED), 96, 8, 1.0, noise_game=int(ids[i]), noise_ply=int(plies[i]))
        assert np.array_equal(visits[i], o["visits"]) and np.array_equal(scores[i], o["scores"]) and depth[i] == o["depth"], i
    # knight shuffle: draws by repetition through the history and each leaf's own path
    pos = orc.startpos()
    hist = [pos.copy()]
    for uci in ["g1f3", "g8f6", "f3g1", "f6g8", "g1f3", "g8f6"]:
        f = (ord(uci[0]) - 97) + 8 * (int(uci[1]) - 1)
        t = (ord(uci[2]) - 97) + 8 * (int(uci[3]) - 1)
        pos = orc.play_encoded(pos, f | (t << 6))
        hist.append(pos.copy())
    h = np.array(hist, orc.POSITION_DTYPE)
    visits, scores, depth, st = eng.search_vl(pos, 200, 8, 1.0, history=h, hist_offsets=np.array([0, len(h)], np.uint32), want_scores=True)
    o = vl.search_vl(pos, vl.stub(SEED), 200, 8, 1.0, history=h)
    assert np.array_equal(visits[0], o["visits"]) and np.array_equal(scores[0], o["scores"]) and depth[0] == o["depth"]
    assert (st.terminal_leaves, st.collisions) == (o["terminal_leaves"], o["collisions"])


def test_roots_are_independent_and_calls_deterministic(eng):
    roots, histories = _roots(64, 9)
    hist, offs = _flat(histories)
    a = eng.search_vl(roots, 128, 16, 1.0, history=hist, hist_offsets=offs, want_scores=True)
    b = eng.search_vl(roots, 128, 16, 1.0, history=hist, hist_offsets=offs, want_scores=True)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)
    assert (a[3].waves, a[3].evaluations, a[3].collisions) == (b[3].waves, b[3].evaluations, b[3].collisions)
    for i in (0, 17, 63):
        v, s, d, _ = eng.search_vl(roots[i], 128, 16, 1.0, history=histories[i], hist_offsets=np.array([0, len(histories[i])], np.uint32),
                                   want_scores=True)
        assert np.array_equal(v[0], a[0][i]) and np.array_equal(s[0], a[1][i]) and d[0] == a[2][i], i


def test_bf16_network_across_the_tower_range_split():
    """64 roots x 64 leaves (up to 4096 boards per wave) and 33 x 63 (up to 2079): the tower walks two board ranges above
    2072 boards.  The oracle, fed the GPU network's outputs for each leaf, reproduces visits and scores bit for bit."""
    sims = 256
    # roots without a move that ends the game: a mating edge never gets a child, so every batch of such a root collides on it
    # after one leaf and the root needs about S waves (profiles/r3_search_vl.md), which would thin out the waves counted below
    positions, _ = random_playouts(256, seed=31, max_plies=30)
    roots = np.array([p for p in positions if orc.outcome(p) == 0 and
                      all(orc.play_move(p, int(i))[1] == 0 for i in orc.legal_moves(p)[1])][:64], orc.POSITION_DTYPE)
    assert len(roots) == 64
    with az.Engine(max_games=64, max_batch=4096, num_simulations=sims, precision=0) as e:
        e.load_weights(az.random_weights(seed=42))
        per_wave = []
        results = {}
        for n, k in ((64, 64), (33, 63)):
            visits, scores, depth, st = e.search_vl(roots[:n], sims, k, 1.0, want_scores=True)
            assert np.all(visits.sum(1) == sims)
            per_wave.append(st.evaluations / st.waves)
            results[(n, k)] = (visits, scores, depth)

        def net_eval(pos):   # the GPU network's own output for each leaf
            p, v = e.forward(pos)
            return p[0], v[0]

        for (n, k), idx in (((64, 64), (0, 40, 63)), ((33, 63), (0, 32))):
            visits, scores, depth = results[(n, k)]
            for i in idx:
                o = vl.search_vl(roots[i], net_eval, sims, k, 1.0)
                assert np.array_equal(visits[i], o["visits"]), (n, k, i)
                assert np.array_equal(scores[i], o["scores"]), (n, k, i)
                assert depth[i] == o["depth"], (n, k, i)
    # more boards than 2072 on average means at least one wave went past the range split
    assert max(per_wave) > 2072, per_wave


def test_errors_leave_the_engine_usable(eng):
    roots, _ = _roots(8, 55)
    for args in ((roots, 32, 300, 1.0), (roots, 32, 0, 1.0), (roots, 32, 4, -0.5), (roots, 32, 4, float("nan")),
                 (roots, 100000, 4, 1.0)):
        with pytest.raises(az.EngineError):
            eng.search_vl(*args)
    with pytest.raises(az.EngineError, match="max_batch"):
        eng.search_vl(roots, 32, 300, 1.0)
    mate = orc.from_fen("7k/6Q1/6K1/8/8/8/8/8 b - - 0 1")
    v, _, d, _ = eng.search_vl(mate, 10, 4, 1.0)
    assert v.sum() == 0 and d[0] == 0
    v, _, _, _ = eng.search_vl(roots, 40, 4, 0.0)
    assert np.all(v.sum(1) == 40)


def test_mcts_player_with_leaves_per_root():
    with az.Engine(max_games=8, max_batch=64, num_simulations=32, seed=5) as e:
        e.load_weights(az.random_weights(seed=42))
        player = ev.MctsPlayer(e, 32, leaves_per_root=8)
        r = ev.evaluate(player, ev.RandomPlayer(e), e, n_games=4, max_plies=12)   # raises if an illegal move is played
        assert len(r["results"]) == 4 and 0.0 <= r["winrate"] <= 1.0
        pos, _ = _roots(3, 12)
        _, index, count = e.movegen(pos)
        hist = [np.array([p]) for p in pos]
        for stochastic in (True, False):
            acts = player.choose(pos, hist, pos["fullmoves"], np.full(3, stochastic), 0, np.arange(3), np.zeros(3, np.int64))
            assert all(a in index[k, : count[k]] for k, a in enumerate(acts))
