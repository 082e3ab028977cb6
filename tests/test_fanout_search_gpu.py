"""Network search at roots with more than 128 legal moves.  The heads scatter the priors of a node's legal moves into the tree, and
moves past the 128th take a separate loop (k_heads_tc: one thread per move of a team of 128; k_heads_mma: one per move of a pair of
warps, 64 at a time).  The oracle, fed the engine's own network outputs for every position it evaluates, must reproduce visits,
scores and depth bit for bit, and must have evaluated enough positions with more than 128 legal moves to tell."""
import numpy as np
import pytest

import alphazero_chess_b200 as az
import vl_oracle as vl
from helpers import orc, random_playouts
from test_edge_cases_gpu import MAX_MOVES_FEN

pytestmark = pytest.mark.gpu

SIMS = 64
WIDE = 20   # high-fanout roots, at the even indices of the batch


def _roots():
    """MAX_MOVES_FEN (218 moves) and 19 positions two plies after it that still have more than 128, each followed by an ordinary
    root: every high-fanout root is evaluated once by itself, so each network of search_networks scatters at least ten of them."""
    top = orc.from_fen(MAX_MOVES_FEN)
    after = []   # most first moves mate or stalemate the boxed-in black king
    for m in orc.legal_moves(top)[0]:
        p1 = orc.play_encoded(top, int(m))
        if orc.outcome(p1) == 0:
            after += [p2 for p2 in (orc.play_encoded(p1, int(m2)) for m2 in orc.legal_moves(p1)[0])
                      if orc.outcome(p2) == 0 and len(orc.legal_moves(p2)[0]) > 128]
    wide = [top] + [after[i] for i in np.linspace(0, len(after) - 1, WIDE - 1).astype(int)]
    positions, _ = random_playouts(3 * WIDE, seed=77, max_plies=40)
    plain = [p for p in positions if orc.outcome(p) == 0][:WIDE]
    return np.array([p for pair in zip(wide, plain) for p in pair], orc.POSITION_DTYPE)


class _Eval:
    """The engine's outputs for one position, counting the evaluated positions with more than 128 legal moves."""

    def __init__(self, forward):
        self.forward, self.wide = forward, 0

    def __call__(self, pos):
        self.wide += len(orc.legal_moves(pos)[0]) > 128
        p, v = self.forward(np.atleast_1d(pos).astype(az.POSITION_DTYPE))
        return p[0], float(v[0])


def _oracle_search(root, ev):
    def cb(ctx, pos_ptr, pol_ptr, val_ptr):
        pos = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_uint8 * 72).from_address(pos_ptr)).view(az.POSITION_DTYPE)
        p, v = ev(pos[0])
        np.ctypeslib.as_array(pol_ptr, (4096,))[:] = p
        val_ptr[0] = v
    f = orc.EVAL_FN(cb)
    return orc.search(root, orc.make_params(num_simulations=SIMS), orc.make_evaluator("callback", callback=f))


def _check(visits, scores, depth, i, o):
    assert np.array_equal(visits[i], o[0]), i
    assert np.array_equal(scores[i], o[1]), i
    assert depth[i] == o[2], i


@pytest.mark.parametrize("heads_tc", ["1", "0"])
def test_search(heads_tc, monkeypatch):
    monkeypatch.setenv("AZ_HEADS_TC", heads_tc)
    roots = _roots()
    with az.Engine(max_games=len(roots), num_simulations=SIMS, precision=0) as e:
        e.load_weights(az.random_weights(seed=21))
        visits, scores, depth = e.search(roots, num_simulations=SIMS, want_scores=True)
        ev = _Eval(e.forward)
        for i, r in enumerate(roots):
            v, s, d, _ = _oracle_search(r, ev)
            _check(visits, scores, depth, i, (v, s, d))
    assert ev.wide >= 10, ev.wide


def test_search_vl():
    roots = _roots()
    with az.Engine(max_games=len(roots), max_batch=8 * len(roots), num_simulations=SIMS, precision=0) as e:
        e.load_weights(az.random_weights(seed=22))
        visits, scores, depth, _ = e.search_vl(roots, SIMS, 8, 1.0, want_scores=True)
        ev = _Eval(e.forward)
        for i, r in enumerate(roots):
            o = vl.search_vl(r, ev, SIMS, 8, 1.0)
            _check(visits, scores, depth, i, (o["visits"], o["scores"], o["depth"]))
    assert ev.wide >= 10, ev.wide


def test_search_networks():
    roots = _roots()
    net = np.array([(i // 2) % 2 for i in range(len(roots))], np.uint8)   # high-fanout roots (even indices) on both networks
    with az.Engine(max_games=len(roots), max_batch=4 * len(roots), num_simulations=SIMS, precision=0) as e:
        e.load_weights(az.random_weights(seed=23))
        e.load_weights(az.random_weights(seed=24), network=1)
        visits, scores, depth, _ = e.search_networks(roots, net, SIMS, 4, 1.0, want_scores=True)
        evs = [_Eval(lambda pos, s=s: e.forward_networks(pos, s)) for s in (0, 1)]
        for i, r in enumerate(roots):
            o = vl.search_vl(r, evs[net[i]], SIMS, 4, 1.0)
            _check(visits, scores, depth, i, (o["visits"], o["scores"], o["depth"]))
    assert min(ev.wide for ev in evs) >= 10, [ev.wide for ev in evs]
