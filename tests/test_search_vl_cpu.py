"""The test restatement of az_search_vl's semantics (tests/vl_oracle.py; leaf-parallel search with virtual loss, not in the
reference): K = 1 is the oracle's reference search bit for bit, every batch makes progress, and the counts add up."""
import numpy as np
import pytest

import vl_oracle as vl
from helpers import orc, random_playouts

SEED = 13


def _roots(n, seed):
    positions, histories = random_playouts(3 * n, seed=seed, max_plies=100)
    keep = [i for i in range(len(positions)) if orc.outcome(positions[i]) == 0][:n]
    return positions[keep], [histories[i] for i in keep]


@pytest.mark.parametrize("sims", [16, 100])
def test_one_leaf_per_root_is_the_reference_search(sims):
    roots, histories = _roots(50, 3 + sims)
    prm = orc.make_params(num_simulations=sims)
    ev = orc.make_evaluator("stub", stub_seed=SEED)
    for i, r in enumerate(roots):
        v, s, d, evals = orc.search(r, prm, ev, history=histories[i])
        out = vl.search_vl(r, vl.stub(SEED), sims, 1, 1.0, history=histories[i])
        assert np.array_equal(out["visits"], v), i
        assert np.array_equal(out["scores"], s), i
        assert out["depth"] == d and out["evaluations"] == evals, i
        assert out["collisions"] == 0, i


@pytest.mark.parametrize("k", [2, 8, 64])
@pytest.mark.parametrize("sims", [16, 100])
def test_visits_sum_to_the_simulations(k, sims):
    roots, histories = _roots(12, 40 + k)
    for i, r in enumerate(roots):
        out = vl.search_vl(r, vl.stub(SEED), sims, k, 1.0, history=histories[i])
        assert out["visits"].sum() == sims, i
        # every leaf was either evaluated or terminal; the root was evaluated once
        assert out["evaluations"] == 1 + sims - out["terminal_leaves"], i
        assert out["depth"] >= 1
        # a batch ends early at most once, so at least ceil(S / K) batches ran
        assert 0 <= out["collisions"] <= sims


def test_single_legal_move_collides_until_the_child_exists():
    root = orc.from_fen("k7/8/8/8/8/8/8/1R5K b - - 0 1")   # Ka7 is the only legal move
    _, idx = orc.legal_moves(root)
    assert len(idx) == 1
    out = vl.search_vl(root, vl.stub(SEED), 16, 8, 1.0)
    # batch 1: the only edge becomes a leaf, the second descent reaches it again before its child exists
    assert out["collisions"] >= 1
    assert out["visits"][idx[0]] == 16 and out["visits"].sum() == 16


def test_terminal_leaves_and_terminal_root():
    mate_in_one = orc.from_fen("6k1/5ppp/8/8/8/8/8/R6K w - - 0 1")
    out = vl.search_vl(mate_in_one, vl.stub(SEED), 32, 8, 1.0)
    assert out["terminal_leaves"] >= 1 and out["visits"].sum() == 32
    mated = orc.from_fen("7k/6Q1/6K1/8/8/8/8/8 b - - 0 1")
    out = vl.search_vl(mated, vl.stub(SEED), 32, 8, 1.0)
    assert out["visits"].sum() == 0 and out["depth"] == 0


def test_zero_virtual_loss_is_accepted_and_differs_from_one():
    roots, histories = _roots(6, 77)
    differ = 0
    for i, r in enumerate(roots):
        a = vl.search_vl(r, vl.stub(SEED), 64, 8, 0.0, history=histories[i])
        b = vl.search_vl(r, vl.stub(SEED), 64, 8, 1.0, history=histories[i])
        assert a["visits"].sum() == 64
        differ += not np.array_equal(a["scores"], b["scores"])
    assert differ > 0
    with pytest.raises(ValueError):
        vl.search_vl(roots[0], vl.stub(SEED), 64, 8, -1.0)
    with pytest.raises(ValueError):
        vl.search_vl(roots[0], vl.stub(SEED), 64, 0, 1.0)
