"""Restatement of az_selfplay_begin_vl's semantics (self-play whose every ply is searched leaf-parallel with virtual loss, NOT in
the reference; DESIGN.md section 5) for the tests, written from the semantics, not from the CUDA code.  One game of run_episode
(training.rs:294-338) in which each ply's search is vl_oracle.search_vl with the game's history and root noise keyed by (seed,
game id, ply); the move is chosen as oracle/api.cpp orc_selfplay_episode chooses it (f32 improved policy, the last maximum from
`anneal` on, WeightedIndex before), played with the oracle's play_move, and the final values are back-filled as there.  With
leaves_per_game = 1 it is orc.selfplay_episode (checked in tests/test_selfplay_vl_cpu.py).

    selfplay_game_vl(game_id, evaluate, num_simulations, leaves_per_game, virtual_loss=1.0, ...)

`evaluate(position) -> (policy [4096] f32, value)` as in vl_oracle.  At ply 0 the root priors are evaluate(start position) (the
shared start-position forward); afterwards they are the child's priors kept by traverse_new, which is evaluate(new root) again.
Neither is a leaf evaluation: `evaluations` counts the boards the searches sent to the network, roots excluded.  Returns dict(
positions, visits [plies, 4096], action, depth, final_value, evaluations, terminal_leaves, collisions)."""
import numpy as np

import vl_oracle as vl
from helpers import orc

F = np.float32
NUM_FULLMOVES = 200   # chess.rs:10


def _choose(improved, fullmoves, seed, game_id, ply, anneal):
    if fullmoves >= anneal:   # Iterator::max_by keeps the LAST maximum (training.rs:311-316)
        return int(np.flatnonzero(improved == improved.max()).max())
    total = F(0.0)   # WeightedIndex: cumulative f32 weights in index order
    for w in improved:
        total = F(total + w)
    h = int(orc.lib().orc_rng_u64(seed, game_id, ply, 1, 0))
    chosen = F(F(h >> 40) * F(1.0 / 16777216.0)) * total
    cum, last = F(0.0), 0
    for i in np.flatnonzero(improved > 0):
        cum = F(cum + improved[i])
        last = int(i)
        if cum > chosen:
            return int(i)
    return last


def selfplay_game_vl(game_id, evaluate, num_simulations, leaves_per_game, virtual_loss=1.0, c_puct=3.0, alpha=0.3, eps=0.25,
                     seed=42, anneal=15, temperature=1.0, max_plies=512):
    pos = orc.startpos()
    history = [pos]
    positions, visits, actions, depths, signs = [], [], [], [], []
    counts = dict(evaluations=0, terminal_leaves=0, collisions=0)
    outcome = F(0.0)
    for ply in range(max_plies):
        r = vl.search_vl(pos, evaluate, num_simulations, leaves_per_game, virtual_loss, history=np.array(history, orc.POSITION_DTYPE),
                         noise_game=game_id, noise_ply=ply, c_puct=c_puct, alpha=alpha, eps=eps, seed=seed)
        counts["evaluations"] += r["evaluations"] - 1   # the root's priors are not a network call of their own
        counts["terminal_leaves"] += r["terminal_leaves"]
        counts["collisions"] += r["collisions"]
        improved = orc.improved_policy(r["visits"], temperature)
        turn = F(1.0) if int(pos["turn"]) == 0 else F(-1.0)
        positions.append(pos)
        visits.append(r["visits"])
        depths.append(r["depth"])
        signs.append(turn)
        action = _choose(improved, int(pos["fullmoves"]), seed, game_id, ply, anneal)
        actions.append(action)
        child, res = orc.play_move(pos, action, np.array(history, orc.POSITION_DTYPE))
        assert res != vl.ILLEGAL
        pos = child
        if res != vl.ONGOING:
            outcome = F(0.0) if res == vl.DRAW else turn
            break
        history.append(child)
    decay = F(F(1.0) - F(F(int(pos["fullmoves"])) / F(2.0 * NUM_FULLMOVES)))
    final = np.array([F(s * F(outcome * decay)) for s in signs], F)
    return dict(positions=np.array(positions, orc.POSITION_DTYPE), visits=np.array(visits, F), action=np.array(actions, np.int64),
                depth=np.array(depths, np.int64), final_value=final, **counts)
