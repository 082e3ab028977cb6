"""Restatement of a resident evaluation match (az_match_*; evaluate of validation.rs:155-282 as alphazero-chess_b200/evaluation.py
plays it; DESIGN.md section 5) under the synthetic evaluator, for the tests, written from the semantics, not from the CUDA code.
One game: each ply the mover (player 1 in game g when g + ply is even) evaluates with the stub of its network slot (seed
stub_seed + slot); an MCTS mover runs vl_oracle.search_vl from a fresh root with the game's history and no noise and weighs the
moves by visits / sum(visits), a BaseModel mover by the stub policy masked to the legal moves; the choice is evaluation.py's own
_weighted_index / _last_argmax with u = _uniform(seed, game, ply), and the move is played with the oracle's play_move.

    match_game(game, kind, networks, stub_seed, ...) -> dict(result (White's side), plies, finished, moves, visits)"""
import numpy as np

import vl_oracle as vl
from alphazero_chess_b200 import evaluation as ev
from helpers import orc

F = np.float32
WHITE_WINS = 2


def match_game(game, kind, networks, stub_seed, num_simulations=16, leaves_per_root=1, virtual_loss=1.0, num_stochastic_moves=15,
               max_plies=450, seed=0, c_puct=3.0):
    pos = orc.startpos()
    history = [pos]
    moves, visits = [], []
    for ply in range(max_plies):
        evaluate = vl.stub(stub_seed + networks[(game + ply) % 2])
        if kind == "mcts":
            r = vl.search_vl(pos, evaluate, num_simulations, leaves_per_root, virtual_loss, history=np.array(history, orc.POSITION_DTYPE),
                             c_puct=c_puct)
            visits.append(r["visits"])
            w = r["visits"] / r["visits"].sum()
        else:
            policy, _ = evaluate(pos)
            _, index = orc.legal_moves(pos)
            w = np.zeros(orc.ACTION_SPACE, F)
            w[index] = policy[index]
        stochastic = int(pos["fullmoves"]) <= num_stochastic_moves
        action = ev._weighted_index(w, ev._uniform(seed, game, ply)) if stochastic else ev._last_argmax(w)
        moves.append(action)
        child, res = orc.play_move(pos, action, np.array(history, orc.POSITION_DTYPE))
        assert res != vl.ILLEGAL
        if res != vl.ONGOING:
            result = 0 if res == vl.DRAW else (1 if res == WHITE_WINS else -1)
            return dict(result=result, plies=ply + 1, finished=True, moves=moves, visits=visits)
        pos = child
        history.append(child)
    return dict(result=0, plies=max_plies, finished=False, moves=moves, visits=visits)
