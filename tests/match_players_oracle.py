"""Restatement of a resident match between two independent players (az_match_begin_players; evaluate of validation.rs:155-282 as
alphazero-chess_b200/evaluation.py plays it on one engine; DESIGN.md section 5) under the synthetic evaluator, for the tests,
written from the semantics, not from the CUDA code.  It extends tests/match_oracle.py (two equal players) to a player per side.
One game: each ply the mover (player 1 in game g when g + ply is even) plays as its kind does:
- MCTS: vl_oracle.search_vl with its own (num_simulations, leaves_per_root, virtual_loss) from a fresh root with the game's history
  and no noise, under the stub of its network slot (seed stub_seed + slot); the weights are visits / sum(visits);
- BaseModel: the stub policy of its slot masked to the legal moves;
- Random: index[int(_uniform(seed ^ 0x5151, game, ply) * count)] over the oracle's legal moves (az_movegen order, under-promotions
  included), the product in double, whatever the fullmove number.
MCTS and BaseModel choose with evaluation.py's own _weighted_index / _last_argmax and u = _uniform(seed, game, ply); every move is
played with the oracle's play_move.

    player(kind, network=0, num_simulations=16, leaves_per_root=1, virtual_loss=1.0)
    match_game(game, players, stub_seed, ...) -> dict(result (White's side), plies, finished, moves, evaluations [2],
                                                      random_underpromotions)"""
import numpy as np

import vl_oracle as vl
from alphazero_chess_b200 import evaluation as ev
from helpers import orc

F = np.float32
WHITE_WINS = 2
KINDS = ("mcts", "base", "random")


def player(kind, network=0, num_simulations=16, leaves_per_root=1, virtual_loss=1.0):
    assert kind in KINDS, kind
    return dict(kind=kind, network=int(network), num_simulations=int(num_simulations), leaves_per_root=int(leaves_per_root),
                virtual_loss=float(virtual_loss))


def random_choice(pos, seed, game, ply):
    """RandomPlayer.choose for one position: (policy index, whether the list entry drawn is an under-promotion)."""
    mv, index = orc.legal_moves(pos)
    i = int(ev._uniform(seed ^ 0x5151, game, ply) * len(index))
    return int(index[i]), int((int(mv[i]) >> 12) & 7) in (1, 2, 3)


def match_game(game, players, stub_seed, num_stochastic_moves=15, max_plies=450, seed=0, c_puct=3.0):
    pos = orc.startpos()
    history = [pos]
    moves, evaluations, under = [], [0, 0], 0
    for ply in range(max_plies):
        p = players[(game + ply) % 2]
        if p["kind"] == "random":
            action, u = random_choice(pos, seed, game, ply)
            under += u
        else:
            evaluate = vl.stub(stub_seed + p["network"])
            if p["kind"] == "mcts":
                r = vl.search_vl(pos, evaluate, p["num_simulations"], p["leaves_per_root"], p["virtual_loss"],
                                 history=np.array(history, orc.POSITION_DTYPE), c_puct=c_puct)
                evaluations[p["network"]] += r["evaluations"]
                w = r["visits"] / r["visits"].sum()
            else:
                policy, _ = evaluate(pos)
                evaluations[p["network"]] += 1
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
            return dict(result=result, plies=ply + 1, finished=True, moves=moves, evaluations=evaluations, random_underpromotions=under)
        pos = child
        history.append(child)
    return dict(result=0, plies=max_plies, finished=False, moves=moves, evaluations=evaluations, random_underpromotions=under)
