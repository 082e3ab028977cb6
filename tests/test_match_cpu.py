"""The test restatement of a resident evaluation match (tests/match_oracle.py): at one leaf per root every ply's search is the
oracle's reference search, the match entry points are exported, and k_match is a plain CUDA-core kernel.  Runs on the CPU box."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
import match_oracle as mo
from helpers import orc

STUB_SEED = 17


@pytest.mark.parametrize("game,networks", [(0, (0, 1)), (3, (1, 0)), (6, (0, 0))])
def test_one_leaf_per_root_is_the_reference_search(game, networks):
    sims = 16
    out = mo.match_game(game, "mcts", networks, STUB_SEED, num_simulations=sims, max_plies=12, seed=5)
    assert len(out["moves"]) == len(out["visits"]) == out["plies"] > 0
    pos = orc.startpos()
    history = [pos]
    prm = orc.make_params(num_simulations=sims)
    for ply, (action, visits) in enumerate(zip(out["moves"], out["visits"])):
        ev = orc.make_evaluator("stub", stub_seed=STUB_SEED + networks[(game + ply) % 2])
        v, _, _, _ = orc.search(pos, prm, ev, history=np.array(history, orc.POSITION_DTYPE))
        assert np.array_equal(visits, v), ply
        assert visits[action] > 0
        pos, res = orc.play_move(pos, action, np.array(history, orc.POSITION_DTYPE))
        history.append(pos)


def test_base_model_plays_legal_moves_until_the_cap():
    out = mo.match_game(2, "base", (0, 1), STUB_SEED, max_plies=40, seed=1)
    assert out["plies"] == len(out["moves"]) and out["visits"] == []
    assert out["finished"] or (out["plies"] == 40 and out["result"] == 0)


def test_match_entry_points_are_exported():
    L = az.lib()
    for name in ("az_match_begin", "az_match_step", "az_match_results"):
        assert getattr(L, name) is not None, name


def test_match_kernel_has_no_tensor_core_instructions():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    az.lib()
    lib = os.path.join(os.path.dirname(az.__file__), "libaz_b200.so")
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = []
        elif cur is not None:
            kernels[cur].append(line)
    hits = [k for k in kernels if "k_match" in k]
    assert hits
    for k in hits:
        assert not re.search(r"\b(UTC[A-Z]*MMA|HMMA|LDTM|STTM|UTMALDG)", "\n".join(kernels[k])), k
