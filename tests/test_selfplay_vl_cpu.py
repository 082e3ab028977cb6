"""The test restatement of az_selfplay_begin_vl's semantics (tests/vl_selfplay_oracle.py; leaf-parallel self-play, not in the
reference): one leaf per game is the oracle's run_episode record for record, larger batches keep every search at S visits with
consistent counts, and k_vl_selfplay is a plain CUDA-core kernel.  Runs on the CPU box."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
import vl_oracle as vl
import vl_selfplay_oracle as vso
from helpers import orc

STUB_SEED = 17


@pytest.mark.parametrize("game_id", [0, 3, 11])
def test_one_leaf_per_game_is_the_reference_episode(game_id):
    sims = 16
    out = vso.selfplay_game_vl(game_id, vl.stub(STUB_SEED), sims, 1, 1.0)
    ep = orc.selfplay_episode(orc.make_params(num_simulations=sims), orc.make_evaluator("stub", stub_seed=STUB_SEED), game_id=game_id)
    n = ep["stats"].n_steps
    assert len(out["action"]) == n
    assert out["positions"].tobytes() == ep["positions"].tobytes()
    assert np.array_equal(out["visits"], ep["visits"])
    assert np.array_equal(out["action"], ep["action"])
    assert np.array_equal(out["depth"], ep["depth"])
    assert np.array_equal(out["final_value"], ep["final_value"])
    assert out["collisions"] == 0
    # the oracle also counts the start-position forward
    assert out["evaluations"] == ep["stats"].evals - 1


@pytest.mark.parametrize("k,lam", [(4, 1.0), (16, 0.25)])
def test_batches_keep_every_search_at_s_visits(k, lam):
    sims = 32
    for game_id in (1, 7):
        out = vso.selfplay_game_vl(game_id, vl.stub(STUB_SEED), sims, k, lam)
        plies = len(out["action"])
        assert plies >= 1 and np.all(out["visits"].sum(axis=1) == sims)
        # every leaf was evaluated or terminal; a batch ends early at most once
        assert out["evaluations"] + out["terminal_leaves"] == plies * sims
        assert 0 <= out["collisions"] <= plies * sims
        # the move played had visits; final values are results scaled by the fullmove decay
        assert all(out["visits"][i][a] > 0 for i, a in enumerate(out["action"]))
        assert np.all(np.abs(out["final_value"]) <= 1.0)


def test_vl_selfplay_entry_points_are_exported():
    L = az.lib()
    for name in ("az_selfplay_begin_vl", "az_selfplay_vl_stats"):
        assert getattr(L, name) is not None, name


def test_vl_selfplay_kernel_has_no_tensor_core_instructions():
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
    hits = [k for k in kernels if "k_vl_selfplay" in k]
    assert hits
    for k in hits:
        s = "\n".join(kernels[k])
        assert not re.search(r"\b(UTC[A-Z]*MMA|HMMA|LDTM|STTM|UTMALDG)", s), k
