"""Leaf-parallel self-play with virtual loss (az_selfplay_begin_vl; not in the reference) on the GPU: byte-identical to the
default path at one leaf per game, bit-exact against the test restatement (tests/vl_selfplay_oracle.py) for larger batches, one
record per game id whatever the slots, and the generation machinery (exactly-N, parking, training, the C++ mirror) unchanged."""
import json
import os
import subprocess

import numpy as np
import pytest

import alphazero_chess_b200 as az
import vl_oracle as vl
import vl_selfplay_oracle as vso
from alphazero_chess_b200 import training as tr
from helpers import ROOT, orc

pytestmark = pytest.mark.gpu

SEED, STUB_SEED = 42, 17
ERR_INVALID, ERR_NO_WEIGHTS, ERR_CAPACITY, ERR_STATE = -1, -5, -6, -8


def _generation(e, slots, first_id, total, k=None, lam=1.0, chunk=32, max_waves=200_000):
    """Plays the exactly-N generation to completion; returns (records sorted by (game id, ply), last stats, max parked)."""
    e.selfplay_begin(slots, first_game_id=first_id, total_games=total, leaves_per_game=k, virtual_loss=lam)
    out, waves, parked = [], 0, 0
    while waves < max_waves:
        st = e.selfplay_step(chunk)
        waves += chunk
        parked = max(parked, int(st.parked_games))
        if st.pending_samples:
            out.append(e.selfplay_drain())
        elif st.active_games == 0:
            break
    assert st.active_games == 0 and st.games_finished == total
    s = np.concatenate(out)
    return s[np.lexsort((s["ply"], s["game_id"]))], st, parked


def _check_game(rec, ref, sims, gid):
    assert len(rec) == len(ref["action"]), gid
    for k in range(len(rec)):
        assert rec[k]["position"].tobytes() == ref["positions"][k].tobytes(), (gid, k)
        assert np.array_equal(az.improved_policy(rec[k], sims) * np.float32(sims), ref["visits"][k]), (gid, k)
        assert rec[k]["action"] == ref["action"][k], (gid, k)
        assert rec[k]["search_depth"] == ref["depth"][k], (gid, k)
        assert rec[k]["final_value"] == ref["final_value"][k], (gid, k)
        assert rec[k]["ply"] == k and rec[k]["game_id"] == gid


def _stub_engine(slots, sims, k_max=1, **kw):
    e = az.Engine(max_games=slots, max_batch=slots * k_max, num_simulations=sims, seed=SEED, **kw)
    e.set_evaluator_stub(1, STUB_SEED)
    return e


def test_one_leaf_per_game_is_byte_identical_to_begin_n():
    sims = 24
    with _stub_engine(16, sims) as e:
        a, sa, _ = _generation(e, 16, 0, 24)
        b, sb, _ = _generation(e, 16, 0, 24, k=1)
        vs = e.selfplay_vl_stats()
    assert a.tobytes() == b.tobytes()
    for f in ("simulations", "positions", "games_finished", "terminal_leaves", "evaluations", "sum_search_depth", "sum_leaf_depth"):
        assert getattr(sa, f) == getattr(sb, f), f
    assert vs.collisions == 0 and vs.evaluations == sb.evaluations and vs.terminal_leaves == sb.terminal_leaves
    assert sb.cache_hits == 0 and sb.sum_edges == 0


@pytest.mark.parametrize("sims", [16, 64])
@pytest.mark.parametrize("lam", [1.0, 0.25])
@pytest.mark.parametrize("k", [2, 8, 32])
def test_records_equal_the_restatement(k, lam, sims):
    first, total = 40, 4
    with _stub_engine(3, sims, k) as e:
        recs, st, _ = _generation(e, 3, first, total, k=k, lam=lam)
        vs = e.selfplay_vl_stats()
    sums = dict(evaluations=0, terminal_leaves=0, collisions=0)
    for gid in range(first, first + total):
        ref = vso.selfplay_game_vl(gid, vl.stub(STUB_SEED), sims, k, lam, seed=SEED)
        _check_game(recs[recs["game_id"] == gid], ref, sims, gid)
        for f in sums:
            sums[f] += ref[f]
    assert (vs.evaluations, vs.terminal_leaves, vs.collisions) == (sums["evaluations"], sums["terminal_leaves"], sums["collisions"])
    assert st.evaluations == vs.evaluations and st.terminal_leaves == vs.terminal_leaves
    assert st.simulations == st.evaluations + st.terminal_leaves and st.cache_hits == 0


def test_records_do_not_depend_on_slots_or_engines():
    sims, k, total = 16, 8, 6
    with _stub_engine(8, sims, k) as e:
        whole, _, _ = _generation(e, 8, 0, total, k=k)
        three, _, _ = _generation(e, 3, 0, total, k=k)
    with _stub_engine(3, sims, k) as e1, _stub_engine(3, sims, k) as e2:
        lo, _, _ = _generation(e1, 3, 0, 3, k=k)
        hi, _, _ = _generation(e2, 3, 3, 3, k=k)
    split = np.concatenate([lo, hi])
    assert whole.tobytes() == three.tobytes() == split.tobytes()
    assert sorted(set(int(g) for g in whole["game_id"])) == list(range(total))


def _net_eval(e):
    def evaluate(pos):
        p, v = e.forward(np.atleast_1d(pos).astype(az.POSITION_DTYPE))
        return p[0], float(v[0])
    return evaluate


def test_bf16_network_records_equal_the_restatement_fed_its_outputs():
    sims, k = 16, 16
    w = az.random_weights(seed=11)
    with az.Engine(max_games=2, max_batch=2 * k, num_simulations=sims, seed=SEED) as e:
        e.load_weights(w)
        recs, _, _ = _generation(e, 2, 500, 2, k=k)
        # az_forward is batch-invariant: the rows the self-play evaluated are the rows forward() returns
        for gid in (500, 501):
            ref = vso.selfplay_game_vl(gid, _net_eval(e), sims, k, 1.0, seed=SEED)
            _check_game(recs[recs["game_id"] == gid], ref, sims, gid)


def test_bf16_waves_larger_than_one_tower_range():
    sims, k, slots = 16, 16, 200
    w = az.random_weights(seed=12)
    with az.Engine(max_games=slots, max_batch=slots * k, num_simulations=sims, seed=SEED) as e:
        e.load_weights(w)
        e.selfplay_begin(slots, first_game_id=0, leaves_per_game=k)
        st = e.selfplay_step(1)
        assert st.evaluations > 2072   # the first wave spans two L2-sized tower ranges
        recs, _, _ = _generation(e, slots, 0, slots, k=k, chunk=64)
        for gid in (0, slots - 1):
            ref = vso.selfplay_game_vl(gid, _net_eval(e), sims, k, 1.0, seed=SEED)
            _check_game(recs[recs["game_id"] == gid], ref, sims, gid)


def test_parking_loses_nothing(monkeypatch):
    sims, k, total = 16, 4, 10
    with _stub_engine(8, sims, k) as e:
        free, _, _ = _generation(e, 8, 0, total, k=k)
    monkeypatch.setenv("AZ_SAMPLE_CAP", "600")
    with _stub_engine(8, sims, k) as e:
        capped, _, parked = _generation(e, 8, 0, total, k=k, chunk=1024)   # drained rarely: games park
    assert parked > 0
    assert free.tobytes() == capped.tobytes()


def _code(err):
    return int(str(err).split(":")[1])


def test_errors_leave_the_engine_usable():
    sims = 16
    with _stub_engine(4, sims, 4) as e:
        with pytest.raises(az.EngineError) as ex:
            e.selfplay_vl_stats()
        assert _code(ex.value) == ERR_STATE
        for k, lam, code in [(0, 1.0, ERR_INVALID), (-3, 1.0, ERR_INVALID), (2, -1.0, ERR_INVALID), (2, float("nan"), ERR_INVALID),
                             (2, float("inf"), ERR_INVALID), (8, 1.0, ERR_CAPACITY)]:
            with pytest.raises(az.EngineError) as ex:
                e.selfplay_begin(4, leaves_per_game=k, virtual_loss=lam)
            assert _code(ex.value) == code, (k, lam)
            e.selfplay_begin(4, leaves_per_game=4, virtual_loss=0.0)
            assert e.selfplay_step(4).simulations > 0
    with _stub_engine(4, sims, 4, cache_log2=10) as e:
        with pytest.raises(az.EngineError) as ex:
            e.selfplay_begin(4, leaves_per_game=2)
        assert _code(ex.value) == ERR_STATE
        e.selfplay_begin(4)
        assert e.selfplay_step(4).simulations > 0
    with az.Engine(max_games=4, max_batch=16, num_simulations=sims) as e:
        with pytest.raises(az.EngineError) as ex:
            e.selfplay_begin(4, leaves_per_game=2)
        assert _code(ex.value) == ERR_NO_WEIGHTS
        e.load_weights(az.random_weights(seed=3))
        e.selfplay_begin(4, leaves_per_game=2)
        assert e.selfplay_step(2).evaluations > 0


def test_other_calls_after_vl_selfplay_are_unchanged():
    sims = 16
    roots = np.array([orc.startpos(), orc.from_fen("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1")],
                     az.POSITION_DTYPE)
    with _stub_engine(8, sims, 8) as fresh:
        v0, s0, d0 = fresh.search(roots, sims, want_scores=True)
        ref, _, _ = _generation(fresh, 8, 0, 8)
    with _stub_engine(8, sims, 8) as e:
        e.selfplay_begin(8, leaves_per_game=8)
        e.selfplay_step(40)
        v1, s1, d1 = e.search(roots, sims, want_scores=True)
        with pytest.raises(az.EngineError):
            e.selfplay_step(1)   # a search ends the self-play in progress
        assert np.array_equal(v0, v1) and np.array_equal(s0, s1) and np.array_equal(d0, d1)
        e.selfplay_begin(8, leaves_per_game=8)
        e.selfplay_step(40)
        got, _, _ = _generation(e, 8, 0, 8)
        with pytest.raises(az.EngineError):
            e.selfplay_vl_stats()   # begin_n ended the leaf-parallel mode
    assert ref.tobytes() == got.tobytes()


def test_run_generation_with_leaves_per_game():
    import torch

    torch.manual_seed(0)
    model = tr.import_weights(tr.AlphaZeroNet(), az.random_weights(seed=42)).cuda()
    opt = tr.make_optimizer(model)
    with az.Engine(max_games=16, max_batch=16 * 8, num_simulations=16, seed=1) as eng:
        replay = az.ReplayBuffer(eng, capacity=20_000, max_batch=64)
        m = tr.run_generation(eng, replay, model, opt, iteration=0, n_games=24, min_replay_size=10**9, num_steps=0, leaves_per_game=8)
        assert m["games"] == 24 and m["positions"] > 24 and m["replay_buffer_size"] == len(replay) > 0
        assert eng.selfplay_vl_stats().evaluations == m["evaluations"]
        replay.close()


def test_cpp_mirror_overload(tmp_path):
    exe = str(tmp_path / "test_selfplay_vl")
    lib_dir = os.path.dirname(az.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_selfplay_vl.cpp"),
                           "-o", exe, "-L", lib_dir, "-laz_b200", f"-Wl,-rpath,{lib_dir}"])
    stub_seed = 5
    out = subprocess.run([exe, str(stub_seed)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    res = {d["test"]: d for d in (json.loads(l) for l in out.stdout.splitlines() if l.startswith("{"))}
    # the records are identical; the number of waves is not: k_advance completes a terminal leaf without the network inside the
    # wave that found it, a leaf-parallel batch waits for k_vl_expand, so avg_batch (evaluations per wave) may be lower at K = 1
    for f in ("steps", "value_sum", "depth_sum"):
        assert res["k1"][f] == res["default"][f], f
    assert 0 < res["k1"]["avg_batch"] <= res["default"]["avg_batch"]
    steps, vsum, dsum = 0, 0.0, 0
    for g in range(4):
        ref = vso.selfplay_game_vl(g, vl.stub(stub_seed), 16, 4, 1.0, seed=42)
        steps += len(ref["action"])
        vsum += float(ref["final_value"].astype(np.float64).sum())
        dsum += int(ref["depth"].sum())
    assert res["k4"]["steps"] == steps and res["k4"]["depth_sum"] == dsum
    assert abs(res["k4"]["value_sum"] - vsum) < 1e-4
