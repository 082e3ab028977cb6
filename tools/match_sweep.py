#!/usr/bin/env python
"""Evaluation matches resident on the device (evaluation.evaluate_on_device, az_match_*) against evaluate()'s host loop, on one GPU.

Random-init bf16 networks (seeds 42 and 43, BatchNorm randomised), 256 games, full length (max_plies 450), seed 3.  Each row runs
its arms alternated in one process, twice each after a 4-ply warm-up match of every arm; wall time is a host clock around the
whole call, which ends in a device synchronise.  Every arm's results and moves (evaluate's captured by wrapping play_move) are
compared with the resident match's.
  mcts K = 1   evaluate_on_device  |  evaluate on one engine (joint path: one search_networks call per ply)  |  evaluate on two
               engines (one engine per network, two searches per ply)
  mcts K = 8   evaluate_on_device  |  evaluate on one engine
  base model   evaluate_on_device  |  evaluate on one engine (one forward_networks + movegen per ply)
    python tools/match_sweep.py OUT_DIR   (writes OUT_DIR/r6_match_1gpu.json and OUT_DIR/r6_match.md)"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _pkg  # noqa: E402,F401
import alphazero_chess_b200 as az  # noqa: E402
from alphazero_chess_b200 import evaluation as ev  # noqa: E402

GAMES, SIMS, MAX_PLIES, SEED, REPS = 256, 256, 450, 3, 2
WARMUP_PLIES = 4


def captured(eng, p1, p2, n_games):
    """evaluate() with every ply's moves captured from play_move"""
    played, orig = [], eng.play_move
    eng.play_move = lambda pos, act, *a, **k: (played.append(np.array(act)), orig(pos, act, *a, **k))[1]
    try:
        return ev.evaluate(p1, p2, eng, n_games=n_games, max_plies=MAX_PLIES, seed=SEED), played
    finally:
        del eng.play_move


def same_games(dev, ref, played):
    if not np.array_equal(dev["results"], ref["results"]) or dev["unfinished"] != ref["unfinished"]:
        return False
    plies = dev["plies"]
    return len(played) == int(plies.max()) and all(np.array_equal(dev["moves"][plies > p, p], a) for p, a in enumerate(played))


def run_row(name, device_players, host_arms):
    """device_players: (p1, p2) on one engine; host_arms: {arm: (p1, p2, rules engine)}"""
    ev.evaluate_on_device(*device_players, n_games=GAMES, max_plies=WARMUP_PLIES, seed=SEED)   # warm-up: every launch shape
    for p1, p2, e in host_arms.values():
        ev.evaluate(p1, p2, e, n_games=GAMES, max_plies=WARMUP_PLIES, seed=SEED)
    times = {"resident": [], **{a: [] for a in host_arms}}
    identical = {a: True for a in host_arms}
    dev = None
    for _ in range(REPS):
        t0 = time.perf_counter()
        dev = ev.evaluate_on_device(*device_players, n_games=GAMES, max_plies=MAX_PLIES, seed=SEED)
        times["resident"].append(time.perf_counter() - t0)
        for a, (p1, p2, e) in host_arms.items():
            t0 = time.perf_counter()
            ref, played = captured(e, p1, p2, GAMES)
            times[a].append(time.perf_counter() - t0)
            identical[a] &= same_games(dev, ref, played)
    st = dev["stats"]
    r = {"row": name, "games": GAMES, "max_plies": MAX_PLIES, "wall_s": times, "plies": int(st.plies), "waves": int(st.waves),
         "evaluations": [int(st.evaluations[0]), int(st.evaluations[1])], "leaves": int(st.leaves), "collisions": int(st.collisions),
         "unfinished": dev["unfinished"], "winrate": dev["winrate"], "results_and_moves_identical": identical}
    r["speedup_min"] = {a: min(times[a]) / min(times["resident"]) for a in host_arms}
    print(json.dumps(r), flush=True)
    return r


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    w0, w1 = az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)
    cfg = dict(max_games=GAMES, max_batch=2 * GAMES * 8, num_simulations=SIMS, seed=42)
    rows = []
    with az.Engine(**cfg) as both, az.Engine(**cfg) as e0, az.Engine(**cfg) as e1:
        both.load_weights(w0)
        both.load_weights(w1, network=1)
        e0.load_weights(w0)
        e1.load_weights(w1)
        mcts = lambda e, k, s: ev.MctsPlayer(e, SIMS, leaves_per_root=k, network=s)  # noqa: E731
        rows.append(run_row("mcts K=1", (mcts(both, 1, 0), mcts(both, 1, 1)),
                            {"evaluate_one_engine": (mcts(both, 1, 0), mcts(both, 1, 1), both),
                             "evaluate_two_engines": (mcts(e0, 1, 0), mcts(e1, 1, 0), e0)}))
        rows.append(run_row("mcts K=8", (mcts(both, 8, 0), mcts(both, 8, 1)),
                            {"evaluate_one_engine": (mcts(both, 8, 0), mcts(both, 8, 1), both)}))
        base = (ev.BasePlayer(both, network=0), ev.BasePlayer(both, network=1))
        rows.append(run_row("base model", base, {"evaluate_one_engine": (*base, both)}))
    doc = {"gpu": gpu, "networks": "random-init bf16, seeds 42 / 43, BatchNorm randomised", "simulations": SIMS, "seed": SEED,
           "reps": REPS, "rows": rows}
    with open(os.path.join(out_dir, "r6_match_1gpu.json"), "w") as f:
        json.dump(doc, f, indent=1)
    with open(os.path.join(out_dir, "r6_match.md"), "w") as f:
        f.write(report(doc))


def report(doc):
    L = ["# Evaluation matches on the device (r6)", "", f"GPU (name, power limit, max SM clock): {doc['gpu']}.  Generated by "
         "`tools/match_sweep.py`; raw numbers in `r6_match_1gpu.json`.  Networks: " + doc["networks"] + f".  {GAMES} games, max_plies "
         f"{MAX_PLIES}, {doc['simulations']} simulations, seed {doc['seed']}; each arm ran {doc['reps']} times, alternated with the "
         "other arms of its row; wall time = host clock around the whole call.", "",
         "| row | arm | wall s (each run) | spread | resident speed-up (best vs best) | results and moves identical |",
         "|---|---|---|---:|---:|---|"]
    for r in doc["rows"]:
        for arm, ts in r["wall_s"].items():
            spread = (max(ts) - min(ts)) / min(ts)
            sp = "" if arm == "resident" else f"{r['speedup_min'][arm]:.2f}"
            same = "" if arm == "resident" else str(r["results_and_moves_identical"][arm])
            L.append(f"| {r['row']} | {arm} | {' / '.join(f'{t:.2f}' for t in ts)} | {100 * spread:.1f} % | {sp} | {same} |")
    L += ["", "Counters of the last resident run (az_match_stats).  `waves` counts the network rounds evaluate_on_device stepped, in "
          "steps of 256: the last step runs on after the final game has ended, with every slot idle.", "",
          "| row | plies | waves | evaluations network 0 / 1 | leaves | collisions | unfinished | player 1 winrate |",
          "|---|---:|---:|---:|---:|---:|---:|---:|"]
    for r in doc["rows"]:
        L.append(f"| {r['row']} | {r['plies']} | {r['waves']} | {r['evaluations'][0]} / {r['evaluations'][1]} | {r['leaves']} | "
                 f"{r['collisions']} | {r['unfinished']} | {r['winrate']:.4f} |")
    return "\n".join(L) + "\n"


if __name__ == "__main__":
    main()
