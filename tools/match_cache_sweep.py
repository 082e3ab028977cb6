#!/usr/bin/env python
"""Resident matches (evaluation.evaluate_on_device, az_match_begin_players) with the match's evaluation cache on (cache_log2 20) and
off (0), on one GPU.

256 games, full length (max_plies 450), seed 3, bf16 networks in slots 0 and 1, two network sets:
  random-init       seeds 42 / 43, BatchNorm randomised
  sharpened         the same with the policy head's last convolution x 8 (logits x 8), the stand-in for a trained network's peaked
                    priors that tools/avoidance_sweep.py uses for self-play
Rows: MCTS(256) vs BaseModel, MCTS(256) vs Random, MCTS(256) vs MCTS(64) (r7's three pairings: player 1 on network 0, player 2 on
network 1), MCTS(256) vs MCTS(256) on networks (0, 1) and on (0, 0).  Each row alternates its two arms, REPS runs each, after a
4-ply warm-up match of each arm; wall time is a host clock around the whole call, which ends in a device synchronise.  Every
cached run's results and moves are compared with the uncached run's, and evaluations + cache_hits with the uncached evaluations.
With --parent-lib, the cache-off runs on the random-init networks are timed again with that library (the parent commit's build) in a child process, alternated
with the cache-off runs of this build in another child, so that the uncached path can be compared with the code it started from.
The parts run as separate calls, each reading the card's name, power limit and max SM clock itself; --report merges them:
    python tools/match_cache_sweep.py OUT_DIR --part random-init|sharpened   (writes OUT_DIR/r8_part_<part>.json)
    python tools/match_cache_sweep.py OUT_DIR --part parent --parent-lib PATH
    python tools/match_cache_sweep.py OUT_DIR --report          (writes OUT_DIR/r8_match_cache_1gpu.json and OUT_DIR/r8_match_cache.md)
    python tools/match_cache_sweep.py --uncached-only [LIB]     (child: one JSON line of cache-off wall times per row)"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import match_sweep  # noqa: E402,F401  (registers the package from the tree)
import alphazero_chess_b200 as az  # noqa: E402
from alphazero_chess_b200 import evaluation as ev  # noqa: E402

GAMES, SIMS, MAX_PLIES, SEED, REPS, CACHE_LOG2, SHARPEN = 256, 256, 450, 3, 2, 20, 8.0
WARMUP_PLIES = 4
ROWS = ["MCTS(256) vs BaseModel", "MCTS(256) vs Random", "MCTS(256) vs MCTS(64)", "MCTS(256) vs MCTS(256), networks 0 / 1",
        "MCTS(256) vs MCTS(256), network 0 / 0"]
NETWORKS = ["random-init", "sharpened"]


def weights(which):
    w = [az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)]
    if which == "sharpened":
        names = az.weight_names()
        w = [[a * np.float32(SHARPEN) if n.startswith("policy_conv_2.") else a for n, a in zip(names, ws)] for ws in w]
    return w


def players(row, e):
    mcts = ev.MctsPlayer(e, SIMS, network=0)
    return {ROWS[0]: (mcts, ev.BasePlayer(e, network=1)), ROWS[1]: (mcts, ev.RandomPlayer(e)),
            ROWS[2]: (mcts, ev.MctsPlayer(e, 64, network=1)), ROWS[3]: (mcts, ev.MctsPlayer(e, SIMS, network=1)),
            ROWS[4]: (mcts, ev.MctsPlayer(e, SIMS, network=0))}[row]


def engine(which):
    e = az.Engine(max_games=GAMES, max_batch=2 * GAMES, num_simulations=SIMS, seed=42)
    w = weights(which)
    e.load_weights(w[0])
    e.load_weights(w[1], network=1)
    return e


def timed(ps, cache_log2):
    kw = {"cache_log2": cache_log2} if cache_log2 else {}   # the parent library's evaluate_on_device has no cache_log2
    t0 = time.perf_counter()
    out = ev.evaluate_on_device(*ps, n_games=GAMES, max_plies=MAX_PLIES, seed=SEED, **kw)
    return time.perf_counter() - t0, out


def uncached_only():
    """child process: the cache-off arm of every row on the random-init networks, one JSON line per row"""
    for which in NETWORKS[:1]:
        with engine(which) as e:
            for row in ROWS:
                ps = players(row, e)
                ev.evaluate_on_device(*ps, n_games=GAMES, max_plies=WARMUP_PLIES, seed=SEED)
                t, _ = timed(ps, 0)
                print(json.dumps({"networks": which, "row": row, "wall_s": t}), flush=True)


def run_row(which, row, e):
    ps = players(row, e)
    for c in (0, CACHE_LOG2):
        ev.evaluate_on_device(*ps, n_games=GAMES, max_plies=WARMUP_PLIES, seed=SEED, cache_log2=c)   # every launch shape
    times = {"off": [], "on": []}
    identical, identity = True, True
    hits = []
    for _ in range(REPS):
        t, off = timed(ps, 0)
        times["off"].append(t)
        t, on = timed(ps, CACHE_LOG2)
        times["on"].append(t)
        identical &= bool(np.array_equal(off["results"], on["results"]) and np.array_equal(off["moves"], on["moves"]) and
                          np.array_equal(off["plies"], on["plies"]))
        so, sc = off["stats"], on["stats"]
        identity &= all(sc.evaluations[s] + sc.cache_hits[s] == so.evaluations[s] for s in range(2))
        hits.append([int(h) for h in sc.cache_hits])
    so, sc = off["stats"], on["stats"]
    ev_off = [int(x) for x in so.evaluations]
    r = {"networks": which, "row": row, "games": GAMES, "max_plies": MAX_PLIES, "wall_s": times, "plies": int(so.plies),
         "waves": {"off": int(so.waves), "on": int(sc.waves)}, "evaluations_off": ev_off,
         "evaluations_on": [int(x) for x in sc.evaluations], "cache_hits_each_run": hits,
         "avoided": [h / e if e else None for h, e in zip(hits[-1], ev_off)],
         "avoided_total": sum(hits[-1]) / max(1, sum(ev_off)), "results_and_moves_identical": identical,
         "evaluations_plus_hits_equal_uncached": identity, "winrate": off["winrate"],
         "speedup_min": min(times["off"]) / min(times["on"])}
    print(json.dumps(r), flush=True)
    return r


def child_times(lib):
    cmd = [sys.executable, os.path.abspath(__file__), "--uncached-only"] + ([lib] if lib else [])
    out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
    return {(d["networks"], d["row"]): d["wall_s"] for d in (json.loads(l) for l in out.splitlines() if l.startswith("{"))}


def gpu_name():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]


def main():
    if sys.argv[1:2] == ["--uncached-only"]:
        if len(sys.argv) > 2:
            az.LIB_PATH = sys.argv[2]
        uncached_only()
        return
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    if "--report" in sys.argv:
        parts = {}
        for name in NETWORKS + ["parent"]:
            with open(os.path.join(out_dir, f"r8_part_{name}.json")) as f:
                parts[name] = json.load(f)
        doc = {"gpu": sorted({p["gpu"] for p in parts.values()}),
               "networks": {"random-init": "bf16, seeds 42 / 43, BatchNorm randomised",
                            "sharpened": f"the same with policy_conv_2 x {SHARPEN:g} (policy logits x {SHARPEN:g})"},
               "simulations": SIMS, "seed": SEED, "reps": REPS, "cache_log2": CACHE_LOG2,
               "rows": [r for name in NETWORKS for r in parts[name]["rows"]], "uncached_vs_parent": parts["parent"]["rows"]}
        with open(os.path.join(out_dir, "r8_match_cache_1gpu.json"), "w") as f:
            json.dump(doc, f, indent=1)
        with open(os.path.join(out_dir, "r8_match_cache.md"), "w") as f:
            f.write(report(doc))
        return
    part = sys.argv[sys.argv.index("--part") + 1]
    gpu = gpu_name()
    print("gpu:", gpu, flush=True)
    if part == "parent":   # the uncached path against the parent build, alternated: this build, parent, this build, parent
        lib = sys.argv[sys.argv.index("--parent-lib") + 1]
        runs = [("this", child_times(None)), ("parent", child_times(lib)), ("this", child_times(None)), ("parent", child_times(lib))]
        rows = [{"networks": w, "row": r, "this_s": [t[(w, r)] for k, t in runs if k == "this"],
                 "parent_s": [t[(w, r)] for k, t in runs if k == "parent"]} for w in NETWORKS[:1] for r in ROWS]
    else:
        with engine(part) as e:
            rows = [run_row(part, row, e) for row in ROWS]
    with open(os.path.join(out_dir, f"r8_part_{part}.json"), "w") as f:
        json.dump({"gpu": gpu, "rows": rows}, f, indent=1)


def report(doc):
    L = ["# Matches with an evaluation cache (r8)", "", f"GPU (name, power limit, max SM clock): {'; '.join(doc['gpu'])}.  Generated by "
         "`tools/match_cache_sweep.py`; raw numbers in `r8_match_cache_1gpu.json`.  " f"{GAMES} games per row, max_plies {MAX_PLIES}, "
         f"seed {doc['seed']}, MCTS with K = 1.  Networks: random-init ({doc['networks']['random-init']}) and sharpened "
         f"({doc['networks']['sharpened']}).  Cache on = `cache_log2` {doc['cache_log2']} (1 GiB); each arm ran {doc['reps']} times, "
         "alternated with the other arm of its row; wall time = host clock around the whole `evaluate_on_device` call.  Each network "
         "set and the comparison with the parent ran in a call of its own, each reading the card's name and power limit.", "",
         "| networks | row | wall s off (each run) | wall s on (each run) | speed-up with the cache (best off / best on) | evaluations off, network 0 / 1 | "
         "cache hits, network 0 / 1 | avoided | results and moves identical | evaluations + hits = off |",
         "|---|---|---|---|---:|---:|---:|---:|---|---|"]
    for r in doc["rows"]:
        t = r["wall_s"]
        L.append(f"| {r['networks']} | {r['row']} | {' / '.join(f'{x:.2f}' for x in t['off'])} | {' / '.join(f'{x:.2f}' for x in t['on'])} | "
                 f"{r['speedup_min']:.3f}x | {r['evaluations_off'][0]} / {r['evaluations_off'][1]} | "
                 f"{r['cache_hits_each_run'][-1][0]} / {r['cache_hits_each_run'][-1][1]} | {100 * r['avoided_total']:.1f} % | "
                 f"{r['results_and_moves_identical']} | {r['evaluations_plus_hits_equal_uncached']} |")
    L += ["", "Hits per run (they may differ between runs: slots race to insert within a wave; the games may not):", ""]
    for r in doc["rows"]:
        L.append(f"- {r['networks']}, {r['row']}: " + ", ".join(f"{a} / {b}" for a, b in r["cache_hits_each_run"]) +
                 f"; waves off {r['waves']['off']}, on {r['waves']['on']}; plies {r['plies']}")
    if "uncached_vs_parent" in doc:
        L += ["", "The uncached path against the parent commit's library: cache-off runs in child processes, this build and the "
              "parent's alternated (this, parent, this, parent), one run per row each time after a 4-ply warm-up.", "",
              "| networks | row | this build, s | parent, s | best this / best parent |", "|---|---|---|---|---:|"]
        for r in doc["uncached_vs_parent"]:
            L.append(f"| {r['networks']} | {r['row']} | {' / '.join(f'{x:.2f}' for x in r['this_s'])} | "
                     f"{' / '.join(f'{x:.2f}' for x in r['parent_s'])} | {min(r['this_s']) / min(r['parent_s']):.3f} |")
    return "\n".join(L) + "\n"


if __name__ == "__main__":
    main()
