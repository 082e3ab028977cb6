#!/usr/bin/env python
"""Leaf-parallel self-play with virtual loss (az_selfplay_begin_vl) against the default self-play (az_selfplay_begin_n) on one GPU.

Random-init bf16 network (seed 42), 256 simulations per move, virtual loss 1.  Reads the GPU's name, power limit and max SM
clock in the same run.  Writes OUT_DIR/r5_selfplay_vl_1gpu.json and OUT_DIR/r5_selfplay_vl.md.
  (a) steady self-play (endless mode) at G concurrent games: begin_n and K in {1, 2, 4, 8, 16, 32} with G * K <= 4096; every arm
      is warmed up, then timed (host clock around az_selfplay_step calls, which end in a device synchronise); the arms run in
      two rounds, forward and reverse order, and a separate profiled pass (az_profile on every forward) gives the split of a
      wave into search kernels and network;
  (b) generations played to completion: 100 games (NUM_EPISODES) and 2048 games on 2048 slots; self-play seconds and the
      seconds after active_games first drops below 256 (the tail);
  (c) agreement: 256 positions from the 100-game generation searched with az_search_vl at each K and with az_search at the same
      budget (total-variation distance of the improved policies, agreement of the last-argmax move);
  (d) bench.py --gpus 1 once: the default path's headline.
    python tools/selfplay_vl_sweep.py OUT_DIR"""
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

SIMS = 256
KS = (1, 2, 4, 8, 16, 32)
WARM_S, TIMED_S = 1.5, 2.5


def steady_point(e, G, k):
    e.selfplay_begin(G, first_game_id=0, leaves_per_game=k)
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < WARM_S:
        e.selfplay_step(16)
    a = e.selfplay_step(0)
    v0 = e.selfplay_vl_stats() if k else None
    waves, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < TIMED_S:
        e.selfplay_step(16)
        waves += 16
    dt = time.perf_counter() - t0
    b = e.selfplay_step(0)
    sims = b.simulations - a.simulations
    row = {"G": G, "arm": "begin_n" if k is None else f"K={k}", "K": k, "seconds": dt, "waves": waves, "sims_per_sec": sims / dt,
           "positions_per_sec": (b.positions - a.positions) / dt, "boards_per_wave": (b.evaluations - a.evaluations) / waves}
    if k:
        v1 = e.selfplay_vl_stats()
        row["collisions_per_1000_sims"] = 1000.0 * (v1.collisions - v0.collisions) / max(sims, 1)
    e.profile_enable(1)
    e.profile_read()
    e.selfplay_step(32)
    p = e.profile_read()
    e.profile_enable(0)
    n = max(p.tower_samples, 1)
    row.update(search_ms_per_wave=p.advance_ms / n, network_ms_per_wave=(p.input_ms + p.tower_ms + p.heads_ms) / n)
    print(json.dumps(row), flush=True)
    return row


def generation(e, games, slots, k, keep=False):
    e.selfplay_begin(slots, first_game_id=0, total_games=games, leaves_per_game=k)
    t0 = time.perf_counter()
    t_tail, kept = None, []
    while True:
        st = e.selfplay_step(16)
        if t_tail is None and st.active_games < 256:
            t_tail = time.perf_counter()
        if st.pending_samples:
            s = e.selfplay_drain()
            if keep:
                kept.append(s)
        elif st.active_games == 0:
            break
    t1 = time.perf_counter()
    row = {"games": games, "slots": slots, "arm": "begin_n" if k is None else f"K={k}", "K": k, "selfplay_seconds": t1 - t0,
           "tail_seconds": t1 - (t_tail or t0), "simulations": int(st.simulations), "positions": int(st.positions),
           "sims_per_sec": st.simulations / (t1 - t0)}
    if k:
        row["collisions"] = int(e.selfplay_vl_stats().collisions)
    print(json.dumps(row), flush=True)
    return row, (np.concatenate(kept) if kept else None)


def agreement(e, positions):
    v0, _, _ = e.search(positions, num_simulations=SIMS)
    p0 = v0 / v0.sum(1, keepdims=True)
    top0 = v0.shape[1] - 1 - np.argmax(v0[:, ::-1], axis=1)
    rows = []
    for k in KS[1:]:
        v, _, _, st = e.search_vl(positions, SIMS, k, 1.0)
        p = v / v.sum(1, keepdims=True)
        top = v.shape[1] - 1 - np.argmax(v[:, ::-1], axis=1)
        rows.append({"K": k, "mean_tv_distance": float(np.mean(0.5 * np.abs(p - p0).sum(1))), "top_move_agreement": float(np.mean(top == top0)),
                     "collisions": int(st.collisions)})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def md(doc):
    L = ["# r5: leaf-parallel self-play (az_selfplay_begin_vl) on one GPU", "",
         f"GPU: {doc['gpu']} (name, power limit, max SM clock, read in the same run).  {doc['network']}, {SIMS} simulations per move, "
         "virtual loss 1.  Written by `tools/selfplay_vl_sweep.py`; raw rows in `r5_selfplay_vl_1gpu.json`.", "",
         "## (a) Steady self-play (endless mode)", "",
         "Two rounds per G (forward, then reverse arm order); each row is one timed window of about 2.5 s after a 1.5 s warm-up.  "
         "Search / network ms per wave come from a separate pass with `az_profile` on every forward.", "",
         "| G | arm | round | M sims/s | positions/s | boards/wave | collisions / 1000 sims | search ms/wave | network ms/wave |",
         "|---:|---|---:|---:|---:|---:|---:|---:|---:|"]
    for r in doc["steady"]:
        L.append(f"| {r['G']} | {r['arm']} | {r['round']} | {r['sims_per_sec'] / 1e6:.3f} | {r['positions_per_sec']:.0f} | {r['boards_per_wave']:.0f} | "
                 f"{r.get('collisions_per_1000_sims', 0):.1f} | {r['search_ms_per_wave']:.3f} | {r['network_ms_per_wave']:.3f} |")
    L += ["", "## (b) Generations played to completion", "",
          "| games | slots | arm | self-play s | tail s (after active < 256) | M sims/s | collisions |", "|---:|---:|---|---:|---:|---:|---:|"]
    for r in doc["generations"]:
        L.append(f"| {r['games']} | {r['slots']} | {r['arm']} | {r['selfplay_seconds']:.2f} | {r['tail_seconds']:.2f} | {r['sims_per_sec'] / 1e6:.3f} | "
                 f"{r.get('collisions', '')} |")
    L += ["", "## (c) Agreement with az_search at the same budget", "",
          "256 positions from the 100-game generation, searched without history or noise.  With a random-init network this is a weak "
          "proxy for playing strength.", "", "| K | mean TV distance | top-move agreement | collisions |", "|---:|---:|---:|---:|"]
    for r in doc["agreement"]:
        L.append(f"| {r['K']} | {r['mean_tv_distance']:.4f} | {r['top_move_agreement']:.3f} | {r['collisions']} |")
    L += ["", "## (d) Headline of the default path", "", "`bench.py --gpus 1`:", "", "```", doc["bench"], "```", ""]
    return "\n".join(L)


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    doc = {"gpu": gpu, "network": "random-init bf16 network (seed 42)", "steady": [], "generations": [], "agreement": []}
    w = az.random_weights(seed=42)
    for G in (100, 256, 1024):
        arms = [None] + [k for k in KS if G * k <= 4096]
        with az.Engine(max_games=G, max_batch=4096, num_simulations=SIMS, seed=42) as e:
            e.load_weights(w)
            for rnd, order in enumerate((arms, arms[::-1])):
                for k in order:
                    doc["steady"].append(dict(steady_point(e, G, k), round=rnd + 1))
    kept = None
    with az.Engine(max_games=100, max_batch=3200, num_simulations=SIMS, seed=42) as e:
        e.load_weights(w)
        for k in (None, 8, 16, 32):
            row, s = generation(e, 100, 100, k, keep=k is None)
            doc["generations"].append(row)
            kept = s if k is None else kept
        idx = np.linspace(0, len(kept) - 1, 256).astype(np.int64)
        with az.Engine(max_games=256, max_batch=256 * 32, num_simulations=SIMS, seed=42) as e2:
            e2.load_weights(w)
            doc["agreement"] = agreement(e2, np.ascontiguousarray(kept["position"][idx]))
    for k in (None, 2, 4, 8):
        with az.Engine(max_games=2048, max_batch=2048 * (k or 1), num_simulations=SIMS, seed=42) as e:
            e.load_weights(w)
            doc["generations"].append(generation(e, 2048, 2048, k)[0])
    b = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"], capture_output=True, text=True)
    doc["bench"] = [l for l in b.stdout.splitlines() if l.startswith("{")][-1] if b.returncode == 0 else f"failed: {b.stderr[-2000:]}"
    print(doc["bench"], flush=True)
    with open(os.path.join(out_dir, "r5_selfplay_vl_1gpu.json"), "w") as f:
        json.dump(doc, f, indent=1)
    with open(os.path.join(out_dir, "r5_selfplay_vl.md"), "w") as f:
        f.write(md(doc))


if __name__ == "__main__":
    main()
