#!/usr/bin/env python
"""Latency sweep of leaf-parallel search with virtual loss (az_search_vl) against az_search on one GPU.

Random-init bf16 network (seed 42), roots reached by seeded random playouts with their histories (tests/helpers), virtual
loss 1.  For n roots x K leaves per root (n * K <= 4096) at 256 simulations, and for one root at 800, each point is warmed
up and then timed for at least 2 s (host clock around complete calls, which end in a device synchronise).  A separate
untimed call with az_profile sampling every forward gives the phase split.  Quality proxy against K = 1 on the same roots:
agreement of the last-argmax move (what MctsPlayer plays) and the mean total-variation distance of the visit distributions.
    python tools/search_vl_sweep.py OUT.json"""
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
from helpers import orc, random_playouts  # noqa: E402

NS = (1, 16, 100, 128, 256)
KS = (1, 2, 4, 8, 16, 32, 64)
MIN_SECONDS = 2.0


def roots_for(n, seed=42):
    positions, histories = random_playouts(4 * n + 8, seed=seed, max_plies=60)
    keep = [i for i in range(len(positions)) if orc.outcome(positions[i]) == 0][:n]
    hist = [histories[i] for i in keep]
    offs = np.zeros(n + 1, np.uint32)
    offs[1:] = np.cumsum([len(h) for h in hist])
    return positions[keep], np.concatenate(hist), offs


def last_argmax(v):
    return v.shape[1] - 1 - np.argmax(v[:, ::-1], axis=1)


def timed(fn):
    fn()   # warm-up
    reps, t0 = 0, time.perf_counter()
    while True:
        out = fn()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= MIN_SECONDS:
            return out, dt / reps, reps


def point(e, n, sims, k, roots, hist, offs, ref_visits):
    if k == 0:   # az_search
        fn = lambda: (*e.search(roots, num_simulations=sims, history=hist, hist_offsets=offs), None)  # noqa: E731
    else:
        fn = lambda: e.search_vl(roots, sims, k, 1.0, history=hist, hist_offsets=offs)  # noqa: E731
    (visits, _, depth, st), sec, reps = timed(fn)
    e.profile_enable(1)
    e.profile_read()
    fn()
    p = e.profile_read()
    e.profile_enable(0)
    row = {"impl": "az_search" if k == 0 else "az_search_vl", "n": n, "sims": sims, "K": k or None, "reps": reps,
           "ms_per_search": sec * 1e3, "sims_per_sec": n * sims / sec, "mean_depth": float(depth.mean()),
           "tower_ms": p.tower_ms, "input_ms": p.input_ms, "heads_ms": p.heads_ms, "search_kernels_ms": p.advance_ms,
           "forwards": p.tower_samples, "boards": p.tower_boards}
    if st is not None:
        row.update(waves=st.waves, evaluations=st.evaluations, boards_per_wave=st.evaluations / st.waves, collisions=st.collisions,
                   collision_fraction=st.collisions / (st.collisions + n * sims), terminal_leaves=st.terminal_leaves)
    if ref_visits is not None:
        p1 = visits / visits.sum(1, keepdims=True)
        p0 = ref_visits / ref_visits.sum(1, keepdims=True)
        row["top_move_agreement"] = float(np.mean(last_argmax(visits) == last_argmax(ref_visits)))
        row["mean_tv_distance"] = float(np.mean(0.5 * np.abs(p1 - p0).sum(1)))
    print(json.dumps(row), flush=True)
    return row, visits


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "search_vl_sweep.json"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    rows = []
    with az.Engine(max_games=256, max_batch=4096, num_simulations=800, seed=42, precision=0) as e:
        e.load_weights(az.random_weights(seed=42))
        for sims, ns in ((256, NS), (800, (1,))):
            for n in ns:
                roots, hist, offs = roots_for(n)
                r, _ = point(e, n, sims, 0, roots, hist, offs, None)
                rows.append(r)
                ref = None
                for k in KS:
                    if n * k > 4096:
                        continue
                    r, v = point(e, n, sims, k, roots, hist, offs, ref)
                    if k == 1:
                        ref = v
                    rows.append(r)
    with open(out_path, "w") as f:
        json.dump({"gpu": gpu, "network": "random-init bf16, seed 42", "virtual_loss": 1.0, "min_seconds_per_point": MIN_SECONDS,
                   "points": rows}, f, indent=1)


if __name__ == "__main__":
    main()
