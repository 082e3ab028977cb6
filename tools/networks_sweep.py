#!/usr/bin/env python
"""Two networks in one engine against one engine per network, on one GPU.

Random-init bf16 networks (seeds 42 and 43, BatchNorm randomised), positions and roots from seeded random playouts
(tests/helpers).  Every point alternates its arms in one process, is warmed up, and each arm runs for at least 2 s (host clock
around complete calls, which end in a device synchronise).  Device times come from az_profile sampling every forward (input
convolution, tower, heads).
  forward  forward_networks of n + n boards (networks interleaved)  |  forward of 2n boards (one network)  |  forward of n boards
           on each of two single-network engines, one after the other
  search   search_networks over 2 x 128 roots (256 simulations, K = 1 and 8)  |  the same roots split over two single-network
           engines: az_search (K = 1) or az_search_vl (K = 8) on each, one after the other
  match    evaluate(MctsPlayer(e, network=0), MctsPlayer(e, network=1))  |  the same match on two engines; 256 games, 256
           simulations, max_plies capped; the results arrays are compared
    python tools/networks_sweep.py OUT_DIR   (writes OUT_DIR/r4_networks_1gpu.json and OUT_DIR/r4_networks.md)"""
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
from helpers import orc, random_playouts  # noqa: E402

FORWARD_NS = (1, 16, 64, 128, 512, 2048)
MIN_SECONDS = 2.0
MATCH_PLIES = 40


def alternate(arms):
    """arms: {name: (fn, engines whose forwards the arm runs)}.  Warm-up, then round-robin until every arm has run >= MIN_SECONDS."""
    for fn, _ in arms.values():
        fn()
    stat = {k: dict(reps=0, sec=0.0, device_ms=0.0, input_ms=0.0, tower_ms=0.0, heads_ms=0.0, forwards=0) for k in arms}
    while min(s["sec"] for s in stat.values()) < MIN_SECONDS:
        for k, (fn, engines) in arms.items():
            for e in engines:
                e.profile_enable(1)
                e.profile_read()
            t0 = time.perf_counter()
            fn()
            stat[k]["sec"] += time.perf_counter() - t0
            stat[k]["reps"] += 1
            for e in engines:
                p = e.profile_read()
                e.profile_enable(0)
                stat[k]["input_ms"] += p.input_ms
                stat[k]["tower_ms"] += p.tower_ms
                stat[k]["heads_ms"] += p.heads_ms
                stat[k]["device_ms"] += p.input_ms + p.tower_ms + p.heads_ms
                stat[k]["forwards"] += p.tower_samples
    out = {}
    for k, s in stat.items():
        r = s["reps"]
        out[k] = {"reps": r, "wall_ms": 1e3 * s["sec"] / r, "device_ms": s["device_ms"] / r, "input_ms": s["input_ms"] / r,
                  "tower_ms": s["tower_ms"] / r, "heads_ms": s["heads_ms"] / r, "forwards_per_call": s["forwards"] / r}
    return out


def roots_for(n, seed):
    positions, histories = random_playouts(4 * n + 8, seed=seed, max_plies=60)
    keep = [i for i in range(len(positions)) if orc.outcome(positions[i]) == 0][:n]
    return positions[keep], [histories[i] for i in keep]


def flat(histories):
    offs = np.zeros(len(histories) + 1, np.uint32)
    offs[1:] = np.cumsum([len(h) for h in histories])
    return np.concatenate(histories), offs


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    w0, w1 = az.random_weights(seed=42, randomize_bn=True), az.random_weights(seed=43, randomize_bn=True)
    cfg = dict(max_games=256, max_batch=4096, num_simulations=256, seed=42)
    rows = {"forward": [], "search": [], "match": []}
    with az.Engine(**cfg) as both, az.Engine(**cfg) as e0, az.Engine(**cfg) as e1:
        both.load_weights(w0)
        both.load_weights(w1, network=1)
        e0.load_weights(w0)
        e1.load_weights(w1)
        pool, _ = random_playouts(4096, seed=7, max_plies=80)
        for n in FORWARD_NS:
            pos = np.resize(pool, 2 * n)
            net = (np.arange(2 * n) % 2).astype(np.uint8)
            a, b = pos[net == 0], pos[net == 1]
            r = alternate({"two_networks": (lambda: both.forward_networks(pos, net), [both]),
                           "one_network_2n": (lambda: both.forward(pos), [both]),
                           "two_engines_sequential": (lambda: (e0.forward(a), e1.forward(b)), [e0, e1])})
            r = {"n": n, **r, "ratio_vs_one_network_2n": r["two_networks"]["device_ms"] / r["one_network_2n"]["device_ms"],
                 "ratio_vs_sequential": r["two_networks"]["device_ms"] / r["two_engines_sequential"]["device_ms"]}
            print(json.dumps(r), flush=True)
            rows["forward"].append(r)
        roots, hists = roots_for(256, seed=11)
        net = (np.arange(256) % 2).astype(np.uint8)
        hist, offs = flat(hists)
        sel = [np.flatnonzero(net == s) for s in (0, 1)]
        part = [flat([hists[i] for i in s]) for s in sel]
        for k in (1, 8):
            def single(e, s):
                if k == 1:
                    return e.search(roots[sel[s]], num_simulations=256, history=part[s][0], hist_offsets=part[s][1])[0]
                return e.search_vl(roots[sel[s]], 256, k, 1.0, history=part[s][0], hist_offsets=part[s][1])[0]
            joint = lambda: both.search_networks(roots, net, 256, k, 1.0, history=hist, hist_offsets=offs)[0]  # noqa: E731
            r = alternate({"search_networks": (joint, [both]), "two_engines_sequential": (lambda: (single(e0, 0), single(e1, 1)), [e0, e1])})
            v = joint()
            same = all(np.array_equal(v[sel[s]], single(e, s)) for s, e in ((0, e0), (1, e1)))
            r = {"roots": "2 x 128", "sims": 256, "K": k, **r, "visits_identical": bool(same),
                 "speedup": r["two_engines_sequential"]["wall_ms"] / r["search_networks"]["wall_ms"]}
            print(json.dumps(r), flush=True)
            rows["search"].append(r)
        times = {"one_engine": [], "two_engines": []}
        res = {}
        for rep in range(2):
            for name in ("one_engine", "two_engines"):
                p1, p2 = ((ev.MctsPlayer(both, 256, network=0), ev.MctsPlayer(both, 256, network=1)) if name == "one_engine"
                          else (ev.MctsPlayer(e0, 256), ev.MctsPlayer(e1, 256)))
                t0 = time.perf_counter()
                out = ev.evaluate(p1, p2, both if name == "one_engine" else e0, n_games=256, max_plies=MATCH_PLIES, seed=3)
                times[name].append(time.perf_counter() - t0)
                res[name] = out["results"]
        r = {"games": 256, "sims": 256, "max_plies": MATCH_PLIES, "wall_s_one_engine": min(times["one_engine"]),
             "wall_s_two_engines": min(times["two_engines"]), "results_identical": bool(np.array_equal(res["one_engine"], res["two_engines"]))}
        r["speedup"] = r["wall_s_two_engines"] / r["wall_s_one_engine"]
        print(json.dumps(r), flush=True)
        rows["match"].append(r)
    doc = {"gpu": gpu, "networks": "random-init bf16, seeds 42 / 43, BatchNorm randomised", "min_seconds_per_arm": MIN_SECONDS, **rows}
    with open(os.path.join(out_dir, "r4_networks_1gpu.json"), "w") as f:
        json.dump(doc, f, indent=1)
    with open(os.path.join(out_dir, "r4_networks.md"), "w") as f:
        f.write(report(doc))


def report(doc):
    L = ["# Two networks in one engine (r4)", "", f"GPU (name, power limit, max SM clock): {doc['gpu']}.  Generated by "
         "`tools/networks_sweep.py`; raw numbers in `r4_networks_1gpu.json`.  Networks: " + doc["networks"] + ".", "",
         "## Forward", "", "Device time per call (az_profile: input convolution + tower + heads, summed over the call's forwards).", "",
         "| n | two networks n + n (ms) | one network 2n (ms) | two engines n, n (ms) | ratio vs 2n | ratio vs sequential | input / tower / heads, two networks (ms) |",
         "|---:|---:|---:|---:|---:|---:|---|"]
    for r in doc["forward"]:
        t = r["two_networks"]
        L.append(f"| {r['n']} | {t['device_ms']:.3f} | {r['one_network_2n']['device_ms']:.3f} | {r['two_engines_sequential']['device_ms']:.3f} | "
                 f"{r['ratio_vs_one_network_2n']:.3f} | {r['ratio_vs_sequential']:.3f} | {t['input_ms']:.3f} / {t['tower_ms']:.3f} / {t['heads_ms']:.3f} |")
    L += ["", "## Search (2 x 128 roots, 256 simulations)", "", "Wall time per call.", "",
          "| K | search_networks (ms) | two engines, sequential (ms) | speed-up | visits identical |", "|---:|---:|---:|---:|---|"]
    for r in doc["search"]:
        L.append(f"| {r['K']} | {r['search_networks']['wall_ms']:.1f} | {r['two_engines_sequential']['wall_ms']:.1f} | {r['speedup']:.2f} | "
                 f"{r['visits_identical']} |")
    L += ["", "## Match", "", "| games | simulations | plies | one engine (s) | two engines (s) | speed-up | results identical |",
          "|---:|---:|---:|---:|---:|---:|---|"]
    for r in doc["match"]:
        L.append(f"| {r['games']} | {r['sims']} | {r['max_plies']} | {r['wall_s_one_engine']:.2f} | {r['wall_s_two_engines']:.2f} | "
                 f"{r['speedup']:.2f} | {r['results_identical']} |")
    return "\n".join(L) + "\n"


if __name__ == "__main__":
    main()
