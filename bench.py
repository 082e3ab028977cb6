#!/usr/bin/env python
"""Benchmark of the self-play hot path (BASELINE.json metric: MCTS simulations/s and self-play positions/s).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference ...                       (the reference algorithm's CPU restatement on host cores)
    python bench.py --mode generation --gpus N ...             (BASELINE configs[4]: the full generation loop)

Default mode.  A step = one ply for every resident game: `sims` network waves, in which each of the `games` concurrent
games completes its PUCT search of `sims` simulations (one simulation in flight per game, as the reference) and plays a
move.  Workload at N = 1: BASELINE configs[2] (4096 games x 800 sims/move, random-init net); every extra GPU adds another
4096 games (N = 8 is configs[3], 32768 games), so scaling is weak and there is no data-path collective: NCCL only
broadcasts the weights at the start of the timed region (one generation).

After the timed region the line is completed by legs that are NOT part of `value`:
  parity_checked   az_search at the benchmark's own size (G roots x S simulations) checked against the oracle on sampled roots
                   (synthetic evaluator: visits and scores bit-equal; the bf16 network: the oracle's tree fed the GPU's outputs)
  rank_identity    (N > 1) every rank plays a few games with the real network, rank 0 replays all of them on its own GPU
                   and compares the records digest by digest (SURVEY section 4: "1 vs N GPUs identical")
  config2_movegen  BASELINE configs[1]: perft depth 6 and 65,536-position move generation with HBM / issue-slot fractions
  eval_avoidance   the same self-play with a briefly trained ("peaked") network and the evaluation cache on: sims/s, evals/s
                   and the avoided fraction separately, next to the bf16 ceiling of one evaluation per simulation
  fp32_path        throughput of the fp32 parity network (precision = 1) beside the bf16 tensor-core path
  cpu_baseline     the oracle port on the host cores: the shared sample of --impl reference plus BASELINE configs[0]
                   (1 game, 256 simulations per move, one thread)
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_SAMPLE_PLIES = 2   # the one CPU sample both arms use: `cores` games x 2 plies x `sims` simulations per step
DUMP_SLOTS = 1024      # game slots whose last EpisodeStep --dump-outputs writes (their dense policies are 16 MB)


def load_pkg():
    import importlib.util

    name = "alphazero_chess_b200"
    if name in sys.modules:
        return sys.modules[name]
    d = os.path.join(ROOT, "alphazero-chess_b200")
    spec = importlib.util.spec_from_file_location(name, os.path.join(d, "__init__.py"), submodule_search_locations=[d])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def profile_constants():
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 8:
                self.rows.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if r[4 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_port_run(weights, sims, seed, games, plies, cores, first_game_id=0):
    """The oracle (CPU restatement of tree.rs / chess.rs / agent.rs / run_episode) on `cores` host threads: `games`
    self-play games x `plies` plies x `sims` simulations, sharing one evaluation cache like the reference."""
    from oracle import pyoracle as orc

    net = orc.Net(weights)
    prm = orc.make_params(num_simulations=sims, seed=seed)
    ev = orc.make_evaluator("net", net=net)
    cache = orc.cache_create()
    stats = [None] * games
    nxt = [0]
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                g = nxt[0]
                nxt[0] += 1
            if g >= games:
                return
            stats[g] = orc.selfplay_episode(prm, ev, game_id=first_game_id + g, max_steps=plies, cache=cache, want_visits=False)["stats"]

    t0 = time.perf_counter()
    th = [threading.Thread(target=work) for _ in range(cores)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    orc.cache_destroy(cache)
    sims_done = sum(s.simulations for s in stats)
    positions = sum(s.n_steps for s in stats)
    evals = sum(s.evals for s in stats)
    return dict(seconds=dt, simulations=sims_done, positions=positions, evals=evals)


def cpu_sample_desc(cores, sims):
    return (f"{cores} games x {CPU_SAMPLE_PLIES} plies x {sims} sims per step, one game per host thread on {cores} threads, shared "
            f"evaluation cache (the same sample in `cpu_baseline` of the GPU arm and in --impl reference)")


def cpu_shared_sample(weights, sims, cores, steps, first_step=0):
    """`steps` repetitions of the shared CPU sample; returns summed work and time."""
    tot = dict(seconds=0.0, simulations=0, positions=0, evals=0)
    for s in range(steps):
        r = cpu_port_run(weights, sims, 42, cores, CPU_SAMPLE_PLIES, cores, first_game_id=(first_step + s) * cores)
        for k in tot:
            tot[k] += r[k]
    return tot


def run_reference(args, rank, world):
    """--impl reference: the reference's own algorithm on the host cores.  The Rust reference cannot be built in this image
    (no cargo/rustc, CUDA backend hard-coded in main.rs:68), so this arm times the oracle port (kind "port").  Nothing of the
    product is imported here: the random-init network comes from the oracle's own weight catalogue."""
    if rank != 0:
        return
    from oracle import pyoracle as orc

    cores = os.cpu_count() or 1
    weights = orc.random_weights(seed=42)
    warm, steps = args.warmup, args.steps   # about 7.5 s of host work per step on 16 threads (20 + 5 steps: 3 minutes)
    cpu_shared_sample(weights, args.sims, cores, warm, first_step=0)
    r = cpu_shared_sample(weights, args.sims, cores, steps, first_step=warm)
    value = r["simulations"] / r["seconds"] if r["seconds"] > 0 else 0.0
    sample = cpu_sample_desc(cores, args.sims)
    line = {
        "impl": "reference", "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * r["seconds"] / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init 10x128 net, seed 42; start position)",
        "config": {"workload": f"reference self-play restated on CPU: {sample}", "sims_per_move": args.sims,
                   "steps_requested": args.steps, "warmup_requested": args.warmup},
        "positions_per_sec": r["positions"] / r["seconds"], "nn_evals_per_sec": r["evals"] / r["seconds"],
        "cpu_baseline": {"value": value, "unit": "sims/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ post-timing legs
def parity_leg(az, eng, G, S, visits_net, roots, ids):
    """Checks the benchmarked code path at its own size against the oracle (VERDICT r1 item 1d)."""
    from oracle import pyoracle as orc

    out = {}
    # (a) the bf16 network path that e2e just ran: the oracle's tree, fed the GPU network's outputs, must give the same visits
    def cb(ctx, pos_ptr, pol_ptr, val_ptr):
        pos = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_uint8 * 72).from_address(pos_ptr)).view(az.POSITION_DTYPE)
        p, v = eng.forward(pos)
        np.ctypeslib.as_array(pol_ptr, (4096,))[:] = p[0]
        val_ptr[0] = float(v[0])

    ev = orc.make_evaluator("callback", callback=orc.EVAL_FN(cb))
    prm = orc.make_params(num_simulations=S)
    net_rows = [0, G - 1]
    ok_net = True
    for i in net_rows:
        v, _, _, _ = orc.search(roots[i], prm, ev, noise_game=int(ids[i]), noise_ply=0)
        ok_net &= bool(np.array_equal(visits_net[i], v))
    out["network_rows_checked"] = len(net_rows)
    out["network_rows_equal"] = ok_net
    # (b) the search kernels with the synthetic evaluator, G roots x S simulations, 48 sampled rows: visits and scores bit-equal
    eng.set_evaluator_stub(1, 97)
    visits, scores, depth = eng.search(roots, num_simulations=S, noise_game_ids=ids, want_scores=True)
    eng.set_evaluator_stub(0, 0)
    evs = orc.make_evaluator("stub", stub_seed=97)
    rows = np.unique(np.concatenate([[0, G - 1], np.random.default_rng(0).choice(G, min(G, 46), replace=False)]))
    ok_stub = True
    h = hashlib.sha256()
    for i in rows:
        v, s, d, _ = orc.search(roots[i], prm, evs, noise_game=int(ids[i]), noise_ply=0)
        ok_stub &= bool(np.array_equal(visits[i], v) and np.array_equal(scores[i], s) and depth[i] == d)
        h.update(visits[i].tobytes())
    out["stub_rows_checked"] = int(len(rows))
    out["stub_rows_equal"] = ok_stub
    out["stub_visits_digest"] = h.hexdigest()[:16]
    out["size"] = f"{G} roots x {S} simulations (az_search)"
    return bool(ok_net and ok_stub), out


def record_digests(samples):
    """sha256 over the raw az_sample records of each game, in ply order."""
    out = {}
    for gid in np.unique(samples["game_id"]):
        rec = samples[samples["game_id"] == gid]
        rec = rec[np.argsort(rec["ply"])]
        out[int(gid)] = hashlib.sha256(rec.tobytes()).digest()
    return out


def play_exact(eng, slots, first_id, total, chunk=64):
    eng.selfplay_begin(slots, first_game_id=first_id, total_games=total)
    out = []
    while True:
        st = eng.selfplay_step(chunk)
        if st.pending_samples:
            out.append(eng.selfplay_drain())
        elif st.active_games == 0:
            break
    return np.concatenate(out)


def rank_identity_leg(az, weights_loader, local_rank, rank, world, dist, torch):
    """Every rank plays `k` complete games with the real network on its own GPU (its own game-id range); rank 0 then replays
    every rank's game ids on ITS GPU and compares per-game record digests: a game's record depends only on (seed, game id,
    weights), never on the device or on which other games share the batch."""
    from alphazero_chess_b200 import sharding

    k, sims = 6, 48
    eng = az.Engine(device=local_rank, max_games=k, num_simulations=sims, seed=42, num_fullmoves=20)
    weights_loader(eng)
    base = sharding.first_game_id(rank) + (1 << 30)
    mine = record_digests(play_exact(eng, k, base, k))
    dev = torch.device("cuda", local_rank)
    buf = torch.zeros(k * 32, dtype=torch.uint8, device=dev)
    buf.copy_(torch.from_numpy(np.frombuffer(b"".join(mine[base + i] for i in range(k)), np.uint8).copy()))
    parts = [torch.zeros_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    result = None
    if rank == 0:
        ok, n = True, 0
        for r in range(world):
            rb = sharding.first_game_id(r) + (1 << 30)
            replay = record_digests(play_exact(eng, k, rb, k))
            theirs = bytes(parts[r].cpu().numpy())
            for i in range(k):
                ok &= replay[rb + i] == theirs[32 * i: 32 * i + 32]
                n += 1
        result = {"games_compared": n, "identical": bool(ok),
                  "how": f"{k} complete games per rank ({sims} sims/move, bf16 network, 20-fullmove limit) replayed on rank 0, sha256 of the az_sample records"}
    eng.close()
    return result


def config2_leg(az, local_rank, peaks, consts):
    """BASELINE configs[1]: perft depth 5-6 and batched move generation, device-timed through the C ABI."""
    from oracle import pyoracle as orc

    eng = az.Engine(device=local_rank, max_games=64, max_batch=65536, num_simulations=16)
    kiwi = az.position_from_fen("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1")
    start = az.start_position()
    eng.perft(kiwi, 4)
    res = {}
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    level = {("kiwipete", 6): (8031647685, 193690690, 4085603), ("startpos", 6): (119060324, 4865609, 197281)}
    for name, pos in (("kiwipete", kiwi), ("startpos", start)):
        want, last_ply, prev_ply = level[(name, 6)]
        eng.timer_start()
        got = int(eng.perft(pos, 6)[0])
        ms = eng.timer_stop()
        # algorithmic bytes (DESIGN.md section 5): interior plies read 64 B and write 64 B per child; the last ply is bulk counted
        # (64 B read + 4 B root id per position, one count per position)
        bytes_alg = (last_ply + prev_ply) * 128 + last_ply * 68
        res[f"perft_{name}_d6"] = {"nodes": got, "equals_public_table": got == want, "ms": ms, "nodes_per_sec": got / (ms * 1e-3),
                                   "positions_expanded_per_sec": last_ply / (ms * 1e-3),
                                   "hbm": {"achieved_gbs": bytes_alg / (ms * 1e-3) / 1e9, "peak_gbs": hbm,
                                           "frac": bytes_alg / (ms * 1e-3) / 1e9 / hbm}}
    wi = consts.get("k_perft_count_warp_insts_per_position")
    if wi:
        clk = 1.9e9
        r = res["perft_kiwipete_d6"]
        r["issue"] = {"warp_insts_per_position": wi, "frac_of_issue_slots": r["positions_expanded_per_sec"] * wi / (148 * 4 * clk),
                      "note": "ncu smsp__inst_executed.sum / positions of k_perft_count (profiles/); 148 SMs x 4 schedulers x 1.9 GHz"}
    roots = np.array([orc.startpos(), orc.from_fen("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1")], orc.POSITION_DTYPE)
    pos, _, _ = orc.playout_corpus(65536, seed=42, max_plies=80, roots=roots, with_history=False)
    eng.movegen(pos[:4096])
    t0 = time.perf_counter()
    moves, index, count = eng.movegen(pos)
    dt = time.perf_counter() - t0
    wm, wi2, wc = orc.legal_moves_batch(pos[:8192])
    res["movegen_65536"] = {"positions_per_sec_e2e": 65536 / dt, "moves": int(count.sum()), "h2d_bytes": 65536 * 72, "d2h_bytes": 65536 * 1028,
                            "first_8192_equal_oracle": bool(np.array_equal(moves[:8192], wm) and np.array_equal(count[:8192], wc))}
    eng.close()
    return res


def peaked_weights(az, local_rank, seconds_budget=40.0):
    """A briefly trained network (two short generations of self-play + AdamW on this GPU): what makes a policy "peaked" is mass on
    LEGAL moves and a value head that separates positions, which a random-init net has not."""
    import torch

    from alphazero_chess_b200 import training as tr

    t0 = time.perf_counter()
    torch.manual_seed(42)
    dev = torch.device("cuda", local_rank)
    eng = az.Engine(device=local_rank, max_games=2048, num_simulations=48, seed=7, num_fullmoves=60)
    model = tr.import_weights(tr.AlphaZeroNet(), az.random_weights(seed=42)).to(dev)
    opt = tr.make_optimizer(model)
    replay = az.ReplayBuffer(eng, capacity=100_000, max_batch=tr.BATCH_SIZE)
    info = []
    for it in range(3):
        m = tr.run_generation(eng, replay, model, opt, it, 2048, min_replay_size=5000, num_steps=60)
        info.append({"positions": m["positions"], "policy_loss": m.get("avg_policy_loss"), "value_loss": m.get("avg_value_loss")})
        if time.perf_counter() - t0 > seconds_budget:
            break
    w = tr.export_weights(model)
    replay.close()
    eng.close()
    del model, opt
    torch.cuda.empty_cache()
    return w, {"generations": info, "seconds": time.perf_counter() - t0,
               "recipe": "2048 games x 48 sims per generation played to completion (60-fullmove limit), 60 AdamW steps of 512 per generation"}


def eval_avoidance_leg(az, local_rank, G, S, peak_tf):
    """Self-play as in the timed region but with the evaluation cache on (2^24 entries, 17 GB), for three networks: the
    random-init one of the headline, a briefly trained one, and the trained one with its policy logits x 4 (a stand-in for the
    peaked priors of a strong network).  sims/s, evals/s and the avoided fraction are reported separately; the headline
    `value` keeps the cache off (every simulation pays a network evaluation)."""
    w_trained, how = peaked_weights(az, local_rank)
    names = az.weight_names()
    w_sharp = [a * np.float32(4.0) if n.startswith("policy_conv_2.") else a for a, n in zip(w_trained, names)]
    out = {"network": how, "cache_log2_slots": 24,
           "note": "3 timed plies after 2 warm-up plies, same games / sims as the headline; profiles/r2_avoidance.md has the longer sweep"}
    for label, w in (("random_init", az.random_weights(seed=42)), ("trained", w_trained), ("trained_policy_logits_x4", w_sharp)):
        eng = az.Engine(device=local_rank, max_games=G, num_simulations=S, seed=42, cache_log2=24)
        eng.load_weights(w)
        eng.selfplay_begin(G, first_game_id=0)
        eng.selfplay_step(2 * S)
        st0 = eng.selfplay_step(0)
        eng.timer_start()
        st1 = eng.selfplay_step(3 * S)
        ms = eng.timer_stop()
        d = {k: getattr(st1, k) - getattr(st0, k) for k in ("simulations", "positions", "evaluations", "terminal_leaves", "cache_hits",
                                                           "cache_evictions", "sum_leaf_depth")}
        out[label] = {"sims_per_sec": d["simulations"] / (ms * 1e-3), "nn_evals_per_sec": d["evaluations"] / (ms * 1e-3),
                      "eval_avoidance_ratio": 1.0 - d["evaluations"] / max(d["simulations"], 1),
                      "cache_hits": int(d["cache_hits"]), "cache_evictions": int(d["cache_evictions"]), "terminal_leaves": int(d["terminal_leaves"]),
                      "mean_leaf_depth": d["sum_leaf_depth"] / max(d["simulations"], 1),
                      "nn_tensor_frac": d["evaluations"] * az.FLOPS_PER_EVAL / (ms * 1e-3) / 1e12 / peak_tf, "waves": 3 * S}
        eng.close()
    return out


def fp32_leg(az, local_rank):
    G, S = 1024, 32
    eng = az.Engine(device=local_rank, max_games=G, num_simulations=S, seed=42, precision=1)
    eng.load_weights(az.random_weights(seed=42))
    eng.selfplay_begin(G)
    eng.selfplay_step(8)
    st0 = eng.selfplay_step(0)
    eng.timer_start()
    st1 = eng.selfplay_step(2 * S)
    ms = eng.timer_stop()
    eng.close()
    sims = st1.simulations - st0.simulations
    return {"sims_per_sec": sims / (ms * 1e-3), "config": f"{G} games x {S} sims/move, precision = 1 (fp32 CUDA-core network, the <= 1e-5 parity path)",
            "max_abs_err_vs_torch_fp32": "<= 1e-5 fp32 / <= 1e-2 bf16 (tests/test_nn_gpu.py, tests/test_bench_size_gpu.py: measured 2e-6 / 1.1e-3)"}


def single_game_leg(az, local_rank):
    """BASELINE configs[0] on the GPU side: one game, 256 simulations per move (batch = 1: latency, not throughput)."""
    eng = az.Engine(device=local_rank, max_games=8, num_simulations=256, seed=42)
    eng.load_weights(az.random_weights(seed=42))
    root = np.array([az.start_position()], az.POSITION_DTYPE)
    eng.search(root, num_simulations=32)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        eng.search(root, num_simulations=256)
    dt = (time.perf_counter() - t0) / reps
    eng.close()
    return {"sims_per_sec": 256 / dt, "ms_per_move": dt * 1e3, "config": "1 game x 256 sims/move through az_search (one evaluation in flight: batch 1)"}


def dump_selfplay_outputs(az, eng, stats, G, S, out_dir):
    """--dump-outputs: what the last timed self-play step handed its caller, as float arrays, so that two builds can be compared
    output for output.  selfplay_stats holds what that az_selfplay_step call returned (running totals since selfplay_begin), in
    az_selfplay_stats order.  The other arrays hold, for a fixed
    seeded sample of game slots, the EpisodeStep that step produced (the last record the slot's game has staged): the searched
    position's 72 bytes, the policy index played, the search depth, the improved policy and the record's ply and game id.  A slot
    whose game ended in that step has nothing staged (its game went to the sample queue): ply -1 and zeros mark it."""
    os.makedirs(out_dir, exist_ok=True)
    slots = np.sort(np.random.default_rng(0).choice(G, min(G, DUMP_SLOTS), replace=False))
    n = len(slots)
    out = {"position": np.zeros((n, az.POSITION_DTYPE.itemsize), np.float32), "action": np.zeros(n, np.float32),
           "search_depth": np.zeros(n, np.float32), "improved_policy": np.zeros((n, az.ACTION_SPACE), np.float32),
           "ply": np.full(n, -1.0), "game_id": np.zeros(n)}
    for k, slot in enumerate(slots):
        staged = eng.selfplay_staged(int(slot))
        if len(staged) == 0:
            continue
        rec = staged[np.argmax(staged["ply"])]
        out["position"][k] = np.frombuffer(rec["position"].tobytes(), np.uint8)
        out["action"][k] = rec["action"]
        out["search_depth"][k] = rec["search_depth"]
        out["improved_policy"][k] = az.improved_policy(rec, S)
        out["ply"][k] = rec["ply"]
        out["game_id"][k] = rec["game_id"]
    out["selfplay_stats"] = np.array([getattr(stats, f) for f, _ in az.SelfplayStats._fields_], np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------ the GPU arm
def run_ours(args, rank, world, local_rank):
    import torch

    az = load_pkg()
    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    G, S = args.games, args.sims
    eng = az.Engine(device=local_rank, max_games=G, num_simulations=S, seed=42, cache_log2=args.cache_log2)

    # ---- weights: rank 0 owns them; one flat NCCL broadcast per generation, then an on-device import
    from alphazero_chess_b200 import sharding

    sizes = az.weight_sizes()
    offs = sharding.weight_offsets(sizes)
    flat = torch.zeros(int(offs[-1]), dtype=torch.float32, device=dev)
    if rank == 0:
        flat.copy_(torch.from_numpy(sharding.flatten_weights(az.random_weights(seed=42))))

    def broadcast_and_load(target=None):
        sharding.broadcast_weights(flat, dist, src=0)
        torch.cuda.synchronize()
        (target or eng).load_weights_dev([flat.data_ptr() + 4 * int(o) for o in offs[:-1]])

    broadcast_and_load()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident self-play: W warm-up steps, K timed steps
    eng.selfplay_begin(G, first_game_id=sharding.first_game_id(rank))
    for _ in range(args.warmup):
        eng.selfplay_step(S)
    st0 = eng.selfplay_step(0)
    eng.profile_enable(16)
    eng.profile_read()
    sampler = ClockSampler(local_rank)
    launches0 = eng.launch_count()
    barrier()
    sampler.start()
    eng.timer_start()
    if world > 1:
        broadcast_and_load()  # the per-generation weight broadcast is inside the timed region
    for _ in range(args.steps):
        st1 = eng.selfplay_step(S)
    ms = eng.timer_stop()
    barrier()
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    prof = eng.profile_read()
    eng.profile_enable(0)
    d = {k: getattr(st1, k) - getattr(st0, k) for k in ("simulations", "positions", "evaluations", "terminal_leaves", "games_finished",
                                                       "sum_leaf_depth", "sum_edges", "cache_hits")}
    if args.dump_outputs and rank == 0:
        dump_selfplay_outputs(az, eng, st1, G, S, args.dump_outputs)
    eng.selfplay_drain()

    # ---- end to end through the reference-facing call: MCTree::init + monte_carlo_tree_search for G host-resident roots
    roots = np.repeat(np.array([az.start_position()], az.POSITION_DTYPE), G)
    ids = np.arange(G, dtype=np.uint64) + np.uint64(sharding.first_game_id(rank))
    e2e_steps = max(1, args.steps // 3)
    eng.search(roots[: min(G, 256)], num_simulations=min(S, 32), noise_game_ids=ids[: min(G, 256)])  # warm the path
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        visits, _, _ = eng.search(roots, num_simulations=S, noise_game_ids=ids)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert float(visits.sum()) == float(G) * S
    h2d = roots.nbytes + ids.nbytes + 4 * G
    d2h = visits.nbytes + 4 * G

    # ---- aggregate over ranks: sums of work, max of time
    vec, tmax = sharding.reduce_metrics([d["simulations"], d["positions"], d["evaluations"], float(G * S * e2e_steps), launches,
                                         d["terminal_leaves"], d["sum_leaf_depth"], d["sum_edges"]], [ms, e2e_s * 1e3], dist)
    sims, positions, evals, e2e_sims = vec[0], vec[1], vec[2], vec[3]
    ms_all, e2e_ms = float(tmax[0]), float(tmax[1])

    # ---- legs outside the timed region
    parity_ok, parity = (None, None)
    if rank == 0 and not args.quick:
        parity_ok, parity = parity_leg(az, eng, G, S, visits, roots, ids)
    eng.close()
    identity = None
    if world > 1 and not args.quick:
        identity = rank_identity_leg(az, lambda e: broadcast_and_load(e), local_rank, rank, world, dist, torch)

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        consts = profile_constants()
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        roof = None
        if prof.tower_samples:
            mode = int(os.environ.get("AZ_TOWER_FUSED", "1"))
            fused = mode != 0
            # fused: one persistent launch runs all 20 convolutions for an L2-sized range of boards (two ranges at 4096 boards);
            # unfused: 20 launches over all boards.  Per launch: its duration, its boards and its algorithmic flops.
            n_launches = max(int(prof.tower_launches), 1)
            launch_ms = prof.tower_ms / n_launches
            layers = 20 if fused else 1
            boards = prof.tower_boards * (20 // layers) / n_launches
            # algorithmic flops: 3x3 128->128 convolutions, plus the input convolution's 19 real channels when it is fused into the
            # same launch (mode 2; the zero-padded channels the MMA also multiplies are not counted)
            flops_per_launch = (az.FLOPS_PER_TOWER_CONV * layers + (az.FLOPS_PER_INPUT_CONV if mode >= 2 else 0)) * boards
            achieved = flops_per_launch / (launch_ms * 1e-3) / 1e12
            traffic = consts.get("conv_tower_kernel_dram_bytes_per_launch" if fused else "conv3x3_tc2_dram_bytes_per_launch")
            kname = ("conv_tower_kernel (input convolution + the 20 3x3 128->128 convolutions of the tower in one persistent tcgen05 "
                     "cta_group::2 launch)" if mode >= 2 else
                     "conv_tower_kernel (the 20 3x3 128->128 convolutions of the tower for an L2-sized range of boards in one persistent tcgen05 cta_group::2 launch)"
                     if fused else "conv3x3_tc2_kernel<2> (tcgen05 cta_group::2 3x3 128->128 convolution, 20 of 23 launches per wave)")
            roof = {"bound": "tensor", "kernel": kname,
                    "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                    "peak_source": f"{peak_kind} bf16_tflops_sustained", "us_per_launch": launch_ms * 1e3, "boards_per_launch": boards,
                    "flops_per_launch": flops_per_launch, "launches_per_wave": n_launches / prof.tower_samples,
                    "peak_burst": float(peaks.get("bf16_tflops", 0.0)) or None,
                    "frac_of_burst": (achieved / float(peaks["bf16_tflops"])) if peaks.get("bf16_tflops") else None,
                    "note": "peak = the driver's back-to-back (sustained) torch.matmul bf16 rate, the figure for a kernel timed inside a "
                            "long step; a frac above 1 means this kernel outruns that GEMM under the same power cap (its activations "
                            "stay in the L2); peak_burst is the best-of-10 rate of the same GEMM timed alone"}
        value = sims / (ms_all * 1e-3)
        ceiling = peak_tf * 1e12 / az.FLOPS_PER_EVAL
        extra = {}
        cpu = None
        if world == 1 and not args.quick:
            extra["config2_movegen"] = config2_leg(az, local_rank, peaks, consts)
            extra["eval_avoidance"] = eval_avoidance_leg(az, local_rank, G, S, peak_tf)
            extra["fp32_path"] = fp32_leg(az, local_rank)
            extra["single_game_gpu"] = single_game_leg(az, local_rank)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as orc

            cores = os.cpu_count() or 1
            w = orc.random_weights(seed=42)
            cpu_shared_sample(w, S, cores, 1, first_step=0)          # warm-up step, as in --impl reference
            r = cpu_shared_sample(w, S, cores, 2, first_step=1)
            c1 = cpu_port_run(w, 256, 42, 1, 12, 1)                     # BASELINE configs[0]: 1 game, 256 sims/move, one thread
            cpu = {"value": r["simulations"] / r["seconds"], "unit": "sims/s", "cores": cores, "kind": "port",
                   "sample": cpu_sample_desc(cores, S) + f"; 2 timed steps after 1 warm-up ({r['seconds']:.1f} s)",
                   "positions_per_sec": r["positions"] / r["seconds"], "evals_per_sec": r["evals"] / r["seconds"],
                   "config1_single_game": {"value": c1["simulations"] / c1["seconds"], "unit": "sims/s", "cores": 1,
                                           "positions_per_sec": c1["positions"] / c1["seconds"],
                                           "sample": f"1 game x 12 plies x 256 sims on one host thread ({c1['seconds']:.1f} s): BASELINE configs[0] with a random-init net"}}
        line = {
            "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_all / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic (random-init 10x128 net, seed 42; games from the start position with Dirichlet noise)",
            "config": {"workload": f"{G} concurrent games x {S} sims/move per GPU (BASELINE configs[2]; x N GPUs = configs[3] at N=8)",
                       "games_per_gpu": G, "sims_per_move": S, "step": "one ply for every game (sims waves)",
                       "l2": "a step streams the tree pools (2.3 GB per 4096 games), planes and priors through HBM: larger than the 126 MB L2, no flush needed; inside a wave the tower keeps each 2048-board range of activations L2-resident by design",
                       "parallelism": f"games sharded {world} x {G}, no data-path collective"},
            "positions_per_sec": positions / (ms_all * 1e-3),
            "nn_evals_per_sec": evals / (ms_all * 1e-3),
            "eval_avoidance_ratio": 1.0 - evals / max(sims, 1.0),
            "cache": {"log2_slots": args.cache_log2, "hits_rank0": int(d["cache_hits"])},
            "mean_leaf_depth": vec[6] / max(sims, 1.0),
            "mean_edges_per_level": vec[7] / max(vec[6], 1.0),
            "nn_tensor_frac_whole_step": evals * az.FLOPS_PER_EVAL / (ms_all * 1e-3) / 1e12 / (peak_tf * world),
            "target": {"north_star_sims_per_sec_8gpu": 1e8, "bf16_ceiling_evals_per_sec_per_gpu": ceiling,
                       "bf16_ceiling_8gpu": 8 * ceiling,
                       "note": "one network evaluation per simulation costs 381,272,192 FLOP, so 100 % of the measured sustained bf16 rate is "
                               f"{ceiling / 1e6:.2f} M evaluations/s per GPU ({8 * ceiling / 1e6:.1f} M on 8): with a random-init network "
                               "(0.2 % of simulations avoid the network) 1e8 simulations/s is unreachable in bf16; it needs >= 71 % of the "
                               "simulations to end in the evaluation cache or a terminal position -- see eval_avoidance for what a "
                               "briefly trained network gives"},
            "e2e": {"value": e2e_sims / (e2e_ms * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "api": "az_search: G host-resident roots in, dense visit counts out"},
            "wave_phases_us": None if not prof.tower_samples else {
                "k_advance": 1e3 * prof.advance_ms / prof.tower_samples, "input_conv": 1e3 * prof.input_ms / prof.tower_samples,
                "tower": 1e3 * prof.tower_ms / prof.tower_samples, "heads": 1e3 * prof.heads_ms / prof.tower_samples,
                "wave_total": 1e3 * ms_all / max(args.steps * S, 1)},
            "gpu_launches": int(vec[4]),
            "clocks": clocks,
            "roofline": roof,
            "parity_checked": parity_ok,
            "parity": parity,
            "rank_identity": identity,
            "cpu_baseline": cpu,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ --mode generation
def run_generation_mode(args, rank, world, local_rank):
    """BASELINE configs[4]: self-play (exactly N games to completion) into the replay buffer, the training update, and a
    BaseModel-vs-BaseModel match for the Elo of the new network (training.rs:70-275 with SKIP_VALIDATION = true), on N GPUs:
    games sharded, samples device -> NCCL all-gather -> device, data-parallel AdamW steps with a gradient all-reduce."""
    import torch

    az = load_pkg()
    from alphazero_chess_b200 import evaluation as evm
    from alphazero_chess_b200 import sharding
    from alphazero_chess_b200 import training as tr

    dist = None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    G, S = args.games, args.sims
    torch.manual_seed(42)
    slots = min(args.slots or G, G, 4096)
    eng = az.Engine(device=local_rank, max_games=max(slots, 256), num_simulations=S, seed=42, cache_log2=args.cache_log2)
    model = tr.import_weights(tr.AlphaZeroNet(), az.random_weights(seed=42)).to(dev)
    if world > 1:
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)   # BatchNorm statistics over the global batch, as the reference's
    opt = tr.make_optimizer(model)
    replay = az.ReplayBuffer(eng, capacity=100_000, max_batch=tr.BATCH_SIZE)
    exchange = sharding.DeviceSampleExchange(eng, dist, dev, max(eng.config.max_games * 128, 1 << 16))
    old = az.Engine(device=local_rank, max_games=256, max_batch=256, num_simulations=S, seed=42) if rank == 0 else None
    rows = []
    for it in range(args.warmup + args.steps):
        if old is not None:
            old.load_weights(tr.export_weights(model))
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m = tr.run_generation_sharded(eng, replay, model, opt, it, G, dist, dev, min_replay_size=args.min_replay, exchange=exchange,
                                      concurrent=slots)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        m["generation_seconds"] = time.perf_counter() - t0
        if rank == 0:
            t1 = time.perf_counter()
            r = evm.evaluate(evm.BasePlayer(eng), evm.BasePlayer(old), eng, n_games=256, seed=it)   # EVALUATION_GAMES (parameters.rs:37)
            m["elo_match"] = {"winrate_vs_previous": r["winrate"], "games": 256, "seconds": time.perf_counter() - t1}
        if it >= args.warmup:
            rows.append(m)
    if rank == 0:
        secs = sum(m["generation_seconds"] for m in rows)
        positions = sum(m["positions"] for m in rows)
        sims = sum(m["simulations"] for m in rows)
        line = {"metric": "selfplay_positions_per_sec", "value": positions / secs, "unit": "positions/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(len(rows), 1), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "mode": "generation",
                "data": "synthetic start (random-init 10x128 net, seed 42), then the loop's own self-play data",
                "config": {"workload": f"BASELINE configs[4]: per generation {G} complete self-play games per GPU x {S} sims/move -> replay buffer "
                                       f"(100,000) -> 40 x 512 AdamW steps (data parallel) -> 256-game BaseModel match", "games_per_gpu": G, "concurrent_games_per_gpu": slots,
                           "sims_per_move": S, "parallelism": f"games sharded {world} x {G}; NCCL: sample all-gather (device to device), gradient all-reduce"},
                "mcts_simulations_per_sec": sims / secs, "sample_bytes_gathered": exchange.bytes_moved, "generations": rows}
        print(json.dumps(line), flush=True)
    replay.close()
    eng.close()
    if old is not None:
        old.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="selfplay", choices=["selfplay", "generation"])
    ap.add_argument("--games", type=int, default=None, help="concurrent games per GPU (selfplay: 4096) / games per GPU and generation (generation: 1024)")
    ap.add_argument("--sims", type=int, default=None, help="simulations per move (selfplay: 800 = BASELINE configs[2]; generation: 256 = parameters.rs:32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="timed region and e2e only (no parity / config-2 / eval-avoidance / fp32 legs)")
    ap.add_argument("--cache-log2", type=int, default=0, help="log2 slots of the GPU evaluation cache (0 = off)")
    ap.add_argument("--min-replay", type=int, default=20_000, help="generation mode: MIN_REPLAY_SIZE (parameters.rs:11)")
    ap.add_argument("--slots", type=int, default=0, help="generation mode: concurrent games per GPU (0 = all games of the generation at once, like the reference's NUM_EPISODES tasks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="selfplay mode: after the timed steps write what the last one computed (rank 0's games) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "selfplay" or args.impl != "ours"):
        ap.error("--dump-outputs writes the GPU self-play path's outputs: it needs --mode selfplay --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.mode == "generation":
        args.games = args.games or 1024
        args.sims = args.sims or 256
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "generation mode has no CPU arm (the oracle restates self-play, not training)"}))
            return
        run_generation_mode(args, rank, world, local_rank)
        return
    args.games = args.games or 4096
    args.sims = args.sims or 800
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
