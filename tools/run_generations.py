#!/usr/bin/env python
"""BASELINE config 5 in miniature: the full generation loop of train() (training.rs:70-275) on one GPU -
self-play on the engine -> device replay buffer -> AdamW steps (PyTorch) -> weights back into the engine -> a short
evaluation match against the previous weights.  Prints one JSON line per iteration.

    python tools/run_generations.py --games 1024 --sims 64 --iterations 3
    torchrun --nproc-per-node 8 tools/run_generations.py --games 1024 --sims 64 --iterations 3     # games sharded; samples
                                   # all-gathered device to device into every rank's replica of the replay buffer; data-parallel
                                   # AdamW steps with one gradient all-reduce each (NCCL)
"""
import argparse
import hashlib
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _pkg  # noqa: E402,F401
import alphazero_chess_b200 as az  # noqa: E402
from alphazero_chess_b200 import evaluation as ev  # noqa: E402
from alphazero_chess_b200 import training as tr  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024, help="games per GPU and iteration")
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--iterations", type=int, default=3)
    ap.add_argument("--eval-games", type=int, default=32)
    ap.add_argument("--min-replay", type=int, default=5000)
    ap.add_argument("--leaves-per-game", type=int, default=None,
                    help="leaf-parallel self-play with virtual loss (not in the reference): up to K leaves per game and network round")
    ap.add_argument("--virtual-loss", type=float, default=1.0, help="virtual loss of --leaves-per-game")
    ap.add_argument("--all-ranks", action="store_true", help="every rank prints its line (replica check)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(42)
    vl = dict(leaves_per_game=args.leaves_per_game, virtual_loss=args.virtual_loss)
    batch = {} if args.leaves_per_game is None else {"max_batch": args.games * args.leaves_per_game}   # one round: games x K boards
    eng = az.Engine(device=local, max_games=args.games, num_simulations=args.sims, seed=42, **batch)
    # every rank holds a replica of the model, the optimizer and the replay buffer; they stay identical because every rank
    # adds the same steps in the same order and applies the same all-reduced gradients
    model = tr.import_weights(tr.AlphaZeroNet(), az.random_weights(seed=42)).to(dev)
    if world > 1:
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
    opt = tr.make_optimizer(model)
    replay = az.ReplayBuffer(eng, capacity=100_000, max_batch=tr.BATCH_SIZE)
    old = None
    if rank == 0 and args.eval_games:
        old = az.Engine(device=local, max_games=args.eval_games, max_batch=args.eval_games, num_simulations=args.sims, seed=42)
    for it in range(args.iterations):
        if old is not None:
            old.load_weights(tr.export_weights(model))
        t0 = time.perf_counter()
        if world == 1:
            m = tr.run_generation(eng, replay, model, opt, it, args.games, min_replay_size=args.min_replay, **vl)
        else:
            m = tr.run_generation_sharded(eng, replay, model, opt, it, args.games, dist, dev, min_replay_size=args.min_replay, **vl)
        torch.cuda.synchronize()
        m["generation_seconds"] = time.perf_counter() - t0
        m["positions_per_sec"] = m["positions"] / m["generation_seconds"]
        if rank == 0 and m["trained"] and args.eval_games:
            t1 = time.perf_counter()
            r = ev.evaluate(ev.MctsPlayer(eng), ev.MctsPlayer(old), eng, n_games=args.eval_games, seed=it)
            m["winrate_vs_previous"] = r["winrate"]
            m["evaluation_seconds"] = time.perf_counter() - t1
        # replica check: digest of the weights and of the oldest 256 replay entries on every rank
        h = hashlib.sha256()
        for a in tr.export_weights(model):
            h.update(a.tobytes())
        pos, pol, val, vis = replay.export(0, 256)
        h.update(pos.tobytes() + pol.tobytes() + val.tobytes() + vis.tobytes())
        m["rank"] = rank
        m["replica_digest"] = h.hexdigest()[:16]
        if world > 1:
            dist.barrier()
        if rank == 0 or args.all_ranks:
            sys.stdout.write(json.dumps(m) + "\n")   # one write per line: the ranks share a pipe
            sys.stdout.flush()
    replay.close()
    if old is not None:
        old.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
