"""Training step and generation loop around the engine (SURVEY section 8(f) #2; training.rs:40-292, 424-440).

Not on the self-play hot path: the network update is ordinary PyTorch (autograd + AdamW on the 10x128 ResNet), the data
comes from the device-resident replay buffer and the new weights go back into the engine through az_load_weights.
Reference semantics restated here (burn 0.18 defaults recalled, not pinned by any reference test):
  loss        = mean_b( -sum_i pi[b,i] * log(p[b,i] + 1e-5) ) + 0.5 * mean_b( (v[b] - z[b])^2 )      training.rs:277-292
  optimizer   = AdamW(beta 0.9/0.999, eps 1e-5, weight decay 1e-4), gradients clipped by value to +-1    training.rs:64-67
  learning rate = triangular cycle 1e-3 <-> 1e-2 over 20 iterations, x0.1 every 1000 iterations            training.rs:424-440
  40 steps of 512 samples per iteration once the buffer holds 20,000 positions                            parameters.rs:11,16-17
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

NUM_RES_BLOCKS, NUM_FILTERS = 10, 128           # parameters.rs:7-8
NUM_TRAIN_STEPS, BATCH_SIZE = 40, 512           # parameters.rs:16-17
MIN_REPLAY_SIZE = 20_000                        # parameters.rs:11
BASE_LEARNING_RATE, MAX_LEARNING_RATE = 1e-3, 1e-2
FULL_CYCLE, HALF_CYCLE, DECAY_INTERVAL = 20, 10, 1000
VALUE_LOSS_WEIGHT, WEIGHT_DECAY = 0.5, 1e-4


class ResidualBlock(nn.Module):                 # agent.rs:11-46
    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(NUM_FILTERS, NUM_FILTERS, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(NUM_FILTERS, eps=1e-5, momentum=0.1)
        self.conv2 = nn.Conv2d(NUM_FILTERS, NUM_FILTERS, 3, padding=1)
        self.bn2 = nn.BatchNorm2d(NUM_FILTERS, eps=1e-5, momentum=0.1)

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        y = self.bn2(self.conv2(y))
        return F.relu(y + x)


class AlphaZeroNet(nn.Module):                  # agent.rs:49-144
    def __init__(self):
        super().__init__()
        self.input_conv = nn.Conv2d(19, NUM_FILTERS, 3, padding=1)
        self.input_bn = nn.BatchNorm2d(NUM_FILTERS)
        self.res_blocks = nn.ModuleList([ResidualBlock() for _ in range(NUM_RES_BLOCKS)])
        self.policy_conv_1 = nn.Conv2d(NUM_FILTERS, 32, 1)
        self.policy_bn = nn.BatchNorm2d(32)
        self.policy_conv_2 = nn.Conv2d(32, 64, 1)
        self.value_conv = nn.Conv2d(NUM_FILTERS, 8, 1)
        self.value_bn = nn.BatchNorm2d(8)
        self.value_linear_1 = nn.Linear(512, 64)
        self.value_linear_2 = nn.Linear(64, 1)

    def forward(self, x):
        x = F.relu(self.input_bn(self.input_conv(x)))
        for blk in self.res_blocks:
            x = blk(x)
        p = F.relu(self.policy_bn(self.policy_conv_1(x)))
        policy = torch.softmax(self.policy_conv_2(p).flatten(1), dim=1)
        v = F.relu(self.value_bn(self.value_conv(x))).flatten(1)
        v = F.relu(self.value_linear_1(v))
        value = torch.tanh(self.value_linear_2(v)).squeeze(1)
        return policy, value


def _modules_in_weight_order(model):
    """(kind, module) in the order of az_weight_name: conv/linear -> weight, bias; bn -> gamma, beta, mean, var."""
    out = [("conv", model.input_conv), ("bn", model.input_bn)]
    for blk in model.res_blocks:
        out += [("conv", blk.conv1), ("bn", blk.bn1), ("conv", blk.conv2), ("bn", blk.bn2)]
    out += [("conv", model.policy_conv_1), ("bn", model.policy_bn), ("conv", model.policy_conv_2), ("conv", model.value_conv),
            ("bn", model.value_bn), ("linear", model.value_linear_1), ("linear", model.value_linear_2)]
    return out


def export_weights(model):
    """The 144 f32 arrays az_load_weights expects (burn layout: Linear weight is [d_in, d_out])."""
    arrays = []
    for kind, m in _modules_in_weight_order(model):
        if kind == "bn":
            arrays += [m.weight, m.bias, m.running_mean, m.running_var]
        elif kind == "linear":
            arrays += [m.weight.t(), m.bias]
        else:
            arrays += [m.weight, m.bias]
    return [a.detach().float().cpu().contiguous().numpy().ravel().copy() for a in arrays]


def import_weights(model, arrays):
    it = iter(arrays)
    with torch.no_grad():
        for kind, m in _modules_in_weight_order(model):
            if kind == "bn":
                for t in (m.weight, m.bias, m.running_mean, m.running_var):
                    t.copy_(torch.from_numpy(np.asarray(next(it), np.float32)).view_as(t))
            elif kind == "linear":
                w = torch.from_numpy(np.asarray(next(it), np.float32)).view(m.in_features, m.out_features)
                m.weight.copy_(w.t())
                m.bias.copy_(torch.from_numpy(np.asarray(next(it), np.float32)))
            else:
                m.weight.copy_(torch.from_numpy(np.asarray(next(it), np.float32)).view_as(m.weight))
                m.bias.copy_(torch.from_numpy(np.asarray(next(it), np.float32)))
    return model


def compute_loss(predicted_policy, target_policy, predicted_value, target_value):
    """compute_gradients (training.rs:277-292) without the backward call."""
    difference = predicted_value - target_value
    policy_loss = -(target_policy * (predicted_policy + 1e-5).log()).sum(1).mean()
    value_loss = (difference * difference).mean()
    return policy_loss, value_loss, policy_loss + value_loss * VALUE_LOSS_WEIGHT


def get_cyclical_lr(iteration):
    """training.rs:424-440."""
    decay_multiplier = 10.0 ** (-(iteration // DECAY_INTERVAL))
    base_lr, max_lr = BASE_LEARNING_RATE * decay_multiplier, MAX_LEARNING_RATE * decay_multiplier
    cur = iteration % FULL_CYCLE
    lr_range = max_lr - base_lr
    if cur <= HALF_CYCLE:
        return base_lr + (cur / HALF_CYCLE) * lr_range
    return max_lr - ((cur - HALF_CYCLE) / HALF_CYCLE) * lr_range


def make_optimizer(model):
    return torch.optim.AdamW(model.parameters(), lr=BASE_LEARNING_RATE, betas=(0.9, 0.999), eps=1e-5, weight_decay=WEIGHT_DECAY)


def train_iteration(model, optimizer, replay, iteration, num_steps=NUM_TRAIN_STEPS, batch_size=BATCH_SIZE, seed=0, dist=None):
    """The inner loop of train() (training.rs:137-200): num_steps batches from the replay buffer, one AdamW step each.
    Returns (avg policy loss, avg value loss).

    With several ranks (dist) the step is data parallel: every rank holds the same replay buffer (DeviceSampleExchange) and
    draws the SAME batch (same seed), computes the loss terms of its own rows rank::world scaled to the global batch, and one
    flat all-reduce sums the gradients, so every rank applies the reference's full-batch update and the replicas stay
    identical.  BatchNorm statistics are per rank slice unless the model was converted with SyncBatchNorm (CUDA only)."""
    from . import sharding

    device = next(model.parameters()).device
    world = dist.get_world_size() if dist is not None and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    model.train()
    lr = get_cyclical_lr(iteration)
    for g in optimizer.param_groups:
        g["lr"] = lr
    params = [p for p in model.parameters() if p.requires_grad]
    flat = None
    tot = torch.zeros(2, dtype=torch.float64, device=device)
    done = 0
    for step in range(num_steps):
        batch_seed = (seed * 1_000_003 + iteration) * 65_537 + step
        if device.type == "cuda" and hasattr(replay, "sample_torch"):   # device-resident: replay buffer -> trainer without a host hop
            planes, policy, value = replay.sample_torch(batch_size, seed=batch_seed)
            n = planes.shape[0]
            if n == 0:
                break
            x, pi, z = planes[rank::world], policy[rank::world], value[rank::world]
        else:
            planes, policy, value = replay.sample(batch_size, seed=batch_seed)
            n = planes.shape[0]
            if n == 0:
                break
            x = torch.from_numpy(planes[rank::world]).to(device)
            pi = torch.from_numpy(policy[rank::world]).to(device)
            z = torch.from_numpy(value[rank::world]).to(device)
        p, v = model(x)
        # compute_gradients (training.rs:277-292) over the GLOBAL batch of n rows: this rank contributes its rows' terms
        difference = v - z
        pl = -(pi * (p + 1e-5).log()).sum() / n
        vl = (difference * difference).sum() / n
        loss = pl + vl * VALUE_LOSS_WEIGHT
        optimizer.zero_grad(set_to_none=True)
        loss.backward()
        flat = sharding.allreduce_gradients(params, dist, flat)
        torch.nn.utils.clip_grad_value_(params, 1.0)
        optimizer.step()
        tot += torch.stack([pl.detach(), vl.detach()]).double()
        done += 1
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    n = max(done, 1)
    return float(tot[0]) / n, float(tot[1]) / n


def run_generation(engine, replay, model, optimizer, iteration, n_games, min_replay_size=MIN_REPLAY_SIZE, waves_per_call=64,
                   num_steps=NUM_TRAIN_STEPS, batch_size=BATCH_SIZE, concurrent=None, leaves_per_game=None, virtual_loss=1.0):
    """One iteration of train() (training.rs:70-200) on the engine: EXACTLY n_games self-play games are played to completion
    (run_all_episodes, training.rs:352-361,376-377: a slot whose game ends takes the next unplayed game or goes idle; nothing
    is cut off), their steps go from device memory straight into the replay buffer, then the training steps, then the new
    weights are loaded into the engine.  Returns a dict of the metrics the reference logs.  leaves_per_game / virtual_loss:
    leaf-parallel self-play (Engine.selfplay_begin; not in the reference), None = the reference's search."""
    engine.load_weights(export_weights(model))
    slots = min(n_games, concurrent or engine.config.max_games, engine.config.max_games)
    engine.selfplay_begin(slots, first_game_id=iteration * (1 << 24), total_games=n_games, leaves_per_game=leaves_per_game,
                          virtual_loss=virtual_loss)
    new_unique = steps = waves = 0
    while True:
        st = engine.selfplay_step(waves_per_call)
        waves += waves_per_call
        if st.pending_samples:
            n, nu = replay.add_pending()
            steps += n
            new_unique += nu
        elif st.active_games == 0:
            break
    assert st.games_finished == n_games, (st.games_finished, n_games)
    out = {"iteration": iteration, "games": int(st.games_finished), "positions": steps, "new_unique_states": new_unique,
           "replay_buffer_size": len(replay), "simulations": int(st.simulations), "evaluations": int(st.evaluations),
           "cache_hits": int(st.cache_hits), "trained": False,
           # what MetricUpdate::SelfPlayFinished logs (training.rs:107-129): mean search depth per step, mean batch per wave
           "avg_search_depth": st.sum_search_depth / max(int(st.positions), 1), "avg_batch_size": st.evaluations / max(waves, 1)}
    if len(replay) >= min_replay_size:
        pl, vl = train_iteration(model, optimizer, replay, iteration, num_steps, batch_size)
        out.update(trained=True, avg_policy_loss=pl, avg_value_loss=vl, learning_rate=get_cyclical_lr(iteration))
        engine.load_weights(export_weights(model))
    return out


def run_generation_sharded(engine, replay, model, optimizer, iteration, games_per_rank, dist, device, min_replay_size=MIN_REPLAY_SIZE,
                           waves_per_call=64, num_steps=NUM_TRAIN_STEPS, batch_size=BATCH_SIZE, concurrent=None, exchange=None,
                           leaves_per_game=None, virtual_loss=1.0):
    """run_generation over several GPUs (BASELINE config 5; SURVEY 8(e)).  Every rank plays EXACTLY games_per_rank games to
    completion (disjoint game ids, no data-path collective) and holds its own replica of the replay buffer, model and
    optimizer.  On CUDA the finished games' steps go device -> NCCL all-gather -> device (sharding.DeviceSampleExchange) and
    every rank adds all ranks' steps in rank order, so the replicas of the FEN-keyed buffer (memory.rs) are identical; the
    training steps are data parallel with one gradient all-reduce each (train_iteration); nothing is broadcast afterwards
    because every rank has applied the same update.  On CPU (gloo tests) the same protocol runs through host arrays."""
    from . import SAMPLE_DTYPE, sharding

    rank = dist.get_rank() if dist is not None and dist.is_initialized() else 0
    world = dist.get_world_size() if dist is not None and dist.is_initialized() else 1
    on_gpu = device is not None and torch.device(device).type == "cuda"
    if iteration == 0 and world > 1:   # replicas start from rank 0's initial weights (afterwards they evolve in lockstep)
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=0)
    engine.load_weights(export_weights(model))
    slots = min(games_per_rank, concurrent or engine.config.max_games, engine.config.max_games)
    engine.selfplay_begin(slots, first_game_id=sharding.first_game_id(rank) + iteration * (1 << 24), total_games=games_per_rank,
                          leaves_per_game=leaves_per_game, virtual_loss=virtual_loss)
    if on_gpu and exchange is None:
        exchange = sharding.DeviceSampleExchange(engine, dist, device, max(engine.config.max_games * 128, 1 << 16))
    import time

    steps = new_unique = 0
    done = False
    st = None
    t_play = t_xchg = 0.0
    while True:
        t0 = time.perf_counter()
        if not done:
            st = engine.selfplay_step(waves_per_call)
        t1 = time.perf_counter()
        t_play += t1 - t0
        if on_gpu:
            for ptr, n in exchange.exchange():
                if n:
                    steps += n
                    new_unique += replay.add_dev(ptr, n)
            t_xchg += time.perf_counter() - t1
        else:
            mine = engine.selfplay_drain() if (st.pending_samples and not done) else np.zeros(0, SAMPLE_DTYPE)
            got = sharding.allgather_samples(mine, dist)
            if len(got):
                steps += len(got)
                new_unique += replay.add(got)
        done = st.active_games == 0
        if sharding.all_done(done, dist, device if on_gpu else None):
            break
    sums, _ = sharding.reduce_metrics([float(st.simulations), float(st.evaluations), float(st.games_finished), float(st.sum_search_depth),
                                       float(st.positions)], [0.0], dist)
    out = {"iteration": iteration, "n_ranks": world, "games": int(sums[2]), "positions": steps, "new_unique_states": new_unique,
           "avg_search_depth": float(sums[3]) / max(float(sums[4]), 1.0),
           "replay_buffer_size": len(replay), "simulations": int(sums[0]), "evaluations": int(sums[1]), "trained": False,
           "sample_gather": "device all-gather (NCCL)" if on_gpu else "host all-gather",
           "seconds_selfplay": t_play, "seconds_sample_exchange_and_replay_add": t_xchg}
    if len(replay) >= min_replay_size:   # identical on every rank: the replicas hold the same entries
        t0 = time.perf_counter()
        pl, vl = train_iteration(model, optimizer, replay, iteration, num_steps, batch_size, dist=dist if world > 1 else None)
        out.update(trained=True, avg_policy_loss=pl, avg_value_loss=vl, learning_rate=get_cyclical_lr(iteration))
        engine.load_weights(export_weights(model))
        out["seconds_training"] = time.perf_counter() - t0
    return out
