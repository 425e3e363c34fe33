#!/usr/bin/env python
"""The training phase of an iteration with the replay memory on the host and on the device, on one GPU.  Prints one JSON
line with the card's name and power limit.

  (a) host path, as a training loop runs it: trainer.ReplayMemory ingests the self-play phase (split_episodes ply by ply,
      6x augmentation), then `steps` x (ReplayMemory.sample(minibatch) + encode_nn_input + omk_train_step), with the
      memory full (600 000 rows, the reference's capacity, src/config.rs)
  (b) device path: the same self-play feeds the context's replay memory; then ONE omk_train_replay of `steps` steps
  (c) self-play ms per ply at `games` x `count` simulations with and without a replay memory attached, two contexts
      alternated in the same process (the spread of each side is reported next to the difference)

The self-play of (a) and (b) is one run: the transitions stream to the host (a) while the driver feeds the device replay
memory (b); the same seeds give the same games either way (tests/test_replay_gpu.py).
    python tools/train_phase_time.py [--games 1024 --count 800 --steps 600 --minibatch 128]"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch

    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except (OSError, ValueError, subprocess.SubprocessError):
        out["power_limit"] = "not read"
    return out


def main(games=1024, count=800, batch=16, steps=600, minibatch=128, capacity=600_000, chunk=20, rounds=4, round_plies=10, seed=0):
    omk = importlib.import_module("omok-ai_b200")
    trainer = importlib.import_module("omok-ai_b200.trainer")
    res = {"tool": "train_phase_time", **card(), "games": games, "sims_per_move": count, "steps": steps, "minibatch": minibatch,
           "capacity": capacity}

    # ---- one self-play phase until both memories hold `capacity` rows ----
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * games, capacity_nodes=4096, seed=seed)
    ctx.net_init_random(seed)
    ctx.replay_reset(capacity)
    ctx.selfplay_begin(games, count, batch, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    mem = trainer.ReplayMemory(capacity=capacity, seed=seed)
    carry, plies, ingest_s, sp_s = None, 0, 0.0, 0.0
    while len(mem) < capacity or ctx.replay_info()[0] < capacity:
        t0 = time.perf_counter()
        _, boards, policy, status, _ = ctx.selfplay_run(chunk, profile=0, want_transitions=True)
        t1 = time.perf_counter()
        for p in range(chunk):  # the host replay's ingest, ply by ply as a driver loop hands them over
            episodes, carry = trainer.split_episodes(boards[p:p + 1], policy[p:p + 1], status[p:p + 1], carry)
            for b, pi, z in episodes:
                mem.add_episode(b, pi, z)
        ingest_s += time.perf_counter() - t1
        sp_s += t1 - t0
        plies += chunk
    n_dev, added, episodes = ctx.replay_info()
    res.update({"selfplay_plies": plies, "selfplay_s": sp_s, "host_ingest_s": ingest_s, "host_rows": len(mem), "device_rows": n_dev,
                "device_rows_added": added, "device_episodes": episodes})

    # ---- (a) host path ----
    b, t, pi, z = mem.sample(minibatch)
    ctx.train_step(trainer.encode_nn_input(b, t), pi, z)  # warm-up: training workspace
    sample_s = encode_s = step_s = 0.0
    host_losses = []
    t_phase = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        b, t, pi, z = mem.sample(minibatch)
        t1 = time.perf_counter()
        img = trainer.encode_nn_input(b, t)
        t2 = time.perf_counter()
        host_losses.append(ctx.train_step(img, pi, z)[2])  # returns after the step's synchronisation
        t3 = time.perf_counter()
        sample_s += t1 - t0
        encode_s += t2 - t1
        step_s += t3 - t2
    host_phase_s = time.perf_counter() - t_phase
    res["host"] = {"train_phase_s": host_phase_s, "sample_s": sample_s, "encode_s": encode_s, "train_step_s": step_s,
                   "sample_ms_per_step": sample_s * 1e3 / steps, "train_step_ms": step_s * 1e3 / steps,
                   "first_loss": host_losses[0], "last_loss": host_losses[-1]}

    # ---- (b) device path ----
    ctx.train_replay(seed, 10**9, 1, minibatch)  # warm-up on a stream the timed call does not use
    h2d0 = ctx.transfer_bytes[0]
    t0 = time.perf_counter()
    losses = ctx.train_replay(seed, 0, steps, minibatch)  # sampling, encoding, steps: one call, one synchronisation
    dev_phase_s = time.perf_counter() - t0
    res["device"] = {"train_phase_s": dev_phase_s, "ms_per_step": dev_phase_s * 1e3 / steps, "h2d_bytes": ctx.transfer_bytes[0] - h2d0,
                     "first_loss": float(losses[0, 2]), "last_loss": float(losses[-1, 2])}
    res["device_phase_over_steps_x_host_step_time"] = dev_phase_s / step_s
    res["host_phase_over_device_phase"] = host_phase_s / dev_phase_s
    ctx.close()

    # ---- (c) self-play with and without the feed, alternated ----
    ctxs = {}
    for name, with_replay in (("without_replay", False), ("with_replay", True)):
        c = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * games, capacity_nodes=4096, seed=seed + 1)
        c.net_init_random(seed)
        if with_replay:
            c.replay_reset(capacity)
        c.selfplay_begin(games, count, batch, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
        c.selfplay_run(2, profile=0, want_transitions=False)  # warm-up
        ctxs[name] = c
    ms = {k: [] for k in ctxs}
    for r in range(rounds):
        for name in (ctxs if r % 2 == 0 else list(ctxs)[::-1]):
            t0 = time.perf_counter()
            ctxs[name].selfplay_run(round_plies, profile=0, want_transitions=False)
            ms[name].append((time.perf_counter() - t0) * 1e3 / round_plies)
    res["selfplay_ms_per_ply"] = {k: {"rounds": v, "mean": float(np.mean(v)), "spread": float(np.max(v) - np.min(v))} for k, v in ms.items()}
    res["selfplay_ms_per_ply"]["with_replay_rows"] = ctxs["with_replay"].replay_info()[0]
    res["selfplay_ms_per_ply"]["plies_per_round"] = round_plies
    for c in ctxs.values():
        c.close()
    print(json.dumps(res), flush=True)
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--count", type=int, default=800)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--minibatch", type=int, default=128)
    ap.add_argument("--capacity", type=int, default=600_000)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--round-plies", type=int, default=10)
    a = ap.parse_args()
    main(games=a.games, count=a.count, steps=a.steps, minibatch=a.minibatch, capacity=a.capacity, rounds=a.rounds,
         round_plies=a.round_plies)
