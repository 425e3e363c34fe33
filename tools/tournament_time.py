#!/usr/bin/env python
"""A round-robin of the benchmark's arena (benchmark/src/main.rs:14-108: half the games each side opening, 800 simulations
per move in rounds of 8, epsilon 0, alpha 1) over 8 random-init networks (omk_net_init_random seeds 0 .. 7) on one GPU:
28 pairings of `games` games each.  Prints one JSON line with the card's name and power limit.

  tournament  one omk_tournament call on one context holding the 8 networks in model slots 0 .. 7: at every half-move each
              network searches the movers of all its 7 pairings as one batch, the networks alternating over the two lanes;
              one 36-byte read-back per half-move
  matches     the 28 pairings as 28 omk_match calls on a second context, the network and the opponent reloaded from the host
              before each call, outside the timed region

The two arms are alternated in one process, `rounds` times each, after one untimed run of each (allocations, lanes), on the
same weights and seed; every game of the tournament must equal its game in the matches.  The tournament's tree pool is
28 pairings x 2 * games trees x `nodes` node slots (5 600 x 4 096 at the defaults).

With --naive, the naive player joins as participant 0 and the arms are
  naive       one omk_tournament_naive call: 36 pairings, the first 8 against the naive player
  separate    one omk_tournament call over the 8 networks, then one omk_eval_naive call of `games` episodes per network (the
              naive player opening every game, epsilon 0, alpha 1), the network reloaded before each, outside the timed region
Every model-model game of the naive tournament must equal its game in the tournament, and the games the naive player opens
must equal the first games // 2 of that network's omk_eval_naive call.  A last, separate run of the naive tournament under
torch.profiler reports the device time of its k_naive_move launches: the naive player's half-moves.
    python tools/tournament_time.py [--naive] [--games 100 --models 8 --count 800 --rounds 2 --out FILE]"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from train_phase_time import card  # noqa: E402


def main(games=100, models=8, count=800, batch=8, rounds=2, nodes=4096, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    pairs = games // 2
    pairings = [(i, j) for i in range(models) for j in range(i + 1, models)]
    P = len(pairings)
    res = {"tool": "tournament_time", **card(), "models": models, "pairings": P, "games_per_pairing": 2 * pairs, "sims_per_move": count,
           "batch_size": batch, "epsilon": 0.0, "alpha": 1.0, "rounds": rounds, "capacity_nodes": nodes,
           "networks": f"random init (omk_net_init_random seeds 0 .. {models - 1}) in slots 0 .. {models - 1}"}
    weights = []
    for s in range(models):
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=seed)
        c.net_init_random(s)
        weights.append(c.net_get_params())
        c.close()
    tour_ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs * P, capacity_nodes=nodes, seed=seed)
    tour_ctx.net_load_params(weights[0])
    for s in range(1, models):
        tour_ctx.model_load_params(s, weights[s])
    match_ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs, capacity_nodes=nodes, seed=seed)
    kw = dict(count=count, batch_size=batch, epsilon=0.0, alpha=1.0, evaluator=omk.EVAL_NET)

    def tournament():
        l0 = tour_ctx.launch_count
        t0 = time.perf_counter()
        result, moves, _, stats = tour_ctx.tournament(list(range(models)), pairs, **kw)
        wall = time.perf_counter() - t0
        return {"wall_s": wall, "gpu_s": stats["gpu_ms"] / 1e3, "simulations": stats["simulations"], "launches": tour_ctx.launch_count - l0,
                "host_syncs": stats["host_syncs"], "moves": stats["moves"]}, result, moves

    def matches():
        run = {"wall_s": 0.0, "gpu_s": 0.0, "simulations": 0, "launches": 0, "host_syncs": 0, "moves": 0}
        result = np.zeros((P, 3), np.int32)
        moves = np.zeros((P, 2 * pairs, 81), np.int8)
        for p, (i, j) in enumerate(pairings):
            match_ctx.net_load_params(weights[i])  # outside the timed region
            match_ctx.opponent_load_params(weights[j])
            l0 = match_ctx.launch_count
            t0 = time.perf_counter()
            r, m, _, stats = match_ctx.match(pairs, **kw)
            run["wall_s"] += time.perf_counter() - t0
            run["gpu_s"] += stats["gpu_ms"] / 1e3
            run["launches"] += match_ctx.launch_count - l0
            for k in ("simulations", "host_syncs", "moves"):
                run[k] += stats[k]
            result[p], moves[p] = r, m
        return run, result, moves

    arms = {"tournament": tournament, "matches": matches}
    ref = {name: fn() for name, fn in arms.items()}  # untimed
    identical = ref["tournament"][1].tobytes() == ref["matches"][1].tobytes() and ref["tournament"][2].tobytes() == ref["matches"][2].tobytes()
    runs = {k: [] for k in arms}
    for r in range(rounds):
        for name in (arms if r % 2 == 0 else list(arms)[::-1]):
            run, result, moves = arms[name]()
            run["sims_per_s"] = run["simulations"] / run["wall_s"]
            runs[name].append(run)
            identical = identical and result.tobytes() == ref["matches"][1].tobytes() and moves.tobytes() == ref["matches"][2].tobytes()
    h2d0 = tour_ctx.transfer_bytes[0]
    tournament()
    res["tournament_h2d_bytes"] = tour_ctx.transfer_bytes[0] - h2d0
    res["games_identical"] = identical
    res["result_table"] = ref["tournament"][1].tolist()
    for name, v in runs.items():
        wall = [x["wall_s"] for x in v]
        res[name] = {"runs": v, "median_wall_s": float(np.median(wall)), "spread_wall_s": float(np.max(wall) - np.min(wall)),
                     "median_gpu_s": float(np.median([x["gpu_s"] for x in v])),
                     "median_sims_per_s": float(np.median([x["sims_per_s"] for x in v]))}
    res["matches_median_over_tournament_median"] = res["matches"]["median_wall_s"] / res["tournament"]["median_wall_s"]
    tour_ctx.close()
    match_ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not identical:
        raise SystemExit("the tournament and the matches played different games")
    return res


def main_naive(games=100, models=8, count=800, batch=8, rounds=2, nodes=4096, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    pairs = games // 2
    n = models + 1
    P, Pm = n * (n - 1) // 2, models * (models - 1) // 2
    res = {"tool": "tournament_time --naive", **card(), "models": models, "pairings": P, "games_per_pairing": 2 * pairs,
           "sims_per_move": count, "batch_size": batch, "epsilon": 0.0, "alpha": 1.0, "rounds": rounds, "capacity_nodes": nodes,
           "naive_seed": seed, "networks": f"random init (omk_net_init_random seeds 0 .. {models - 1}) in slots 0 .. {models - 1}"}
    weights = []
    for s in range(models):
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=seed)
        c.net_init_random(s)
        weights.append(c.net_get_params())
        c.close()

    def loaded(trees):
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=trees, capacity_nodes=nodes, seed=seed)
        c.net_load_params(weights[0])
        for s in range(1, models):
            c.model_load_params(s, weights[s])
        return c

    naive_ctx, sep_ctx = loaded(4 * pairs * P), loaded(max(4 * pairs * Pm, 2 * pairs))
    kw = dict(count=count, batch_size=batch, epsilon=0.0, alpha=1.0, evaluator=omk.EVAL_NET)
    slots = list(range(models))

    def naive():
        l0 = naive_ctx.launch_count
        t0 = time.perf_counter()
        result, moves, _, stats = naive_ctx.tournament_naive(slots, pairs, seed=seed, **kw)
        wall = time.perf_counter() - t0
        return {"wall_s": wall, "gpu_s": stats["gpu_ms"] / 1e3, "simulations": stats["simulations"], "launches": naive_ctx.launch_count - l0,
                "host_syncs": stats["host_syncs"], "moves": stats["moves"]}, (result, moves)

    def separate():
        l0 = sep_ctx.launch_count
        t0 = time.perf_counter()
        result, moves, _, stats = sep_ctx.tournament(slots, pairs, **kw)
        run = {"wall_s": time.perf_counter() - t0, "gpu_s": stats["gpu_ms"] / 1e3, "launches": sep_ctx.launch_count - l0,
               **{k: stats[k] for k in ("simulations", "host_syncs", "moves")}}
        evals = []
        for s in range(models):
            sep_ctx.net_load_params(weights[s])  # outside the timed region
            l0 = sep_ctx.launch_count
            t0 = time.perf_counter()
            r, m, _, st = sep_ctx.eval_naive(2 * pairs, seed=seed, **kw)
            run["wall_s"] += time.perf_counter() - t0
            run["gpu_s"] += st["gpu_ms"] / 1e3
            run["launches"] += sep_ctx.launch_count - l0
            for k in ("simulations", "host_syncs", "moves"):
                run[k] += st[k]
            evals.append((r, m))
        sep_ctx.net_load_params(weights[0])
        return run, (result, moves, evals)

    def same(a, b):  # the naive tournament's games against the tournament's and the evaluations' games
        (nr, nm), (tr, tm, evals) = a, b
        ok = nr[models:].tobytes() == tr.tobytes() and nm[models:].tobytes() == tm.tobytes()
        return ok and all(nm[s, :pairs].tobytes() == evals[s][1][:pairs].tobytes() for s in range(models))

    arms = {"naive": naive, "separate": separate}
    ref = {name: fn()[1] for name, fn in arms.items()}  # untimed
    identical = same(ref["naive"], ref["separate"])
    runs = {k: [] for k in arms}
    for r in range(rounds):
        for name in (arms if r % 2 == 0 else list(arms)[::-1]):
            run, outs = arms[name]()
            run["sims_per_s"] = run["simulations"] / run["wall_s"]
            runs[name].append(run)
            if name == "naive":
                identical = identical and outs[0].tobytes() == ref["naive"][0].tobytes() and outs[1].tobytes() == ref["naive"][1].tobytes()
            else:
                identical = identical and same(ref["naive"], outs)
    h2d0 = naive_ctx.transfer_bytes[0]
    naive()
    res["naive_h2d_bytes"] = naive_ctx.transfer_bytes[0] - h2d0
    res["games_identical"] = identical
    res["result_table"] = ref["naive"][0].tolist()
    for name, v in runs.items():
        wall = [x["wall_s"] for x in v]
        res[name] = {"runs": v, "median_wall_s": float(np.median(wall)), "spread_wall_s": float(np.max(wall) - np.min(wall)),
                     "median_gpu_s": float(np.median([x["gpu_s"] for x in v])),
                     "median_sims_per_s": float(np.median([x["sims_per_s"] for x in v]))}
    res["separate_median_over_naive_median"] = res["separate"]["median_wall_s"] / res["naive"]["median_wall_s"]
    res["naive_half_moves"] = profile_naive_moves(naive_ctx, lambda: naive_ctx.tournament_naive(slots, pairs, seed=seed, **kw))
    naive_ctx.close()
    sep_ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not identical:
        raise SystemExit("the naive tournament and the separate calls played different games")
    return res


def profile_naive_moves(ctx, call):
    """Device time of the k_naive_move launches of one call, from torch.profiler's CUDA activity (a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, _, _, stats = call()
        ctx.synchronize()
        torch.cuda.synchronize()
    device = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [e for e in device if "k_naive_move" in e.name]
    us = sum(e.device_time_total for e in kernels)
    return {"launches": len(kernels), "device_ms": us / 1e3, "mean_us_per_launch": us / len(kernels) if kernels else None,
            "call_gpu_ms": stats["gpu_ms"], "share_of_call": us / 1e3 / stats["gpu_ms"] if stats["gpu_ms"] else None,
            "kernels_captured": len(device), "kernel_device_ms_captured": sum(e.device_time_total for e in device) / 1e3}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=100, help="games per pairing (half of them each side opens)")
    ap.add_argument("--models", type=int, default=8)
    ap.add_argument("--count", type=int, default=800)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--nodes", type=int, default=4096)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--naive", action="store_true", help="time omk_tournament_naive against omk_tournament + omk_eval_naive calls")
    a = ap.parse_args()
    (main_naive if a.naive else main)(games=a.games, models=a.models, count=a.count, rounds=a.rounds, nodes=a.nodes, out=a.out)
