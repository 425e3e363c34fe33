#!/usr/bin/env python
"""The benchmark's arena (benchmark/src/main.rs:14-108: two networks, half the games each opening, 800 simulations per move
in rounds of 8, epsilon 0, alpha 1) on one GPU, driven from the host and on the device, with two random-init networks.
Prints one JSON line with the card's name and power limit.

  host path    arena.play_match on two contexts, one network each: the leg the left network opens, then the other;
               per half-move five entry points (pool_search, pool_sample, pool_play, pool_ensure_action, pool_play), each
               with its own synchronisation
  device path  arena.play_match_device: one omk_match call on one context holding both networks (the network and the
               opponent); both legs at once, each model's half-move on its own search lane, one 8-byte read-back per half-move

The two paths are alternated in one process, `rounds` times each, after one untimed run of each (allocations, lanes), on
the same weights and seed; every run's move lists must be identical across the paths.
    python tools/match_time.py [--games 100,1024 --count 800 --rounds 3 --out FILE]"""
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


def main(games=(100, 1024), count=800, batch=8, rounds=3, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    arena = importlib.import_module("omok-ai_b200.arena")
    res = {"tool": "match_time", **card(), "sims_per_move": count, "batch_size": batch, "epsilon": 0.0, "alpha": 1.0, "rounds": rounds,
           "networks": f"random init (omk_net_init_random seeds {seed + 1} left / network, {seed + 2} right / opponent)", "shapes": []}
    for game_count in games:
        pairs = game_count // 2
        left, right = (omk.Context(device=0, capacity_envs=1, capacity_trees=pairs, capacity_nodes=4096, seed=seed) for _ in range(2))
        dev = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs, capacity_nodes=4096, seed=seed)
        left.net_init_random(seed + 1)
        right.net_init_random(seed + 2)
        dev.net_init_random(seed + 1)
        dev.opponent_load_params(right.net_get_params())
        kw = dict(game_count=game_count, count=count, batch_size=batch, epsilon=0.0, alpha=1.0, evaluator=omk.EVAL_NET)
        paths = {"host": lambda moves: arena.play_match(left, right, moves_out=moves, **kw),
                 "device": lambda moves: arena.play_match_device(dev, moves_out=moves, **kw)}
        ref = {}
        for name, fn in paths.items():  # untimed
            ref[name] = []
            fn(ref[name])
        runs = {k: [] for k in paths}
        identical = ref["host"] == ref["device"]
        for r in range(rounds):
            for name in (paths if r % 2 == 0 else list(paths)[::-1]):
                moves = []
                t0 = time.perf_counter()
                wld = paths[name](moves)
                runs[name].append({"s": time.perf_counter() - t0, "left_network_wins": wld[0], "right_opponent_wins": wld[1], "draws": wld[2]})
                identical = identical and moves == ref["host"]
        h2d0 = dev.transfer_bytes[0]
        _, _, _, stats = dev.match(pairs, count=count, batch_size=batch, epsilon=0.0, alpha=1.0, evaluator=omk.EVAL_NET)
        entry = {"games": 2 * pairs, "move_lists_identical": identical, "moves": sum(len(m) for m in ref["host"]),
                 "device_call_stats": stats, "device_call_h2d_bytes": dev.transfer_bytes[0] - h2d0}
        for name, v in runs.items():
            s = [x["s"] for x in v]
            entry[name] = {"runs": v, "median_s": float(np.median(s)), "spread_s": float(np.max(s) - np.min(s))}
        entry["host_median_over_device_median"] = entry["host"]["median_s"] / entry["device"]["median_s"]
        res["shapes"].append(entry)
        for c in (left, right, dev):
            c.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not all(e["move_lists_identical"] for e in res["shapes"]):
        raise SystemExit("the host and device matches played different games")
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", default="100,1024", help="comma-separated game counts (half of them each side opens)")
    ap.add_argument("--count", type=int, default=800)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    main(games=[int(x) for x in a.games.split(",")], count=a.count, rounds=a.rounds, out=a.out)
