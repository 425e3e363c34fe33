#!/usr/bin/env python
"""The evaluation phase of an iteration (src/trainer.rs:487-603: the model against the naive player) on one GPU, driven
from the host and on the device, with the random-init network.  Prints one JSON line with the card's name and power limit.

  host path    arena.play_against_naive_player: per move pair a Python loop over the live games and about eight entry
               points (pool_get_envs, env_set + env_step on 162 candidate boards per game, ensure_action, play, search,
               sample, play), each with its own synchronisation
  device path  arena.play_against_naive_player_device: one omk_eval_naive call, one 4-byte read-back per half-move

The two paths are alternated in one process, `rounds` times each, after one untimed run of each (allocations, lanes).
Their naive players draw from different generators (numpy / the specified stream), so their games differ; the W/L/D of
every run is reported next to its time.
    python tools/eval_phase_time.py [--shapes 100x800,1024x800 --rounds 3 --out FILE]"""
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


def main(shapes=((100, 800), (1024, 800)), batch=16, epsilon=0.25, alpha=0.03, rounds=3, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    arena = importlib.import_module("omok-ai_b200.arena")
    res = {"tool": "eval_phase_time", **card(), "batch_size": batch, "epsilon": epsilon, "alpha": alpha, "rounds": rounds,
           "network": "random init (omk_net_init_random)", "shapes": []}
    for episodes, count in shapes:
        host = omk.Context(device=0, capacity_envs=162 * episodes, capacity_trees=episodes, capacity_nodes=4096, seed=seed)
        dev = omk.Context(device=0, capacity_envs=1, capacity_trees=episodes, capacity_nodes=4096, seed=seed)
        for c in (host, dev):
            c.net_init_random(seed)
        kw = dict(episode_count=episodes, count=count, batch_size=batch, epsilon=epsilon, alpha=alpha, evaluator=omk.EVAL_NET)
        paths = {"host": lambda r: arena.play_against_naive_player(host, seed=r, **kw),
                 "device": lambda r: arena.play_against_naive_player_device(dev, seed=r, **kw)}
        for fn in paths.values():
            fn(10**6)  # untimed
        runs = {k: [] for k in paths}
        for r in range(rounds):
            for name in (paths if r % 2 == 0 else list(paths)[::-1]):
                t0 = time.perf_counter()
                wld = paths[name](r)
                runs[name].append({"s": time.perf_counter() - t0, "black_naive_wins": wld[0], "white_model_wins": wld[1], "draws": wld[2]})
        h2d0 = dev.transfer_bytes[0]
        _, _, _, stats = dev.eval_naive(episodes, count=count, batch_size=batch, epsilon=epsilon, alpha=alpha, evaluator=omk.EVAL_NET,
                                        seed=rounds)
        entry = {"episodes": episodes, "sims_per_move": count, "device_call_stats": stats,
                 "device_call_h2d_bytes": dev.transfer_bytes[0] - h2d0}
        for name, v in runs.items():
            s = [x["s"] for x in v]
            entry[name] = {"runs": v, "median_s": float(np.median(s)), "spread_s": float(np.max(s) - np.min(s))}
        entry["host_median_over_device_median"] = entry["host"]["median_s"] / entry["device"]["median_s"]
        res["shapes"].append(entry)
        host.close()
        dev.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="100x800,1024x800", help="comma-separated EPISODESxSIMULATIONS")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    shapes = [tuple(int(x) for x in s.split("x")) for s in a.shapes.split(",")]
    main(shapes=shapes, rounds=a.rounds, out=a.out)
