#!/usr/bin/env python
"""Self-play with the driver on the network (slot 0) vs on model slot 1 holding the same weights, on one GPU.  Prints one
JSON line with the card's name and power limit.

One context, `games` games x `count` simulations a move in rounds of 16 (the iteration's shape), random-init network copied
into slot 1 (omk_model_from_net).  After `warm` untimed plies, the two arms alternate `rounds` times on the same running
games: omk_selfplay_set_model(slot), then one omk_selfplay_run of `plies` plies, timed on the host around the call (which
ends in a synchronisation) and on the device (the call's gpu_ms).  Both arms evaluate with the same weights, so the games
are those of a driver that never switched.
    python tools/selfplay_slot_time.py [--games 1024 --count 800 --plies 8 --rounds 6 --out FILE]"""
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


def main(games=1024, count=800, batch=16, plies=8, rounds=6, warm=4, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    res = {"tool": "selfplay_slot_time", **card(), "games": games, "sims_per_move": count, "batch": batch, "plies_per_run": plies,
           "rounds": rounds, "network": "random init (omk_net_init_random seed 0), copied into slot 1"}
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * games, capacity_nodes=4096, seed=seed)
    ctx.net_init_random(0)
    ctx.model_from_net(1)
    ctx.selfplay_begin(games, count, batch, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    ctx.selfplay_run(warm, want_transitions=False)  # allocations, lane set-up

    def arm(slot):
        ctx.selfplay_set_model(slot)
        t = time.perf_counter()
        stats = ctx.selfplay_run(plies, want_transitions=False)[0]
        return (time.perf_counter() - t) * 1e3 / plies, stats.gpu_ms / plies, stats.simulations

    times = {0: [], 1: []}
    for r in range(rounds):
        for slot in ((0, 1) if r % 2 == 0 else (1, 0)):
            times[slot].append(arm(slot))
    for slot, v in times.items():
        wall, gpu = [x[0] for x in v], [x[1] for x in v]
        res[f"slot{slot}"] = {"ms_per_ply": wall, "gpu_ms_per_ply": gpu, "median_ms_per_ply": float(np.median(wall)),
                              "spread_ms_per_ply": float(np.max(wall) - np.min(wall)), "median_gpu_ms_per_ply": float(np.median(gpu)),
                              "simulations_per_s": float(sum(x[2] for x in v) / (sum(wall) * plies / 1e3))}
    res["slot1_median_over_slot0_median"] = res["slot1"]["median_ms_per_ply"] / res["slot0"]["median_ms_per_ply"]
    ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--count", type=int, default=800, help="simulations per move")
    ap.add_argument("--plies", type=int, default=8, help="plies per timed run")
    ap.add_argument("--rounds", type=int, default=6, help="timed runs per arm, alternated")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    main(games=a.games, count=a.count, plies=a.plies, rounds=a.rounds, out=a.out)
