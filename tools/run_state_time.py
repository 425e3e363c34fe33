#!/usr/bin/env python
"""Save and load time of a full run state (run_state.save / run_state.load) on one GPU: a 600 000-row device replay memory
(src/config.rs) filled by the self-play driver, the weights and the Adadelta accumulators after a few training steps.  Prints
one JSON line with the card's name and power limit.

  save  run_state.save: omk_net_get_params, omk_train_get_optimizer, omk_replay_get in chunks, np.savez to a file, fsync
  load  run_state.load into a fresh context: np.load, omk_net_load_params, omk_train_set_optimizer, omk_replay_reset,
        omk_replay_append

The file goes to a temporary directory (or --dir) and is removed at the end; its disk is part of the numbers.  Save and load
alternate `rounds` times; after each load the rows, weights and accumulators must equal the saved context's bit for bit.
    python tools/run_state_time.py [--rows 600000 --games 1024 --count 16 --rounds 3 --dir DIR --out FILE]"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from train_phase_time import card  # noqa: E402


def main(rows=600_000, games=1024, count=16, rounds=3, seed=0, directory=None, out=None):
    omk = importlib.import_module("omok-ai_b200")
    run_state = importlib.import_module("omok-ai_b200.run_state")
    res = {"tool": "run_state_time", **card(), "rows": rows, "selfplay_games": games, "sims_per_move": count, "rounds": rounds}
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * games, capacity_nodes=1024, seed=seed)
    ctx.net_init_random(0)
    ctx.replay_reset(rows)
    ctx.selfplay_begin(games, count, 8, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    for _ in range(200):
        if ctx.replay_info()[0] == rows:
            break
        ctx.selfplay_run(40, want_transitions=False)
    n, added, episodes = ctx.replay_info()
    if n != rows:
        raise SystemExit(f"the replay memory holds {n} of {rows} rows after self-play")
    ctx.train_replay(1, 0, 5, 128)  # non-zero accumulators
    want = (ctx.replay_get(np.arange(n)), ctx.net_get_params(), ctx.train_get_optimizer())
    tmp = tempfile.mkdtemp(prefix="run_state_time_", dir=directory)
    path = os.path.join(tmp, "state")
    times = {"save": [], "load": []}
    same = True
    try:
        for _ in range(rounds):
            t = time.perf_counter()
            run_state.save(ctx, path, seed=seed, sampler_seed=1, step=5, iteration=1, world=1, rank=0)
            times["save"].append(time.perf_counter() - t)
            fresh = omk.Context(device=0, capacity_envs=1, capacity_trees=4, capacity_nodes=64, seed=seed)
            t = time.perf_counter()
            run_state.load(fresh, path)
            times["load"].append(time.perf_counter() - t)
            got = (fresh.replay_get(np.arange(n)), fresh.net_get_params(), fresh.train_get_optimizer())
            same &= all(a.tobytes() == b.tobytes() for a, b in zip(want[0], got[0]))
            same &= all(a.tobytes() == b.tobytes() for a, b in zip(want[1], got[1]))
            same &= all(a.tobytes() == b.tobytes() for a, b in zip(want[2][0] + want[2][1], got[2][0] + got[2][1]))
            same &= fresh.replay_info() == (n, n, episodes)
            fresh.close()
        res["file_bytes"] = os.path.getsize(path)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    res.update({"rows_added": added, "episodes": episodes, "round_trip_bit_identical": bool(same)})
    for k, v in times.items():
        res[k] = {"wall_s": v, "median_wall_s": float(np.median(v)), "spread_wall_s": float(np.max(v) - np.min(v))}
    ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not same:
        raise SystemExit("a loaded state differs from the saved context")
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=600_000, help="replay capacity, filled to the brim (src/config.rs: 600 000)")
    ap.add_argument("--games", type=int, default=1024, help="self-play games that fill it")
    ap.add_argument("--count", type=int, default=16, help="simulations per self-play move")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--dir", default=None, help="directory of the temporary state file (default: the system's temporary directory)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    main(rows=a.rows, games=a.games, count=a.count, rounds=a.rounds, directory=a.dir, out=a.out)
