#!/usr/bin/env python
"""The trainer's loss terms of the network on a full device replay memory (600 000 rows, src/config.rs), two ways, on one
GPU.  Prints one JSON line with the card's name and power limit.

  device  one omk_replay_score call over all rows (rows == NULL: the range form)
  host    omk_replay_get of all rows, omk_net_eval of their boards (Player mode) in chunks of 16 384 rows, and the losses in
          numpy: p_loss = -sum pi log P, v_loss = (z - V)^2, top1 = argmax P == argmax pi

The memory is filled by the self-play driver (random-init network, `count` simulations a move) until it is full.  The two
arms are alternated `rounds` times after one untimed run of each (allocations); each timed run ends in a synchronisation.
The per-row losses must agree: p_loss to 1e-5 relative (absolutely below 1) on the rows where P >= 1e-30 on pi's support,
v_loss to 1e-6.
    python tools/replay_score_time.py [--rows 600000 --games 1024 --count 16 --rounds 3 --out FILE]"""
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

CHUNK = 16384


def main(rows=600_000, games=1024, count=16, rounds=3, seed=0, out=None):
    omk = importlib.import_module("omok-ai_b200")
    res = {"tool": "replay_score_time", **card(), "rows": rows, "selfplay_games": games, "sims_per_move": count, "rounds": rounds,
           "network": "random init (omk_net_init_random seed 0)", "host_chunk_rows": CHUNK}
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * games, capacity_nodes=1024, seed=seed)
    ctx.net_init_random(0)
    ctx.replay_reset(rows)
    ctx.selfplay_begin(games, count, 8, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    t0 = time.perf_counter()
    for _ in range(200):
        if ctx.replay_info()[0] == rows:
            break
        ctx.selfplay_run(40, want_transitions=False)
    n, added, episodes = ctx.replay_info()
    if n != rows:
        raise SystemExit(f"the replay memory holds {n} of {rows} rows after self-play")
    res.update({"fill_s": time.perf_counter() - t0, "rows_added": added, "episodes": episodes})

    def device():
        t = time.perf_counter()
        means, p, v, top1 = ctx.replay_score(0, first=0, n=n, per_row=True)
        return time.perf_counter() - t, (means, p, v, top1)

    def host():
        t = time.perf_counter()
        boards, turns, pi, z = ctx.replay_get(np.arange(n))
        P = np.empty((n, 81), np.float32)
        V = np.empty(n, np.float32)
        for a in range(0, n, CHUNK):
            P[a:a + CHUNK], V[a:a + CHUNK] = ctx.net_eval(boards[a:a + CHUNK], turns[a:a + CHUNK], mode=0)
        support = pi > 0
        p = -(pi.astype(np.float64) * np.log(np.where(support, P, 1.0).astype(np.float64))).sum(1)
        v = (z.astype(np.float64) - V.astype(np.float64)) ** 2
        top1 = (P.argmax(1) == pi.argmax(1)).astype(np.uint8)
        means = (p.mean(), v.mean(), p.mean() + v.mean(), top1.mean())
        usable = np.all(np.where(support, P >= 1e-30, True), axis=1)
        return time.perf_counter() - t, (means, p, v, top1, usable)

    arms = {"device": device, "host": host}
    ref = {k: fn()[1] for k, fn in arms.items()}  # untimed
    times = {k: [] for k in arms}
    for r in range(rounds):
        for k in (arms if r % 2 == 0 else list(arms)[::-1]):
            times[k].append(arms[k]()[0])
    (dm, dp, dv, dt), (hm, hp, hv, ht, usable) = ref["device"], ref["host"]
    p_err = np.abs(dp[usable] - hp[usable]) / np.maximum(np.abs(hp[usable]), 1.0)
    v_err = np.abs(dv - hv)
    agree = bool(p_err.max() <= 1e-5 and v_err.max() <= 1e-6)
    h2d0 = ctx.transfer_bytes[0]
    device()
    res.update({"device_h2d_bytes": ctx.transfer_bytes[0] - h2d0, "device_means": list(dm), "host_means": [float(x) for x in hm],
                "rows_compared_p_loss": int(usable.sum()), "max_p_loss_error": float(p_err.max()), "max_v_loss_error": float(v_err.max()),
                "top1_rows_differing": int((dt != ht).sum()), "per_row_losses_agree": agree})
    for k, v in times.items():
        res[k] = {"wall_s": v, "median_wall_s": float(np.median(v)), "spread_wall_s": float(np.max(v) - np.min(v)),
                  "median_rows_per_s": n / float(np.median(v))}
    res["host_median_over_device_median"] = res["host"]["median_wall_s"] / res["device"]["median_wall_s"]
    ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not agree:
        raise SystemExit("the device and host per-row losses differ")
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=600_000, help="replay capacity, filled to the brim (src/config.rs: 600 000)")
    ap.add_argument("--games", type=int, default=1024, help="self-play games that fill it")
    ap.add_argument("--count", type=int, default=16, help="simulations per self-play move")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    main(rows=a.rows, games=a.games, count=a.count, rounds=a.rounds, out=a.out)
