#!/usr/bin/env python
"""Rate up to 16 checkpoints on one scale whose zero is the naive player (DESIGN.md 4): the files (`model_io` format) go
into model slots 0 .. K-1 of one context, and one omk_tournament_naive call plays the benchmark's arena (half the games each
side opening, `count` simulations per move in rounds of 8, epsilon 0, alpha 1) between every pair of the K + 1 participants.
`arena.ratings` then rates the naive player at 0 Elo, so ratings from separate runs of this tool, with the same seed and
settings, share their zero.  Prints one line per file: its Elo and its score against the naive player (wins, losses,
draws, and (wins + draws / 2) / games).  With no files it rates `--random` seeded random-init networks (omk_net_init_random
seeds 0 .. n-1), so it runs anywhere there is a GPU.
    python tools/rate_checkpoints.py [FILE ...] [--games 100 --count 800 --seed 0 --nodes 4096 --random 4]"""
from __future__ import annotations

import argparse
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(files=(), games=100, count=800, batch=8, seed=0, nodes=4096, random_models=4, quiet=False):
    omk = importlib.import_module("omok-ai_b200")
    arena = importlib.import_module("omok-ai_b200.arena")
    model_io = importlib.import_module("omok-ai_b200.model_io")
    files = list(files)
    if len(files) > 16:
        raise SystemExit("at most 16 checkpoints fit in one context's model slots")
    if not files and not 1 <= random_models <= 16:
        raise SystemExit("--random must be in 1 .. 16 when no checkpoint file is given")
    if files:
        names = files
        weights = [model_io.load(f)[1] for f in files]
    else:
        names = [f"random-init seed {s}" for s in range(random_models)]
        weights = []
        for s in range(random_models):
            c = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=seed)
            c.net_init_random(s)
            weights.append(c.net_get_params())
            c.close()
    k = len(weights)
    n = k + 1
    pairs = games // 2
    P = n * (n - 1) // 2
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs * P, capacity_nodes=nodes, seed=seed)
    ctx.net_load_params(weights[0])
    for s in range(1, k):
        ctx.model_load_params(s, weights[s])
    table = arena.play_tournament_naive_device(ctx, list(range(k)), seed=seed, game_count=2 * pairs, count=count, batch_size=batch)
    ctx.close()
    elo = arena.ratings(table, n)
    rows = []
    for i, name in enumerate(names):
        naive_wins, wins, draws = (int(x) for x in table[i])  # pairing i is (naive, slot i): the naive player is left
        rows.append({"file": name, "elo": float(elo[i + 1]), "wins": wins, "losses": naive_wins, "draws": draws,
                     "score": (wins + 0.5 * draws) / (2 * pairs)})
    if not quiet:
        print(f"{k} models and the naive player (0 Elo), {2 * pairs} games per pairing, {count} simulations per move, seed {seed}")
        for r in rows:
            print(f"{r['elo']:9.1f} Elo  vs naive {r['wins']:4d} W {r['losses']:4d} L {r['draws']:4d} D  score {r['score']:.3f}  {r['file']}")
    return {"table": table.tolist(), "ratings": [float(x) for x in elo], "models": rows}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("files", nargs="*", help="checkpoint files (model_io format), at most 16")
    ap.add_argument("--games", type=int, default=100, help="games per pairing (half of them each side opens)")
    ap.add_argument("--count", type=int, default=800, help="simulations per move")
    ap.add_argument("--seed", type=int, default=0, help="the context's seed and the naive player's")
    ap.add_argument("--nodes", type=int, default=4096, help="node slots per tree")
    ap.add_argument("--random", type=int, default=4, help="random-init networks to rate when no file is given")
    a = ap.parse_args()
    main(a.files, games=a.games, count=a.count, seed=a.seed, nodes=a.nodes, random_models=a.random)
