#!/usr/bin/env python
"""One AlphaZero iteration (BASELINE configs[4]): sharded self-play on every GPU with the transitions streamed to the
host replay memory (no collective on that path), then the trainer's gradient steps through the C ABI (omk_train_step)
with ONE NCCL all-reduce of the 22.6 MB gradient per step, the weights going live for the next self-play phase inside
the same call.  Single GPU: `python tools/iteration.py`; N GPUs of one node:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/iteration.py
Defaults are the reference trainer's: 800 simulations per move here (BASELINE) in rounds of 16, minibatch 128
(src/config.rs:89-100).  Prints one JSON line (rank 0): self-play throughput, the trainer step time with and without
the all-reduce (device timed, max over ranks), the all-reduce of the same 22.6 MB timed alone, and the losses.
With --device-replay the replay memory lives in the context instead (omk_replay_reset before omk_selfplay_begin): the
self-play driver feeds it on the device, no transition is streamed, and the whole training phase -- sampling, encoding and
the steps -- is ONE omk_train_replay call, timed as such (train_phase_s); every rank samples its own replay memory.
With --evaluate EPISODES the trained weights then play the trainer's evaluation against the naive player
(src/trainer.rs:487-603) as ONE omk_eval_naive call on trees past the self-play driver's 2 * games, so the driver stays
active for the next iteration; it reports eval_phase_s and the naive player's wins, the model's wins and the draws.
With --gate GAMES the network is copied into the context's opponent before the training phase (omk_opponent_from_net), and
after training the trained network plays GAMES games against that snapshot at the benchmark's constants (800 simulations,
batch 8, epsilon 0, alpha 1; benchmark/src/main.rs) as ONE omk_match call on trees past the driver's and the evaluation's:
AlphaZero's gating question, whether this iteration's network beats the last one.
With --device-replay --score the rows this phase's self-play committed, which no step has trained on yet, are a held-out
set: the network's loss terms on them (policy cross-entropy, value MSE, their sum, and top-1 agreement of the policy with
the visit distribution) are measured by ONE omk_replay_score call before the training phase and one after it, and with
--gate also for the snapshot; no game is played.  Under torchrun every rank scores its own memory and the means are
combined weighted by rows.
With --device-replay --state PATH the run is resumable across processes: if PATH exists, the weights, the Adadelta
accumulators and the replay memory are loaded from it (run_state.load) instead of a random initialisation, the context gets
the saved seed and the trainer's sampler streams continue at the saved step; after the training phase (and the evaluation
and the gating match, if they run) the state is saved to PATH again.  Running the command K times continues one run over K
processes.  Under torchrun every rank keeps its own file, PATH.rank{r}, and a file written with another world size is
refused.  It reports state_load_s and state_save_s.
With --device-replay --gate GAMES --gated the run acts on the gating answer, as AlphaGo Zero does: the context's opponent
(model slot 1) holds the BEST network, self-play reads it (omk_selfplay_set_model(1)) and the network (slot 0) is the
candidate the trainer keeps changing.  A fresh run starts with best = the initial network; with --state the best is saved
and resumed with the rest, and a state file without one is refused.  No snapshot is taken before training: the gating match
is the candidate against the best, and if the candidate's score (wins + draws / 2) / games over all ranks reaches
--promote-at (default 0.55) every rank copies it into slot 1, so the next self-play phase plays the new best.  A resumed
gated run does not reuse the saved context seed: it derives the next one from it and the iteration
(sharding.iteration_seed), because a kept best network with the same random streams would replay the previous process's
games and append them to the replay memory again.  It reports gate_score and promoted, the gating match's wins as
gate_trained_wins / gate_best_wins, and --score labels slot 1's terms "best"."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_PARAMS = 5_643_250


def run(games_per_gpu=1024, plies=12, count=800, batch=16, steps=20, minibatch=128, seed=0, quiet=False, gather=False, torch_step=False,
        device_replay=False, replay_capacity=600_000, evaluate=0, gate=0, score=False, state=None, gated=False, promote_at=0.55):
    omk = importlib.import_module("omok-ai_b200")
    run_state = importlib.import_module("omok-ai_b200.run_state")
    trainer = importlib.import_module("omok-ai_b200.trainer")
    sharding = importlib.import_module("omok-ai_b200.sharding")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if device_replay and (torch_step or gather):
        raise ValueError("--device-replay trains through omk_train_replay: it excludes --torch-step and --gather")
    if score and not device_replay:
        raise ValueError("--score reads the device replay memory: it needs --device-replay")
    if gate and gate < 2:
        raise ValueError("--gate GAMES needs at least 2 games: one opened by each side")
    if state and not device_replay:
        raise ValueError("--state saves the device replay memory: it needs --device-replay")
    if gated and not (device_replay and gate):
        raise ValueError("--gated acts on the gating match of the device-replay run: it needs --device-replay and --gate GAMES")
    state_path = (f"{state}.rank{rank}" if world > 1 else state) if state else None
    resume = None
    if state_path and os.path.exists(state_path):
        resume = run_state.read_meta(state_path)
        if resume["world"] != world:
            raise ValueError(f"{state_path} was written by a run of {resume['world']} ranks, this one has {world}")
        if gated and not resume.get("best"):
            raise ValueError(f"{state_path} holds no best network: it was not written by a --gated run")
    my_games = games_per_gpu
    ctx_seed = resume["seed"] if resume else sharding.rank_seed(seed, rank)
    if resume and gated:                            # fresh self-play streams: the best network may be the one that played last time
        ctx_seed = sharding.iteration_seed(ctx_seed, resume["iteration"] + 1)
    ctx = omk.Context(device=local, capacity_envs=4, capacity_trees=2 * my_games + evaluate + 4 * (gate // 2),
                      capacity_nodes=4096, seed=ctx_seed)
    load_s = None
    if resume:                                      # weights, accumulators and replay memory of the last iteration
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_state.load(ctx, state_path, world=world, rank=rank, best_slot=1 if gated else None)
        load_s = time.perf_counter() - t0
    else:
        ctx.net_init_random(seed)                   # identical weights on every rank
        if gated:
            ctx.opponent_from_net()                 # the best network so far: the initial one
    if torch_step:
        step = trainer.TrainStep(ctx.net_get_params(), device=f"cuda:{local}")
    else:
        uid = None
        if world > 1:                               # rank 0's NCCL unique id reaches the others over the process group
            t = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                t.copy_(torch.frombuffer(bytearray(ctx.train_comm_unique_id()), dtype=torch.uint8))
            dist.broadcast(t, src=0)
            uid = bytes(t.cpu().numpy().tobytes())
        step = trainer.AbiTrainStep(ctx, world=world, rank=rank, unique_id=uid)
        if resume:
            step.steps = resume["step"]             # the sampler streams continue where the saved run stopped
    if device_replay:
        if not resume:
            ctx.replay_reset(replay_capacity)       # before selfplay_begin: the driver feeds the replay that exists then
        return _run_device_replay(ctx, step, sharding, dist, rank, world, games_per_gpu, plies, count, batch, steps, minibatch,
                                  seed, quiet, evaluate, gate, score, state_path, resume, load_s, gated, promote_at)
    mem = trainer.ReplayMemory(capacity=600_000, seed=seed + rank)

    # ---- self-play phase: per-GPU game pools, transitions streamed to the host (pinned ring inside the library) ----
    ctx.selfplay_begin(my_games, count, batch, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    ctx.selfplay_run(2, profile=0, want_transitions=False)        # warm-up: allocations, lane set-up
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    stats, boards, policy, status, _ = ctx.selfplay_run(plies, profile=0, want_transitions=True)
    sp_s = time.perf_counter() - t0
    merged = None
    merge_s = 0.0
    if gather and dist:                             # config 4's host replay merge: every rank's block lands on rank 0
        t1 = time.perf_counter()
        merged = sharding.gather_replay(torch.from_numpy(boards).cuda(), torch.from_numpy(policy).cuda(), torch.from_numpy(status).cuda())
        torch.cuda.synchronize()
        merge_s = time.perf_counter() - t1
    episodes, _carry = trainer.split_episodes(boards, policy, status)   # unfinished tails wait for the next phase (trainer.rs:206-215)
    for b, p, z in episodes:
        mem.add_episode(b, p, z)
    if len(mem) == 0:                               # too few plies for any game to end: train on the raw transitions (benchmark shape only)
        flat_b, flat_p = boards.reshape(-1, 81), policy.reshape(-1, 81)
        mem.add_episode(flat_b[: 4 * minibatch], flat_p[: 4 * minibatch], 0.0)

    # ---- training phase: data parallel over the minibatch, one gradient all-reduce per step ----
    if gate:
        ctx.opponent_from_net()                     # the snapshot the trained network has to beat
    per_rank = max(1, minibatch // world)
    batches = [mem.sample(per_rank) for _ in range(steps + 2)]
    enc = [(trainer.encode_nn_input(b, t), pi, z) for b, t, pi, z in batches]

    def timed(fn, n_warm=2):
        for i in range(n_warm):
            fn(i)
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        t = time.perf_counter()
        out = [fn(n_warm + i) for i in range(steps)]
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3 / steps, out

    step_ms, losses = timed(lambda i: step.train(*enc[i]))
    # the same 22.6 MB all-reduce alone (torch.distributed over the same NCCL / NVLink path), CUDA-event timed
    ar_ms = 0.0
    if dist:
        g = torch.zeros(N_PARAMS, dtype=torch.float32, device="cuda")
        for _ in range(3):
            dist.all_reduce(g)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        dist.barrier()
        e0.record()
        for _ in range(20):
            dist.all_reduce(g)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / 20
    # ... and the step without the collective (communicator detached): the difference is what data parallelism costs
    local_ms = step_ms
    if dist and not torch_step:
        ctx.train_comm_destroy()
        local_ms, _ = timed(lambda i: step.train(*enc[i]), n_warm=1)
    if torch_step:
        step.sync_to(ctx)
    b, t = batches[-1][0], batches[-1][1]
    p, _ = ctx.net_eval_images(trainer.encode_nn_input(b[:4], t[:4]))
    times, work = sharding.reduce_measurements({"step_ms": step_ms, "local_ms": local_ms, "selfplay_s": sp_s, "allreduce_ms": ar_ms,
                                                "merge_s": merge_s, "selfplay_gpu_ms": float(stats.gpu_ms)},
                                               {"sims": int(stats.simulations), "positions": int(stats.positions),
                                                "episodes": len(episodes), "replay": len(mem), "d2h": int(stats.d2h_bytes)},
                                               device="cuda" if dist else "cpu")
    out = {"config": "AlphaZero iteration (BASELINE configs[4])", "n_gpus": world, "games_per_gpu": games_per_gpu, "plies": plies,
           "sims_per_move": count, "selfplay_sims_per_s": work["sims"] / times["selfplay_s"],
           "selfplay_positions_per_s": work["positions"] / times["selfplay_s"], "selfplay_wall_s": times["selfplay_s"],
           "selfplay_gpu_ms": times["selfplay_gpu_ms"], "transitions_streamed_to_host": True, "d2h_bytes": work["d2h"],
           "replay_merge_s": times["merge_s"] if gather else None, "merged_games_on_rank0": int(merged[0].shape[1]) if merged else None,
           "episodes_finished": work["episodes"], "replay_transitions": work["replay"], "train_steps": steps,
           "global_minibatch": per_rank * world, "train_step": "omk_train_step (C ABI, fp32 CUDA kernels)" if not torch_step else "PyTorch autograd",
           "train_step_ms": times["step_ms"], "train_step_ms_without_allreduce": times["local_ms"],
           "allreduce_22.6MB_alone_ms": times["allreduce_ms"], "allreduce_bytes_per_step": N_PARAMS * 4 if world > 1 else 0,
           "first_loss": losses[0][2], "last_loss": losses[-1][2], "policy_sums_to_one": bool(abs(float(p[0].sum()) - 1) < 1e-3)}
    if evaluate:
        out.update(_evaluate(ctx, evaluate, 2 * my_games, count, batch, seed))
    if gate:
        out.update(_gate(ctx, gate, 2 * my_games + evaluate))
    if rank == 0 and not quiet:
        print(json.dumps(out), flush=True)
    ctx.close()
    if dist:
        dist.destroy_process_group()
    return out


def _evaluate(ctx, episodes, first_tree, count, batch, seed):
    """The evaluation phase: the current weights against the naive player, one omk_eval_naive call."""
    omk = importlib.import_module("omok-ai_b200")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    (black, white, draw), _, _, stats = ctx.eval_naive(episodes, count=count, batch_size=batch, epsilon=0.25, alpha=0.03,
                                                       evaluator=omk.EVAL_NET, seed=seed, first_tree=first_tree)
    return {"eval_episodes": episodes, "eval_phase_s": time.perf_counter() - t0, "eval_naive_wins": black, "eval_model_wins": white,
            "eval_draws": draw, "eval_moves": stats["moves"], "eval_host_syncs": stats["host_syncs"], "eval_gpu_ms": stats["gpu_ms"]}


def _gate(ctx, games, first_tree, opponent="snapshot"):
    """The gating match: the trained network against the opponent (the snapshot taken before training, or the best network
    of a gated run), one omk_match call at the benchmark's constants."""
    omk = importlib.import_module("omok-ai_b200")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    (net, snap, draw), _, _, stats = ctx.match(games // 2, first_tree=first_tree, count=800, batch_size=8, epsilon=0.0, alpha=1.0,
                                               evaluator=omk.EVAL_NET)
    return {"gate_games": 2 * (games // 2), "gate_phase_s": time.perf_counter() - t0, "gate_trained_wins": net, f"gate_{opponent}_wins": snap,
            "gate_draws": draw, "gate_moves": stats["moves"], "gate_host_syncs": stats["host_syncs"], "gate_gpu_ms": stats["gpu_ms"]}


SCORE_TERMS = ("p_loss", "v_loss", "loss", "top1")


def _score(ctx, slot, first, n):
    """Model slot `slot`'s loss terms on the logical replay rows [first, first + n): one omk_replay_score call, and its wall
    time."""
    if n == 0:
        return (0.0,) * 4, 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    means = ctx.replay_score(slot, first=first, n=n)
    return means, time.perf_counter() - t0


def _run_device_replay(ctx, step, sharding, dist, rank, world, games, plies, count, batch, steps, minibatch, seed, quiet,
                       evaluate=0, gate=0, score=False, state_path=None, resume=None, load_s=None, gated=False, promote_at=0.55):
    omk = importlib.import_module("omok-ai_b200")
    run_state = importlib.import_module("omok-ai_b200.run_state")
    trainer = importlib.import_module("omok-ai_b200.trainer")
    rows_at_start = ctx.replay_info()[0]
    if gated:
        ctx.selfplay_set_model(1)                   # the best network (slot 1) generates the self-play data
    ctx.selfplay_begin(games, count, batch, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    ctx.selfplay_run(2, profile=0, want_transitions=False)        # warm-up: allocations, lane set-up
    if dist:
        dist.barrier()
    added_before = ctx.replay_info()[1]
    t0 = time.perf_counter()
    stats = ctx.selfplay_run(plies, profile=0, want_transitions=False)[0]
    sp_s = time.perf_counter() - t0
    rows, added, episodes = ctx.replay_info()
    if rows == 0:
        raise SystemExit("no game finished during self-play, so the replay memory is empty: raise --plies")
    fresh = min(rows, added - added_before)         # this phase's rows: the newest, not trained on yet
    scores = {}
    if score:
        scores["before"] = _score(ctx, 0, rows - fresh, fresh)
    per_rank = max(1, minibatch // world)
    sampler_seed = resume["sampler_seed"] if resume else sharding.rank_seed(seed, rank)   # every rank samples its own replay memory
    if gate and not gated:
        ctx.opponent_from_net()                     # the snapshot the trained network has to beat
    step.train_replay(2, per_rank, sampler_seed)   # warm-up: training workspace, split-K scratch
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t1 = time.perf_counter()
    losses = step.train_replay(steps, per_rank, sampler_seed)   # the whole training phase: one call, one synchronisation
    phase_s = time.perf_counter() - t1
    h2d, _ = ctx.transfer_bytes
    if score:
        scores["after"] = _score(ctx, 0, rows - fresh, fresh)
        if gate:
            scores["best" if gated else "snapshot"] = _score(ctx, 1, rows - fresh, fresh)
    score_times = {f"score_{k}_s": s for k, (_, s) in scores.items()}
    score_work = {f"score_{k}_{t}": float(x) * fresh for k, (m, _) in scores.items() for t, x in zip(SCORE_TERMS, m)}
    if scores:
        score_work["score_rows"] = fresh
    times, work = sharding.reduce_measurements({"train_phase_s": phase_s, "selfplay_s": sp_s, "selfplay_gpu_ms": float(stats.gpu_ms),
                                                **score_times},
                                               {"sims": int(stats.simulations), "positions": int(stats.positions),
                                                "rows": rows, "episodes": episodes, **score_work},
                                               device="cuda" if dist else "cpu")
    out = {"config": "AlphaZero iteration (BASELINE configs[4]), device replay memory", "n_gpus": world, "games_per_gpu": games,
           "plies": plies, "sims_per_move": count, "selfplay_sims_per_s": work["sims"] / times["selfplay_s"],
           "selfplay_positions_per_s": work["positions"] / times["selfplay_s"], "selfplay_wall_s": times["selfplay_s"],
           "selfplay_gpu_ms": times["selfplay_gpu_ms"], "transitions_streamed_to_host": False,
           "replay_capacity_per_gpu": ctx.replay_capacity, "replay_rows": work["rows"], "replay_episodes": work["episodes"],
           "train_steps": steps, "global_minibatch": per_rank * world, "train_step": "omk_train_replay (C ABI, fp32 CUDA kernels)",
           "train_phase_s": times["train_phase_s"], "train_step_ms": times["train_phase_s"] * 1e3 / steps,
           "first_loss": float(losses[0, 2]), "last_loss": float(losses[-1, 2]), "h2d_bytes_total": h2d}
    if scores:  # means over every rank's rows; the wall time of the slowest rank's call
        n_scored = work["score_rows"]
        out["score_rows"] = n_scored
        for k in scores:
            out[f"score_{k}"] = {t: work[f"score_{k}_{t}"] / n_scored if n_scored else float("nan") for t in SCORE_TERMS}
            out[f"score_{k}_s"] = times[f"score_{k}_s"]
    if evaluate:
        out.update(_evaluate(ctx, evaluate, 2 * games, count, batch, seed))
    if gate:
        g = _gate(ctx, gate, 2 * games + evaluate, "best" if gated else "snapshot")
        out.update(g)
        if gated:  # every rank decides on the same sums, so the best stays identical across ranks
            _, summed = sharding.reduce_measurements({"gate_phase_s": g["gate_phase_s"]},
                                                     {k: g[k] for k in ("gate_trained_wins", "gate_best_wins", "gate_draws")},
                                                     device="cuda" if dist else "cpu")
            gate_score, promoted = trainer.gate_decision(
                [(summed["gate_trained_wins"], summed["gate_best_wins"], summed["gate_draws"])], promote_at)
            if promoted:
                ctx.opponent_from_net()             # the candidate becomes the best; the driver's restart prior follows
            out.update({"gate_score": gate_score, "promote_at": promote_at, "promoted": promoted})
    if state_path:
        iteration = resume["iteration"] + 1 if resume else 1
        t0 = time.perf_counter()
        run_state.save(ctx, state_path, seed=ctx.seed, sampler_seed=sampler_seed, step=step.steps, iteration=iteration, world=world,
                       rank=rank, best_slot=1 if gated else None)
        save_s = time.perf_counter() - t0
        st, sw = sharding.reduce_measurements({"state_load_s": load_s or 0.0, "state_save_s": save_s}, {"rows_at_start": rows_at_start},
                                              device="cuda" if dist else "cpu")
        out.update({"iteration": iteration, "replay_rows_at_start": sw["rows_at_start"],
                    "state_load_s": st["state_load_s"] if resume else None, "state_save_s": st["state_save_s"]})
    if rank == 0 and not quiet:
        print(json.dumps(out), flush=True)
    ctx.close()
    if dist:
        dist.destroy_process_group()
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--games-per-gpu", type=int, default=1024)
    ap.add_argument("--plies", type=int, default=12)
    ap.add_argument("--count", type=int, default=800)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--minibatch", type=int, default=128)
    ap.add_argument("--gather", action="store_true", help="merge every rank's transitions on rank 0 (config 4's host replay buffer)")
    ap.add_argument("--torch-step", action="store_true", help="PyTorch-autograd step instead of omk_train_step")
    ap.add_argument("--device-replay", action="store_true",
                    help="replay memory on the device, fed by the self-play driver; the training phase is one omk_train_replay call")
    ap.add_argument("--replay-capacity", type=int, default=600_000, help="rows of the device replay memory per GPU (src/config.rs: 600 000)")
    ap.add_argument("--evaluate", type=int, default=0, metavar="EPISODES",
                    help="after training, play EPISODES games against the naive player on the device (omk_eval_naive)")
    ap.add_argument("--gate", type=int, default=0, metavar="GAMES",
                    help="after training, play GAMES games of the trained network against its pre-training snapshot (omk_match)")
    ap.add_argument("--score", action="store_true",
                    help="with --device-replay: the loss terms of the network on this phase's new replay rows before and after "
                         "training (and of the snapshot with --gate), one omk_replay_score call each")
    ap.add_argument("--state", metavar="PATH",
                    help="with --device-replay: resume from PATH if it exists (weights, Adadelta accumulators, replay memory) and "
                         "save there after the iteration (PATH.rank{r} per rank under torchrun)")
    ap.add_argument("--gated", action="store_true",
                    help="with --device-replay --gate GAMES: the best network (slot 1) plays self-play and is replaced by the "
                         "trained one when its gating score reaches --promote-at")
    ap.add_argument("--promote-at", type=float, default=0.55, metavar="X",
                    help="with --gated: the candidate's score (wins + draws / 2) / games that promotes it (AlphaGo Zero: 0.55)")
    a = ap.parse_args()
    run(games_per_gpu=a.games_per_gpu, plies=a.plies, count=a.count, steps=a.steps, minibatch=a.minibatch, gather=a.gather, torch_step=a.torch_step,
        device_replay=a.device_replay, replay_capacity=a.replay_capacity, evaluate=a.evaluate,
        gate=a.gate, score=a.score, state=a.state, gated=a.gated, promote_at=a.promote_at)
