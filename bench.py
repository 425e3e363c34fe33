#!/usr/bin/env python
"""bench.py -- headline benchmark of the self-play hot path (BASELINE.json configs[2]).

Workload (per GPU): 1024 concurrent self-play games, two trees per game as in the reference trainer
(src/trainer.rs:86-94), 800 simulations per move in rounds of 16 per tree (epsilon 0.25, alpha 0.03,
Boltzmann(1.0) for the first 30 plies then Best), random-init residual policy/value network.
One "step" = one ply on every game = 1024 positions = 1024 x 800 simulations.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun: one process per GPU, per-GPU game pools, NO data-path collective
(games are independent units -> weak scaling); only the timing barrier / max-over-ranks uses NCCL.

The line's `value` is device-resident throughput (omk_selfplay_run, CUDA events) WITH the transition stream on: every
ply's positions (board, visit policy, action, status: 410 B each) leave for the host replay buffer through the pinned
ring inside the timed region (BASELINE configs[3]); `e2e` drives the same ply through the granular C-ABI calls a Rust
`alpha-zero` shim would make (host id/action buffers in, actions/policies/status out, every call synchronising) -- that
is the headline against the reference arm; its byte counts are the library's own transfer counters.
`--impl reference` times the CPU oracle (C restatement, all host cores) with the PyTorch-CPU fp32 network
standing in for TensorFlow-CPU, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import contextlib
import importlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAMES_PER_GPU = 1024
COUNT, BATCH, EPS, ALPHA, TEMP, TEMP_THRESHOLD = 800, 16, 0.25, 0.03, 1.0, 30
CAP_NODES = 4096
FLOP_FC0 = 2 * 10368 * 512
FLOP_TOWER = 2 * (81 * 3 * 128 + 3 * 81 * (128 * 32 + 9 * 32 + 32 * 32 + 32 * 128))
FLOP_POSITION = 15_906_240
CPU_SAMPLE_TREES = 64


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the network kernels, from the committed
    `ncu --set full` capture of this same workload (profiles/r01_ncu_traffic.json; tools/ncu_summary.py wrote it)."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        try:
            return {k: v["dram_bytes_per_launch"] for k, v in json.load(open(path)).items()}
        except Exception:
            continue
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [x.strip() for x in line.split(",")]))

    def mark_start(self):
        self.t0 = time.monotonic()

    def mark_end(self):
        self.t1 = time.monotonic()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        # samples taken inside the timed region; nvidia-smi needs up to a second to start on an 8-GPU box, so it is started
        # before the warm-up and, should a short region hold no sample, the nearest ones (+-1 s, same load) stand in
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        window = "timed region"
        if not rows:
            rows = [r for t, r in self.rows if t0 - 1.0 <= t <= t1 + 1.0]
            window = "within 1 s of the timed region (same workload running)"
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: CPU oracle + PyTorch-CPU fp32 network on the box's host cores
# --------------------------------------------------------------------------------------------------
def cpu_selfplay_sample(steps: int, warmup: int, trees: int = CPU_SAMPLE_TREES):
    """Each step: one ply (800 sims/move, rounds of 16) on `trees` concurrent trees, trainer semantics."""
    import numpy as np
    import torch

    from oracle import net_oracle, oracle as orc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    params = net_oracle.random_params(0)
    ev = orc.TorchEvaluator(params)
    games = trees
    black = [orc.Agent(ev, 0, 2 * g) for g in range(games)]
    white = [orc.Agent(ev, 0, 2 * g + 1) for g in range(games)]
    ply = [0] * games

    def one_ply():
        movers = [black[g] if ply[g] % 2 == 0 else white[g] for g in range(games)]
        others = [white[g] if ply[g] % 2 == 0 else black[g] for g in range(games)]
        sims = orc.execute(movers, COUNT, BATCH, EPS, ALPHA, ev, n_threads=cores)
        for g in range(games):
            act, _ = movers[g].sample_action(1 if ply[g] < TEMP_THRESHOLD else 0, TEMP)
            st = movers[g].play_action(act)
            others[g].ensure_action_exists(act, ev)
            others[g].play_action(act)
            if st != 0:
                black[g], white[g], ply[g] = orc.Agent(ev, 0, 2 * g), orc.Agent(ev, 0, 2 * g + 1), 0
            else:
                ply[g] += 1
        return sims

    for _ in range(warmup):
        one_ply()
    t0 = time.perf_counter()
    sims = 0
    for _ in range(steps):
        sims += one_ply()
    dt = time.perf_counter() - t0
    return {"sims": sims, "positions": steps * games, "seconds": dt, "cores": cores, "trees": trees,
            "nn_positions": ev.positions}


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps = args.steps
    warm = max(0, args.warmup)  # the same W untimed plies as the repo arm is asked for
    r = cpu_selfplay_sample(steps, warm)
    value = r["sims"] / r["seconds"]
    line = {
        "impl": "reference",
        "metric": "mcts_simulations_per_sec", "value": value, "unit": "simulations/s",
        "positions_per_sec": r["positions"] / r["seconds"],
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * r["seconds"] / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": reference_config(args.gpus, r["trees"]),
        "cpu_baseline": {"value": value, "unit": "simulations/s", "cores": r["cores"], "kind": "port",
                         "sample": f"{r['trees']} concurrent trees x {steps} plies x {COUNT} sims/move (rounds of {BATCH}); "
                                   "C oracle on all host cores + PyTorch-CPU fp32 network in place of TensorFlow-CPU"},
        "e2e": {"value": value, "unit": "simulations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_config(n_gpus, trees):
    """The reference arm runs a BOUNDED SAMPLE of the workload: `trees` concurrent games instead of 1024 per GPU (one
    ply of 1024 games is ~50 s of CPU work on 16 cores), everything else identical; its NN batches are trees x 16 rows."""
    cfg = workload_config(n_gpus)
    cfg["workload"] = (f"bounded sample of BASELINE configs[2] on the host CPU: {trees} concurrent games (of {GAMES_PER_GPU}) x {COUNT} "
                       f"sims/move, rounds of {BATCH}, eps {EPS}, alpha {ALPHA}, the same random-init network in PyTorch-CPU fp32; "
                       "trainer-shaped self-play (2 trees per game, ensure_action_exists + re-root each ply); C restatement of the "
                       "reference's Rust on all host cores (the Rust/TensorFlow binary cannot be built here)")
    # the structured keys keep naming the workload both arms are quoted on; what this arm actually ran is in `sample_*`
    cfg["sample_games"], cfg["sample_trees"], cfg["sample_nn_rows_per_call"] = trees, 2 * trees, trees * BATCH
    cfg["sample_parallelism"] = "one process, pthreads over trees (rayon stand-in) + PyTorch intra-op threads; rank 0 only"
    return cfg


def workload_config(n_gpus, games=GAMES_PER_GPU):
    which = "BASELINE configs[2]" if games == GAMES_PER_GPU else f"BASELINE configs[2] shape at {games} games per GPU"
    lanes = f"two search lanes (streams) of {games // 2} games each" if games >= 768 else "one search lane"
    return {"workload": f"{which}: batched MCTS, {games} concurrent trees per GPU x {COUNT} sims/move, "
                        f"rounds of {BATCH}, eps {EPS}, alpha {ALPHA}, random-init residual policy/value net; "
                        "trainer-shaped self-play (2 trees per game, ensure_action_exists + re-root each ply); every ply's "
                        "transitions (board, visit policy, action, status) stream to the host replay buffer inside the timed region",
            "games_per_gpu": games, "trees_per_gpu": 2 * games, "sims_per_move": COUNT,
            "nn_batch_per_tree": BATCH, "capacity_nodes": CAP_NODES,
            "parallelism": f"games sharded x{n_gpus}, no collective; per GPU {lanes}",
            "l2": "no flush: each network launch streams a 333 MB fc0 input (>> 126 MB L2) and ~2.9 GB of tree records are resident"}


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, games):
    """Writes each [games, ...] array as out_dir/<name>.npy in float32, with game_index.npy naming the games kept. Above
    DUMP_LIMIT_BYTES in all, a fixed seeded sample of games is kept, so two builds run with the same arguments write
    the same games."""
    import numpy as np

    per_game = 8 + sum(4 * (a.size // games) for a in arrays.values())  # float32 rows + the float64 index
    budget = DUMP_LIMIT_BYTES - 128 * (len(arrays) + 1)  # less one .npy header per file
    idx = np.arange(games)
    if games * per_game > budget:
        idx = np.sort(np.random.default_rng(0).choice(games, budget // per_game, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "game_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a[idx], dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=GAMES_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", action="store_true", help="N > 1: also merge every rank's streamed transitions on rank 0 (BASELINE configs[3]'s host replay buffer) and report the merge time")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the run, write what the last timed ply returned to its caller "
                    "(rank 0's games) as DIR/<name>.npy in float32: selfplay_* from the device-resident arm, e2e_* from the "
                    "C-ABI arm; the inputs are seeded, so two builds run with the same arguments can be compared array for array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; the reference arm has none")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch

    omk = importlib.import_module("omok-ai_b200")
    sharding = importlib.import_module("omok-ai_b200.sharding")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    games = args.games
    warm = max(3, args.warmup)
    steps = args.steps
    ctx = omk.Context(device=local_rank, capacity_envs=4, capacity_trees=2 * games, capacity_nodes=CAP_NODES, seed=sharding.rank_seed(1000, rank))
    ctx.net_init_random(0)  # same random-init weights on every rank (no broadcast needed)
    ctx.selfplay_begin(games, COUNT, BATCH, EPS, ALPHA, TEMP, TEMP_THRESHOLD, omk.EVAL_NET)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    # ---- device-resident arm: `value` ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    ctx.selfplay_run(warm, profile=0, want_transitions=True)
    launches0 = ctx.launch_count
    barrier()
    sampler.mark_start()
    # BASELINE configs[3]: "positions streamed to host replay buffer" -- the pinned transition ring is ON in the timed region
    stats, t_boards, t_policy, t_status, t_actions = ctx.selfplay_run(steps, profile=0, want_transitions=True)
    barrier()
    sampler.mark_end()
    launches = ctx.launch_count - launches0
    assert t_boards.shape == (steps, games, 81) and int(stats.d2h_bytes) == steps * games * (81 + 81 * 4 + 4 + 1)
    stream_d2h = int(stats.d2h_bytes)
    merge = None
    if args.gather and dist:  # the host replay buffer of configs[3]: all ranks' blocks of the timed region land on rank 0
        barrier()
        tm = time.perf_counter()
        merged = sharding.gather_replay(torch.from_numpy(t_boards).cuda(), torch.from_numpy(t_policy).cuda(), torch.from_numpy(t_status).cuda())
        host = [m.cpu() for m in merged] if merged is not None else None
        barrier()
        merge = {"seconds": time.perf_counter() - tm, "games_on_rank0": int(host[0].shape[1]) if host else None,
                 "bytes_on_rank0": int(sum(h.numel() * h.element_size() for h in host)) if host else None,
                 "path": "sharding.gather_replay: per-rank [plies, games, ...] blocks all-gathered over NCCL, concatenated along the game axis on rank 0, copied to host",
                 "in_timed_region": False}
    ctx.selfplay_run(1, profile=0, want_transitions=False)  # keeps the load on while the last samples arrive (untimed)
    barrier()
    clocks = sampler.stop()
    ms = float(stats.gpu_ms)
    sims, positions, nn_evals = int(stats.simulations), int(stats.positions), int(stats.nn_evals)
    # Kernel durations for the rooflines: the timed region above runs two search lanes on two streams, where a CUDA-event
    # span around one kernel also contains its wait for the other lane's kernels.  The SAME workload is therefore stepped
    # on with the second lane disabled (one stream, whole 16k-row batches) and event spans around the network kernels.
    ctx.debug_set_lane_min_trees(0)
    ctx.selfplay_run(1, profile=0, want_transitions=False)
    kstats, *_ = ctx.selfplay_run(max(2, steps // 2), profile=2, want_transitions=False)
    ctx.debug_set_lane_min_trees(768)
    fc0_ms, fc0_launches = kstats.by_kind()["fc0"]

    # ---- e2e arm: granular C-ABI calls with host buffers, as the Rust alpha-zero shim would issue them ----
    e2e_steps = steps
    ids_b = np.arange(0, 2 * games, 2, dtype=np.int32)
    ids_w = ids_b + 1
    ctx.pool_new_games(n=2 * games, evaluator=omk.EVAL_NET)
    barrier()
    h2d0, d2h0 = ctx.transfer_bytes  # the library counts every host <-> device copy its entry points make
    t0 = time.perf_counter()
    e2e_sims = 0
    for p in range(e2e_steps):
        mover, other = (ids_b, ids_w) if p % 2 == 0 else (ids_w, ids_b)
        ctx.pool_search(ids=mover, count=COUNT, batch_size=BATCH, epsilon=EPS, alpha=ALPHA, evaluator=omk.EVAL_NET)
        e2e_sims += games * (-(-COUNT // BATCH) * BATCH)
        modes = np.full(games, 1 if p < TEMP_THRESHOLD else 0, np.uint8)
        acts, pol = ctx.pool_sample(ids=mover, modes=modes, temperatures=np.full(games, TEMP, np.float32))
        st = ctx.pool_play(acts, ids=mover)
        ctx.pool_ensure_action(acts, ids=other, evaluator=omk.EVAL_NET)
        ctx.pool_play(acts, ids=other)
        assert (st == 0).all() or p >= 8, "a game ended implausibly early"
        done = np.nonzero(st != 0)[0]
        if len(done):  # a finished game starts over with two fresh agents, as the trainer's episode loop does (src/trainer.rs:101-121)
            fresh = np.concatenate([ids_b[done], ids_w[done]]).astype(np.int32)
            ctx.pool_new_games(ids=fresh, evaluator=omk.EVAL_NET)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_last = {"e2e_actions": acts, "e2e_policy": pol, "e2e_status": st}  # the last timed ply's results, as the caller got them
    h2d1, d2h1 = ctx.transfer_bytes
    h2d, d2h = h2d1 - h2d0, d2h1 - d2h0

    # ---- aggregate over ranks: max time, summed work (the only cross-rank traffic of the whole run) ----
    times, work = sharding.reduce_measurements(
        {"ms": ms, "e2e_s": e2e_s},
        {"sims": sims, "positions": positions, "nn_evals": nn_evals, "launches": launches, "e2e_sims": e2e_sims},
        device="cuda" if dist else "cpu")
    ms, e2e_s = times["ms"], times["e2e_s"]
    sims, positions, nn_evals, launches, e2e_sims = (work[k] for k in ("sims", "positions", "nn_evals", "launches", "e2e_sims"))

    if rank == 0:
        peaks = read_peaks()
        kinds = kstats.by_kind()
        tower_ms, tower_launches = kinds["tower"]
        rows_per_launch = (int(kstats.nn_evals) / max(1, fc0_launches))
        # launches also cover the (small) ensure_action batches; algorithmic flops = rows actually evaluated
        fc0_tflops = (int(kstats.nn_evals) * FLOP_FC0) / (fc0_ms * 1e-3) / 1e12 if fc0_ms > 0 else 0.0
        tower_tflops = (int(kstats.nn_evals) * FLOP_TOWER) / (tower_ms * 1e-3) / 1e12 if tower_ms > 0 else 0.0
        peak = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
        fc0_mode = os.environ.get("OMK_FC0", "f16")
        tower_mode = os.environ.get("OMK_TOWER", "f16")
        passes = {"f16": 3, "simt": 0}
        traffic = ncu_traffic()
        fc0_names = {"f16": "k_fc16 (fc0 10368->512: tcgen05 kind::f16 cta_group::2, 3-pass fp16 hi/lo split, TMA-fed, TMEM chunk promotion)",
                     "simt": "k_gemm (fc0 10368->512, fp32 CUDA cores)"}
        tower_names = {"f16": "k_tower16 (stem + 3 bottleneck blocks: 1x1 convs on tcgen05 kind::f16 3-pass with the activations as TMEM A "
                              "operand, depthwise 3x3 + epilogues on CUDA cores, two CTAs per SM)",
                       "simt": "k_tower (fp32 CUDA cores in shared memory)"}
        note = (f"{peaks['src']} bf16/fp16 dense sustained (MEASURED_PEAKS.json); the fp32-accurate path issues 3 fp16 MMAs per "
                "product (hi.hi + hi.lo + lo.hi), so frac <= 1/3 by construction; tensor_pipe_tflops = 3 x achieved is what the "
                "tensor pipe executes (DESIGN.md 3)")
        roof_fc0 = {"bound": "tensor", "kernel": fc0_names.get(fc0_mode, fc0_mode),
                    "achieved": fc0_tflops, "peak": peak, "unit": "TFLOP/s", "frac": fc0_tflops / peak,
                    "tensor_pipe_tflops": passes.get(fc0_mode, 3) * fc0_tflops,
                    "tensor_pipe_frac": passes.get(fc0_mode, 3) * fc0_tflops / peak,
                    "peak_source": note,
                    "avg_launch_ms": fc0_ms / max(1, fc0_launches), "rows_per_launch": rows_per_launch,
                    "share_of_step": fc0_ms / float(kstats.gpu_ms) if kstats.gpu_ms else None,
                    "measured": "NOT in the timed region: second pass of the same workload with one search lane, CUDA-event spans per kernel (in the two-lane timed region a span would include waits for the other lane); shares agree with the ncu launch list of the two-lane command under profiles/",
                    "in_timed_region": False,
                    "traffic": traffic.get("k_fc16") if fc0_mode == "f16" else None}
        roof_tower = {"bound": "tensor", "kernel": tower_names.get(tower_mode, tower_mode),
                      "achieved": tower_tflops, "peak": peak, "unit": "TFLOP/s", "frac": tower_tflops / peak,
                      "tensor_pipe_tflops": passes.get(tower_mode, 3) * tower_tflops,
                      "peak_source": note + "; this kernel is bound by its CUDA-core epilogues (issue slots), not by the tensor pipe",
                      "avg_launch_ms": tower_ms / max(1, tower_launches), "rows_per_launch": rows_per_launch,
                      "share_of_step": tower_ms / float(kstats.gpu_ms) if kstats.gpu_ms else None,
                      "measured": "NOT in the timed region: second pass of the same workload with one search lane, CUDA-event spans per kernel (in the two-lane timed region a span would include waits for the other lane); shares agree with the ncu launch list of the two-lane command under profiles/",
                    "in_timed_region": False,
                      "traffic": traffic.get("k_tower16") if tower_mode == "f16" else None}
        # K2 tree kernels of this workload (one-lane pass) and K1 environment step (measured here, 16 Mi boards = 512 MB of
        # records, far beyond L2) against the HBM roofline: SURVEY 8d byte models, 1672 B per simulation, 78 B per board-step
        sel_ms, _ = kinds["select_expand"]
        app_ms, _ = kinds["apply"]
        tree_gbs = int(kstats.simulations) * 1672 / ((sel_ms + app_ms) * 1e-3) / 1e9 if sel_ms + app_ms > 0 else 0.0
        roof_tree = {"bound": "hbm", "kernel": "k_select_expand + k_apply (warp per tree; 1024 searching trees per launch)",
                     "achieved": tree_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": tree_gbs / peaks["hbm_gbs"],
                     "note": "algorithmic 1672 B/simulation; at this pool size the kernels are bound by the latency of one serial "
                             "chain per tree, at 65 536 trees k_select_expand by issue slots (66 %) and k_apply by memory (36 % of DRAM "
                             "throughput by ncu, 43 % of HBM by this byte model: DESIGN.md 3, profiles/r02_tree_pool_sweep.json); the PUCT "
                             "descent is reused inside a round and the expansions at a leaf run lane-parallel; "
                             "hidden behind the other search lane's fc0 in the timed region",
                     # one k_select_expand + one k_apply launch at 1024 searching trees (ncu capture with the hash evaluator)
                     "traffic": (traffic.get("k_select_expand", 0.0) + traffic.get("k_apply", 0.0)) or None}
        roof_env = None
        try:
            n_env = 1 << 24
            ectx = omk.Context(device=local_rank, capacity_envs=n_env, capacity_trees=1, capacity_nodes=16, seed=0)
            ectx.env_reset(n=n_env)
            acts = [torch.randint(0, 81, (n_env,), dtype=torch.uint8, device="cuda") for _ in range(8)]
            st = torch.empty(n_env, dtype=torch.int8, device="cuda")
            legal = torch.empty((n_env, 3), dtype=torch.int32, device="cuda")
            es = torch.cuda.ExternalStream(ectx.stream)
            with torch.cuda.stream(es):
                for a in acts[:3]:
                    ectx.env_step_device(a.data_ptr(), n_env, st.data_ptr(), legal.data_ptr())
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record(es)
                for a in acts[3:]:
                    ectx.env_step_device(a.data_ptr(), n_env, st.data_ptr(), legal.data_ptr())
                ev1.record(es)
            ectx.synchronize()
            env_ms = ev0.elapsed_time(ev1) / 5
            env_gbs = n_env * 78 / (env_ms * 1e-3) / 1e9
            roof_env = {"bound": "hbm", "kernel": "k_env_step (lane per board, 32-byte packed records; BASELINE configs[1] shape scaled to 16 Mi boards)",
                        "achieved": env_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": env_gbs / peaks["hbm_gbs"],
                        "avg_launch_ms": env_ms, "board_steps_per_s": n_env / (env_ms * 1e-3), "traffic": traffic.get("k_env_step")}
            ectx.close()
            del acts, st, legal
        except Exception as exc:  # the headline line must still print
            roof_env = {"error": str(exc)}
        # the whole network (tower + fc0 + fc1 + heads) against the tensor pipe: algorithmic flops and the 3-pass MMA rate
        net_ms = sum(kinds[k][0] for k in ("tower", "fc0", "fc1", "heads"))
        net_tflops = int(kstats.nn_evals) * FLOP_POSITION / (net_ms * 1e-3) / 1e12 if net_ms > 0 else 0.0
        roof_net = {"bound": "tensor", "kernel": "whole network forward: k_tower16 + k_fc16 (fc0, fc1, heads)",
                    "achieved": net_tflops, "peak": peak, "unit": "TFLOP/s", "frac": net_tflops / peak,
                    "tensor_pipe_tflops": 3 * net_tflops, "tensor_pipe_frac": 3 * net_tflops / peak,
                    "evals_per_s": int(kstats.nn_evals) / (net_ms * 1e-3) if net_ms > 0 else 0.0,
                    "note": "15 906 240 flop per position; every product is three fp16 MMAs (hi.hi + hi.lo + lo.hi), so "
                            "tensor_pipe_* is what the tensor cores execute; one-lane pass"}
        dominant, other = (roof_tower, roof_fc0) if tower_ms >= fc0_ms else (roof_fc0, roof_tower)
        line = {
            "metric": "mcts_simulations_per_sec", "value": sims / (ms * 1e-3), "unit": "simulations/s",
            "positions_per_sec": positions / (ms * 1e-3), "nn_evals_per_sec": nn_evals / (ms * 1e-3),
            "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": ms / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, games),
            "clocks": clocks,
            "e2e": {"value": e2e_sims / e2e_s, "unit": "simulations/s", "h2d_bytes_per_step": h2d // e2e_steps,
                    "d2h_bytes_per_step": d2h // e2e_steps,
                    "path": "omk_pool_search/sample/play/ensure_action/play per ply with host id+action buffers",
                    "bytes_source": "omk_ctx_transfer_bytes (the library's own counters)"},
            "transition_stream": {"in_timed_region": True, "d2h_bytes_per_step": stream_d2h // steps,
                                  "bytes_per_position": 81 + 81 * 4 + 4 + 1,
                                  "path": "omk_selfplay_run: four-slot device ring -> pinned host mirror on a copy stream -> caller's arrays"},
            "gpu_launches": launches,
            "replay_merge": merge,
            "roofline": dominant,
            "roofline_second": other,
            "roofline_network": roof_net,
            "roofline_tree": roof_tree,
            "roofline_env": roof_env,
        }
        if not args.no_cpu_baseline and world == 1:
            r = cpu_selfplay_sample(4, 0)  # ~12 s of CPU work on 16 cores
            line["cpu_baseline"] = {
                "value": r["sims"] / r["seconds"], "unit": "simulations/s", "cores": r["cores"], "kind": "port",
                "sample": f"{r['trees']} concurrent trees x 4 plies x {COUNT} sims/move; C oracle (pthreads over trees) + "
                          "PyTorch-CPU fp32 network standing in for TensorFlow-CPU"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"selfplay_boards": t_boards[-1], "selfplay_policy": t_policy[-1],
                                             "selfplay_status": t_status[-1], "selfplay_actions": t_actions[-1], **e2e_last}, games)
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    # ONE JSON line on stdout: libraries (NCCL prints its version banner to the C stdout of rank 0) write to stderr instead
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _buf = io.StringIO()
    with contextlib.redirect_stdout(_buf):
        main()
    sys.stdout.flush()
    os.dup2(_real_stdout, 1)
    out = [l for l in _buf.getvalue().splitlines() if l.startswith("{")]
    if out:
        print(out[-1], flush=True)
