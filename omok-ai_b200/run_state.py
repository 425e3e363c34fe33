"""Save and restore everything a training run needs to resume exactly: the network's 31 weight tensors, the trainer's two
Adadelta accumulators and the device replay memory (capacity, rows and episode count), with the run's position.

The state is one `.npz` (numpy's zip of `.npy` arrays, read with allow_pickle=False), written at an iteration boundary.  The
self-play driver's unfinished games are not part of it: the resumed process calls `selfplay_begin`, which restarts every
game.  To resume, recreate the context with the saved `seed`, call `load`, and continue the trainer's sampler streams at the
saved `step` (`AbiTrainStep.steps = step`).  A run that is resumed then produces the replay rows, losses, weights and
accumulators of a run that was never stopped but restarted its driver at the same boundary, bit for bit (DESIGN.md 2).

A gated run (tools/iteration.py --gated) also keeps its best network, the weights of a model slot other than the network,
as `best_00 .. best_30`; a file without them is a run that has none.  `read_meta` and `load` report a best network as the
metadata key `best` (True), present only when the file holds one, so that a file without one yields exactly the metadata
it always did: test it with `meta.get("best", False)`.

The reference's checkpoint (model_io.py) still holds the weights only.
"""
from __future__ import annotations

import os

import numpy as np

from .binding import CELLS, NET_SHAPES

FORMAT_VERSION = 1
META = ("seed", "sampler_seed", "step", "iteration", "world", "rank")
REPLAY_CHUNK = 65536  # rows per replay_get call while saving


class RunStateError(ValueError):
    pass


def _key(kind: str, i: int) -> str:
    return f"{kind}_{i:02d}"


def save(ctx, path, *, seed: int, sampler_seed: int, step: int, iteration: int, world: int, rank: int,
         best_slot: int | None = None) -> None:
    """Write the state of `ctx` with the run's metadata to `path` (the file is replaced only once it is complete).  With
    `best_slot`, that model slot's weights are saved too, as the run's best network."""
    meta = dict(seed=seed, sampler_seed=sampler_seed, step=step, iteration=iteration, world=world, rank=rank)
    for k, v in meta.items():
        if not 0 <= int(v) < 2**64:
            raise RunStateError(f"{k} = {v} is not an unsigned 64-bit integer")
    arrays = {"version": np.array(FORMAT_VERSION, np.int64)}
    arrays.update({k: np.array(int(v), np.uint64) for k, v in meta.items()})
    accum, accum_update = ctx.train_get_optimizer()
    for i, (p, a, u) in enumerate(zip(ctx.net_get_params(), accum, accum_update)):
        arrays[_key("param", i)], arrays[_key("accum", i)], arrays[_key("accum_update", i)] = p, a, u
    if best_slot is not None:
        arrays.update({_key("best", i): p for i, p in enumerate(ctx.model_get_params(best_slot))})
    n, _, episodes = ctx.replay_info()
    boards = np.empty((n, CELLS), np.uint8)
    turns = np.empty(n, np.uint8)
    policy = np.empty((n, CELLS), np.float32)
    z = np.empty(n, np.float32)
    for first in range(0, n, REPLAY_CHUNK):
        last = min(n, first + REPLAY_CHUNK)
        boards[first:last], turns[first:last], policy[first:last], z[first:last] = ctx.replay_get(np.arange(first, last))
    arrays.update(replay_capacity=np.array(ctx.replay_capacity, np.int64), replay_episodes=np.array(episodes, np.int64),
                  replay_boards=boards, replay_turns=turns, replay_policy=policy, replay_z=z)
    path = os.fspath(path)
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:  # a file object: np.savez would append ".npz" to a name
        np.savez(f, **arrays)
        f.flush()
        os.fsync(f.fileno())
    os.replace(tmp, path)


def _expect(f, key: str, shape, dtype) -> np.ndarray:
    if key not in f.files:
        raise RunStateError(f"run state lacks {key}")
    a = f[key]
    if a.shape != tuple(shape) or a.dtype != np.dtype(dtype):
        raise RunStateError(f"{key}: {a.dtype}{list(a.shape)}, expected {np.dtype(dtype)}{list(shape)}")
    return a


def read_meta(path) -> dict:
    """The metadata of a run state file ({seed, sampler_seed, step, iteration, world, rank}, and best = True if it holds a
    best network), after its version check."""
    with np.load(path, allow_pickle=False) as f:
        return _meta(f)


def _meta(f) -> dict:
    version = int(_expect(f, "version", (), np.int64))
    if version != FORMAT_VERSION:
        raise RunStateError(f"run state format {version}; this version reads format {FORMAT_VERSION}")
    meta = {k: int(_expect(f, k, (), np.uint64)) for k in META}
    if _has_best(f):
        meta["best"] = True
    return meta


def _has_best(f) -> bool:
    return any(k.startswith("best_") for k in f.files)


def load(ctx, path, *, world: int | None = None, rank: int | None = None, best_slot: int | None = None) -> dict:
    """Restore the state in `path` into `ctx`: net_load_params, the best network with model_load_params(best_slot) if the
    file holds one and `best_slot` is given, train_set_optimizer, replay_reset(capacity), replay_append.  Every array is
    checked before the context is touched: a best network must be complete.  With `world` / `rank` given, a file written by
    another world size or rank is refused.  Returns the metadata, with best = True if the file holds a best network."""
    with np.load(path, allow_pickle=False) as f:
        meta = _meta(f)
        for k, want in (("world", world), ("rank", rank)):
            if want is not None and meta[k] != want:
                raise RunStateError(f"run state written with {k} {meta[k]}, this run has {k} {want}")
        params, accum, accum_update = ([_expect(f, _key(kind, i), s, np.float32) for i, s in enumerate(NET_SHAPES)]
                                       for kind in ("param", "accum", "accum_update"))
        best = [_expect(f, _key("best", i), s, np.float32) for i, s in enumerate(NET_SHAPES)] if _has_best(f) else None
        capacity = int(_expect(f, "replay_capacity", (), np.int64))
        episodes = int(_expect(f, "replay_episodes", (), np.int64))
        z = f["replay_z"] if "replay_z" in f.files else None
        n = z.shape[0] if z is not None and z.ndim == 1 else -1
        if not 0 <= n <= capacity or episodes < 0 or (capacity == 0 and episodes):
            raise RunStateError(f"replay: {n} rows and {episodes} episodes in a capacity of {capacity}")
        boards = _expect(f, "replay_boards", (n, CELLS), np.uint8)
        turns = _expect(f, "replay_turns", (n,), np.uint8)
        policy = _expect(f, "replay_policy", (n, CELLS), np.float32)
        z = _expect(f, "replay_z", (n,), np.float32)
    ctx.net_load_params(params)
    if best is not None and best_slot is not None:
        ctx.model_load_params(best_slot, best)
    ctx.train_set_optimizer(accum, accum_update)
    ctx.replay_reset(capacity)
    if n or episodes:
        ctx.replay_append(boards, turns, policy, z, episodes=episodes)
    return meta
