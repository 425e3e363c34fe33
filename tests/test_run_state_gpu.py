"""Exact resume of a training run: the Adadelta accumulators out of and into a context (omk_train_get_optimizer /
omk_train_set_optimizer), rows appended to the device replay memory (omk_replay_append) against a numpy model of the ring,
the self-play driver and the trainer on appended rows, and run_state's save / load end to end against a run that was never
stopped."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ERR_INVALID, ERR_STATE = -1, -4


@pytest.fixture(scope="module")
def trainer():
    return importlib.import_module("omok-ai_b200.trainer")


@pytest.fixture(scope="module")
def run_state():
    return importlib.import_module("omok-ai_b200.run_state")


def synthetic_rows(rng, n):
    """n replay rows in replay_get's layout; a third of the z are -0.0, as a draw's are."""
    boards = rng.integers(0, 3, (n, 81)).astype(np.uint8)
    turns = rng.integers(0, 2, n).astype(np.uint8)
    policy = rng.random((n, 81)).astype(np.float32)
    policy /= policy.sum(axis=1, keepdims=True)
    z = rng.choice(np.array([1.0, -1.0, -0.0, 0.0], np.float32), n)
    return boards, turns, policy, z


def all_rows(ctx):
    n = ctx.replay_info()[0]
    return ctx.replay_get(np.arange(n)) if n else tuple(np.zeros((0,) + s, d) for s, d in (((81,), np.uint8), ((), np.uint8),
                                                                                          ((81,), np.float32), ((), np.float32)))


def same_bytes(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and x.tobytes() == y.tobytes() for x, y in zip(a, b))


def cat(*parts):
    return tuple(np.concatenate(col) for col in zip(*parts))


def expect_error(omk, code, fn, *args, **kw):
    with pytest.raises(omk.OmkError) as e:
        fn(*args, **kw)
    assert e.value.code == code, e.value


# ------------------------------------------------------------------ the optimizer state
def minibatch(trainer, rng, n=16):
    boards, turns, policy, z = synthetic_rows(rng, n)
    return trainer.encode_nn_input(boards, turns), policy, np.where(z == 0, 0.0, z).astype(np.float32)


@gpu
def test_optimizer_round_trip_resumes_the_step_bit_for_bit(omk, trainer):
    rng = np.random.default_rng(0)
    batches = [minibatch(trainer, rng) for _ in range(4)]
    mk = lambda: omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)  # noqa: E731
    a, b, c = mk(), mk(), mk()
    for x in (a, b, c):
        assert all(not t.any() for t in sum(x.train_get_optimizer(), [])), "a context that has not stepped reports zeros"
    a.net_init_random(3)
    for i in range(3):
        a.train_step(*batches[i])
    accum, update = a.train_get_optimizer()
    assert all(np.isfinite(t).all() and (t >= 0).all() for t in accum + update) and any(t.any() for t in update)
    for x in (b, c):
        x.net_load_params(a.net_get_params())
    b.train_set_optimizer(accum, update)  # allocates the optimizer state of a context that never stepped
    got = b.train_get_optimizer()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(got[0] + got[1], accum + update))
    la, lb, lc = (np.array(x.train_step(*batches[3]), np.float32) for x in (a, b, c))
    assert la.tobytes() == lb.tobytes()
    for x, y in zip(a.net_get_params(), b.net_get_params()):
        assert x.tobytes() == y.tobytes()
    oa, ob = a.train_get_optimizer(), b.train_get_optimizer()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(oa[0] + oa[1], ob[0] + ob[1]))
    # without the accumulators the first update after a restart is a different one
    assert la.tobytes() != lc.tobytes()
    assert any(x.tobytes() != y.tobytes() for x, y in zip(a.net_get_params(), c.net_get_params()))
    # invalid entries: refused whole, the state unchanged
    for tensor, which, value in ((5, 0, np.nan), (23, 1, -1e-6), (30, 0, np.inf), (0, 1, -np.inf)):
        bad = [[t.copy() for t in ob[0]], [t.copy() for t in ob[1]]]
        bad[which][tensor].reshape(-1)[-1] = value
        expect_error(omk, ERR_INVALID, b.train_set_optimizer, *bad)
    wrong = [[t.copy() for t in ob[0]], [t.copy() for t in ob[1]]]
    for w in wrong:
        w[23] = w[23][:-1]
    expect_error(omk, ERR_INVALID, b.train_set_optimizer, *wrong)  # a tensor length the network does not have
    with pytest.raises(ValueError):
        b.train_set_optimizer(ob[0], wrong[1])  # one length list serves both sets: they must agree
    now = b.train_get_optimizer()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(now[0] + now[1], ob[0] + ob[1]))
    for x in (a, b, c):
        x.close()


# ------------------------------------------------------------------ appending rows
class RingModel:
    """The replay memory's logical rows and counters as numpy sees them."""

    def __init__(self, cap, rows=None, added=0, episodes=0):
        self.cap, self.rows = cap, rows
        self.added, self.episodes = added, episodes

    def append(self, rows, episodes=0):
        self.rows = rows if self.rows is None else cat(self.rows, rows)
        self.rows = tuple(col[max(0, len(col) - self.cap):] for col in self.rows)
        self.added += len(rows[0])
        self.episodes += episodes

    def check(self, ctx):
        assert ctx.replay_info() == (len(self.rows[0]), self.added, self.episodes)
        assert same_bytes(all_rows(ctx), self.rows)


@gpu
def test_append_follows_the_ring_model(omk):
    rng = np.random.default_rng(1)
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    expect_error(omk, ERR_STATE, ctx.replay_append, *synthetic_rows(rng, 3))  # no replay memory
    ctx.replay_reset(50)
    model = RingModel(50)
    for n, episodes in ((20, 2), (45, 1), (0, 3), (120, 4), (50, 0), (7, 0)):  # empty, beyond the free room, only
        rows = synthetic_rows(rng, n)                                           # episodes, beyond the capacity, exactly it
        ctx.replay_append(*rows, episodes=episodes)
        model.append(rows, episodes)
        model.check(ctx)
    assert np.signbit(all_rows(ctx)[3]).any()
    # invalid rows: all or nothing
    for col, index, value in ((0, (3, 40), 3), (0, (0, 0), 255), (1, 5, 2), (2, (6, 80), np.nan), (2, (1, 2), np.inf),
                              (3, 4, np.nan), (3, 0, -np.inf)):
        rows = [x.copy() for x in synthetic_rows(rng, 8)]
        rows[col][index] = value
        expect_error(omk, ERR_INVALID, ctx.replay_append, *rows)
        model.check(ctx)
    expect_error(omk, ERR_INVALID, ctx.replay_append, *synthetic_rows(rng, 2), episodes=-1)
    model.check(ctx)
    ctx.close()


@gpu
def test_append_after_self_play_wrapped_the_ring(omk):
    rng = np.random.default_rng(2)
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=64, capacity_nodes=1024, seed=4)
    ctx.replay_reset(300)
    ctx.selfplay_begin(32, 32, 16, 0.25, 0.03, 1.0, 6, omk.EVAL_HASH)
    ctx.selfplay_run(60, want_transitions=False)
    n, added, episodes = ctx.replay_info()
    assert n == 300 and added % 300 != 0, "the write position should not be slot 0"
    model = RingModel(300, all_rows(ctx), added, episodes)
    for k in (37, 263, 301):  # the memory is full: each append drops the oldest rows; 301 rows exceed the capacity
        rows = synthetic_rows(rng, k)
        ctx.replay_append(*rows, episodes=1)
        model.append(rows, 1)
        model.check(ctx)
    ctx.close()


# ------------------------------------------------------------------ the driver and the trainer on appended rows
def driver(omk, lanes, capacity=600_000, seed=4, G=32):
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=1024, seed=seed)
    ctx.debug_set_lane_min_trees(2 if lanes == 2 else 0)
    ctx.replay_reset(capacity)
    ctx.selfplay_begin(G, 32, 16, 0.25, 0.03, 1.0, 6, omk.EVAL_HASH)
    return ctx


@gpu
@pytest.mark.parametrize("lanes", [1, 2])
def test_the_driver_commits_after_appended_rows(omk, lanes):
    """Rows appended before the first ply and between two runs (the games' staged tails kept): the driver's rows are those
    of a context without the appends, shifted past the appended rows."""
    rng = np.random.default_rng(3)
    a, b = driver(omk, lanes), driver(omk, lanes)
    first, second = synthetic_rows(rng, 53), synthetic_rows(rng, 211)
    a.replay_append(*first, episodes=5)
    for x in (a, b):
        x.selfplay_run(30, want_transitions=False)
    n1 = b.replay_info()[0]
    assert n1 > 0
    a.replay_append(*second, episodes=7)
    for x in (a, b):
        x.selfplay_run(50, want_transitions=False)
    ra, rb = all_rows(a), all_rows(b)
    nb, added_b, eps_b = b.replay_info()
    assert a.replay_info() == (nb + 264, added_b + 264, eps_b + 12)
    head = tuple(col[:n1] for col in rb)
    tail = tuple(col[n1:] for col in rb)
    assert same_bytes(ra, cat(first, head, second, tail))
    for x in (a, b):
        x.close()


@gpu
def test_training_on_appended_rows_equals_training_on_self_played_rows(omk):
    """omk_train_replay on rows self-play committed (context A) and on the same rows appended into context B, at another
    ring offset: the same losses, weights and accumulators, bit for bit."""
    rng = np.random.default_rng(4)
    a = driver(omk, 1, capacity=500)
    a.selfplay_run(90, want_transitions=False)
    n, added_a, episodes = a.replay_info()
    assert n == 500
    rows = all_rows(a)
    b = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=9)
    b.replay_reset(500)
    b.replay_append(*synthetic_rows(rng, 23))
    b.replay_append(*rows, episodes=episodes)  # pushes the 23 out: the ring holds A's rows from slot 23 on
    assert b.replay_info() == (500, 523, episodes) and added_a % 500 != 23
    for x in (a, b):
        x.net_init_random(3)
    la, lb = (x.train_replay(17, 5, 3, 64) for x in (a, b))
    assert la.tobytes() == lb.tobytes()
    for x, y in zip(a.net_get_params(), b.net_get_params()):
        assert x.tobytes() == y.tobytes()
    oa, ob = a.train_get_optimizer(), b.train_get_optimizer()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(oa[0] + oa[1], ob[0] + ob[1]))
    for x in (a, b):
        x.close()


# ------------------------------------------------------------------ end to end
@gpu
def test_a_resumed_run_equals_one_that_was_never_stopped(omk, run_state, tmp_path):
    """A: self-play, S steps, save, then selfplay_begin, self-play and S more steps.  B: a fresh context with the saved seed
    loads the file, then the same.  Network evaluator, 64 games, count 32, batch 8, a ring that wraps."""
    G, S, SEED, SAMPLER, CAP = 64, 4, 21, 77, 2000
    cfg = (G, 32, 8, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    mk = lambda seed: omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=4096, seed=seed)  # noqa: E731
    a = mk(SEED)
    a.net_init_random(7)
    a.replay_reset(CAP)
    a.selfplay_begin(*cfg)
    a.selfplay_run(60, want_transitions=False)
    assert a.replay_info()[1] > CAP, "the ring should have wrapped"
    a.train_replay(SAMPLER, 0, S, 8)
    path = tmp_path / "run.state"
    run_state.save(a, path, seed=SEED, sampler_seed=SAMPLER, step=S, iteration=1, world=1, rank=0)
    a.selfplay_begin(*cfg)
    a.selfplay_run(40, want_transitions=False)
    la = a.train_replay(SAMPLER, S, S, 8)

    meta = run_state.read_meta(path)
    assert meta == dict(seed=SEED, sampler_seed=SAMPLER, step=S, iteration=1, world=1, rank=0)
    b = mk(meta["seed"])
    assert run_state.load(b, path, world=1, rank=0) == meta
    n_saved = b.replay_info()[0]
    assert b.replay_info() == (n_saved, n_saved, b.replay_info()[2]), "rows_added counts from the restore"
    b.selfplay_begin(*cfg)
    b.selfplay_run(40, want_transitions=False)
    lb = b.train_replay(meta["sampler_seed"], meta["step"], S, 8)

    (na, _, ea), (nb, _, eb) = a.replay_info(), b.replay_info()
    assert (na, ea) == (nb, eb)
    assert same_bytes(all_rows(a), all_rows(b))
    assert la.tobytes() == lb.tobytes() and np.isfinite(la).all()
    for x, y in zip(a.net_get_params(), b.net_get_params()):
        assert x.tobytes() == y.tobytes()
    oa, ob = a.train_get_optimizer(), b.train_get_optimizer()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(oa[0] + oa[1], ob[0] + ob[1]))
    for x in (a, b):
        x.close()


@gpu
def test_iteration_tool_continues_a_run_across_processes(tmp_path):
    """tools/iteration.py --device-replay --state twice: the second run loads the first one's state (its replay length,
    its trainer step) and saves the next iteration."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    iteration = importlib.import_module("iteration")
    run_state = importlib.import_module("omok-ai_b200.run_state")
    path = str(tmp_path / "it.state")
    kw = dict(games_per_gpu=16, plies=80, count=16, batch=16, steps=5, minibatch=64, quiet=True, device_replay=True,
              replay_capacity=1000, state=path)
    first = iteration.run(**kw)
    assert first["iteration"] == 1 and first["state_load_s"] is None and first["state_save_s"] > 0
    assert first["replay_rows_at_start"] == 0
    second = iteration.run(**kw)
    assert second["iteration"] == 2 and second["state_load_s"] > 0
    assert second["replay_rows_at_start"] == first["replay_rows"]
    assert run_state.read_meta(path)["step"] == 2 * (2 + 5) and run_state.read_meta(path)["iteration"] == 2
