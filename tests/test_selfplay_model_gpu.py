"""The self-play driver on a model slot other than the network (omk_selfplay_set_model) and a slot's weights read back
(omk_model_get_params): a driver on slot s with weights W is bit for bit a driver on the network with weights W, in one lane
and in two; changes to other slots leave its games alone; the restarted games' cached prior follows the driver's slot;
switching slots mid-run equals swapping the network's weights at the same boundaries, also onto a network training left
stale; and the gated iteration of tools/iteration.py promotes, keeps and resumes its best network on fresh random streams."""
import importlib
import os
import sys

import numpy as np
import pytest

from oracle import net_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_STATE = -1, -4
G, COUNT, BATCH, NODES, CAPACITY = 8, 32, 8, 4096, 20_000
EMPTY = np.zeros((1, 81), np.uint8), np.zeros(1, np.uint8)


def context(omk, net, lanes=1, slots=None, model=0, seed=11):
    """A context with the network `net`, model slots {slot: params}, a replay memory and the driver on `model`."""
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=NODES, seed=seed)
    ctx.net_load_params(net)
    for s, p in (slots or {}).items():
        ctx.model_load_params(s, p)
    ctx.debug_set_lane_min_trees(2 if lanes == 2 else 0)
    ctx.replay_reset(CAPACITY)
    if model:
        ctx.selfplay_set_model(model)
    ctx.selfplay_begin(G, COUNT, BATCH, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    return ctx


def play(ctx, plies):
    """One selfplay_run: the streamed transitions and the call's statistics."""
    stats, boards, policy, status, actions = ctx.selfplay_run(plies, profile=0, want_transitions=True)
    counts = (stats.simulations, stats.nn_evals, stats.positions, stats.games_finished)
    return [boards, policy, status, actions, np.array(counts, np.int64)]


def state(ctx):
    """The replay memory (rows and counters) and every tree's root statistics."""
    n = ctx.replay_info()[0]
    out = [np.array(ctx.replay_info(), np.int64)] + (list(ctx.replay_get(np.arange(n))) if n else [])
    for t in range(2 * G):
        rn, rw, rp, st, pol = ctx.pool_root_stats(t)
        out += [np.array([rn, st], np.int64), np.array([rw, rp], np.float32), pol]
    return out


def same(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and x.tobytes() == y.tobytes() for x, y in zip(a, b))


def expect_error(omk, code, fn, *args):
    with pytest.raises(omk.OmkError) as e:
        fn(*args)
    assert e.value.code == code, e.value


def minibatch(seed, n=16):
    trainer = importlib.import_module("omok-ai_b200.trainer")
    rng = np.random.default_rng(seed)
    boards = rng.integers(0, 3, (n, 81)).astype(np.uint8)
    turns = rng.integers(0, 2, n).astype(np.uint8)
    pi = rng.random((n, 81)).astype(np.float32)
    pi /= pi.sum(axis=1, keepdims=True)
    return trainer.encode_nn_input(boards, turns), pi, rng.choice(np.array([1.0, -1.0], np.float32), n)


@pytest.mark.parametrize("lanes", [1, 2])
@pytest.mark.parametrize("slot", [1, 2, 15])
def test_a_driver_on_a_slot_equals_a_driver_on_the_network_with_its_weights(omk, slot, lanes):
    w0, w = net_oracle.random_params(0), net_oracle.random_params(1)
    a = context(omk, w0, lanes, {slot: w}, model=slot)
    b = context(omk, w, lanes)
    got, want = play(a, 81) + play(a, 20), play(b, 81) + play(b, 20)  # every game ends at least once in 81 plies
    assert got[4][3] > 0 and a.replay_info()[0] > 0
    assert same(got, want), "streamed boards, policies, status, actions or statistics differ"
    assert same(state(a), state(b)), "replay rows or root statistics differ"
    for x in (a, b):
        x.close()


def test_changes_to_the_network_leave_a_driver_on_another_slot_alone(omk):
    w0, w = net_oracle.random_params(0), net_oracle.random_params(1)
    a, b = (context(omk, w0, 1, {1: w}, model=1) for _ in range(2))
    got, want = play(a, 81), play(b, 81)
    before = a.net_get_params()
    a.train_replay(7, 0, 3, 32)      # trains slot 0 on the rows the driver fed
    a.train_step(*minibatch(0))
    trained = a.net_get_params()
    assert not same(before, trained), "the steps changed the network"
    got += play(a, 30)
    a.net_load_params(net_oracle.random_params(2))
    got += play(a, 30)
    want += play(b, 30) + play(b, 30)
    assert same(got, want) and same(state(a), state(b))
    # (evaluated only now: net_eval's positions are counted in the nn_evals of the driver's next call)
    p_a, p_b = a.net_eval(*EMPTY)[0], b.net_eval(*EMPTY)[0]
    assert not np.array_equal(p_a, p_b), "the network of the first context changed"
    assert a.model_eval(1, *EMPTY)[0].tobytes() == b.model_eval(1, *EMPTY)[0].tobytes()
    for x in (a, b):
        x.close()


def restarted_prior(ctx, max_plies=200):
    """Play one ply at a time until a game ends; the root prior of its restarted Black tree."""
    for _ in range(max_plies):
        status = ctx.selfplay_run(1, profile=0, want_transitions=True)[3]
        done = np.flatnonzero(status[0] > 0)
        if done.size:
            g = int(done[0])
            board, turn, legal = ctx.pool_get_env(2 * g)
            assert legal == 81 and turn == 0 and not board.any()
            assert ctx.pool_root_stats(2 * g)[4].tobytes() == ctx.pool_root_stats(2 * g + 1)[4].tobytes()
            return ctx.pool_root_stats(2 * g)[4]
    pytest.fail(f"no game ended within {max_plies} plies")


def test_the_cached_restart_prior_follows_the_drivers_slot(omk):
    ctx = context(omk, net_oracle.random_params(1), 1, {1: net_oracle.random_params(0)}, model=1)
    ctx.model_load_params(1, net_oracle.random_params(2))  # the best network changes while the driver is active
    p_new, _ = ctx.model_eval(1, *EMPTY)
    assert restarted_prior(ctx).tobytes() == p_new[0].tobytes()
    ctx.net_load_params(net_oracle.random_params(3))        # slot 0 changes: not the driver's
    ctx.train_step(*minibatch(1))
    assert not np.array_equal(ctx.net_eval(*EMPTY)[0], p_new)
    assert restarted_prior(ctx).tobytes() == p_new[0].tobytes()
    ctx.model_from_net(1)                                   # promotion: slot 1 becomes the trained network
    p_net, _ = ctx.net_eval(*EMPTY)
    assert ctx.model_eval(1, *EMPTY)[0].tobytes() == p_net.tobytes()
    assert restarted_prior(ctx).tobytes() == p_net[0].tobytes()
    ctx.close()


@pytest.mark.parametrize("lanes", [1, 2])
def test_switching_slots_mid_run_equals_swapping_the_networks_weights(omk, lanes):
    w0, w1 = net_oracle.random_params(0), net_oracle.random_params(1)
    a = context(omk, w0, lanes, {1: w1}, model=1)
    b = context(omk, w1, lanes)
    got, want = play(a, 7), play(b, 7)
    a.selfplay_set_model(0)
    b.net_load_params(w0)
    got += play(a, 60)
    want += play(b, 60)
    a.selfplay_set_model(1)
    b.net_load_params(w1)
    got += play(a, 40)
    want += play(b, 40)
    assert same(got, want) and same(state(a), state(b))
    for x in (a, b):
        x.close()


@pytest.mark.parametrize("lanes", [1, 2])
def test_switching_to_a_network_that_training_left_stale(omk, lanes):
    """The driver on slot 1 while the network trains (its operand images stale), then omk_selfplay_set_model(0): the
    network is re-packed and the restart prior re-evaluated inside the call, so the games equal those of a driver on the
    network that loaded the trained weights at the same boundary."""
    w0, w1 = net_oracle.random_params(0), net_oracle.random_params(1)
    a = context(omk, w0, lanes, {1: w1}, model=1)
    b = context(omk, w1, lanes)
    got, want = play(a, 81), play(b, 81)
    a.train_replay(3, 0, 4, 32)
    a.train_step(*minibatch(2))
    trained = a.net_get_params()
    assert not same(trained, [np.asarray(p, np.float32).reshape(t.shape) for p, t in zip(w0, trained)])
    a.selfplay_set_model(0)
    b.net_load_params(trained)
    got += play(a, 60)
    want += play(b, 60)
    assert same(got, want) and same(state(a), state(b))
    for x in (a, b):
        x.close()


def test_errors(omk):
    w = net_oracle.random_params(0)
    a, b = (context(omk, w) for _ in range(2))
    for bad in (-1, 16):
        expect_error(omk, ERR_INVALID, a.selfplay_set_model, bad)
    expect_error(omk, ERR_STATE, a.selfplay_set_model, 5)  # unloaded, with a network driver active: nothing changes
    assert same(play(a, 40), play(b, 40)) and same(state(a), state(b))
    for x in (a, b):
        x.close()
    # no driver: the slot is recorded, and selfplay_begin refuses it while it is unloaded
    c = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=NODES, seed=11)
    c.net_load_params(w)
    c.selfplay_set_model(3)
    expect_error(omk, ERR_STATE, c.selfplay_begin, G, COUNT, BATCH, 0.25, 0.03, 1.0, 30, omk.EVAL_NET)
    c.close()
    # the hash evaluator never reads the slot
    outs = []
    for slot in (0, 7, 1):
        h = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=NODES, seed=11)
        h.selfplay_set_model(slot)
        h.selfplay_begin(G, COUNT, BATCH, 0.25, 0.03, 1.0, 30, omk.EVAL_HASH)
        out = play(h, 30)
        h.selfplay_set_model(12)  # an active hash driver accepts an unloaded slot
        outs.append(out + play(h, 30) + state(h))
        h.close()
    assert same(outs[0], outs[1]) and same(outs[0], outs[2])


def test_model_get_params_round_trips_every_slot(omk):
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    expect_error(omk, ERR_STATE, ctx.model_get_params, 0)
    w0, w1 = net_oracle.random_params(0), net_oracle.random_params(1)
    ctx.net_load_params(w0)
    ctx.model_load_params(1, w1)
    ctx.model_from_net(2)
    for slot, want in ((0, w0), (1, w1), (2, w0)):
        got = ctx.model_get_params(slot)
        assert same(got, [np.asarray(p, np.float32).reshape(g.shape) for p, g in zip(want, got)])
    assert same(ctx.model_get_params(0), ctx.net_get_params())
    expect_error(omk, ERR_STATE, ctx.model_get_params, 3)
    for bad in (-1, 16):
        expect_error(omk, ERR_INVALID, ctx.model_get_params, bad)
    ctx.close()


def test_gated_iterations_promote_keep_and_resume_the_best_network(tmp_path):
    """Three tools/iteration.py --gated runs chained through one state file: the first promotes the candidate whatever the
    match (promote_at 0), the others never do (promote_at above 1), so they save the best they resumed.  The last two play
    self-play with the same best network, yet each resumed run draws fresh random streams: the rows they add differ."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    iteration = importlib.import_module("iteration")
    run_state = importlib.import_module("omok-ai_b200.run_state")
    path = str(tmp_path / "gated.state")
    kw = dict(games_per_gpu=16, plies=80, count=16, batch=16, steps=4, minibatch=64, quiet=True, device_replay=True,
              replay_capacity=100_000, gate=2, gated=True, score=True, state=path)

    def arrays():
        with np.load(path, allow_pickle=False) as f:
            return ([f[f"param_{i:02d}"] for i in range(31)], [f[f"best_{i:02d}"] for i in range(31)],
                    [f[k] for k in ("replay_boards", "replay_turns", "replay_policy", "replay_z")])

    first = iteration.run(promote_at=0.0, **kw)
    assert first["promoted"] is True and 0.0 <= first["gate_score"] <= 1.0 and "score_best" in first
    assert first["gate_trained_wins"] + first["gate_best_wins"] + first["gate_draws"] == 2 and "gate_snapshot_wins" not in first
    params, best, rows1 = arrays()
    assert same(params, best), "the promoted best is the trained network"
    seeds = [run_state.read_meta(path)["seed"]]
    second = iteration.run(promote_at=1.01, **kw)
    assert second["promoted"] is False and second["iteration"] == 2
    params2, best2, rows2 = arrays()
    assert same(best2, best), "the best network resumed from the file and kept"
    assert not same(params2, best2)
    seeds.append(run_state.read_meta(path)["seed"])
    third = iteration.run(promote_at=1.01, **kw)
    assert third["promoted"] is False and third["iteration"] == 3
    _, best3, rows3 = arrays()
    assert same(best3, best)
    seeds.append(run_state.read_meta(path)["seed"])
    assert len(set(seeds)) == 3, "every gated iteration runs on a context seed of its own"
    n1, n2 = len(rows1[3]), len(rows2[3])
    assert len(rows3[3]) <= 100_000 and same([r[:n2] for r in rows3], rows2) and same([r[:n1] for r in rows2], rows1)
    added2, added3 = [r[n1:n2] for r in rows2], [r[n2:] for r in rows3]
    assert len(added2[3]) and len(added3[3])
    assert not same(added2, added3), "the same best network replayed the previous iteration's games"
    assert third["score_best"] != second["score_best"]
    plain = str(tmp_path / "plain.state")
    iteration.run(**{**kw, "gated": False, "state": plain})
    with pytest.raises(ValueError, match="best"):
        iteration.run(**{**kw, "state": plain})
