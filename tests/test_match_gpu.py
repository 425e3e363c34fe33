"""The opponent network and the arena on the device (omk_opponent_*, omk_match): the opponent's forward pass against a
context holding the same weights as its network, whole matches against `arena.play_match` on two contexts (hash and
network evaluators, one lane and two), the snapshot taken before training, coexistence with the self-play driver, and the
call's errors and accounting."""
import importlib

import numpy as np
import pytest

from oracle import net_oracle

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_CAPACITY, ERR_STATE, ERR_NUMERIC = -1, -3, -4, -5


@pytest.fixture(scope="module")
def arena():
    return importlib.import_module("omok-ai_b200.arena")


def _positions(n, seed):
    """n boards of 0 .. 60 alternating stones at random cells, with either turn."""
    rng = np.random.default_rng(seed)
    boards = np.zeros((n, 81), np.uint8)
    for b in range(n):
        k = int(rng.integers(0, 61))
        cells = rng.permutation(81)[:k]
        boards[b, cells] = 1 + (np.arange(k) % 2)
    return boards, rng.integers(0, 2, n).astype(np.uint8)


def _final_status(omk, moves):
    """Each game's last GameStatus, replaying its move list on an env pool."""
    n = len(moves)
    ctx = omk.Context(device=0, capacity_envs=n, capacity_trees=1, capacity_nodes=16, seed=0)
    ctx.env_reset(n=n)
    final = np.zeros(n, np.int8)
    for p in range(max(len(m) for m in moves)):
        ids = np.array([g for g in range(n) if len(moves[g]) > p], np.int32)
        status, _ = ctx.env_step(np.array([moves[g][p] for g in ids], np.uint8), ids=ids, want_legal=False)
        final[ids] = status
    ctx.close()
    return final


def _tally(status, pairs):
    """(network wins, opponent wins, draws) from the final statuses: BlackWin counts for the side that opened."""
    s = np.asarray(status)
    opened, answered = s[:pairs], s[pairs:]
    return (int(np.count_nonzero(opened == 2) + np.count_nonzero(answered == 3)),
            int(np.count_nonzero(opened == 3) + np.count_nonzero(answered == 2)), int(np.count_nonzero(s == 1)))


def _host_match(omk, arena, left_params, right_params, pairs, seed, count, batch, evaluator):
    """arena.play_match on two contexts with the match context's seed: (result, move lists)."""
    ctxs = []
    for params in (left_params, right_params):
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=pairs, capacity_nodes=2048, seed=seed)
        if params is not None:
            c.net_load_params(params)
        ctxs.append(c)
    moves = []
    result = arena.play_match(ctxs[0], ctxs[1], game_count=2 * pairs, count=count, batch_size=batch, evaluator=evaluator, moves_out=moves)
    for c in ctxs:
        c.close()
    return result, moves


def _check_same(omk, got, want_result, want_moves, pairs):
    result, moves, status, stats = got
    listed = [[int(a) for a in row if a >= 0] for row in moves]
    assert listed == want_moves
    for g in range(2 * pairs):
        assert (moves[g, len(listed[g]):] == -1).all()
    assert status.tolist() == _final_status(omk, want_moves).tolist()
    assert result == want_result == _tally(status, pairs)
    assert stats["moves"] == sum(len(m) for m in want_moves)


def test_opponent_forward_is_the_network_forward_on_other_weights(omk):
    w1, w2 = net_oracle.random_params(1), net_oracle.random_params(2)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
    ref = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
    ctx.net_load_params(w1)
    ref.net_load_params(w2)
    cases = [(n, mode, _positions(n, seed=n + 7 * mode)) for n in (1, 5, 300, 4096) for mode in (0, 1)]
    before = [ctx.net_eval(b, t, mode=mode) for _, mode, (b, t) in cases]
    ctx.opponent_load_params(w2)
    for (n, mode, (b, t)), (p1, v1) in zip(cases, before):
        p, v = ctx.opponent_eval(b, t, mode=mode)
        rp, rv = ref.net_eval(b, t, mode=mode)
        assert p.tobytes() == rp.tobytes() and v.tobytes() == rv.tobytes(), (n, mode)
        p, v = ctx.net_eval(b, t, mode=mode)
        assert p.tobytes() == p1.tobytes() and v.tobytes() == v1.tobytes(), (n, mode)
    ctx.close()
    ref.close()


@pytest.mark.parametrize("pairs", [3, 8])
@pytest.mark.parametrize("first_tree", [0, 5])
def test_match_hash_evaluator_matches_the_host_match(omk, arena, pairs, first_tree):
    seed, count, batch = 13, 32, 8
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=first_tree + 4 * pairs, capacity_nodes=2048, seed=seed)
    got = ctx.match(pairs, first_tree=first_tree, count=count, batch_size=batch, evaluator=omk.EVAL_HASH)
    listed = []
    assert arena.play_match_device(ctx, game_count=2 * pairs, count=count, batch_size=batch, evaluator=omk.EVAL_HASH,
                                   first_tree=first_tree, moves_out=listed) == got[0]
    ctx.close()
    want_result, want_moves = _host_match(omk, arena, None, None, pairs, seed, count, batch, omk.EVAL_HASH)
    assert listed == want_moves
    _check_same(omk, got, want_result, want_moves, pairs)


def test_match_network_evaluator_matches_the_host_match_on_one_and_two_lanes(omk, arena):
    pairs, seed, count, batch = 8, 5, 16, 8
    w1, w2 = net_oracle.random_params(3), net_oracle.random_params(4)
    runs = []
    for min_trees in (None, 0):
        ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs, capacity_nodes=2048, seed=seed)
        ctx.net_load_params(w1)
        ctx.opponent_load_params(w2)
        if min_trees is not None:
            ctx.debug_set_lane_min_trees(min_trees)
        runs.append(ctx.match(pairs, count=count, batch_size=batch, evaluator=omk.EVAL_NET))
        ctx.close()
    want_result, want_moves = _host_match(omk, arena, w1, w2, pairs, seed, count, batch, omk.EVAL_NET)
    for got in runs:
        _check_same(omk, got, want_result, want_moves, pairs)


def test_match_after_training_plays_the_trained_network_against_the_snapshot(omk, arena):
    pairs, seed, count, batch = 4, 9, 16, 8
    w1 = net_oracle.random_params(5)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs, capacity_nodes=2048, seed=seed)
    ctx.net_load_params(w1)
    ctx.opponent_from_net()
    rng = np.random.default_rng(0)
    for _ in range(3):
        images = (rng.random((64, 243)) < 0.2).astype(np.float32)
        pi = rng.random((64, 81)).astype(np.float32)
        pi /= pi.sum(axis=1, keepdims=True)
        ctx.train_step(images, pi, rng.choice([-1.0, 1.0], 64).astype(np.float32))
    got = ctx.match(pairs, count=count, batch_size=batch, evaluator=omk.EVAL_NET)  # the network's images are stale until here
    trained = ctx.net_get_params()
    assert any(not np.array_equal(a, b) for a, b in zip(trained, w1))
    boards, turns = _positions(300, seed=1)
    for params, fn in ((w1, ctx.opponent_eval), (trained, ctx.net_eval)):
        fresh = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
        fresh.net_load_params(params)
        p, v = fn(boards, turns)
        rp, rv = fresh.net_eval(boards, turns)
        assert p.tobytes() == rp.tobytes() and v.tobytes() == rv.tobytes()
        fresh.close()
    want_result, want_moves = _host_match(omk, arena, trained, w1, pairs, seed, count, batch, omk.EVAL_NET)
    _check_same(omk, got, want_result, want_moves, pairs)
    ctx.close()


def test_match_between_selfplay_runs_leaves_self_play_unchanged(omk):
    n_games, plies, cap, pairs = 8, 30, 4096, 2

    def make():
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * n_games + 4 * pairs, capacity_nodes=1024, seed=21)
        c.net_init_random(2)
        c.replay_reset(cap)
        c.selfplay_begin(n_games, 16, 8, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        return c

    a, b = make(), make()
    out_a = [a.selfplay_run(plies)[1:]]
    out_b = [b.selfplay_run(plies)[1:]]
    a.opponent_load_params(net_oracle.random_params(6))
    res = a.match(pairs, first_tree=2 * n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert sum(res[0]) == 2 * pairs
    with pytest.raises(omk.OmkError) as e:
        a.match(pairs, first_tree=2 * n_games - 1, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert e.value.code == ERR_STATE
    out_a.append(a.selfplay_run(plies)[1:])
    out_b.append(b.selfplay_run(plies)[1:])
    for xa, xb in zip(out_a, out_b):
        for u, v in zip(xa, xb):
            assert u.tobytes() == v.tobytes()
    assert a.replay_info() == b.replay_info() and a.replay_info()[0] > 0
    rows = np.arange(a.replay_info()[0])
    for u, v in zip(a.replay_get(rows), b.replay_get(rows)):
        assert u.tobytes() == v.tobytes()
    a.close()
    b.close()


def test_match_errors_and_accounting(omk):
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=16, capacity_nodes=2048, seed=3)
    H, N = omk.EVAL_HASH, omk.EVAL_NET
    for kw in (dict(pairs=0), dict(pairs=5), dict(pairs=2, first_tree=9), dict(pairs=2, first_tree=-1), dict(pairs=2, batch_size=0),
               dict(pairs=2, batch_size=65), dict(pairs=2, count=0), dict(pairs=2, evaluator=7)):
        args = dict(count=16, batch_size=8, evaluator=H)
        args.update(kw)
        with pytest.raises(omk.OmkError) as e:
            ctx.match(**args)
        assert e.value.code == ERR_INVALID, kw
    assert ctx.L.omk_match(ctx.h, 2, 0, 16, 8, 0.0, 1.0, H, None, None, None, None, None) == ERR_INVALID
    w = net_oracle.random_params(7)
    with pytest.raises(omk.OmkError) as e:  # a tensor of the wrong length
        ctx.opponent_load_params(w[:3] + [w[3][:-1]] + w[4:])
    assert e.value.code == ERR_INVALID
    for call in (lambda: ctx.match(2, count=16, evaluator=N),                 # no network
                 lambda: ctx.opponent_from_net(),                              # no network to copy
                 lambda: ctx.opponent_eval(np.zeros((1, 81), np.uint8), [0])):  # no opponent
        with pytest.raises(omk.OmkError) as e:
            call()
        assert e.value.code == ERR_STATE
    ctx.net_load_params(w)
    with pytest.raises(omk.OmkError) as e:  # a network but no opponent
        ctx.match(2, count=16, evaluator=N)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(True)
    with pytest.raises(omk.OmkError) as e:
        ctx.match(2, count=16, evaluator=H)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(False)
    # accounting
    h2d0 = ctx.transfer_bytes[0]
    result, moves, status, stats = ctx.match(4, count=48, batch_size=16, evaluator=H)
    assert ctx.transfer_bytes[0] == h2d0
    assert sum(result) == 8 and result == _tally(status, 4)
    played = (moves >= 0).sum(axis=1)
    assert stats["moves"] == int(played.sum())
    assert stats["host_syncs"] == int(played.max()) + 1
    assert all((moves[g, : played[g]] >= 0).all() and (moves[g, played[g]:] == -1).all() for g in range(8))
    assert stats["simulations"] > 0 and stats["nn_evals"] > 0 and stats["gpu_ms"] > 0
    ctx.close()
    small = omk.Context(device=0, capacity_envs=1, capacity_trees=8, capacity_nodes=8, seed=3)
    with pytest.raises(omk.OmkError) as e:
        small.match(2, count=64, batch_size=16, evaluator=H)
    assert e.value.code == ERR_CAPACITY
    small.close()


def test_match_and_opponent_eval_report_a_non_finite_opponent(omk):
    """An opponent whose activations leave the fp16 operand range answers OMK_ERR_NUMERIC in omk_opponent_eval and stops
    omk_match at the half-move that produced it; the network and a sound opponent then work as before."""
    params = net_oracle.random_params(0)
    bad = [p.copy() for p in params]
    bad[0] = bad[0] * np.float32(1e5)  # stem weights x 1e5: the residual stream leaves the fp16 range
    boards, turns = _positions(5, seed=3)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=8, capacity_nodes=2048, seed=1)
    ctx.net_load_params(params)
    ctx.opponent_load_params(bad)
    with pytest.raises(omk.OmkError) as e:
        ctx.opponent_eval(boards, turns)
    assert e.value.code == ERR_NUMERIC
    with pytest.raises(omk.OmkError) as e:
        ctx.match(2, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert e.value.code == ERR_NUMERIC
    p, v = ctx.net_eval(boards, turns)
    assert np.isfinite(p).all() and np.isfinite(v).all()
    ctx.opponent_load_params(params)
    result, _, _, _ = ctx.match(2, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert sum(result) == 4
    ctx.close()


def test_iteration_with_a_gating_match():
    """tools/iteration.py --device-replay --gate at a small size: the trained network plays every game against its snapshot."""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    iteration = importlib.import_module("iteration")
    out = iteration.run(games_per_gpu=16, plies=80, count=16, batch=16, steps=4, minibatch=64, quiet=True, device_replay=True,
                        replay_capacity=256, gate=8)
    assert out["gate_trained_wins"] + out["gate_snapshot_wins"] + out["gate_draws"] == 8
    assert out["gate_phase_s"] > 0 and out["gate_host_syncs"] <= out["gate_moves"] + 1
    with pytest.raises(ValueError):
        iteration.run(games_per_gpu=16, plies=80, count=16, batch=16, steps=4, minibatch=64, quiet=True, device_replay=True,
                      replay_capacity=256, gate=1)
