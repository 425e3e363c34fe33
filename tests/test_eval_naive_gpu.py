"""The trainer's evaluation against the naive player on the device (omk_naive_move, omk_eval_naive): the naive player's
move against the restatement of DESIGN.md 4, whole evaluations against the oracle loop and against the host-driven loop,
coexistence with the self-play driver and the replay memory, and the call's errors and accounting."""
import importlib

import numpy as np
import pytest

import naive_ref

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_CAPACITY, ERR_STATE = -1, -3, -4


@pytest.fixture(scope="module")
def arena():
    return importlib.import_module("omok-ai_b200.arena")


def _drawn_board():
    """Every cell but 80 filled with no run longer than two: the last cell is a Draw for either side."""
    b = np.zeros(81, np.uint8)
    for y in range(9):
        for x in range(9):
            b[y * 9 + x] = 1 + ((x // 2 + y) % 2)
    b[80] = 0
    return b


def test_naive_move_kats_and_random_positions(omk):
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
    boards = np.zeros((6, 81), np.uint8)
    turns = np.zeros(6, np.uint8)
    boards[0, [0, 1, 2, 3]] = 1          # black completes five at 4
    boards[0, [9, 10, 11]] = 2
    boards[1, [20, 21, 22, 23]] = 1      # white must block: 19 comes first
    boards[1, [40, 41, 50]] = 2
    turns[1] = 1
    boards[2, [0, 1, 2, 3, 5]] = 1       # 4 would make six (no win); black blocks white's four at 29
    boards[2, [30, 31, 32, 33]] = 2
    boards[2, 60] = 2
    boards[3, 40] = 1                    # nothing to win or block: random
    turns[3] = 1
    boards[4] = _drawn_board()           # one empty cell: Draw, forced
    boards[5, [0, 20, 42, 66]] = 1       # white to move completes its column at 1
    boards[5, [10, 19, 28, 37]] = 2
    turns[5] = 1
    assert naive_ref.naive_move(boards[4], 0, 0, 0) == (80, 1)
    seed = 17
    streams = np.array([0, 1, 2, 3 + 81 * 7, 4, 5], np.uint32)
    actions, forced = ctx.naive_move(boards, turns, seed, streams=streams)
    assert actions.tolist()[:3] == [4, 19, 29] and actions[4] == 80 and actions[5] == 1
    assert forced.tolist() == [1, 1, 1, 0, 1, 1]
    assert (int(actions[3]), 0) == naive_ref.naive_move(boards[3], 1, seed, int(streams[3]))
    # a few thousand positions from random playouts, both turns, against the restatement bit for bit
    boards, turns = naive_ref.random_positions(3000, seed=11)
    streams = np.random.default_rng(3).integers(0, 2**32, 3000, dtype=np.uint64).astype(np.uint32)
    for s, strm in ((5, None), (2**63 + 9, streams)):
        got_a, got_f = ctx.naive_move(boards, turns, s, streams=strm)
        want = [naive_ref.naive_move(b, t, s, i if strm is None else int(strm[i])) for i, (b, t) in enumerate(zip(boards, turns))]
        assert got_a.tolist() == [w[0] for w in want]
        assert got_f.tolist() == [w[1] for w in want]
    full = np.ones((1, 81), np.uint8)
    assert ctx.naive_move(full, [0], 0)[0].tolist() == [-1]
    with pytest.raises(omk.OmkError) as e:
        ctx.naive_move(np.full((1, 81), 3, np.uint8), [0], 0)
    assert e.value.code == ERR_INVALID
    ctx.close()


def _oracle_eval(orc, games, count, batch, eps, alpha, ctx_seed, naive_seed, first_tree):
    """test_arena_gpu's oracle loop with the naive player's random move on the restated stream and the agents on the
    streams of their tree ids."""
    ev = orc.NativeHashEvaluator()
    agents = {g: orc.Agent(ev, ctx_seed, first_tree + g) for g in range(games)}
    moves = [[] for _ in range(games)]
    final = [0] * games
    tally = {1: 0, 2: 0, 3: 0}

    def play(g, a):
        moves[g].append(a)
        st = agents[g].play_action(a)
        if st != 0:
            tally[st] += 1
            final[g] = st
        return st == 0

    live = list(range(games))
    while live:
        nxt = []
        for g in live:
            a, _ = naive_ref.naive_move(agents[g].board(), agents[g].env.turn, naive_seed, g * 81 + len(moves[g]))
            agents[g].ensure_action_exists(a, ev)
            if play(g, a):
                nxt.append(g)
        live = nxt
        if not live:
            break
        orc.execute([agents[g] for g in live], count, batch, eps, alpha, ev)
        live = [g for g in live if play(g, agents[g].sample_action(0)[0])]
    return moves, final, (tally[2], tally[3], tally[1])


@pytest.mark.parametrize("first_tree", [0, 5])
def test_eval_naive_matches_the_oracle_loop(omk, orc, arena, first_tree):
    games, count, batch, eps, alpha, seed, nseed = 10, 64, 16, 0.25, 0.03, 11, 5
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=first_tree + games, capacity_nodes=2048, seed=seed)
    result, moves, status, stats = ctx.eval_naive(games, count=count, batch_size=batch, epsilon=eps, alpha=alpha,
                                                  evaluator=omk.EVAL_HASH, seed=nseed, first_tree=first_tree)
    listed = []
    assert arena.play_against_naive_player_device(ctx, episode_count=games, count=count, batch_size=batch, epsilon=eps, alpha=alpha,
                                                  evaluator=omk.EVAL_HASH, seed=nseed, first_tree=first_tree, moves_out=listed) == result
    ctx.close()
    want_moves, want_final, want_result = _oracle_eval(orc, games, count, batch, eps, alpha, seed, nseed, first_tree)
    assert listed == want_moves
    for g in range(games):
        row = moves[g].tolist()
        assert row[: len(want_moves[g])] == want_moves[g] and all(a == -1 for a in row[len(want_moves[g]):])
    assert status.tolist() == want_final
    assert result == want_result
    assert stats["moves"] == sum(len(m) for m in want_moves)


def _host_eval(omk, ctx, games, count, batch, nseed):
    """The same evaluation driven from the host, one entry point per step."""
    ids = np.arange(games, dtype=np.int32)
    ctx.pool_new_games(ids=ids, evaluator=omk.EVAL_NET)
    moves = [[] for _ in range(games)]
    final = np.zeros(games, np.int8)
    live = ids

    def record(actions, status):
        for g, a, st in zip(live, actions, status):
            moves[g].append(int(a))
            final[g] = st
        return live[status == 0]

    while live.size:
        boards, turns, _, _ = ctx.pool_get_envs(ids=live)
        streams = np.array([g * 81 + len(moves[g]) for g in live], np.uint32)
        actions, _ = ctx.naive_move(boards, turns, nseed, streams=streams)
        ctx.pool_ensure_action(actions, ids=live, evaluator=omk.EVAL_NET)
        live = record(actions, ctx.pool_play(actions, ids=live))
        if not live.size:
            break
        ctx.pool_search(ids=live, count=count, batch_size=batch, epsilon=0.25, alpha=0.03, evaluator=omk.EVAL_NET)
        actions, _ = ctx.pool_sample(ids=live, modes=np.zeros(live.size, np.uint8))
        live = record(actions, ctx.pool_play(actions, ids=live))
    result = tuple(int(np.count_nonzero(final == s)) for s in (2, 3, 1))
    return result, moves, final


def test_eval_naive_network_matches_the_host_loop_on_one_and_two_lanes(omk):
    games, count, batch, nseed = 64, 32, 16, 8
    runs = []
    for lanes in (1, 2):
        ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=games, capacity_nodes=1024, seed=4)
        ctx.net_init_random(6)
        if lanes == 2:
            ctx.debug_set_lane_min_trees(2)
        runs.append(ctx.eval_naive(games, count=count, batch_size=batch, evaluator=omk.EVAL_NET, seed=nseed))
        ctx.close()
    (r1, m1, s1, _), (r2, m2, s2, _) = runs
    assert r1 == r2 and np.array_equal(m1, m2) and np.array_equal(s1, s2)
    host = omk.Context(device=0, capacity_envs=1, capacity_trees=games, capacity_nodes=1024, seed=4)
    host.net_init_random(6)
    want_result, want_moves, want_final = _host_eval(omk, host, games, count, batch, nseed)
    host.close()
    assert r1 == want_result and sum(r1) == games
    assert [[int(a) for a in row if a >= 0] for row in m1] == want_moves
    assert np.array_equal(s1, want_final)


def test_eval_naive_between_selfplay_runs_and_after_training(omk):
    n_games, plies, cap = 8, 30, 4096

    def make():
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=3 * n_games, capacity_nodes=1024, seed=21)
        c.net_init_random(2)
        c.replay_reset(cap)
        c.selfplay_begin(n_games, 16, 8, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        return c

    a, b = make(), make()
    out_a = [a.selfplay_run(plies)[1:]]
    out_b = [b.selfplay_run(plies)[1:]]
    res = a.eval_naive(n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET, seed=1, first_tree=2 * n_games)
    assert sum(res[0]) == n_games
    with pytest.raises(omk.OmkError) as e:
        a.eval_naive(n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET, first_tree=2 * n_games - 1)
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
    # an evaluation right after a training phase plays the trained weights
    a.train_replay(3, 0, 4, 64)
    got = a.eval_naive(n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET, seed=2, first_tree=2 * n_games)
    fresh = omk.Context(device=0, capacity_envs=1, capacity_trees=3 * n_games, capacity_nodes=1024, seed=21)
    fresh.net_load_params(a.net_get_params())
    want = fresh.eval_naive(n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET, seed=2, first_tree=2 * n_games)
    assert got[0] == want[0] and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2])
    for c in (a, b, fresh):
        c.close()


def test_eval_naive_errors_and_accounting(omk):
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=8, capacity_nodes=2048, seed=3)
    H = omk.EVAL_HASH
    for kw in (dict(episodes=0), dict(episodes=9), dict(episodes=4, first_tree=5), dict(episodes=4, first_tree=-1),
               dict(episodes=4, batch_size=0), dict(episodes=4, batch_size=65), dict(episodes=4, count=0),
               dict(episodes=4, evaluator=7)):
        args = dict(count=16, batch_size=8, evaluator=H)
        args.update(kw)
        with pytest.raises(omk.OmkError) as e:
            ctx.eval_naive(**args)
        assert e.value.code == ERR_INVALID, kw
    with pytest.raises(omk.OmkError) as e:  # no weights loaded
        ctx.eval_naive(4, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(True)
    with pytest.raises(omk.OmkError) as e:
        ctx.eval_naive(4, count=16, batch_size=8, evaluator=H)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(False)
    # accounting on a context with a single env slot
    h2d0 = ctx.transfer_bytes[0]
    result, moves, status, stats = ctx.eval_naive(8, count=48, batch_size=16, evaluator=H, seed=9)
    assert ctx.transfer_bytes[0] == h2d0
    assert sum(result) == 8
    assert result == tuple(int(np.count_nonzero(status == s)) for s in (2, 3, 1))
    played = (moves >= 0).sum(axis=1)
    assert stats["moves"] == int(played.sum()) and stats["host_syncs"] <= stats["moves"] + 2
    assert all((moves[g, : played[g]] >= 0).all() and (moves[g, played[g]:] == -1).all() for g in range(8))
    assert stats["simulations"] > 0 and stats["nn_evals"] > 0 and stats["gpu_ms"] > 0
    ctx.close()
    small = omk.Context(device=0, capacity_envs=1, capacity_trees=4, capacity_nodes=8, seed=3)
    with pytest.raises(omk.OmkError) as e:
        small.eval_naive(4, count=64, batch_size=16, evaluator=H)
    assert e.value.code == ERR_CAPACITY
    small.close()


def test_iteration_with_an_evaluation_phase():
    """tools/iteration.py --device-replay --evaluate at a small size: the trained weights play every game to its end."""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    iteration = importlib.import_module("iteration")
    out = iteration.run(games_per_gpu=16, plies=80, count=16, batch=16, steps=4, minibatch=64, quiet=True, device_replay=True,
                        replay_capacity=256, evaluate=8)
    assert out["eval_naive_wins"] + out["eval_model_wins"] + out["eval_draws"] == 8
    assert out["eval_phase_s"] > 0 and out["eval_host_syncs"] <= out["eval_moves"] + 2
