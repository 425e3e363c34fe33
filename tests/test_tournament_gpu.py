"""Model slots and the tournament on the device (omk_model_*, omk_tournament): each slot's forward pass against a context
holding the same weights as its network, every pairing of a tournament against the omk_match call it stands for (hash and
network evaluators, two lanes and one), two models as a match, coexistence with the self-play driver, and the call's
errors and accounting."""
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


def _pairings(n):
    return [(i, j) for i in range(n) for j in range(i + 1, n)]


def _assert_pairing_is_the_match(tour, p, match):
    result, moves, status, _ = tour
    m_result, m_moves, m_status, _ = match
    assert tuple(int(x) for x in result[p]) == m_result, p
    assert moves[p].tobytes() == m_moves.tobytes(), p
    assert status[p].tobytes() == m_status.tobytes(), p


def _same_eval(got, want):
    return got[0].tobytes() == want[0].tobytes() and got[1].tobytes() == want[1].tobytes()


def test_model_slots_hold_the_weights_they_were_given(omk):
    weights = {s: net_oracle.random_params(10 + s) for s in range(16)}
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
    ctx.net_load_params(weights[0])
    ctx.opponent_load_params(weights[1])
    cases = [(n, mode, _positions(n, seed=n + 7 * mode)) for n in (1, 5, 300, 4096) for mode in (0, 1)]
    before = [(ctx.net_eval(b, t, mode=mode), ctx.opponent_eval(b, t, mode=mode)) for _, mode, (b, t) in cases]
    for s in range(2, 16):
        ctx.model_load_params(s, weights[s])
    for s in (0, 1, 2, 9, 15):
        ref = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
        ref.net_load_params(weights[s])
        for n, mode, (b, t) in cases:
            assert _same_eval(ctx.model_eval(s, b, t, mode=mode), ref.net_eval(b, t, mode=mode)), (s, n, mode)
        ref.close()
    for (n, mode, (b, t)), (net_out, opp_out) in zip(cases, before):  # loading slots 2 .. 15 changed neither
        assert _same_eval(ctx.net_eval(b, t, mode=mode), net_out), (n, mode)
        assert _same_eval(ctx.opponent_eval(b, t, mode=mode), opp_out), (n, mode)
        assert _same_eval(ctx.model_eval(1, b, t, mode=mode), opp_out), (n, mode)
    ctx.close()


def test_a_slot_snapshot_of_the_network_survives_training(omk):
    w = net_oracle.random_params(5)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
    ctx.net_load_params(w)
    ctx.model_from_net(5)
    rng = np.random.default_rng(0)
    for _ in range(3):
        images = (rng.random((64, 243)) < 0.2).astype(np.float32)
        pi = rng.random((64, 81)).astype(np.float32)
        pi /= pi.sum(axis=1, keepdims=True)
        ctx.train_step(images, pi, rng.choice([-1.0, 1.0], 64).astype(np.float32))
    trained = ctx.net_get_params()
    assert any(not np.array_equal(a, b) for a, b in zip(trained, w))
    boards, turns = _positions(300, seed=1)
    for params, slot in ((w, 5), (trained, 0)):  # slot 0: the trained weights, packed on the way in
        fresh = omk.Context(device=0, capacity_envs=1, capacity_trees=1, capacity_nodes=16, seed=0)
        fresh.net_load_params(params)
        assert _same_eval(ctx.model_eval(slot, boards, turns), fresh.net_eval(boards, turns)), slot
        fresh.close()
    ctx.close()


@pytest.mark.parametrize("n_models", [2, 3, 5])
@pytest.mark.parametrize("pairs", [1, 3])
@pytest.mark.parametrize("first_tree", [0, 7])
def test_tournament_hash_evaluator_is_one_match_per_pairing(omk, arena, n_models, pairs, first_tree):
    seed, count, batch = 13, 32, 8
    P = n_models * (n_models - 1) // 2
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=first_tree + 4 * pairs * P, capacity_nodes=2048, seed=seed)
    slots = list(range(n_models))[::-1]
    tour = ctx.tournament(slots, pairs, first_tree=first_tree, count=count, batch_size=batch, evaluator=omk.EVAL_HASH)
    listed = []
    table = arena.play_tournament_device(ctx, slots, game_count=2 * pairs, count=count, batch_size=batch, evaluator=omk.EVAL_HASH,
                                         first_tree=first_tree, moves_out=listed)
    assert table.tobytes() == tour[0].tobytes()
    total = {"simulations": 0, "nn_evals": 0, "moves": 0}
    for p in range(P):
        match = ctx.match(pairs, first_tree=first_tree + 4 * pairs * p, count=count, batch_size=batch, evaluator=omk.EVAL_HASH)
        _assert_pairing_is_the_match(tour, p, match)
        assert listed[p] == [[int(a) for a in row if a >= 0] for row in match[1]]
        for k in total:
            total[k] += match[3][k]
        assert sum(match[0]) == 2 * pairs
    for k in total:
        assert tour[3][k] == total[k], k
    ctx.close()


@pytest.mark.parametrize("min_trees", [None, 0], ids=["lanes", "one_lane"])
def test_tournament_network_evaluator_is_one_match_per_pairing(omk, min_trees):
    slots, pairs, seed, count, batch = (3, 0, 2, 7), 3, 5, 16, 8
    P = len(slots) * (len(slots) - 1) // 2
    weights = {s: net_oracle.random_params(30 + s) for s in slots}
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs * P, capacity_nodes=2048, seed=seed)
    ctx.net_load_params(weights[0])
    for s in slots:
        if s:
            ctx.model_load_params(s, weights[s])
    if min_trees is not None:
        ctx.debug_set_lane_min_trees(min_trees)
    tour = ctx.tournament(slots, pairs, count=count, batch_size=batch, evaluator=omk.EVAL_NET)
    ctx.close()
    ref = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs * P, capacity_nodes=2048, seed=seed)
    for p, (i, j) in enumerate(_pairings(len(slots))):
        ref.net_load_params(weights[slots[i]])
        ref.opponent_load_params(weights[slots[j]])
        _assert_pairing_is_the_match(tour, p, ref.match(pairs, first_tree=4 * pairs * p, count=count, batch_size=batch,
                                                        evaluator=omk.EVAL_NET))
    ref.close()


def test_two_models_are_a_match(omk):
    pairs, seed, count, batch = 4, 9, 16, 8
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * pairs, capacity_nodes=2048, seed=seed)
    ctx.net_load_params(net_oracle.random_params(1))
    ctx.opponent_load_params(net_oracle.random_params(2))
    tour = ctx.tournament([0, 1], pairs, count=count, batch_size=batch, evaluator=omk.EVAL_NET)
    match = ctx.match(pairs, count=count, batch_size=batch, evaluator=omk.EVAL_NET)
    _assert_pairing_is_the_match(tour, 0, match)
    for k in ("simulations", "nn_evals", "moves", "host_syncs"):
        assert tour[3][k] == match[3][k], k
    ctx.close()


def test_tournament_between_selfplay_runs_leaves_self_play_unchanged(omk):
    n_games, plies, cap, pairs = 8, 30, 4096, 2

    def make():
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * n_games + 12 * pairs, capacity_nodes=1024, seed=21)
        c.net_init_random(2)
        c.replay_reset(cap)
        c.selfplay_begin(n_games, 16, 8, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        return c

    a, b = make(), make()
    out_a = [a.selfplay_run(plies)[1:]]
    out_b = [b.selfplay_run(plies)[1:]]
    a.opponent_load_params(net_oracle.random_params(6))
    a.model_load_params(4, net_oracle.random_params(7))
    res = a.tournament([0, 1, 4], pairs, first_tree=2 * n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert (res[0].sum(axis=1) == 2 * pairs).all()
    with pytest.raises(omk.OmkError) as e:
        a.tournament([0, 1, 4], pairs, first_tree=2 * n_games - 1, count=16, batch_size=8, evaluator=omk.EVAL_NET)
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


def test_tournament_errors_and_accounting(omk):
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=40, capacity_nodes=2048, seed=3)
    H, N = omk.EVAL_HASH, omk.EVAL_NET
    for kw in (dict(slots=[0]), dict(slots=list(range(17))), dict(slots=[0, 2, 0]), dict(slots=[0, 16]), dict(slots=[-1, 0]),
               dict(pairs=0), dict(pairs=4), dict(first_tree=5), dict(first_tree=-1), dict(batch_size=0), dict(batch_size=65),
               dict(count=0), dict(evaluator=7)):
        args = dict(slots=[0, 1, 2], pairs=3, count=16, batch_size=8, evaluator=H)  # 3 pairings x 12 trees = 36 of 40
        args.update(kw)
        with pytest.raises(omk.OmkError) as e:
            ctx.tournament(**args)
        assert e.value.code == ERR_INVALID, kw
    slots = np.array([0, 1, 2], np.int32)  # a NULL out_result
    assert ctx.L.omk_tournament(ctx.h, 3, slots.ctypes.data, 3, 0, 16, 8, 0.0, 1.0, H, None, None, None, None, None) == ERR_INVALID
    w = net_oracle.random_params(7)
    for call in (lambda: ctx.model_load_params(0, w), lambda: ctx.model_load_params(16, w), lambda: ctx.model_from_net(0),
                 lambda: ctx.model_load_params(3, w[:3] + [w[3][:-1]] + w[4:]),  # a tensor of the wrong length
                 lambda: ctx.model_eval(16, np.zeros((1, 81), np.uint8), [0])):
        with pytest.raises(omk.OmkError) as e:
            call()
        assert e.value.code == ERR_INVALID
    for call in (lambda: ctx.tournament([0, 1], 2, count=16, evaluator=N),           # no network
                 lambda: ctx.model_from_net(3),                                      # no network to copy
                 lambda: ctx.model_eval(3, np.zeros((1, 81), np.uint8), [0])):       # an empty slot
        with pytest.raises(omk.OmkError) as e:
            call()
        assert e.value.code == ERR_STATE
    ctx.net_load_params(w)
    ctx.model_load_params(3, net_oracle.random_params(8))
    with pytest.raises(omk.OmkError) as e:  # slot 1 was never loaded
        ctx.tournament([0, 3, 1], 2, count=16, evaluator=N)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(True)
    with pytest.raises(omk.OmkError) as e:
        ctx.tournament([0, 3], 2, count=16, evaluator=H)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(False)
    # accounting
    h2d0 = ctx.transfer_bytes[0]
    result, moves, status, stats = ctx.tournament([3, 0, 5], 3, count=48, batch_size=16, evaluator=H)
    assert ctx.transfer_bytes[0] == h2d0
    assert (result.sum(axis=1) == 6).all()
    played = (moves >= 0).sum(axis=2)
    assert stats["moves"] == int(played.sum())
    assert stats["host_syncs"] == int(played.max()) + 1
    for p in range(3):
        for g in range(6):
            assert (moves[p, g, : played[p, g]] >= 0).all() and (moves[p, g, played[p, g]:] == -1).all()
            assert status[p, g] in (1, 2, 3)
    assert stats["simulations"] > 0 and stats["nn_evals"] > 0 and stats["gpu_ms"] > 0
    ctx.close()
    small = omk.Context(device=0, capacity_envs=1, capacity_trees=24, capacity_nodes=8, seed=3)
    with pytest.raises(omk.OmkError) as e:
        small.tournament([0, 1, 2], 2, count=64, batch_size=16, evaluator=H)
    assert e.value.code == ERR_CAPACITY
    small.close()


def test_tournament_reports_a_non_finite_model(omk):
    """A slot whose activations leave the fp16 operand range answers OMK_ERR_NUMERIC in omk_model_eval and stops
    omk_tournament at the half-move that produced it; the network and the other slots then play as before."""
    params = net_oracle.random_params(0)
    bad = [p.copy() for p in params]
    bad[0] = bad[0] * np.float32(1e5)  # stem weights x 1e5: the residual stream leaves the fp16 range
    boards, turns = _positions(5, seed=3)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=24, capacity_nodes=2048, seed=1)
    ctx.net_load_params(params)
    ctx.model_load_params(2, net_oracle.random_params(1))
    ctx.model_load_params(6, bad)
    with pytest.raises(omk.OmkError) as e:
        ctx.model_eval(6, boards, turns)
    assert e.value.code == ERR_NUMERIC
    with pytest.raises(omk.OmkError) as e:
        ctx.tournament([0, 6, 2], 2, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert e.value.code == ERR_NUMERIC
    for s in (0, 2):
        p, v = ctx.model_eval(s, boards, turns)
        assert np.isfinite(p).all() and np.isfinite(v).all()
    result, _, _, _ = ctx.tournament([2, 0], 2, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert result.sum() == 4
    ctx.close()
