"""The tournament with the naive player as participant 0 (omk_tournament_naive): its model-model pairings against
omk_tournament, the games the naive player opens against omk_eval_naive, both legs of its pairings against the oracle loop
(hash evaluator) and against granular host loops (network evaluator, two lanes and one), independence of the slot order,
the naive side's reserved trees left alone, coexistence with the self-play driver, the call's errors and accounting, and
tools/rate_checkpoints.py."""
import importlib
import os
import sys

import numpy as np
import pytest

import naive_ref
from oracle import net_oracle
from test_eval_naive_gpu import _oracle_eval

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_CAPACITY, ERR_STATE, ERR_NUMERIC = -1, -3, -4, -5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def arena():
    return importlib.import_module("omok-ai_b200.arena")


def _pairings(n):
    return [(i, j) for i in range(n) for j in range(i + 1, n)]


def _rows(moves):
    return [[int(a) for a in row if a >= 0] for row in moves]


def _tally(status, pairs):
    """{left wins, right wins, draws} of one pairing from its games' final statuses: BlackWin is the opener's."""
    out = [0, 0, 0]
    for g, st in enumerate(status.tolist()):
        if st == 1:
            out[2] += 1
        else:
            opener = 0 if g < pairs else 1
            out[opener if st == 2 else 1 - opener] += 1
    return out


def _oracle_model_opens(orc, pairs, count, batch, eps, alpha, ctx_seed, naive_seed):
    """Leg 1 of a naive pairing in the oracle: game pairs + g, the model opening on its agent of stream g, the naive player
    answering on stream (pairs + g) * 81 + ply."""
    ev = orc.NativeHashEvaluator()
    agents = {g: orc.Agent(ev, ctx_seed, g) for g in range(pairs)}
    moves = [[] for _ in range(pairs)]
    final = [0] * pairs

    def play(g, a):
        moves[g].append(a)
        st = agents[g].play_action(a)
        final[g] = st
        return st == 0

    live = list(range(pairs))
    while live:
        orc.execute([agents[g] for g in live], count, batch, eps, alpha, ev)
        live = [g for g in live if play(g, agents[g].sample_action(0)[0])]
        nxt = []
        for g in live:
            a, _ = naive_ref.naive_move(agents[g].board(), agents[g].env.turn, naive_seed, (pairs + g) * 81 + len(moves[g]))
            agents[g].ensure_action_exists(a, ev)
            if play(g, a):
                nxt.append(g)
        live = nxt
    return moves, final


def _host_naive_pairing(omk, ctx, pairs, count, batch, eps, alpha, nseed, evaluator):
    """Both legs of a naive pairing driven from the host, one entry point per step, with the context's network as the model:
    `arena.play_match`'s loop with the naive player's side replaced by naive_move on stream g * 81 + h.  Trees 0 .. pairs - 1,
    tree g on stream g, serve game g of each leg in turn.  Returns (move lists, final statuses) of the 2 * pairs games."""
    moves = [[] for _ in range(2 * pairs)]
    final = np.zeros(2 * pairs, np.int8)
    for leg in (0, 1):
        ids = np.arange(pairs, dtype=np.int32)
        ctx.pool_new_games(ids=ids, evaluator=evaluator)
        live = ids
        naive_turn = leg == 0
        while live.size:
            games = leg * pairs + live
            if naive_turn:
                boards, turns, _, _ = ctx.pool_get_envs(ids=live)
                streams = np.array([g * 81 + len(moves[g]) for g in games], np.uint32)
                actions, _ = ctx.naive_move(boards, turns, nseed, streams=streams)
                ctx.pool_ensure_action(actions, ids=live, evaluator=evaluator)
            else:
                ctx.pool_search(ids=live, count=count, batch_size=batch, epsilon=eps, alpha=alpha, evaluator=evaluator)
                actions, _ = ctx.pool_sample(ids=live, modes=np.zeros(live.size, np.uint8))
            status = ctx.pool_play(actions, ids=live)
            for g, a, st in zip(games, actions, status):
                moves[g].append(int(a))
                final[g] = st
            live = live[status == 0]
            naive_turn = not naive_turn
    return moves, final


@pytest.mark.parametrize("n_models", [1, 2, 4])
@pytest.mark.parametrize("pairs", [3, 8])
@pytest.mark.parametrize("first_tree", [0, 5])
def test_tournament_naive_hash_evaluator(omk, orc, arena, n_models, pairs, first_tree):
    seed, nseed, count, batch, eps, alpha = 13, 29, 32, 8, 0.25, 0.03
    N = n_models + 1
    P = N * (N - 1) // 2
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=first_tree + 4 * pairs * P, capacity_nodes=2048, seed=seed)
    slots = list(range(n_models))[::-1]
    kw = dict(count=count, batch_size=batch, epsilon=eps, alpha=alpha, evaluator=omk.EVAL_HASH)
    result, moves, status, stats = ctx.tournament_naive(slots, pairs, seed=nseed, first_tree=first_tree, **kw)
    listed = []
    table = arena.play_tournament_naive_device(ctx, slots, seed=nseed, game_count=2 * pairs, first_tree=first_tree, moves_out=listed, **kw)
    assert table.tobytes() == result.tobytes()
    assert listed == [_rows(m) for m in moves]
    # model-model pairings: omk_tournament's, game by game
    if n_models >= 2:
        tour = ctx.tournament(slots, pairs, first_tree=first_tree, **kw)
        assert result[n_models:].tobytes() == tour[0].tobytes()
        assert moves[n_models:].tobytes() == tour[1].tobytes() and status[n_models:].tobytes() == tour[2].tobytes()
    ctx.close()
    # the games the naive player opens: omk_eval_naive's, on a second context with the same seed
    ref = omk.Context(device=0, capacity_envs=1, capacity_trees=pairs, capacity_nodes=2048, seed=seed)
    ev = ref.eval_naive(pairs, seed=nseed, **kw)
    ref.close()
    want0, final0, _ = _oracle_eval(orc, pairs, count, batch, eps, alpha, seed, nseed, 0)
    want1, final1 = _oracle_model_opens(orc, pairs, count, batch, eps, alpha, seed, nseed)
    for k in range(n_models):
        assert moves[k, :pairs].tobytes() == ev[1].tobytes() and status[k, :pairs].tobytes() == ev[2].tobytes(), k
        assert _rows(moves[k]) == want0 + want1, k
        assert status[k].tolist() == final0 + final1, k
        assert result[k].tolist() == _tally(status[k], pairs), k
    assert (result.sum(axis=1) == 2 * pairs).all()
    assert stats["moves"] == int((moves >= 0).sum())
    assert stats["host_syncs"] == int((moves >= 0).sum(axis=2).max()) + 1


def _net_ctx(omk, weights, trees, seed, network):
    c = omk.Context(device=0, capacity_envs=1, capacity_trees=trees, capacity_nodes=2048, seed=seed)
    c.net_load_params(weights[network])
    return c


@pytest.mark.parametrize("min_trees", [None, 0], ids=["lanes", "one_lane"])
def test_tournament_naive_network_evaluator_is_the_host_loops(omk, arena, min_trees):
    slots, pairs, seed, nseed, count, batch = (3, 0, 2), 3, 5, 41, 16, 8
    N = len(slots) + 1
    P = N * (N - 1) // 2
    weights = {s: net_oracle.random_params(30 + s) for s in slots}
    kw = dict(count=count, batch_size=batch, epsilon=0.0, alpha=1.0, evaluator=omk.EVAL_NET)

    def play(order):
        ctx = _net_ctx(omk, weights, 4 * pairs * P, seed, 0)
        for s in order:
            if s:
                ctx.model_load_params(s, weights[s])
        if min_trees is not None:
            ctx.debug_set_lane_min_trees(min_trees)
        out = ctx.tournament_naive(list(order), pairs, seed=nseed, **kw)
        ctx.close()
        return out

    result, moves, status, _ = play(slots)
    pairings = _pairings(N)
    for p, (a, b) in enumerate(pairings):
        if a == 0:  # the naive player against slots[b - 1]
            host = _net_ctx(omk, weights, pairs, seed, slots[b - 1])
            want_moves, want_final = _host_naive_pairing(omk, host, pairs, count, batch, 0.0, 1.0, nseed, omk.EVAL_NET)
            host.close()
            assert status[p].tobytes() == want_final.tobytes(), p
            # leg 0 is omk_eval_naive's evaluation with this network
            ref = _net_ctx(omk, weights, pairs, seed, slots[b - 1])
            ev = ref.eval_naive(pairs, seed=nseed, **kw)
            ref.close()
            assert moves[p, :pairs].tobytes() == ev[1].tobytes() and status[p, :pairs].tobytes() == ev[2].tobytes(), p
        else:  # slots[a - 1] against slots[b - 1]: arena.play_match on two contexts
            left = _net_ctx(omk, weights, pairs, seed, slots[a - 1])
            right = _net_ctx(omk, weights, pairs, seed, slots[b - 1])
            want_moves = []
            want = arena.play_match(left, right, game_count=2 * pairs, moves_out=want_moves, **kw)
            left.close()
            right.close()
            assert tuple(int(x) for x in result[p]) == want, p
        assert _rows(moves[p]) == want_moves, p
        assert result[p].tolist() == _tally(status[p], pairs), p
    # another order of the same slots: the same games, the table permuted (a pairing whose sides swap swaps its legs)
    order = (2, 3, 0)
    r2, m2, s2, _ = play(order)
    part = lambda o, k: 0 if k == 0 else 1 + list(o).index(slots[k - 1])  # noqa: E731  participant of `o` for slots' k
    index = {pr: q for q, pr in enumerate(pairings)}
    for p, (a, b) in enumerate(pairings):
        x, y = part(order, a), part(order, b)
        q = index[(min(x, y), max(x, y))]
        if x < y:
            assert r2[q].tolist() == result[p].tolist() and m2[q].tobytes() == moves[p].tobytes() and s2[q].tobytes() == status[p].tobytes()
        else:
            assert r2[q].tolist() == [result[p][1], result[p][0], result[p][2]]
            assert m2[q].tobytes() == np.roll(moves[p], pairs, axis=0).tobytes()
            assert s2[q].tobytes() == np.roll(status[p], pairs).tobytes()


def test_tournament_naive_leaves_the_naive_sides_trees_alone(omk):
    n_models, pairs, seed = 2, 3, 7
    N = n_models + 1
    P = N * (N - 1) // 2
    trees = 4 * pairs * P
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=trees, capacity_nodes=2048, seed=seed)
    ids = np.arange(trees, dtype=np.int32)
    ctx.pool_new_games(ids=ids, evaluator=omk.EVAL_HASH)  # earlier games on every tree: a search and a move
    ctx.pool_search(ids=ids, count=24, batch_size=8, epsilon=0.25, alpha=0.03, evaluator=omk.EVAL_HASH)
    actions, _ = ctx.pool_sample(ids=ids, modes=np.zeros(trees, np.uint8))
    ctx.pool_play(actions, ids=ids)
    ctx.pool_search(ids=ids, count=8, batch_size=8, epsilon=0.25, alpha=0.03, evaluator=omk.EVAL_HASH)
    reserved = [4 * pairs * p + i for p in range(n_models) for i in range(2 * pairs)]

    def snapshot():
        return [(ctx.pool_tree_info(t), [np.asarray(x).tobytes() for x in ctx.pool_root_stats(t)], ctx.pool_get_env(t)[0].tobytes())
                for t in reserved]

    before = snapshot()
    result, _, _, _ = ctx.tournament_naive(list(range(n_models)), pairs, seed=3, count=32, batch_size=8, evaluator=omk.EVAL_HASH)
    assert (result.sum(axis=1) == 2 * pairs).all()
    assert snapshot() == before
    ctx.close()


def test_tournament_naive_between_selfplay_runs_leaves_self_play_unchanged(omk):
    n_games, plies, cap, pairs = 8, 30, 4096, 2

    def make():
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * n_games + 24 * pairs, capacity_nodes=1024, seed=21)
        c.net_init_random(2)
        c.replay_reset(cap)
        c.selfplay_begin(n_games, 16, 8, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        return c

    a, b = make(), make()
    out_a = [a.selfplay_run(plies)[1:]]
    out_b = [b.selfplay_run(plies)[1:]]
    a.opponent_load_params(net_oracle.random_params(6))
    a.model_load_params(4, net_oracle.random_params(7))
    res = a.tournament_naive([0, 1, 4], pairs, seed=5, first_tree=2 * n_games, count=16, batch_size=8, evaluator=omk.EVAL_NET)
    assert (res[0].sum(axis=1) == 2 * pairs).all()
    with pytest.raises(omk.OmkError) as e:
        a.tournament_naive([0, 1, 4], pairs, first_tree=2 * n_games - 1, count=16, batch_size=8, evaluator=omk.EVAL_NET)
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


def test_tournament_naive_errors_and_accounting(omk, arena):
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=40, capacity_nodes=2048, seed=3)
    H, N = omk.EVAL_HASH, omk.EVAL_NET
    for kw in (dict(slots=[]), dict(slots=list(range(17))), dict(slots=[0, 2, 0]), dict(slots=[0, 16]), dict(slots=[-1, 0]),
               dict(pairs=0), dict(pairs=4), dict(first_tree=5), dict(first_tree=-1), dict(batch_size=0), dict(batch_size=65),
               dict(count=0), dict(evaluator=7)):
        args = dict(slots=[0, 1], pairs=3, count=16, batch_size=8, evaluator=H)  # 3 participants: 3 pairings x 12 trees = 36 of 40
        args.update(kw)
        with pytest.raises(omk.OmkError) as e:
            ctx.tournament_naive(**args)
        assert e.value.code == ERR_INVALID, kw
    slots = np.array([0, 1], np.int32)  # a NULL out_result
    assert ctx.L.omk_tournament_naive(ctx.h, 2, slots.ctypes.data, 3, 0, 16, 8, 0.0, 1.0, H, 0, None, None, None, None, None) == ERR_INVALID
    # the hash evaluator needs no weights at all: the naive player never evaluates
    result, _, _, _ = ctx.tournament_naive([9], 2, count=16, batch_size=8, evaluator=H)
    assert result.shape == (1, 3) and result.sum() == 4
    with pytest.raises(omk.OmkError) as e:  # no network
        ctx.tournament_naive([0], 2, count=16, evaluator=N)
    assert e.value.code == ERR_STATE
    ctx.net_load_params(net_oracle.random_params(7))
    ctx.model_load_params(3, net_oracle.random_params(8))
    with pytest.raises(omk.OmkError) as e:  # slot 1 was never loaded
        ctx.tournament_naive([3, 1], 2, count=16, evaluator=N)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(True)
    with pytest.raises(omk.OmkError) as e:
        ctx.tournament_naive([3], 2, count=16, evaluator=H)
    assert e.value.code == ERR_STATE
    ctx.search_set_virtual_loss(False)
    # accounting
    h2d0 = ctx.transfer_bytes[0]
    result, moves, status, stats = ctx.tournament_naive([3, 0], 3, seed=4, count=48, batch_size=16, evaluator=H)
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
    elo = arena.ratings(result, 3)
    assert elo[0] == 0.0 and np.isfinite(elo).all()
    ctx.close()
    small = omk.Context(device=0, capacity_envs=1, capacity_trees=24, capacity_nodes=8, seed=3)
    with pytest.raises(omk.OmkError) as e:
        small.tournament_naive([0, 1], 2, count=64, batch_size=16, evaluator=H)
    assert e.value.code == ERR_CAPACITY
    small.close()
    # a slot whose activations leave the fp16 operand range stops the call at the half-move that produced it
    params = net_oracle.random_params(0)
    bad = [p.copy() for p in params]
    bad[0] = bad[0] * np.float32(1e5)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=24, capacity_nodes=2048, seed=1)
    ctx.net_load_params(params)
    ctx.model_load_params(6, bad)
    with pytest.raises(omk.OmkError) as e:
        ctx.tournament_naive([0, 6], 2, count=16, batch_size=8, evaluator=N)
    assert e.value.code == ERR_NUMERIC
    result, _, _, _ = ctx.tournament_naive([0], 2, count=16, batch_size=8, evaluator=N)
    assert result.sum() == 4
    ctx.close()


def test_rate_checkpoints_rates_two_files_as_the_call_it_wraps(omk, arena, tmp_path):
    model_io = importlib.import_module("omok-ai_b200.model_io")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    rate = importlib.import_module("rate_checkpoints")
    weights = [net_oracle.random_params(50 + k) for k in range(2)]
    files = []
    for k, w in enumerate(weights):
        files.append(str(tmp_path / f"ckpt{k}.bin"))
        model_io.save(files[-1], w)
    games, count, seed = 6, 16, 3
    out = rate.main(files, games=games, count=count, seed=seed, nodes=1024, quiet=True)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=4 * (games // 2) * 3, capacity_nodes=1024, seed=seed)
    ctx.net_load_params(weights[0])
    ctx.model_load_params(1, weights[1])
    result, _, _, _ = ctx.tournament_naive([0, 1], games // 2, seed=seed, count=count, batch_size=8, evaluator=omk.EVAL_NET)
    ctx.close()
    assert out["table"] == result.tolist()
    elo = arena.ratings(result, 3)
    assert out["ratings"] == [float(x) for x in elo] and out["ratings"][0] == 0.0
    for k, row in enumerate(out["models"]):
        assert row["file"] == files[k] and row["elo"] == float(elo[k + 1])
        assert (row["losses"], row["wins"], row["draws"]) == tuple(int(x) for x in result[k])
