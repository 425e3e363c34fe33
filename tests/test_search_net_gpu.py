"""Network-evaluated search (EVAL_NET, the self-play path) against the oracle, bit for bit, at the pool sizes and in the
late-game regime self-play runs in.

Recorded mode: the oracle (orc.Agent / orc.execute) is driven by the same context's network through `net_eval`, which rests
on the network's batch invariance (tests/test_net_gpu.py::test_batch_invariance).  The recorder evaluates the oracle's rows
in batches of at most 128, so a reference row always comes from the split-K fc0 and the first 128-row tile: never from the
fc0 path, tile or row index the search's own launch gave the same position.  A search round reserves its evaluator rows on
the device (atomicAdd on n_req) and every network kernel clamps to that count, while the launches are sized on the host by
trees x batch; terminal leaves, full nodes and terminal children leave the count below that bound, which `net_eval` alone
never does.  The recorder logs (rows, mode) per call so that each test can show it reached the regime it is about."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_oracle_env import draw_moves, win81_moves  # noqa: E402
from test_tree_gpu import assert_tree_equal  # noqa: E402

pytestmark = pytest.mark.gpu

BATCH, EPS, ALPHA = 16, 0.25, 0.03  # the reference trainer's search settings (rounds of 16 requests per tree)
LANE_MIN_TREES = 768  # a context's default: searches over at least this many trees run as two lanes (omk_internal.h)
SPLIT_K_MAX_ROWS = 2048  # fc0 launches up to this bound take the split-K kernel, larger ones the CTA-pair kernel (fc_f16.cu)
REF_ROWS = 128  # the recorder's batch: one fc0 tile


@pytest.fixture(scope="module")
def params():
    from oracle import net_oracle

    return net_oracle.random_params(0)


def net_context(omk, params, trees, nodes, seed, lane_min=LANE_MIN_TREES):
    c = omk.Context(device=0, capacity_envs=4, capacity_trees=trees, capacity_nodes=nodes, seed=seed)
    c.net_load_params(params)
    if lane_min != LANE_MIN_TREES:
        c.debug_set_lane_min_trees(lane_min)
    return c


class Recorder:
    """The oracle's evaluator: `ctx.net_eval` on the oracle's rows, REF_ROWS at a time; `log` holds (rows, mode) per call."""

    def __init__(self, orc, ctx):
        self.log = []

        def evaluate(boards, turns, mode):
            self.log.append((len(boards), int(mode)))
            out = [ctx.net_eval(boards[i : i + REF_ROWS], turns[i : i + REF_ROWS], mode=mode) for i in range(0, len(boards), REF_ROWS)]
            return np.concatenate([p for p, _ in out]), np.concatenate([v for _, v in out])

        self.ev = orc.CallbackEvaluator(evaluate)


def lanes_of(ids, lane_min):
    """The trees of each search lane: the two halves of the id list, the first one larger (omk_api.cu search_rounds)."""
    if lane_min <= 0 or len(ids) < max(lane_min, 2):
        return [ids]
    h = (len(ids) + 1) // 2
    return [ids[:h], ids[h:]]


def search(ctx, omk, orc, rec, agents, ids, count, lane_min):
    """execute(count, 16, 0.25, 0.03) on the trees `ids` on the device, and lane by lane on their oracle agents (a tree's
    result does not depend on the other trees of its batch, so the oracle's rounds can follow the device's lanes).  Returns
    (rows, bound) for every round of every lane: rows the round evaluated, bound = the lane's trees x 16, the row count the
    network launches are sized for.  A round without requests evaluates nothing on the oracle and counts as 0 rows."""
    ctx.pool_search(ids=ids, count=count, batch_size=BATCH, epsilon=EPS, alpha=ALPHA, evaluator=omk.EVAL_NET)
    rounds = []
    for lane in lanes_of(ids, lane_min):
        first = len(rec.log)
        orc.execute([agents[t] for t in lane], count, BATCH, EPS, ALPHA, rec.ev)
        calls = rec.log[first:]
        assert all(mode == 0 for _, mode in calls), "search rounds evaluate in EnvTurnMode::Player"
        rows = [r for r, _ in calls] + [0] * (-(-count // BATCH) - len(calls))
        rounds += [(r, len(lane) * BATCH) for r in rows]
    return rounds


def sample_best_and_play(ctx, agents, ids, where):
    """pool_sample Best + pool_play on the trees `ids` and on their agents; returns the statuses."""
    acts, pol = ctx.pool_sample(ids=ids)
    ref = [agents[t].sample_action(0) for t in ids]
    assert [int(a) for a in acts] == [r[0] for r in ref], f"{where}: sampled actions"
    assert pol.tobytes() == np.stack([r[1] for r in ref]).tobytes(), f"{where}: visit policies"
    st = [int(s) for s in ctx.pool_play(acts, ids=ids)]
    assert st == [agents[t].play_action(int(a)) for t, a in zip(ids, acts)], f"{where}: play statuses"
    return st


def test_product_pool_two_lanes_matches_oracle(omk, orc, params):
    """1024 trees on the default lane threshold: two lanes of 512 trees, 8192 rows each, so fc0 runs as CTA pairs.  The
    reference trainer's search (800 simulations, rounds of 16, eps 0.25, alpha 0.03) from Agent::new's evaluation, then
    Best, play and 160 more simulations on the re-rooted trees; every tree compared with the oracle after each step."""
    T = 1024
    ctx = net_context(omk, params, T, 2048, seed=31)
    rec = Recorder(orc, ctx)
    agents = [orc.Agent(rec.ev, ctx.seed, t) for t in range(T)]  # stream == tree id
    ctx.pool_new_games(n=T, evaluator=omk.EVAL_NET)
    ids = list(range(T))
    assert len(lanes_of(ids, LANE_MIN_TREES)) == 2
    for t in ids:
        assert_tree_equal(ctx, t, agents[t], f"new game, tree {t}")
    rounds = search(ctx, omk, orc, rec, agents, ids, 800, LANE_MIN_TREES)
    for t in ids:
        assert_tree_equal(ctx, t, agents[t], f"800 simulations, tree {t}")
    st = sample_best_and_play(ctx, agents, ids, "first move")
    assert not any(st)
    for t in ids:
        assert_tree_equal(ctx, t, agents[t], f"re-rooted, tree {t}")
    rounds += search(ctx, omk, orc, rec, agents, ids, 160, LANE_MIN_TREES)
    for t in ids:
        assert_tree_equal(ctx, t, agents[t], f"160 more simulations, tree {t}")
    ctx.close()
    assert max(r for r, _ in rounds) > SPLIT_K_MAX_ROWS, "no round took the CTA-pair fc0"


def late_sequences(orc, n, seed):
    """n move sequences of 50..74 stones in which no move ends the game: random cells (seeded), each sequence kept only if it
    reaches its drawn length with every move InProgress; the first two are prefixes of the reference-derived draw /
    win-on-move-81 boards (tests/test_oracle_env.py)."""
    rng = np.random.default_rng(seed)
    out = [draw_moves()[:66], win81_moves()[:70]]
    while len(out) < n:
        k = int(rng.integers(50, 75))
        env = orc.Environment()
        moves = []
        for cell in rng.permutation(81)[:k]:
            if env.place_stone(int(cell)) != 0:
                break
            moves.append(int(cell))
        if len(moves) == k:
            out.append(moves)
    return out[:n]


def ceil_div(a, b):
    return -(-a // b)


@pytest.mark.parametrize(
    "trees,lane_min,fc0",
    [
        (48, LANE_MIN_TREES, "split-K"),  # 768-row bound: split-K fc0, six 128-row tiles
        (192, LANE_MIN_TREES, "pair"),  # 3072-row bound: CTA-pair fc0
        (320, 2, "pair"),  # two lanes of 160 trees, 2560 rows each: CTA pairs on both
    ],
)
def test_late_positions_fewer_rows_than_the_bound(omk, orc, params, trees, lane_min, fc0):
    """Late positions (50..74 stones) fed in move by move (pool_ensure_action + pool_play against ensure_action_exists +
    play_action: the ensure evaluations' rows), then every game played to its end by one tree: search (96 simulations in
    rounds of 16), Best, play.  Terminal leaves and terminal children are the rule there, so rounds evaluate fewer rows than
    their launches are sized for, and whole tiles / CTA pairs of the network kernels leave on the device's row count alone.
    Finished games leave the id list (ragged explicit ids); every tree is compared after every search and every play."""
    seqs = late_sequences(orc, trees, seed=trees)
    ctx = net_context(omk, params, trees, 4096, seed=1000 + trees, lane_min=lane_min)
    rec = Recorder(orc, ctx)
    agents = [orc.Agent(rec.ev, ctx.seed, t) for t in range(trees)]  # stream == tree id
    ctx.pool_new_games(n=trees, evaluator=omk.EVAL_NET)
    for k in range(max(len(s) for s in seqs)):
        ids = [g for g in range(trees) if k < len(seqs[g])]
        acts = [seqs[g][k] for g in ids]
        ctx.pool_ensure_action(acts, ids=ids, evaluator=omk.EVAL_NET)
        assert not np.any(ctx.pool_play(acts, ids=ids)), f"opening move {k}"
        for g, a in zip(ids, acts):
            agents[g].ensure_action_exists(a, rec.ev)
            assert agents[g].play_action(a) == 0
    for g in range(trees):
        assert_tree_equal(ctx, g, agents[g], f"game {g} after its {len(seqs[g])} opening moves")
    live = list(range(trees))
    rounds = []
    ply = 0
    while live:
        rounds += search(ctx, omk, orc, rec, agents, live, 96, lane_min)
        for g in live:
            assert_tree_equal(ctx, g, agents[g], f"game {g}, move {ply} after the opening: searched")
        st = sample_best_and_play(ctx, agents, live, f"move {ply} after the opening")
        for g in live:
            assert_tree_equal(ctx, g, agents[g], f"game {g}, move {ply} after the opening: played")
        live = [g for g, s in zip(live, st) if s == 0]
        ply += 1
    ctx.close()

    first = f"(rows, bound) of the first rounds: {rounds[:12]}"
    assert any(r < b for r, b in rounds), f"no round evaluated fewer rows than its trees x 16; {first}"
    if fc0 == "split-K":
        assert all(b <= SPLIT_K_MAX_ROWS for _, b in rounds)
        assert any(ceil_div(r, 128) < ceil_div(b, 128) for r, b in rounds), f"no 128-row tile of a bound was left empty; {first}"
    else:
        assert rounds[0][1] > SPLIT_K_MAX_ROWS
        pair = [(r, b) for r, b in rounds if b > SPLIT_K_MAX_ROWS and ceil_div(r, 256) < ceil_div(b, 256)]
        assert pair, f"no CTA-pair round left a whole 256-row pair of its bound empty; {first}"


@pytest.mark.parametrize("games,lane_min", [(800, LANE_MIN_TREES), (24, 2)])
def test_selfplay_driver_with_the_network_matches_granular_calls(omk, params, games, lane_min):
    """tests/test_tree_gpu.py::test_selfplay_driver_ring_matches_granular_calls with the network: seven plies (more than the
    driver's four-slot ring, Boltzmann for the first three) of the device-resident driver give, ply by ply, the boards /
    visit policies / actions / statuses of the same games played through the granular calls, which
    test_late_positions_fewer_rows_than_the_bound compares with the oracle.  800 games search 800 movers: two lanes of 400
    trees, 6400 rows each (CTA-pair fc0); 24 games run on two lanes forced by a threshold of 2.  No game can end within
    seven plies."""
    G, plies, count, batch, eps, alpha, temp, threshold = games, 7, 64, BATCH, EPS, ALPHA, 1.0, 3
    a = net_context(omk, params, 2 * G, 2048, seed=77, lane_min=lane_min)
    a.selfplay_begin(G, count, batch, eps, alpha, temp, threshold, omk.EVAL_NET)
    stats, boards, policy, status, actions = a.selfplay_run(plies, profile=0, want_transitions=True)
    a.close()
    assert int(stats.positions) == G * plies and int(stats.d2h_bytes) == G * plies * (81 + 81 * 4 + 4 + 1)
    boards, policy = boards.reshape(plies, G, 81), policy.reshape(plies, G, 81)
    status, actions = status.reshape(plies, G), actions.reshape(plies, G)

    b = net_context(omk, params, 2 * G, 2048, seed=77, lane_min=lane_min)
    b.pool_new_games(n=2 * G, evaluator=omk.EVAL_NET)  # black = tree 2g, white = 2g + 1, stream id = tree id
    for ply in range(plies):
        mids = [2 * g + (ply % 2) for g in range(G)]
        oids = [2 * g + 1 - (ply % 2) for g in range(G)]
        b.pool_search(ids=mids, count=count, batch_size=batch, epsilon=eps, alpha=alpha, evaluator=omk.EVAL_NET)
        before = b.pool_get_envs(ids=mids)[0]
        acts, pol = b.pool_sample(ids=mids, modes=[1 if ply < threshold else 0] * G, temperatures=[temp] * G)
        st = b.pool_play(acts, ids=mids)
        b.pool_ensure_action(acts, ids=oids, evaluator=omk.EVAL_NET)
        b.pool_play(acts, ids=oids)
        assert [int(x) for x in acts] == [int(x) for x in actions[ply]], f"ply {ply}: actions"
        assert pol.tobytes() == policy[ply].tobytes(), f"ply {ply}: visit policies"
        assert np.array_equal(before, boards[ply]), f"ply {ply}: boards (state the move was chosen in)"
        assert [int(x) for x in st] == [int(x) for x in status[ply]], f"ply {ply}: status"
        assert all(int(x) == 0 for x in st), "the horizon is too short for a game to end"
    b.close()
