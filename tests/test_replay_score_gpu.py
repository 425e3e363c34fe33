"""omk_replay_score: the trainer's loss terms of a model slot on device replay rows.  The per-row terms against an fp64
forward, against the product heads' probabilities and against the trainer's own reporting losses; their invariance to the
call's shape (row list or range, chunks, lanes, repeats) and the specified fp64 order of the means; the slots; no effect
on self-play; the CUDA-core debug kernels; and the error codes."""
import importlib
import os
import sys

import numpy as np
import pytest

from oracle import net_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
ERR_INVALID, ERR_STATE, ERR_NUMERIC = -1, -4, -5
CHUNK = 16384  # omk_api.cu kScoreChunk


def fill(omk, games=32, plies=(90,), capacity=600_000, seed=4, net_seed=1, lanes=1, count=16):
    """A context whose replay memory the self-play driver filled, playing with random network weights `net_seed` (`count`
    simulations a move).  Returns (ctx, params)."""
    params = net_oracle.random_params(net_seed)
    ctx = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * games, capacity_nodes=1024, seed=seed)
    ctx.debug_set_lane_min_trees(2 if lanes == 2 else 0)
    ctx.net_load_params(params)
    ctx.replay_reset(capacity)
    ctx.selfplay_begin(games, count, 8, 0.25, 0.03, 1.0, 6, omk.EVAL_NET)
    for p in plies:
        ctx.selfplay_run(p, want_transitions=False)
    assert ctx.replay_info()[0] > 0
    return ctx, params


def score_rows(ctx, slot=0, **kw):
    means, p, v, top1 = ctx.replay_score(slot, per_row=True, **kw)
    return np.array(means, np.float64), p, v, top1


def same(a, b):
    (ma, pa, va, ta), (mb, pb, vb, tb) = a, b
    assert ma.tobytes() == mb.tobytes(), (ma, mb)
    assert pa.tobytes() == pb.tobytes() and va.tobytes() == vb.tobytes() and ta.tobytes() == tb.tobytes()


def block_means(p, v, top1, block=1024):
    """The specified order in fp64: rows [block b, block b + block) added in row order from 0.0, then the block sums in
    ascending b, divided by n."""
    sums = []
    for x in (p, v, top1):
        total = 0.0
        for b in range(0, x.size, block):
            s = 0.0
            for y in x[b:b + block].astype(np.float64).tolist():
                s += y
            total += s
        sums.append(total / x.size)
    return np.array([sums[0], sums[1], sums[0] + sums[1], sums[2]], np.float64)


@pytest.fixture(scope="module")
def wrapped(omk):
    """A capacity-1000 memory the driver has wrapped many times.  64 simulations a move: with 16 in rounds of 8 the visit
    counts of a root tie at the top, so pi has no first maximum apart from its ties to compare top-1 on."""
    ctx, params = fill(omk, capacity=1000, plies=(90, 40), count=64)
    n, added, _ = ctx.replay_info()
    assert n == 1000 and added > 3000
    yield ctx, params
    ctx.close()


@pytest.fixture(scope="module")
def large(omk):
    """A 60 000-row memory that has wrapped: one call over it is four chunks."""
    ctx, params = fill(omk, games=128, plies=(200,), capacity=60_000, seed=9, net_seed=2)
    n, added, _ = ctx.replay_info()
    assert n == 60_000 and added > n and n > 3 * CHUNK
    yield ctx, params
    ctx.close()


# ------------------------------------------------------------------ accuracy
def fp64_terms(params, boards, turns, pi, z):
    """p_loss, v_loss, top1 of the formulas in omok_b200.h from the fp64 forward (logits and value logit kept in fp64),
    and each row's top-two gaps of the logits and of pi."""
    import torch

    out = net_oracle.forward_layers(params, net_oracle_images(boards, turns), dtype=torch.float64)
    l, v = out["logits"], np.tanh(out["vlogit"])
    assert l.dtype == v.dtype == np.float64
    mx = l.max(1, keepdims=True)
    lse = mx + np.log(np.exp(l - mx).sum(1, keepdims=True))
    p_loss = -(pi.astype(np.float64) * (l - lse)).sum(1)
    v_loss = (z.astype(np.float64) - v.astype(np.float64)) ** 2
    top1 = (l.argmax(1) == pi.argmax(1)).astype(np.uint8)  # argmax: the first maximum
    gap = lambda a: np.diff(np.sort(a, 1)[:, -2:], axis=1)[:, 0]  # noqa: E731
    return p_loss, v_loss, top1, gap(l), gap(pi.astype(np.float64))


def net_oracle_images(boards, turns):
    return importlib.import_module("omok-ai_b200.trainer").encode_nn_input(boards, turns)


def check_fp64(p, v, t, ref):
    """p_loss within 1e-3 relative (absolute below 1); v_loss within 5e-4 (DESIGN 3's 8.3e-5 value error times
    2|z - v| <= 4, rounded up); top1 equal wherever both top-two gaps exceed 1e-3."""
    rp, rv, rt, gl, gp = ref
    assert np.all(np.abs(p - rp) <= 1e-3 * np.maximum(np.abs(rp), 1.0)), np.max(np.abs(p - rp) / np.maximum(np.abs(rp), 1.0))
    assert np.max(np.abs(v - rv)) <= 5e-4, np.max(np.abs(v - rv))
    clear = (gl > 1e-3) & (gp > 1e-3)
    assert np.array_equal(t[clear], rt[clear])
    return int(clear.sum())


def test_per_row_terms_match_an_fp64_forward(wrapped, large):
    top1_compared = 0
    for ctx, params in (wrapped, large):
        n = ctx.replay_info()[0]
        rows = np.arange(n) if n <= 1000 else np.random.default_rng(0).choice(n, 1500, replace=False)
        boards, turns, pi, z = ctx.replay_get(rows)
        _, p, v, t = score_rows(ctx, rows=rows)
        top1_compared += check_fp64(p, v, t, fp64_terms(params, boards, turns, pi, z))
    assert top1_compared >= 100, top1_compared


def test_per_row_terms_match_the_product_heads(wrapped, omk):
    """p_loss = -sum pi log P and v_loss = (z - V)^2 with P, V from omk_model_eval of the same slot: the logits
    instantiation of the heads kernel is the kernel that plays.  p_loss compares to 1e-5 relative, absolutely below 1 (both
    sides hold l - logsumexp(l) in f32 at a logit scale of ~20, whose rounding is ~1e-6)."""
    ctx, _ = wrapped
    ctx.model_load_params(3, net_oracle.random_params(5))
    rows = np.arange(ctx.replay_info()[0])
    boards, turns, pi, z = ctx.replay_get(rows)
    for slot in (0, 3):
        P, V = ctx.model_eval(slot, boards, turns, mode=0)
        _, p, v, _ = score_rows(ctx, slot, rows=rows)
        support = pi > 0
        ok = np.all(np.where(support, P >= 1e-30, True), axis=1)
        assert ok.mean() > 0.5
        ref = -(pi.astype(np.float64) * np.log(np.where(support, P, 1.0).astype(np.float64))).sum(1)
        assert np.all(np.abs(p[ok] - ref[ok]) <= 1e-5 * np.maximum(np.abs(ref[ok]), 1.0))
        vref = (z.astype(np.float64) - V.astype(np.float64)) ** 2
        assert np.max(np.abs(v - vref)) <= 1e-6


def test_means_match_the_trainers_reporting_losses(omk):
    """omk_train_replay(1 step of 128) reports its losses after the update on its rows (fp32 CUDA-core forward); the score
    of slot 0 on the same rows (tensor-core forward) agrees to 1e-3 relative."""
    ctx, _ = fill(omk, seed=12)
    for seed in (3, 4):
        losses, rows = ctx.train_replay(seed, 0, 1, 128, want_rows=True)
        means = ctx.replay_score(0, rows=rows[0])
        assert np.allclose(means[:3], losses[0], rtol=1e-3, atol=0), (means, losses[0])
    ctx.close()


# ------------------------------------------------------------------ shape invariance and the order of the means
def test_the_result_depends_on_the_rows_only(large):
    ctx, _ = large
    n = ctx.replay_info()[0]
    full = score_rows(ctx, first=0, n=n)  # four chunks over the wrapped ring
    same(full, score_rows(ctx, rows=np.arange(n)))
    same(full, score_rows(ctx, first=0, n=n))
    pieces = [0, 1, 1000, 17_000, 40_000, n]
    parts = [score_rows(ctx, first=a, n=b - a) for a, b in zip(pieces[:-1], pieces[1:])]
    for k in (1, 2, 3):
        assert np.concatenate([x[k] for x in parts]).tobytes() == full[k].tobytes()
    pick = np.random.default_rng(1).choice(n, 5000, replace=False)
    _, p, v, t = score_rows(ctx, rows=pick)
    assert p.tobytes() == full[1][pick].tobytes() and v.tobytes() == full[2][pick].tobytes() and t.tobytes() == full[3][pick].tobytes()
    # omk_replay_score runs on the main stream only and has no lane split: this case records that a context set to split
    # searches over two lanes scores the same
    ctx.debug_set_lane_min_trees(2)
    try:
        same(full, score_rows(ctx, first=0, n=n))
    finally:
        ctx.debug_set_lane_min_trees(0)
    # the fp64 means are exactly the specified order over the returned per-row terms ...
    assert full[0].tobytes() == block_means(*full[1:]).tobytes()
    for x in parts[1:]:
        assert x[0].tobytes() == block_means(*x[1:]).tobytes()
    # ... and on these rows other orders give other fp64 sums, so the comparison above sees the order
    for other in (block_means(*full[1:], block=n), block_means(*full[1:], block=512)):
        assert other.tobytes() != full[0].tobytes()
    assert ctx.replay_score(0, first=0, n=n) == tuple(float(x) for x in full[0])


# ------------------------------------------------------------------ slots
def test_slots_score_the_weights_they_hold(omk):
    ctx, params = fill(omk, seed=21)
    twin, _ = fill(omk, seed=21)  # the same rows
    n = ctx.replay_info()[0]
    assert twin.replay_info() == ctx.replay_info()
    for x, y in zip(ctx.replay_get(np.arange(n)), twin.replay_get(np.arange(n))):
        assert x.tobytes() == y.tobytes()
    other = net_oracle.random_params(8)
    ctx.model_load_params(5, params)
    ctx.model_load_params(2, other)
    net = score_rows(ctx, 0)
    same(net, score_rows(ctx, 5))
    in_slot = score_rows(ctx, 2)
    twin.net_load_params(other)
    same(in_slot, score_rows(twin, 0))
    # the snapshot taken before a training phase scores, after it, what the network scored before it
    ctx.opponent_from_net()
    ctx.train_replay(7, 0, 3, 128)
    trained = score_rows(ctx, 0)
    same(net, score_rows(ctx, 1))
    assert trained[0].tobytes() != net[0].tobytes()
    # slot 0 after training (re-packed) == a context loaded with the trained weights
    twin.net_load_params(ctx.net_get_params())
    same(trained, score_rows(twin, 0))
    ctx.close()
    twin.close()


# ------------------------------------------------------------------ no side effects
def test_scoring_between_selfplay_runs_changes_nothing(omk):
    games = 16

    def make():
        c = omk.Context(device=0, capacity_envs=1, capacity_trees=2 * games, capacity_nodes=1024, seed=33)
        c.net_load_params(net_oracle.random_params(3))
        c.model_load_params(4, net_oracle.random_params(4))
        c.replay_reset(4096)
        c.selfplay_begin(games, 16, 8, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        return c

    a, b = make(), make()
    out_a, out_b = [a.selfplay_run(70)], [b.selfplay_run(70)]
    h2d = a.transfer_bytes[0]
    for slot in (0, 4):
        a.replay_score(slot)
    assert a.transfer_bytes[0] == h2d, "the range form copied bytes host -> device"
    a.replay_score(0, rows=[0, 5, 3])
    out_a.append(a.selfplay_run(40))
    out_b.append(b.selfplay_run(40))
    for ra, rb in zip(out_a, out_b):
        for x, y in zip(ra[1:], rb[1:]):
            assert x.tobytes() == y.tobytes()
        for f in ("simulations", "positions", "nn_evals", "games_finished"):
            assert getattr(ra[0], f) == getattr(rb[0], f), f
    assert a.replay_info() == b.replay_info()
    rows = np.arange(a.replay_info()[0])
    for x, y in zip(a.replay_get(rows), b.replay_get(rows)):
        assert x.tobytes() == y.tobytes()
    for tree in range(2 * games):
        for x, y in zip(a.pool_root_stats(tree), b.pool_root_stats(tree)):
            assert np.asarray(x).tobytes() == np.asarray(y).tobytes()
        assert a.pool_tree_info(tree) == b.pool_tree_info(tree)
    boards, turns = a.replay_get(rows[:64])[:2]
    for x, y in zip(a.net_eval(boards, turns), b.net_eval(boards, turns)):
        assert x.tobytes() == y.tobytes()
    a.close()
    b.close()


# ------------------------------------------------------------------ the CUDA-core debug kernels
def test_cuda_core_kernels_hold_the_tolerance(wrapped):
    """With the fp32 CUDA-core tower and fc layers, k_loss reads the logits the heads GEMM wrote: per-row terms within the
    tolerances the fp64 comparison uses."""
    ctx, _ = wrapped
    ref = score_rows(ctx)
    try:
        ctx.debug_set_tower_mode(0)
        ctx.debug_set_fc0_mode(0)
        _, p, v, _ = score_rows(ctx)
    finally:
        ctx.debug_set_tower_mode(1)
        ctx.debug_set_fc0_mode(1)
    assert np.all(np.abs(p - ref[1]) <= 1e-3 * np.maximum(np.abs(ref[1]), 1.0))
    assert np.max(np.abs(v - ref[2])) <= 5e-4
    same(ref, score_rows(ctx))


# ------------------------------------------------------------------ errors
def test_errors(omk):
    bare = omk.Context(device=0, capacity_envs=1, capacity_trees=2, capacity_nodes=64, seed=0)
    bare.net_load_params(net_oracle.random_params(0))
    for cap in (0, 1000):  # no memory, an empty one
        bare.replay_reset(cap)
        with pytest.raises(omk.OmkError) as e:
            bare.replay_score(0, first=0, n=1)
        assert e.value.code == ERR_STATE
    bare.close()

    ctx, _ = fill(omk, games=16, seed=5)
    n = ctx.replay_info()[0]
    want = score_rows(ctx)
    bad = [p.copy() for p in net_oracle.random_params(6)]
    bad[30][7] = np.nan  # a policy bias: a non-finite logit
    ctx.model_load_params(4, bad)
    cases = [(ERR_INVALID, dict(rows=[n])), (ERR_INVALID, dict(rows=[0, -1])), (ERR_INVALID, dict(first=n - 5, n=10)),
             (ERR_INVALID, dict(first=-1, n=2)), (ERR_INVALID, dict(first=0, n=0)), (ERR_INVALID, dict(rows=[])),
             (ERR_INVALID, dict(slot=16)), (ERR_INVALID, dict(slot=-1)), (ERR_STATE, dict(slot=9)), (ERR_NUMERIC, dict(slot=4))]
    for code, kw in cases:
        with pytest.raises(omk.OmkError) as e:
            ctx.replay_score(**kw)
        assert e.value.code == code, kw
        same(want, score_rows(ctx))
    ctx.close()


# ------------------------------------------------------------------ end to end
def test_one_small_iteration_scores_the_new_rows():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    iteration = importlib.import_module("iteration")
    out = iteration.run(games_per_gpu=16, plies=80, count=16, batch=16, steps=30, minibatch=256, quiet=True, device_replay=True,
                        replay_capacity=2048, gate=2, score=True)
    assert 0 < out["score_rows"] <= out["replay_rows"]
    for k in ("before", "after", "snapshot"):
        m = out[f"score_{k}"]
        assert all(np.isfinite(m[t]) for t in iteration.SCORE_TERMS), m
        assert m["loss"] == pytest.approx(m["p_loss"] + m["v_loss"], rel=1e-6) and 0 <= m["top1"] <= 1
        assert out[f"score_{k}_s"] > 0
    assert out["score_snapshot"] == out["score_before"]
