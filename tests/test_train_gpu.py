"""The C-ABI trainer step (omk_train_step / omk_train_backward / omk_train_apply; AgentModel::train,
alpha-zero/src/agent_model.rs:26-103,136-168) on cuda against the oracle: gradients vs fp64 autograd over
oracle/net_oracle.py, the update vs oracle/trainer_oracle.py's Adadelta (tensorflow ApplyAdadelta), the reported losses vs
`losses_fp64`.  Tolerances are written at each assertion."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def make_batch(no, n, seed):
    rng = np.random.default_rng(seed)
    boards = np.zeros((n, 81), np.uint8)
    turns = np.zeros(n, np.uint8)
    for b in range(n):
        k = int(rng.integers(0, 70))
        cells = rng.permutation(81)[:k]
        boards[b, cells[0::2]] = 1
        boards[b, cells[1::2]] = 2
        turns[b] = k % 2
    images = np.stack([no.encode_image(bb, int(tt)) for bb, tt in zip(boards, turns)])
    pi = rng.random((n, 81)).astype(np.float32) * (boards == 0)
    pi /= pi.sum(1, keepdims=True)
    z = rng.choice(np.array([-1.0, 0.0, 1.0], np.float32), n)
    return images, pi.astype(np.float32), z


def params_with_biases(no, seed):
    """Random-init weights (biases are zero in the recipe) plus small random biases, so every tensor carries signal."""
    rng = np.random.default_rng(1000 + seed)
    params = no.random_params(seed)
    for i, (name, shape) in enumerate(no.PARAM_SPECS):
        if len(shape) == 1:
            params[i] = (0.05 * rng.standard_normal(shape)).astype(np.float32)
    return params


@pytest.fixture(scope="module")
def no():
    from oracle import net_oracle

    return net_oracle


def test_gradients_match_fp64_autograd(omk, no):
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    params = params_with_biases(no, 0)
    ctx.net_load_params(params)
    images, pi, z = make_batch(no, 24, 1)
    ptr, count = ctx.train_backward(images, pi, z)
    assert ptr != 0 and count == 5_643_250
    got = ctx.train_get_grads()
    (_, _, _), want = no.loss_and_grads(params, images, pi, z)
    for (name, _), g, w in zip(no.PARAM_SPECS, got, want):
        scale = float(np.abs(w).max())
        assert scale > 0, name
        err = float(np.abs(g.astype(np.float64) - w).max())
        # bar: 1e-4 of the tensor's largest gradient.  The value head's own tensors get 5e-4: d tanh = 1 - tanh^2 has a
        # relative sensitivity of 2 |tanh| per unit of logit error, and an fp32 forward errs by ~1e-4 on logits of scale 20.
        bar = 5e-4 if name in ("v_w", "v_b") else 1e-4
        assert err <= bar * scale, f"{name}: gradient differs from fp64 autograd by {err / scale:.2e} of its max (bar {bar:g})"
    ctx.close()


def test_two_steps_match_the_adadelta_oracle(omk, no):
    """Two steps on cuda vs fp64 gradients + oracle Adadelta: parameters within 1e-4 relative of their tensor's scale,
    the UPDATE itself (after - before) within 2e-2 of the oracle's update norm per tensor (an fp32 parameter keeps only
    ~7 bits of a 4.5e-6 first-step update, so the update is compared as a whole, not element by element), reported
    losses within 1e-4 relative of `losses_fp64` on the updated weights."""
    from oracle import trainer_oracle as to

    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    params = params_with_biases(no, 1)
    ctx.net_load_params(params)
    opt = to.Adadelta(params, lr=0.01, rho=0.95, eps=1e-8)
    cur = [np.asarray(p, np.float64) for p in params]
    for step in range(2):
        images, pi, z = make_batch(no, 32, 10 + step)
        before = [p.astype(np.float64) for p in ctx.net_get_params()]
        p_loss, v_loss, loss = ctx.train_step(images, pi, z)
        after = ctx.net_get_params()
        _, grads = no.loss_and_grads([c.astype(np.float32) for c in cur], images, pi, z)
        new = opt.step(grads)
        for (name, _), b, a, o_old, o_new in zip(no.PARAM_SPECS, before, after, cur, new):
            scale = max(float(np.abs(o_new).max()), 1e-3)
            assert float(np.abs(a - o_new).max()) <= 1e-4 * scale, f"step {step} {name}: parameters"
            d_got, d_want = (a.astype(np.float64) - b).reshape(-1), (o_new - o_old).reshape(-1)
            assert np.linalg.norm(d_got - d_want) <= 2e-2 * np.linalg.norm(d_want) + 1e-12, f"step {step} {name}: update"
            assert np.sign(d_got[np.abs(d_want) > 1e-6]).tolist() == np.sign(d_want[np.abs(d_want) > 1e-6]).tolist(), name
        cur = [np.asarray(x, np.float64) for x in new]
        rp, rv, rl = to.losses_fp64([x.astype(np.float32) for x in after], images, pi, z)
        assert abs(p_loss - rp) <= 1e-4 * abs(rp) and abs(v_loss - rv) <= 1e-4 * max(abs(rv), 1e-2) and abs(loss - rl) <= 1e-4 * abs(rl)
    ctx.close()


def test_split_calls_equal_the_fused_step_and_weights_reach_the_kernels(omk, no):
    """omk_train_backward + omk_train_apply == omk_train_step bit for bit; after a step the tensor-core kernels answer
    with the NEW weights (omk_net_eval vs the fp64 oracle on omk_net_get_params, 1e-3 relative); repeated steps on one
    batch lower its loss."""
    import torch

    a = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    b = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    params = params_with_biases(no, 2)
    a.net_load_params(params)
    b.net_load_params(params)
    images, pi, z = make_batch(no, 16, 3)
    la = a.train_step(images, pi, z)
    b.train_backward(images, pi, z)
    lb = b.train_apply()
    assert la == lb
    for x, y in zip(a.net_get_params(), b.net_get_params()):
        assert x.tobytes() == y.tobytes()
    with pytest.raises(omk.OmkError):
        b.train_apply()  # one gradient, one update
    first = la[2]
    for _ in range(30):
        last = a.train_step(images, pi, z)[2]
    assert last < first, (first, last)
    boards = np.zeros((8, 81), np.uint8)
    boards[np.arange(8), np.arange(8) * 7] = 1
    turns = np.ones(8, np.uint8)
    p, v = a.net_eval(boards, turns)
    rp, rv, _ = no.forward_boards(a.net_get_params(), boards, turns, dtype=torch.float64)
    big = rp > 1e-12
    assert np.max(np.abs(p[big] - rp[big]) / rp[big]) < 1e-3
    # values: tanh of a logit of scale ~20 -- relative error only where it is well conditioned (DESIGN.md 3, "Values")
    assert np.max(np.abs(v - rv)) < 2e-4
    far = np.abs(rv) >= 0.1
    assert np.max(np.abs(v - rv)[far] / np.abs(rv)[far]) < 1e-3
    a.close()
    b.close()


def test_two_rank_nccl_step_equals_the_full_batch_step(omk, no):
    """BASELINE config 5's collective: two ranks (two GPUs, one context each, one host thread each) with half the
    minibatch each and an attached NCCL communicator land on the single-context full-batch step: all-reduced gradient
    within 1e-5 of the full-batch gradient's scale per tensor, parameters after the step within 1e-6 of their scale,
    identical on both ranks bit for bit, losses equal to the mean of the halves."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    params = params_with_biases(no, 4)
    images, pi, z = make_batch(no, 32, 5)
    full = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    full.net_load_params(params)
    full.train_backward(images, pi, z)
    g_full = full.train_get_grads()
    l_full = full.train_apply()
    p_full = full.net_get_params()
    full.close()

    ranks = [omk.Context(device=r, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0) for r in range(2)]
    uid = ranks[0].train_comm_unique_id()
    out = [None, None]

    def work(r):
        try:
            c = ranks[r]
            c.net_load_params(params)
            c.train_comm_init(uid, 2, r)
            sl = slice(16 * r, 16 * (r + 1))
            c.train_backward(images[sl], pi[sl], z[sl])
            losses = c.train_apply()
            out[r] = (losses, c.train_get_grads(), c.net_get_params())
        except Exception as e:  # noqa: BLE001
            out[r] = e

    threads = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=300)
    for r in range(2):
        assert not isinstance(out[r], Exception), out[r]
        assert out[r] is not None, "a rank hung"
    for (name, _), gf, g0, g1, pf, p0, p1 in zip(no.PARAM_SPECS, g_full, out[0][1], out[1][1], p_full, out[0][2], out[1][2]):
        assert g0.tobytes() == g1.tobytes() and p0.tobytes() == p1.tobytes(), f"{name}: the ranks disagree"
        gs, ps = float(np.abs(gf).max()), max(float(np.abs(pf).max()), 1e-3)
        assert float(np.abs(g0 - gf).max()) <= 1e-5 * gs, f"{name}: all-reduced gradient"
        assert float(np.abs(p0 - pf).max()) <= 1e-6 * ps, f"{name}: parameters after the step"
    assert out[0][0] == out[1][0]
    assert all(abs(a - b) <= 1e-5 * abs(b) for a, b in zip(out[0][0], l_full))
    for c in ranks:
        c.train_comm_destroy()
        c.close()


@pytest.mark.parametrize("n", [1, 3, 17, 67, 130])
def test_ragged_minibatch_sizes(omk, no, n):
    """Tile edges of the training GEMMs (64 x 64 x 16 tiles, K slices) and ragged last slices of the sliced reductions (17
    positions: two position slices of the depthwise weight gradient, 9 + 8; 67: 21 row slices of the bias gradients, the last
    one short): minibatches of 1 ... 130 positions give gradients within the same bars as the 24-position case, and a step
    returns finite losses."""
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    params = params_with_biases(no, 7)
    ctx.net_load_params(params)
    images, pi, z = make_batch(no, n, 40 + n)
    ctx.train_backward(images, pi, z)
    got = ctx.train_get_grads()
    _, want = no.loss_and_grads(params, images, pi, z)
    for (name, _), g, w in zip(no.PARAM_SPECS, got, want):
        scale = float(np.abs(w).max())
        if scale == 0.0:
            assert not g.any(), name
            continue
        bar = 5e-4 if name in ("v_w", "v_b") else 1e-4
        assert float(np.abs(g.astype(np.float64) - w).max()) <= bar * scale, name
    losses = ctx.train_apply()
    assert all(np.isfinite(losses)) and abs(losses[0] + losses[1] - losses[2]) <= 1e-5 * abs(losses[2])
    ctx.close()


def test_gradient_is_deterministic_across_calls(omk, no):
    """The sliced reductions (bias gradients, depthwise weight gradients: the last CTA to finish adds the slice sums in slice
    order; arrival counters re-arm themselves) and the K-sliced GEMMs use no floating-point atomics: the same minibatch on the
    same weights gives the same gradient bits, call after call and across minibatch sizes that change the slice counts in
    between."""
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    ctx.net_load_params(params_with_biases(no, 11))
    images, pi, z = make_batch(no, 96, 5)
    ctx.train_backward(images, pi, z)
    first = [g.copy() for g in ctx.train_get_grads()]
    for other in (40, 96, 9):
        oi, op, oz = make_batch(no, other, 6 + other)
        ctx.train_backward(oi, op, oz)  # another slice count in between
        ctx.train_backward(images, pi, z)
        for (name, _), a, b in zip(no.PARAM_SPECS, first, ctx.train_get_grads()):
            assert a.tobytes() == b.tobytes(), name
    ctx.close()


def test_transfer_counters_follow_the_calls(omk, no):
    """omk_ctx_transfer_bytes (bench.py's e2e byte counts): a network call on n boards copies n * 82 bytes in and n * 82
    floats out; a train step copies n * (243 + 81 + 1) floats in and 3 floats out."""
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    ctx.net_init_random(0)
    h0, d0 = ctx.transfer_bytes
    boards = np.zeros((10, 81), np.uint8)
    ctx.net_eval(boards, np.zeros(10, np.uint8))
    h1, d1 = ctx.transfer_bytes
    assert 10 * 82 <= h1 - h0 <= 10 * 82 + 64 and 10 * 82 * 4 <= d1 - d0 <= 10 * 82 * 4 + 64, (h1 - h0, d1 - d0)
    images, pi, z = make_batch(no, 6, 1)
    ctx.train_step(images, pi, z)
    h2, d2 = ctx.transfer_bytes
    assert 6 * 325 * 4 <= h2 - h1 <= 6 * 325 * 4 + 64 and 12 <= d2 - d1 <= 12 + 64, (h2 - h1, d2 - d1)
    ctx.close()
