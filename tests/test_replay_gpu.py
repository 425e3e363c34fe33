"""The replay memory on the device (omk_replay_* / omk_train_replay): the rows the self-play driver commits against
trainer.ReplayMemory fed ply by ply, the sampler against a host restatement of its specified stream, the training
phase against omk_train_step on the same rows, and the state rules of the C ABI.  The sampler restatement is also
checked on the CPU."""
import importlib
import os
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

SAMPLER_KEY = 0x2545F4914F6CDD1D  # replay_kernels.cu kReplaySamplerKey
ERR_INVALID, ERR_STATE = -1, -4


# ------------------------------------------------------------------ host restatement of the sampler (DESIGN.md 4)
def floyd_rows(seed: int, step: int, length: int, n: int) -> list[int]:
    """Floyd's sample without replacement of m = min(n, length) rows on the stream (mix64(seed ^ K), step, 0..)."""
    import pyref

    st = pyref.Stream(pyref._mix64(seed ^ SAMPLER_KEY), step & 0xFFFFFFFF)
    m = min(n, length)
    out = []
    for j in range(length - m, length):
        t = st.below(j + 1)
        out.append(j if t in out else t)
    return out


def test_sampler_restatement_is_a_uniform_sample_without_replacement():
    for length, n in ((1, 1), (5, 128), (50, 10), (1000, 128), (7, 7)):
        for step in range(20):
            rows = floyd_rows(11, step, length, n)
            assert len(rows) == min(n, length) and len(set(rows)) == len(rows)
            assert all(0 <= r < length for r in rows)
    assert sorted(floyd_rows(3, 0, 9, 9)) == list(range(9))
    from scipy.stats import chisquare

    counts = np.zeros(50, np.int64)
    for step in range(2000):
        for r in floyd_rows(5, step, 50, 10):
            counts[r] += 1
    assert chisquare(counts).pvalue > 1e-3, counts
    assert floyd_rows(5, 1, 1000, 16) != floyd_rows(5, 2, 1000, 16) != floyd_rows(6, 1, 1000, 16)


# ------------------------------------------------------------------ helpers
def play(omk, G=32, plies=(60, 60), capacity=600_000, seed=4, lanes=1, transitions=True, replay=True):
    """Hash-evaluator self-play with an optional device replay; returns (ctx, per-run (stats, boards, policy, status))."""
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=2 * G, capacity_nodes=1024, seed=seed)
    ctx.debug_set_lane_min_trees(2 if lanes == 2 else 0)
    if replay:
        ctx.replay_reset(capacity)
    ctx.selfplay_begin(G, 32, 16, 0.25, 0.03, 1.0, 6, omk.EVAL_HASH)
    runs = [ctx.selfplay_run(p, profile=0, want_transitions=transitions)[:4] for p in plies]
    return ctx, runs


def host_memory(runs, capacity, trainer, mem=None, carry=None):
    """trainer.ReplayMemory fed with split_episodes ONE PLY AT A TIME (with carry) from the streamed transitions."""
    mem = mem if mem is not None else trainer.ReplayMemory(capacity=capacity)
    for _, boards, policy, status in runs:
        for p in range(status.shape[0]):
            episodes, carry = trainer.split_episodes(boards[p:p + 1], policy[p:p + 1], status[p:p + 1], carry)
            for b, pi, z in episodes:
                mem.add_episode(b, pi, z)
    return mem, carry


def assert_same_rows(ctx, mem):
    n, added, episodes = ctx.replay_info()
    assert n == len(mem) and added >= n
    if n == 0:
        return
    boards, turns, policy, z = ctx.replay_get(np.arange(n))
    assert boards.tobytes() == np.stack(mem.boards).astype(np.uint8).tobytes(), "boards"
    assert turns.tobytes() == np.array(mem.turns, np.uint8).tobytes(), "turns"
    assert policy.tobytes() == np.stack(mem.policies).astype(np.float32).tobytes(), "policies"
    assert z.tobytes() == np.array(mem.zs, np.float32).tobytes(), "z (bit for bit, -0.0 included)"


@pytest.fixture(scope="module")
def trainer():
    return importlib.import_module("omok-ai_b200.trainer")


# ------------------------------------------------------------------ ingest
@gpu
@pytest.mark.parametrize("capacity", [600_000, 1000, 300])
def test_ingest_matches_the_host_replay_memory(omk, trainer, capacity):
    """32 games x 2 runs of 60 plies: the device rows equal trainer.ReplayMemory's bit for bit, with the capacity's
    drop-oldest rule (1000 rows wraps the ring many times; 300 rows is below one long episode's 6T rows)."""
    ctx, runs = play(omk, capacity=capacity)
    mem, _ = host_memory(runs, capacity, trainer)
    assert_same_rows(ctx, mem)
    assert ctx.replay_info()[2] >= 32  # every game ends within 81 plies
    if capacity == 600_000:
        assert ctx.replay_info()[1] == len(mem)
    ctx.close()


@gpu
def test_two_search_lanes_and_the_feed_leave_self_play_unchanged(omk):
    """Two lanes give the same replay rows as one; with and without a replay the same seeds stream byte-identical
    transitions and statistics."""
    one, runs1 = play(omk, lanes=1)
    two, runs2 = play(omk, lanes=2)
    bare, runs0 = play(omk, lanes=1, replay=False)
    n1, n2 = one.replay_info(), two.replay_info()
    assert n1 == n2
    rows = np.arange(n1[0])
    for a, b in zip(one.replay_get(rows), two.replay_get(rows)):
        assert a.tobytes() == b.tobytes()
    for (s1, *t1), (s0, *t0) in zip(runs1, runs0):
        for x, y in zip(t1, t0):
            assert x.tobytes() == y.tobytes()
        for f in ("simulations", "positions", "nn_evals", "games_finished", "d2h_bytes"):
            assert getattr(s1, f) == getattr(s0, f), f
    for c in (one, two, bare):
        c.close()


# ------------------------------------------------------------------ sampler and training
@gpu
def test_sampled_rows_follow_the_specified_stream(omk):
    ctx, _ = play(omk, plies=(90,), capacity=100, transitions=False)
    ctx.net_init_random(1)
    length = ctx.replay_info()[0]
    assert length == 100
    for seed, step, n in ((0, 0, 16), (7, 3, 64), (2**63 + 5, 2**32 + 1, 100), (1, 9, 128)):
        losses, rows = ctx.train_replay(seed, step, 2, n, want_rows=True)
        for s in range(2):
            want = floyd_rows(seed, step + s, length, n)
            assert rows[s, : len(want)].tolist() == want, (seed, step, n, s)
            assert (rows[s, len(want):] == -1).all()
        assert np.isfinite(losses).all()
    ctx.close()


def _encode(trainer, boards, turns):
    return trainer.encode_nn_input(boards, turns)


@gpu
def test_training_on_the_replay_equals_omk_train_step_on_its_rows(omk, trainer):
    """omk_train_replay(seed, s0, 3 steps, 128) == 3 x omk_train_step on the host-encoded rows it reports, bit for bit
    (losses and all 31 tensors); one call of 3 steps == three calls of 1 step; no minibatch byte goes host -> device."""
    a, _ = play(omk, plies=(90,), transitions=False)
    c, _ = play(omk, plies=(90,), transitions=False)
    b = omk.Context(device=0, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
    for x in (a, b, c):
        x.net_init_random(3)
    h2d0 = a.transfer_bytes[0]
    la, rows = a.train_replay(17, 40, 3, 128, want_rows=True)
    assert a.transfer_bytes[0] == h2d0, "the replay path copied bytes host -> device"
    lc = np.concatenate([c.train_replay(17, 40 + s, 1, 128) for s in range(3)])
    for s in range(3):
        boards, turns, pi, z = a.replay_get(rows[s])
        lb = b.train_step(_encode(trainer, boards, turns), pi, z)
        assert np.array_equal(np.array(lb, np.float32), la[s]), (s, lb, la[s])
    assert la.tobytes() == lc.tobytes()
    for x, y, w in zip(a.net_get_params(), b.net_get_params(), c.net_get_params()):
        assert x.tobytes() == y.tobytes() == w.tobytes()
    for x in (a, b, c):
        x.close()


@gpu
def test_abi_train_step_continues_the_sampler_streams(omk, trainer):
    a, _ = play(omk, plies=(90,), transitions=False)
    a.net_init_random(0)
    step = trainer.AbiTrainStep(a)
    first = step.train_replay(2, 32, seed=5)
    assert first.shape == (2, 3) and step.steps == 2 and np.isfinite(first).all()
    _, rows = a.train_replay(5, 2, 1, 32, want_rows=True)  # the stream the next call of `step` uses
    assert rows[0].tolist() == floyd_rows(5, 2, a.replay_info()[0], 32)
    a.close()


@gpu
def test_two_rank_replay_training_equals_the_host_path_per_rank(omk, trainer):
    """With a NCCL communicator on two GPUs, each rank's omk_train_replay equals that rank's omk_train_step on the same
    rows (losses and weights bit for bit)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    reps, hosts = [], []
    for r in range(2):
        ctx = omk.Context(device=r, capacity_envs=4, capacity_trees=64, capacity_nodes=1024, seed=10 + r)
        ctx.replay_reset(600_000)
        ctx.selfplay_begin(32, 32, 16, 0.25, 0.03, 1.0, 6, omk.EVAL_HASH)
        ctx.selfplay_run(90, want_transitions=False)
        ctx.net_init_random(2)
        reps.append(ctx)
        h = omk.Context(device=r, capacity_envs=4, capacity_trees=4, capacity_nodes=64, seed=0)
        h.net_init_random(2)
        hosts.append(h)
    out = [None, None]

    def work(r, uid_rep, uid_host):
        try:
            reps[r].train_comm_init(uid_rep, 2, r)
            losses, rows = reps[r].train_replay(100 + r, 0, 3, 64, want_rows=True)
            hosts[r].train_comm_init(uid_host, 2, r)
            hl = []
            for s in range(3):
                boards, turns, pi, z = reps[r].replay_get(rows[s])
                hl.append(hosts[r].train_step(_encode(trainer, boards, turns), pi, z))
            out[r] = (losses, np.array(hl, np.float32), reps[r].net_get_params(), hosts[r].net_get_params())
        except Exception as e:  # noqa: BLE001
            out[r] = e

    uid_rep, uid_host = reps[0].train_comm_unique_id(), hosts[0].train_comm_unique_id()
    threads = [threading.Thread(target=work, args=(r, uid_rep, uid_host)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=300)
    for r in range(2):
        assert out[r] is not None and not isinstance(out[r], Exception), out[r]
        losses, hl, pr, ph = out[r]
        assert losses.tobytes() == hl.tobytes()
        for x, y in zip(pr, ph):
            assert x.tobytes() == y.tobytes()
    for c in reps + hosts:
        c.train_comm_destroy()
        c.close()


# ------------------------------------------------------------------ states and errors
@gpu
def test_states_and_errors(omk, trainer):
    ctx = omk.Context(device=0, capacity_envs=4, capacity_trees=64, capacity_nodes=1024, seed=4)
    ctx.net_init_random(0)
    with pytest.raises(omk.OmkError) as e:
        ctx.train_replay(0, 0, 1, 8)  # no replay
    assert e.value.code == ERR_STATE
    ctx.replay_reset(1000)
    with pytest.raises(omk.OmkError) as e:
        ctx.train_replay(0, 0, 1, 8)  # empty replay
    assert e.value.code == ERR_STATE
    assert ctx.replay_info() == (0, 0, 0)
    with pytest.raises(omk.OmkError) as e:
        ctx.replay_reset(-1)
    assert e.value.code == ERR_INVALID
    ctx.replay_reset(0)
    ctx.selfplay_begin(32, 32, 16, 0.25, 0.03, 1.0, 6, omk.EVAL_HASH)
    with pytest.raises(omk.OmkError) as e:
        ctx.replay_reset(1000)  # creating one while the driver is active
    assert e.value.code == ERR_STATE
    ctx.selfplay_run(90, want_transitions=False)
    assert ctx.replay_info() == (0, 0, 0)  # no replay, nothing fed
    ctx.close()


@gpu
def test_emptying_keeps_the_staged_tails_and_capacity_zero_stops_the_feed(omk, trainer):
    G = 32
    ctx, runs = play(omk, G=G, plies=(37,))
    mem, carry = host_memory(runs, 600_000, trainer)
    assert_same_rows(ctx, mem)
    ctx.replay_reset(600_000)  # empty it mid-game: the games' tails stay staged
    assert ctx.replay_info() == (0, 0, 0)
    more = [ctx.selfplay_run(50, want_transitions=True)[:4]]
    fresh, _ = host_memory(more, 600_000, trainer, carry=carry)  # a new host memory, the carry kept
    assert_same_rows(ctx, fresh)
    # bad arguments
    n = ctx.replay_info()[0]
    for rows in ([n], [-1]):
        with pytest.raises(omk.OmkError) as e:
            ctx.replay_get(rows)
        assert e.value.code == ERR_INVALID
    ctx.net_init_random(0)
    for steps, bs in ((0, 8), (1, 0)):
        with pytest.raises(omk.OmkError) as e:
            ctx.train_replay(0, 0, steps, bs)
        assert e.value.code == ERR_INVALID
    # capacity 0: freed, the driver stops feeding
    ctx.replay_reset(0)
    ctx.selfplay_run(30, want_transitions=False)
    assert ctx.replay_info() == (0, 0, 0)
    with pytest.raises(omk.OmkError) as e:
        ctx.replay_get([0])
    assert e.value.code == ERR_STATE
    with pytest.raises(omk.OmkError) as e:
        ctx.replay_reset(10)  # re-creating it while the driver is active
    assert e.value.code == ERR_STATE
    ctx.close()


# ------------------------------------------------------------------ end to end
@gpu
def test_one_small_iteration_with_the_device_replay():
    """tools/iteration.py --device-replay at a small size: every game ends within the 2 + 80 plies, the replay is not
    empty, and 30 steps on minibatches that cover the whole (256-row) replay lower its loss."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    iteration = importlib.import_module("iteration")
    out = iteration.run(games_per_gpu=16, plies=80, count=16, batch=16, steps=30, minibatch=256, quiet=True, device_replay=True,
                        replay_capacity=256)
    assert out["replay_rows"] == 256 and out["replay_episodes"] >= 16
    assert np.isfinite(out["first_loss"]) and np.isfinite(out["last_loss"]) and out["last_loss"] < out["first_loss"]
    assert out["train_phase_s"] > 0 and out["train_step"].startswith("omk_train_replay")
