"""Ownership of the context's device buffers: a failed omk_ctx_create releases what it allocated and leaves no pending
runtime error, and each search lane's evaluator state (activation buffers, their tensor maps, fc0 scratch) belongs to that
lane's workspace, so two lanes give the results of one on the network evaluator, across regrown workspaces."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_failed_create_releases_everything(omk):
    import torch

    torch.cuda.init()
    torch.zeros(1, device="cuda:0")  # the primary context exists before the first reading
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info(0)
    for _ in range(8):
        # a 256 MiB env pool (allocated), then a 378 GB tree pool that the device refuses: an ordinary error return
        with pytest.raises(omk.OmkError) as e:
            omk.Context(device=0, capacity_envs=8 << 20, capacity_trees=4096, capacity_nodes=65535, seed=1)
        assert e.value.code == -2, str(e.value)
    free_after, _ = torch.cuda.mem_get_info(0)
    assert free_before - free_after <= 512 << 20, f"{(free_before - free_after) >> 20} MiB not released by 8 failed creates"
    # the failed calls' allocation error must not surface in a later call on another context
    c = omk.Context(device=0, capacity_envs=8, capacity_trees=8, capacity_nodes=2048, seed=3)
    c.env_reset(n=2)
    c.env_step([40, 41], ids=[0, 1])
    c.pool_new_games(n=4, evaluator=omk.EVAL_HASH)
    c.pool_search(n=4, count=32, batch_size=16, epsilon=0.25, alpha=0.03, evaluator=omk.EVAL_HASH)
    c.close()


def _run(omk, lanes):
    c = omk.Context(device=0, capacity_envs=4, capacity_trees=128, capacity_nodes=4096, seed=31)
    c.debug_set_lane_min_trees(2 if lanes == 2 else 0)
    c.net_init_random(7)
    out = []
    # the second begin regrows both lanes' workspaces and activation buffers: stale maps or scratch would show
    for games, plies in ((16, 3), (64, 3)):
        c.selfplay_begin(games, 32, 16, 0.25, 0.03, 1.0, 4, omk.EVAL_NET)
        stats, boards, policy, status, actions = c.selfplay_run(plies, profile=0, want_transitions=True)
        out.append((boards.tobytes(), policy.tobytes(), status.tobytes(), actions.tobytes(), int(stats.simulations),
                    int(stats.nn_evals)))
    for n in (24, 96):
        c.pool_new_games(n=n, evaluator=omk.EVAL_NET)
        c.pool_search(n=n, count=48, batch_size=16, epsilon=0.25, alpha=0.03, evaluator=omk.EVAL_NET)
        for t in range(n):
            a, visits, w, p = c.pool_root_children(t)
            out.append((a.tobytes(), visits.tobytes(), w.tobytes(), p.tobytes()))
    c.close()
    return out


def test_two_lanes_equal_one_lane_on_the_network(omk):
    """The network is batch-invariant (test_net_gpu.py::test_batch_invariance), so splitting the trees over two lanes must
    not change a byte."""
    two, one = _run(omk, 2), _run(omk, 1)
    assert len(two) == len(one)
    for i, (a, b) in enumerate(zip(two, one)):
        assert a == b, f"result {i} differs between two lanes and one"
