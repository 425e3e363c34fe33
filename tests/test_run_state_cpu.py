"""run_state's file round trip and its refusals, on the CPU: a stand-in context holds synthetic weights, accumulators and
replay rows, and records the calls `load` makes."""
import importlib

import numpy as np
import pytest

run_state = importlib.import_module("omok-ai_b200.run_state")
binding = importlib.import_module("omok-ai_b200.binding")

META = dict(seed=2**64 - 3, sampler_seed=12345, step=602, iteration=3, world=2, rank=1)


class FakeContext:
    """The Context calls run_state uses, over host arrays; replay_get counts its calls."""

    def __init__(self, rng=None, rows=0, capacity=0, episodes=0):
        rng = rng or np.random.default_rng(0)
        self.params = [rng.standard_normal(s).astype(np.float32) for s in binding.NET_SHAPES]
        self.accum = [rng.random(s).astype(np.float32) for s in binding.NET_SHAPES]
        self.accum_update = [rng.random(s).astype(np.float32) for s in binding.NET_SHAPES]
        self.boards = rng.integers(0, 3, (rows, 81)).astype(np.uint8)
        self.turns = rng.integers(0, 2, rows).astype(np.uint8)
        self.policy = rng.random((rows, 81)).astype(np.float32)
        self.z = np.where(rng.random(rows) < 0.5, -1.0, 1.0).astype(np.float32)
        self.z[::7] = -0.0
        self.replay_capacity, self.episodes, self.calls, self.gets = capacity, episodes, [], 0

    def net_get_params(self):
        return [p.copy() for p in self.params]

    def train_get_optimizer(self):
        return [a.copy() for a in self.accum], [u.copy() for u in self.accum_update]

    def replay_info(self):
        return len(self.z), len(self.z), self.episodes

    def replay_get(self, rows):
        self.gets += 1
        return self.boards[rows], self.turns[rows], self.policy[rows], self.z[rows]

    def net_load_params(self, params):
        self.calls.append("net_load_params")
        self.params = params

    def train_set_optimizer(self, accum, accum_update):
        self.calls.append("train_set_optimizer")
        self.accum, self.accum_update = accum, accum_update

    def replay_reset(self, capacity):
        self.calls.append("replay_reset")
        self.replay_capacity, self.episodes = capacity, 0
        self.boards, self.turns, self.policy, self.z = self.boards[:0], self.turns[:0], self.policy[:0], self.z[:0]

    def replay_append(self, boards, turns, policy, z, episodes=0):
        self.calls.append("replay_append")
        self.boards, self.turns, self.policy, self.z = boards, turns, policy, z
        self.episodes += episodes


def assert_same_state(a, b):
    for x, y in zip(a.params + a.accum + a.accum_update, b.params + b.accum + b.accum_update):
        assert x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes()
    for x, y in ((a.boards, b.boards), (a.turns, b.turns), (a.policy, b.policy), (a.z, b.z)):
        assert x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes()
    assert (a.replay_capacity, a.episodes) == (b.replay_capacity, b.episodes)


@pytest.mark.parametrize("rows", [0, 1, run_state.REPLAY_CHUNK + 5])
def test_round_trip_restores_every_array_bit_for_bit(tmp_path, rows):
    src = FakeContext(np.random.default_rng(rows), rows=rows, capacity=rows + 100, episodes=rows // 40)
    path = tmp_path / "state"  # no .npz suffix: the file is written under exactly this name
    run_state.save(src, path, **META)
    assert path.exists() and not (tmp_path / "state.npz").exists() and not (tmp_path / "state.tmp").exists()
    assert src.gets == -(-rows // run_state.REPLAY_CHUNK)
    dst = FakeContext(np.random.default_rng(99), rows=3, capacity=7, episodes=1)
    assert run_state.load(dst, path, world=2, rank=1) == META
    want = ["net_load_params", "train_set_optimizer", "replay_reset"] + (["replay_append"] if rows or src.episodes else [])
    assert dst.calls == want
    assert_same_state(src, dst)
    assert np.signbit(dst.z).tolist() == np.signbit(src.z).tolist()  # -0.0 stays -0.0
    assert run_state.read_meta(path) == META


def test_no_replay_memory_round_trips(tmp_path):
    src = FakeContext()
    run_state.save(src, tmp_path / "s", **META)
    dst = FakeContext(np.random.default_rng(1), rows=5, capacity=9)
    run_state.load(dst, tmp_path / "s")
    assert dst.calls == ["net_load_params", "train_set_optimizer", "replay_reset"] and dst.replay_capacity == 0
    assert_same_state(src, dst)


def _rewrite(path, **changes):
    with np.load(path, allow_pickle=False) as f:
        arrays = {k: f[k] for k in f.files}
    for k, v in changes.items():
        if v is None:
            del arrays[k]
        else:
            arrays[k] = v
    with open(path, "wb") as f:
        np.savez(f, **arrays)


@pytest.mark.parametrize("change", [
    dict(version=np.array(2, np.int64)),
    dict(version=None),
    dict(step=None),
    dict(param_23=np.zeros((512, 10368), np.float32)),       # transposed
    dict(accum_05=np.zeros((1, 1, 32, 32), np.float64)),     # wrong dtype
    dict(accum_update_30=None),
    dict(replay_boards=np.zeros((10, 80), np.uint8)),
    dict(replay_turns=np.zeros(11, np.uint8)),
    dict(replay_policy=np.zeros((10, 81), np.float16)),
    dict(replay_capacity=np.array(9, np.int64)),             # fewer than the 10 rows held
    dict(replay_episodes=np.array(-1, np.int64)),
])
def test_refuses_a_wrong_version_or_shape_and_touches_nothing(tmp_path, change):
    path = tmp_path / "s"
    run_state.save(FakeContext(rows=10, capacity=20, episodes=2), path, **META)
    _rewrite(path, **change)
    dst = FakeContext(np.random.default_rng(5), rows=3, capacity=4)
    with pytest.raises(run_state.RunStateError):
        run_state.load(dst, path)
    assert dst.calls == []


@pytest.mark.parametrize("kw", [dict(world=1), dict(world=4), dict(rank=0), dict(world=2, rank=0)])
def test_refuses_another_world_size_or_rank(tmp_path, kw):
    path = tmp_path / "s"
    run_state.save(FakeContext(rows=4, capacity=8), path, **META)
    dst = FakeContext()
    with pytest.raises(run_state.RunStateError, match="world|rank"):
        run_state.load(dst, path, **kw)
    assert dst.calls == []


def test_refuses_metadata_that_is_not_an_unsigned_64_bit_integer(tmp_path):
    for bad in (dict(step=-1), dict(seed=2**64)):
        with pytest.raises(run_state.RunStateError):
            run_state.save(FakeContext(), tmp_path / "s", **{**META, **bad})
    assert not (tmp_path / "s").exists()


def test_a_failed_save_leaves_the_previous_file(tmp_path):
    path = tmp_path / "s"
    run_state.save(FakeContext(rows=2, capacity=2), path, **META)
    before = path.read_bytes()

    class Broken(FakeContext):
        def replay_get(self, rows):
            raise RuntimeError("device lost")

    with pytest.raises(RuntimeError):
        run_state.save(Broken(rows=3, capacity=3), path, **META)
    assert path.read_bytes() == before
