"""The gated run's host side on the CPU: the best network's round trip through run_state (a stand-in context with model
slots records the calls `load` makes), the refusal of an incomplete best network, old files without one, the
promotion rule trainer.gate_decision and the fresh context seed of each resumed gated iteration."""
import importlib

import numpy as np
import pytest

run_state = importlib.import_module("omok-ai_b200.run_state")
binding = importlib.import_module("omok-ai_b200.binding")
trainer = importlib.import_module("omok-ai_b200.trainer")
sharding = importlib.import_module("omok-ai_b200.sharding")

META = dict(seed=7, sampler_seed=8, step=40, iteration=2, world=1, rank=0)


def weights(rng):
    return [rng.standard_normal(s).astype(np.float32) for s in binding.NET_SHAPES]


class SlotContext:
    """The Context calls run_state uses, over host arrays, with model slots."""

    def __init__(self, seed=0, rows=4, capacity=10):
        rng = np.random.default_rng(seed)
        self.slots = {0: weights(rng), 1: weights(rng), 2: weights(rng)}
        self.accum, self.accum_update = weights(rng), weights(rng)
        self.boards = rng.integers(0, 3, (rows, 81)).astype(np.uint8)
        self.turns = rng.integers(0, 2, rows).astype(np.uint8)
        self.policy = rng.random((rows, 81)).astype(np.float32)
        self.z = np.ones(rows, np.float32)
        self.replay_capacity, self.episodes, self.calls = capacity, 1, []

    def net_get_params(self):
        return self.model_get_params(0)

    def model_get_params(self, slot):
        return [p.copy() for p in self.slots[slot]]

    def train_get_optimizer(self):
        return [a.copy() for a in self.accum], [u.copy() for u in self.accum_update]

    def replay_info(self):
        return len(self.z), len(self.z), self.episodes

    def replay_get(self, rows):
        return self.boards[rows], self.turns[rows], self.policy[rows], self.z[rows]

    def net_load_params(self, params):
        self.calls.append("net_load_params")
        self.slots[0] = params

    def model_load_params(self, slot, params):
        self.calls.append(f"model_load_params({slot})")
        self.slots[slot] = params

    def train_set_optimizer(self, accum, accum_update):
        self.calls.append("train_set_optimizer")
        self.accum, self.accum_update = accum, accum_update

    def replay_reset(self, capacity):
        self.calls.append("replay_reset")
        self.replay_capacity = capacity

    def replay_append(self, boards, turns, policy, z, episodes=0):
        self.calls.append("replay_append")
        self.boards, self.turns, self.policy, self.z = boards, turns, policy, z


def same(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes() for x, y in zip(a, b))


def test_the_best_network_round_trips_bit_for_bit(tmp_path):
    src = SlotContext(0)
    path = tmp_path / "s"
    run_state.save(src, path, **META, best_slot=2)
    assert run_state.read_meta(path) == {**META, "best": True}
    dst = SlotContext(1)
    assert run_state.load(dst, path, best_slot=1) == {**META, "best": True}
    assert dst.calls == ["net_load_params", "model_load_params(1)", "train_set_optimizer", "replay_reset", "replay_append"]
    assert same(dst.slots[0], src.slots[0]) and same(dst.slots[1], src.slots[2])
    other = SlotContext(2)
    run_state.load(other, path)  # no slot named: the best network is checked but not restored
    assert "model_load_params(1)" not in " ".join(other.calls) and same(other.slots[0], src.slots[0])


def test_a_file_without_a_best_network_loads_as_before(tmp_path):
    path = tmp_path / "s"
    run_state.save(SlotContext(0), path, **META)
    with np.load(path) as f:
        assert not any(k.startswith("best_") for k in f.files)
    dst = SlotContext(1)
    meta = run_state.load(dst, path, best_slot=1)
    assert meta == META and not meta.get("best", False) and run_state.read_meta(path) == META
    assert dst.calls == ["net_load_params", "train_set_optimizer", "replay_reset", "replay_append"]


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
    dict(best_00=None),                                      # one tensor missing
    dict(best_30=None),
    dict(best_23=np.zeros((512, 10368), np.float32)),         # transposed
    dict(best_05=np.zeros((1, 1, 32, 32), np.float64)),       # wrong dtype
    dict(best_12=np.zeros(7, np.float32)),
])
def test_an_incomplete_best_network_is_refused_before_the_context_is_touched(tmp_path, change):
    path = tmp_path / "s"
    run_state.save(SlotContext(0), path, **META, best_slot=1)
    _rewrite(path, **change)
    for best_slot in (None, 1):
        dst = SlotContext(1)
        with pytest.raises(run_state.RunStateError, match="best"):
            run_state.load(dst, path, best_slot=best_slot)
        assert dst.calls == []


def test_a_lone_best_tensor_makes_the_set_incomplete(tmp_path):
    path = tmp_path / "s"
    run_state.save(SlotContext(0), path, **META)
    _rewrite(path, best_07=np.zeros(binding.NET_SHAPES[7], np.float32))
    dst = SlotContext(1)
    with pytest.raises(run_state.RunStateError, match="best_00"):
        run_state.load(dst, path, best_slot=1)
    assert dst.calls == []


def test_gate_decision_counts_draws_half():
    assert trainer.gate_decision([(3, 3, 4)], 0.5) == (0.5, True)
    assert trainer.gate_decision([(0, 0, 10)], 0.55) == (0.5, False)
    assert trainer.gate_decision([(10, 0, 0)]) == (1.0, True)
    assert trainer.gate_decision([(0, 10, 0)]) == (0.0, False)


def test_gate_decision_promotes_at_exactly_the_threshold():
    # 11 wins of 20 is 0.55 exactly in binary arithmetic as (11 + 0) / 20
    score, promoted = trainer.gate_decision([(11, 9, 0)], 11 / 20)
    assert score == 11 / 20 and promoted
    assert trainer.gate_decision([(10, 9, 1)], 0.5) == (0.525, True)
    assert trainer.gate_decision([(21, 19, 0)], 0.55) == (0.525, False)
    assert trainer.gate_decision([(1, 0, 1)], 0.75) == (0.75, True)
    assert trainer.gate_decision([(1, 0, 1)], np.nextafter(0.75, 1.0))[1] is False


def test_gate_decision_sums_over_ranks():
    # each rank alone would promote (rank 0) or not (rank 1); the verdict is the sum's
    ranks = [(6, 4, 0), (2, 6, 2)]
    assert trainer.gate_decision(ranks, 0.55) == ((8 + 1) / 20, False)
    assert trainer.gate_decision(ranks, 0.45) == (0.45, True)
    assert trainer.gate_decision(ranks, 0.55) == trainer.gate_decision([(8, 10, 2)], 0.55)
    with pytest.raises(ValueError):
        trainer.gate_decision([(0, 0, 0), (0, 0, 0)], 0.55)


def test_every_gated_iteration_gets_a_seed_of_its_own():
    world, iterations = 8, 50
    chains = [[sharding.rank_seed(0, r)] for r in range(world)]
    for it in range(2, iterations + 2):
        for c in chains:
            c.append(sharding.iteration_seed(c[-1], it))
    seeds = [s for c in chains for s in c]
    assert all(0 <= s < 2**64 for s in seeds)
    assert len(set(seeds)) == len(seeds), "no two ranks or iterations share a context seed"
    assert sharding.iteration_seed(12345, 7) == sharding.iteration_seed(12345, 7)
