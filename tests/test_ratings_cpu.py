"""arena.ratings: the Bradley-Terry fit, in Elo units, of a tournament's pairwise table (left wins, right wins, draws)."""
import importlib

import numpy as np
import pytest


@pytest.fixture(scope="module")
def arena():
    return importlib.import_module("omok-ai_b200.arena")


def _pairings(n):
    return [(i, j) for i in range(n) for j in range(i + 1, n)]


def test_symmetric_results_give_equal_ratings(arena):
    even = np.tile([10, 10, 5], (6, 1))  # four models, every pairing level
    assert np.abs(arena.ratings(even, 4)).max() < 1e-9
    # a cycle: 0 beats 1, 1 beats 2, 2 beats 0, each 7-3
    cycle = np.array([[7, 3, 0], [3, 7, 0], [7, 3, 0]])
    assert np.abs(arena.ratings(cycle, 3)).max() < 1e-9
    # nothing played: the virtual draws alone
    assert np.abs(arena.ratings(np.zeros((10, 3)), 5)).max() < 1e-9


@pytest.mark.parametrize("w, l, d", [(7, 2, 1), (0, 0, 0), (50, 0, 0), (0, 13, 4), (3, 3, 94)])
def test_two_models_give_the_closed_form(arena, w, l, d):
    r = arena.ratings([[w, l, d]], 2)
    assert r[0] == 0.0
    want = 400.0 * np.log10((w + d / 2 + 0.5) / (l + d / 2 + 0.5))
    assert abs((r[0] - r[1]) - want) < 1e-9
    assert np.isfinite(r).all()


def test_a_clean_sweep_stays_finite(arena):
    sweep = np.array([[100, 0, 0]] * 3)  # every left side wins every game: 0 sweeps 1 and 2, 1 sweeps 2
    r = arena.ratings(sweep, 3)
    assert np.isfinite(r).all() and r[0] == 0.0 and r[1] < 0 and r[2] < r[1]


def test_ratings_drawn_from_known_ratings_are_recovered(arena):
    """Every pairing plays 20 000 games with draws: a draw with probability 0.1, and the expected score of the stronger side
    equals the Bradley-Terry (Elo) expectation.  With that many games the fit's standard error is below 3 Elo per model; the
    bar is 10 Elo."""
    true = np.array([0.0, 150.0, -100.0, 250.0, 50.0, -150.0])
    n, games, q = len(true), 20000, 0.1
    rng = np.random.default_rng(20261021)
    table = []
    for i, j in _pairings(n):
        p = 1.0 / (1.0 + 10.0 ** ((true[j] - true[i]) / 400.0))  # left's expected score
        w, l, d = rng.multinomial(games, [p - q / 2, 1.0 - p - q / 2, q])
        table.append((w, l, d))
    r = arena.ratings(np.array(table), n)
    assert r[0] == 0.0
    assert np.abs(r - true).max() < 10.0, r - true


def test_ratings_are_deterministic_and_check_their_input(arena):
    rng = np.random.default_rng(3)
    table = rng.integers(0, 40, (10, 3))
    assert arena.ratings(table, 5).tobytes() == arena.ratings(table.copy(), 5).tobytes()
    with pytest.raises(ValueError):
        arena.ratings(table, 4)  # 6 pairings expected
    with pytest.raises(ValueError):
        arena.ratings([[1, -1, 0]], 2)
