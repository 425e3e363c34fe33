"""The naive player's rule (DESIGN.md 4) as restated in tests/naive_ref.py: its forced moves against the oracle's
restatement of src/trainer.rs:506-537, and its random moves on the specified stream."""
import ctypes as C
import os
import re

import numpy as np

import naive_ref
import pyref
from test_arena_gpu import _oracle_naive_move

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _NoDraw:
    """Stands in for the oracle loop's generator: records whether the rule fell through to a random move."""

    def __init__(self):
        self.called = False

    def integers(self, lo, hi):
        self.called = True
        return 0


def test_forced_moves_match_the_oracle_rule(orc):
    boards, turns = naive_ref.random_positions(3000, seed=7)
    forced_seen = 0
    for b, t in zip(boards, turns):
        e = orc.Environment()
        C.memmove(e.e.board, b.ctypes.data, 81)
        e.e.turn = int(t)
        e.e.legal_move_count = int(np.count_nonzero(b == 0))
        stub = _NoDraw()
        want = _oracle_naive_move(orc, e.e, stub)
        got, forced = naive_ref.naive_move(b, t, seed=1, stream=0)
        assert forced == (0 if stub.called else 1)
        if forced:
            assert got == want
            forced_seen += 1
        else:
            assert b[got] == 0
    assert 300 < forced_seen < 2700  # both branches are well represented


def test_random_moves_follow_the_naive_stream():
    board = np.zeros(81, np.uint8)
    board[[40, 41]] = (1, 2)
    legal = [a for a in range(81) if board[a] == 0]
    for seed, stream in ((0, 0), (3, 1), (2**64 - 1, 81 * 5 + 2), (12345, 2**32 - 1)):
        st = pyref.Stream(pyref._mix64(seed ^ 0xA0761D6478BD642F), stream)
        assert naive_ref.naive_move(board, 0, seed, stream) == (legal[st.below(79)], 0)
    # uniform over the 79 legal cells across streams (chi-square, 78 degrees of freedom: p < 1e-4 beyond 131)
    hits = np.zeros(81, np.int64)
    for s in range(7900):
        hits[naive_ref.naive_move(board, 0, 9, s)[0]] += 1
    assert hits[40] == 0 and hits[41] == 0
    obs = hits[legal]
    assert float(((obs - 100.0) ** 2 / 100.0).sum()) < 131.0


def test_naive_key_is_the_librarys_and_distinct_from_the_other_keys():
    src = open(os.path.join(ROOT, "omok-ai_b200", "csrc", "omk_device.cuh")).read()
    key = int(re.search(r"kNaiveKey\s*=\s*(0x[0-9A-Fa-f]+)ull", src).group(1), 16)
    assert key == naive_ref.K_NAIVE
    assert key not in (0x2545F4914F6CDD1D, 0xD1B54A32D192ED03, 0x5EED5EED5EED)
