"""The naive player's rule of DESIGN.md 4, restated on tests/pyref (test infrastructure): src/trainer.rs:506-537 with its
random move on the specified stream instead of thread_rng()."""
from __future__ import annotations

import numpy as np

import pyref

K_NAIVE = 0xA0761D6478BD642F  # omk_device.cuh kNaiveKey


def env_of(board, turn):
    env = pyref.Environment()
    env.board = [int(x) for x in board]
    env.turn = int(turn)
    env.legal_move_count = env.board.count(pyref.EMPTY)
    return env


def naive_move(board, turn, seed, stream):
    """(action, forced) for the position `board` (81 cells) with `turn` to move: the first empty cell, ascending, where
    place_stone is terminal for the mover or, with the turn flipped, for the opponent (forced = 1); else
    legal[below(len(legal))] on the stream (mix64(seed ^ K_NAIVE), stream, counter from 0) (forced = 0)."""
    env = env_of(board, turn)
    legal = [a for a in range(pyref.CELLS) if env.board[a] == pyref.EMPTY]
    for a in legal:
        for flip in (0, 1):
            e = env.clone()
            e.turn = int(turn) ^ flip
            if e.place_stone(a) != pyref.IN_PROGRESS:
                return a, 1
    if not legal:
        return -1, 0
    st = pyref.Stream(pyref._mix64((int(seed) ^ K_NAIVE) & pyref.M64), int(stream) & 0xFFFFFFFF)
    return legal[st.below(len(legal))], 0


def random_positions(count, seed):
    """`count` unfinished positions from seeded random playouts (between 0 and 80 stones), each with the turn of its
    stone counts or, for every other position, the opposite turn."""
    rng = np.random.default_rng(seed)
    boards = np.zeros((count, pyref.CELLS), np.uint8)
    turns = np.zeros(count, np.uint8)
    i = 0
    while i < count:
        env = pyref.Environment()
        target = int(rng.integers(0, 81))
        for a in rng.permutation(pyref.CELLS)[:target]:
            probe = env.clone()
            if probe.place_stone(int(a)) != pyref.IN_PROGRESS:
                break
            env.place_stone(int(a))
        boards[i] = env.board
        turns[i] = env.turn ^ (i & 1)
        i += 1
    return boards, turns
