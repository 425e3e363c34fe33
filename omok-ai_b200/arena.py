"""Evaluation play (SURVEY.md 8f row 3), batched over games on the tree / env pools of `binding.Context`.

  * `play_match`                 benchmark/src/main.rs:14-108 + benchmark/src/agent.rs:14-47: two models, GAME_COUNT games,
                                 half with each side moving first; every move = MCTSExecutor::run(800, 8, eps 0, alpha 1)
                                 then `sample_action(Best)`; the opponent follows with ensure_action_exists + play_action.
  * `play_match_device`          the same match as ONE call (omk_match) between the context's network (left) and its
                                 opponent network (right): both legs run at once, each model's half-move on its own lane.
  * `play_tournament_device`     a round-robin of that match over up to 16 model slots of one context as ONE call
                                 (omk_tournament); each model searches all its pairings' movers as one batch per half-move.
  * `play_tournament_naive_device`  the same round-robin with the naive player below as participant 0 (omk_tournament_naive),
                                 so `ratings` puts every model on one scale, with the naive player at 0 Elo.
  * `ratings`                    a Bradley-Terry fit, in Elo units, of a tournament's pairwise results.
  * `play_against_naive_player`  src/trainer.rs:487-603: the naive player takes the first legal move (ascending) that ends
                                 the game for itself, or that would end it for the opponent (a block); else a random
                                 legal move.  The model answers with ParallelMCTSExecutor::execute + Best.
  * `play_against_naive_player_device`  the same evaluation as ONE call (omk_eval_naive): the naive player's move is a
                                 kernel, and its random moves follow the specified stream of DESIGN.md 4.

The reference plays its games one after another; games are independent, so all of them run concurrently here (one tree
per game and model), which changes nothing for any single game.  The naive player's "does this move end the game?" test
is the environment kernel itself: every (game, empty cell, perspective) candidate is one board of the env pool, stepped
in a single `omk_env_step` call -- a pure K1 workload.
"""
from __future__ import annotations

import numpy as np

from . import binding as B

CELLS = 81


def _play_moves(ctx, ids, actions, evaluator):
    """ensure_action_exists + play_action on the trees `ids` (the opponent's move arriving in this model's trees)."""
    ctx.pool_ensure_action(actions, ids=ids, evaluator=evaluator)
    return ctx.pool_play(actions, ids=ids)


def play_match(ctx_left, ctx_right, game_count: int = 100, count: int = 800, batch_size: int = 8, epsilon: float = 0.0,
               alpha: float = 1.0, evaluator: int = B.EVAL_NET, moves_out: list | None = None):
    """Returns (left_wins, right_wins, draws).  Each context holds one model; it needs `game_count // 2` trees.
    `moves_out`, if given, receives one move list per game: first the `half` games left opens, then those right opens."""
    half = game_count // 2
    wins = {"left": 0, "right": 0, "draw": 0}
    log = [[] for _ in range(2 * half)]
    for leg, (first, second, first_name, second_name) in enumerate(((ctx_left, ctx_right, "left", "right"), (ctx_right, ctx_left, "right", "left"))):
        ids = np.arange(half, dtype=np.int32)
        first.pool_new_games(ids=ids, evaluator=evaluator)
        second.pool_new_games(ids=ids, evaluator=evaluator)
        live = ids.copy()
        mover, other, mover_name, other_name = first, second, first_name, second_name
        while live.size:
            mover.pool_search(ids=live, count=count, batch_size=batch_size, epsilon=epsilon, alpha=alpha, evaluator=evaluator)
            actions, _ = mover.pool_sample(ids=live, modes=np.full(live.size, B.SAMPLE_BEST, np.uint8))
            for g, a in zip(live, actions):
                log[leg * half + int(g)].append(int(a))
            status = mover.pool_play(actions, ids=live)
            # BlackWin / WhiteWin: the player who just moved made five (main.rs:61-75 maps it to the side to move first)
            done = status != 0
            wins[mover_name] += int(np.count_nonzero(status >= 2))
            wins["draw"] += int(np.count_nonzero(status == 1))
            keep = ~done
            if keep.any():
                _play_moves(other, live[keep], actions[keep], evaluator)
            live = live[keep]
            mover, other, mover_name, other_name = other, mover, other_name, mover_name
    if moves_out is not None:
        moves_out[:] = log
    return wins["left"], wins["right"], wins["draw"]


def play_match_device(ctx, game_count: int = 100, count: int = 800, batch_size: int = 8, epsilon: float = 0.0, alpha: float = 1.0,
                      evaluator: int = B.EVAL_NET, first_tree: int = 0, moves_out: list | None = None):
    """Returns (network wins, opponent wins, draws) like `play_match` with left = the network and right = the opponent
    (`Context.opponent_load_params` / `opponent_from_net`), from one `omk_match` call of `game_count // 2` pairs on the trees
    first_tree .. first_tree + 2 * game_count - 1.  `play_match` on two contexts with this context's seed replays it game
    by game.  `moves_out`, if given, receives one move list per game in `play_match`'s order."""
    result, moves, _, _ = ctx.match(game_count // 2, first_tree=first_tree, count=count, batch_size=batch_size, epsilon=epsilon,
                                    alpha=alpha, evaluator=evaluator)
    if moves_out is not None:
        moves_out[:] = [[int(a) for a in row if a >= 0] for row in moves]
    return result


def play_tournament_device(ctx, slots, game_count: int = 100, count: int = 800, batch_size: int = 8, epsilon: float = 0.0,
                           alpha: float = 1.0, evaluator: int = B.EVAL_NET, first_tree: int = 0, moves_out: list | None = None):
    """A round-robin of `play_match_device` over the model slots `slots` (`Context.model_load_params` / `model_from_net`; slot 0
    is the network, slot 1 the opponent) from one `omk_tournament` call of `game_count // 2` pairs per pairing, on the trees
    first_tree .. first_tree + 2 * game_count * P - 1.  Pairing p = (i, j), i < j in lexicographic order, is
    `play_match_device` with slots[i] left and slots[j] right.  Returns the [P, 3] table of (left wins, right wins, draws).
    `moves_out`, if given, receives per pairing one move list per game in `play_match`'s order."""
    result, moves, _, _ = ctx.tournament(slots, game_count // 2, first_tree=first_tree, count=count, batch_size=batch_size,
                                         epsilon=epsilon, alpha=alpha, evaluator=evaluator)
    if moves_out is not None:
        moves_out[:] = [[[int(a) for a in row if a >= 0] for row in pairing] for pairing in moves]
    return result


def play_tournament_naive_device(ctx, slots, seed: int = 0, game_count: int = 100, count: int = 800, batch_size: int = 8,
                                 epsilon: float = 0.0, alpha: float = 1.0, evaluator: int = B.EVAL_NET, first_tree: int = 0,
                                 moves_out: list | None = None):
    """`play_tournament_device` with the naive player as participant 0 and slots[k] as participant k + 1, from one
    `omk_tournament_naive` call of `game_count // 2` pairs per pairing on the trees first_tree .. first_tree + 2 * game_count * P - 1,
    P = N(N-1)/2 over the N = len(slots) + 1 participants.  The first len(slots) pairings are (naive, slots[k]), the naive
    player left and opening the first half of the games; its random moves draw on stream g * 81 + h of key
    mix64(seed ^ K_NAIVE) (DESIGN.md 4).  Returns the [P, 3] table of (left wins, right wins, draws), so
    `ratings(table, len(slots) + 1)` rates the naive player at 0 Elo and slots[k] at entry k + 1: every tournament against the
    naive player shares that zero.  `moves_out` as in `play_tournament_device`."""
    result, moves, _, _ = ctx.tournament_naive(slots, game_count // 2, seed=seed, first_tree=first_tree, count=count,
                                               batch_size=batch_size, epsilon=epsilon, alpha=alpha, evaluator=evaluator)
    if moves_out is not None:
        moves_out[:] = [[[int(a) for a in row if a >= 0] for row in pairing] for pairing in moves]
    return result


def ratings(result, n_models: int, iterations: int = 100000, tol: float = 1e-12) -> np.ndarray:
    """Elo ratings of the n_models models of a tournament from its [P, 3] table of (left wins, right wins, draws), pairings
    (i, j), i < j, in lexicographic order: the maximum-likelihood Bradley-Terry strengths (Hunter's MM iteration), each
    reported as 400 * log10(strength / strength of model 0), so model 0 (slots[0]) is rated 0.  A draw counts as half a win
    to each side, and every pairing gets one virtual draw, which keeps a clean sweep finite.  Deterministic; with two models
    the rating difference is 400 * log10((w + d/2 + 0.5) / (l + d/2 + 0.5))."""
    r = np.asarray(result, dtype=np.float64).reshape(-1, 3)
    n = int(n_models)
    if n < 2 or r.shape[0] != n * (n - 1) // 2:
        raise ValueError(f"need n_models >= 2 and n(n-1)/2 = {n * (n - 1) // 2} pairings, got {r.shape[0]}")
    if (r < 0).any():
        raise ValueError("negative game counts")
    games = np.zeros((n, n))   # games[i, j]: games between i and j, the virtual draw included
    score = np.zeros(n)        # each model's wins + draws / 2, virtual draws included
    p = 0
    for i in range(n):
        for j in range(i + 1, n):
            w, l, d = r[p]
            games[i, j] = games[j, i] = w + l + d + 1.0
            score[i] += w + 0.5 * d + 0.5
            score[j] += l + 0.5 * d + 0.5
            p += 1
    gamma = np.ones(n)
    for _ in range(iterations):
        nxt = score / (games / (gamma[:, None] + gamma[None, :])).sum(axis=1)
        nxt /= nxt[0]
        done = np.max(np.abs(np.log(nxt) - np.log(gamma))) < tol
        gamma = nxt
        if done:
            break
    return 400.0 * np.log10(gamma)


def naive_moves(ctx, boards: np.ndarray, turns: np.ndarray, rng: np.random.Generator) -> np.ndarray:
    """The naive player's move for every board (trainer.rs:506-534).  Needs 162 * n env slots in `ctx`."""
    boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
    turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
    n = boards.shape[0]
    # candidate (game g, perspective s in {own, opponent}, cell a): board g with the turn of perspective s, move a
    cand_boards = np.repeat(boards, 2 * CELLS, axis=0)
    cand_turns = np.repeat(np.stack([turns, turns ^ 1], axis=1).reshape(-1), CELLS)
    cand_actions = np.tile(np.arange(CELLS, dtype=np.uint8), 2 * n)
    ids = np.arange(cand_boards.shape[0], dtype=np.int32)
    ctx.env_set(cand_boards, cand_turns, ids=ids)
    status, _ = ctx.env_step(cand_actions, ids=ids, want_legal=False)
    status = status.reshape(n, 2, CELLS)
    terminal = (status != B.NONE) & (status != 0)          # occupied cells answer NONE; Draw counts as terminal (:517,:525)
    ends = terminal[:, 0, :] | terminal[:, 1, :]            # per action: own win checked first, then the block -- same action
    out = np.empty(n, dtype=np.int32)
    for g in range(n):
        hits = np.flatnonzero(ends[g])
        if hits.size:
            out[g] = hits[0]
        else:
            legal = np.flatnonzero(boards[g] == 0)
            out[g] = legal[rng.integers(0, legal.size)]     # :536-537 uniform over the legal moves
    return out


def play_against_naive_player(ctx, episode_count: int = 100, count: int = 800, batch_size: int = 16, epsilon: float = 0.25,
                              alpha: float = 0.03, evaluator: int = B.EVAL_NET, seed: int = 0, moves_out: list | None = None):
    """Returns (black_win, white_win, draw): the naive player moves first (Black), the model answers (White).

    The naive player's random choices come from `numpy.random.default_rng(seed)`, one draw per live game without a
    forced move, games in ascending id order (the reference draws from thread_rng() in its swap_remove order,
    trainer.rs:498-563: unreproducible; the order of independent games does not change any single game).
    `moves_out`, if given, receives one list of actions per game (both players' moves in playing order)."""
    rng = np.random.default_rng(seed)
    ids = np.arange(episode_count, dtype=np.int32)
    ctx.pool_new_games(ids=ids, evaluator=evaluator)
    result = np.zeros(4, dtype=np.int64)
    log = [[] for _ in range(episode_count)]
    live = ids
    while live.size:
        boards, turns, _, _ = ctx.pool_get_envs(ids=live)  # one launch + one synchronisation for all live games
        actions = naive_moves(ctx, boards, turns, rng)
        for g, a in zip(live, actions):
            log[int(g)].append(int(a))
        status = _play_moves(ctx, live, actions, evaluator)
        np.add.at(result, status[status != 0].astype(np.int64), 1)
        live = live[status == 0]
        if not live.size:
            break
        ctx.pool_search(ids=live, count=count, batch_size=batch_size, epsilon=epsilon, alpha=alpha, evaluator=evaluator)
        actions, _ = ctx.pool_sample(ids=live, modes=np.full(live.size, B.SAMPLE_BEST, np.uint8))
        for g, a in zip(live, actions):
            log[int(g)].append(int(a))
        status = ctx.pool_play(actions, ids=live)
        np.add.at(result, status[status != 0].astype(np.int64), 1)
        live = live[status == 0]
    if moves_out is not None:
        moves_out[:] = log
    return int(result[2]), int(result[3]), int(result[1])


def play_against_naive_player_device(ctx, episode_count: int = 100, count: int = 800, batch_size: int = 16, epsilon: float = 0.25,
                                     alpha: float = 0.03, evaluator: int = B.EVAL_NET, seed: int = 0, first_tree: int = 0,
                                     moves_out: list | None = None):
    """Returns (black_win, white_win, draw) like `play_against_naive_player`, from one `omk_eval_naive` call on the trees
    first_tree .. first_tree + episode_count - 1 (no env slot is used).

    The naive player's random choices do NOT come from numpy: game g's move at ply p (moves already played) draws
    legal[below(legal_count)] on the specified stream (mix64(seed ^ K_NAIVE), g * 81 + p) (DESIGN.md 4), so any
    implementation of that stream replays the games.  `moves_out`, if given, receives one list of actions per game."""
    result, moves, _, _ = ctx.eval_naive(episode_count, count=count, batch_size=batch_size, epsilon=epsilon, alpha=alpha,
                                         evaluator=evaluator, seed=seed, first_tree=first_tree)
    if moves_out is not None:
        moves_out[:] = [[int(a) for a in row if a >= 0] for row in moves]
    return result
