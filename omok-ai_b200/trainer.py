"""Trainer side of an AlphaZero iteration (SURVEY.md 8f row 1; BASELINE config 5): what the reference's `Trainer::train`
does between two self-play phases, fed by this library's self-play driver.

  * episode bookkeeping + value targets     src/trainer.rs:141-215   (z of the last ply, sign alternating backwards)
  * 6x symmetry augmentation                src/trainer.rs:216-318, src/utils.rs:1-64
  * replay memory + uniform minibatches     src/trainer.rs:320-352
  * encode_nn_input / encode_nn_targets     alpha-zero/src/encoder.rs:10-68
  * AgentModel::train                       alpha-zero/src/agent_model.rs:26-103,136-168 + network.rs:249-253
        loss = mean((z - v)^2) + mean(softmax_cross_entropy(logits, pi)); tensorflow AdadeltaOptimizer, lr 0.01,
        rho 0.95, epsilon 1e-8 (the crate's defaults); one step, then a SECOND forward that reports the losses
  * data parallelism (config 5)             gradients averaged with one all-reduce per step (NCCL over NVLink on
                                            GPUs, gloo in the CPU tests); every rank then applies the same update

The self-play hot path is the hand-written CUDA of csrc/.  The gradient step is not on that path (600 steps of 128
positions per iteration against ~10^8 network evaluations of self-play).  On a GPU it is `AbiTrainStep`: the C ABI's
omk_train_step (csrc/train_kernels.cu: fp32 forward / backward / Adadelta kernels, NCCL all-reduce of the flat gradient
through an attached communicator) -- the call the Rust `AgentModel::train` shim makes.  `TrainStep` is the same step on
PyTorch autograd over tensors in the reference's variable layout; it runs anywhere (the CPU tests check it against a float64 restatement and check the
data-parallel logic over gloo) and hands weights to the kernels with `sync_to`.
"""
from __future__ import annotations

import collections

import numpy as np
import torch
import torch.nn.functional as F

from .model_io import PARAM_SHAPES

BOARD = 9
CELLS = 81
LRELU = 0.2  # TensorFlow LeakyRelu default alpha (network.rs:77,108,148,161 never set it)


# ---------------------------------------------------------------------------------------------- symmetries
def _perm(fn) -> np.ndarray:
    """Gather indices of a board symmetry: dst[k] = src[perm[k]]."""
    perm = np.empty(CELLS, dtype=np.int64)
    for i in range(BOARD):
        for j in range(BOARD):
            perm[i * BOARD + j] = fn(i, j)
    return perm


# dst[i*size + j] = src[...] exactly as src/utils.rs:1-64 index them
SYMMETRIES = {
    "rotate_90": _perm(lambda i, j: (BOARD - j - 1) * BOARD + i),
    "rotate_180": _perm(lambda i, j: (BOARD - i - 1) * BOARD + (BOARD - j - 1)),
    "rotate_270": _perm(lambda i, j: j * BOARD + (BOARD - i - 1)),
    "flip_horizontal": _perm(lambda i, j: i * BOARD + (BOARD - j - 1)),
    "flip_vertical": _perm(lambda i, j: (BOARD - i - 1) * BOARD + j),
}
AUGMENT_ORDER = ("rotate_90", "rotate_180", "rotate_270", "flip_horizontal", "flip_vertical")  # trainer.rs:223-315


def apply_symmetry(name: str, x: np.ndarray) -> np.ndarray:
    """Apply one symmetry to boards or policies of shape [..., 81]."""
    return np.asarray(x)[..., SYMMETRIES[name]]


# ---------------------------------------------------------------------------------------------- replay memory
class ReplayMemory:
    """The reference's `VecDeque<Transition>` (trainer.rs:27,320-324): (board before the move, turn, pi, z), capped by
    dropping the oldest entries."""

    def __init__(self, capacity: int = 600_000, seed: int = 0):
        self.capacity = capacity
        self.boards = collections.deque()
        self.turns = collections.deque()
        self.policies = collections.deque()
        self.zs = collections.deque()
        self.rng = np.random.default_rng(seed)

    def __len__(self) -> int:
        return len(self.zs)

    def add_episode(self, boards: np.ndarray, policies: np.ndarray, final_z: float) -> int:
        """One finished game: boards [T,81] (0 empty, 1 black, 2 white; Black moves first), policies [T,81],
        `final_z` = z of the LAST ply (1 for a win of its mover, 0 for a draw, trainer.rs:157-162).  Value targets
        alternate sign backwards (:208-214); then the five symmetric copies of every transition follow the originals
        (:216-318)."""
        boards = np.asarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        policies = np.asarray(policies, dtype=np.float32).reshape(-1, CELLS)
        T = boards.shape[0]
        z = np.empty(T, dtype=np.float32)
        cur = np.float32(final_z)
        for t in range(T - 1, -1, -1):
            z[t] = cur
            cur = -cur
        turns = ((boards == 1).sum(1) != (boards == 2).sum(1)).astype(np.uint8)  # 0 = black to move
        for t in range(T):
            self._push(boards[t], turns[t], policies[t], z[t])
        for t in range(T):
            for name in AUGMENT_ORDER:
                self._push(apply_symmetry(name, boards[t]), turns[t], apply_symmetry(name, policies[t]), z[t])
        while len(self) > self.capacity:
            for d in (self.boards, self.turns, self.policies, self.zs):
                d.popleft()
        return 6 * T

    def _push(self, board, turn, policy, z):
        self.boards.append(np.array(board, dtype=np.uint8))
        self.turns.append(int(turn))
        self.policies.append(np.array(policy, dtype=np.float32))
        self.zs.append(float(z))

    def sample(self, batch_size: int):
        """`choose_multiple` (trainer.rs:331-334): a uniform sample without replacement of min(batch, len) transitions."""
        n = min(batch_size, len(self))
        idx = self.rng.choice(len(self), size=n, replace=False)
        boards = np.stack([self.boards[i] for i in idx])
        turns = np.array([self.turns[i] for i in idx], dtype=np.uint8)
        pi = np.stack([self.policies[i] for i in idx])
        z = np.array([self.zs[i] for i in idx], dtype=np.float32)
        return boards, turns, pi, z


def split_episodes(boards: np.ndarray, policy: np.ndarray, status: np.ndarray, carry=None):
    """Cut the (ply, game)-ordered transition blocks of `Context.selfplay_run` into finished games.

    boards [P,G,81], policy [P,G,81], status [P,G] (status AFTER the move; a finished game restarts on the next ply).
    Returns (episodes, carry): episodes = list of (boards[T,81], policies[T,81], final_z); `carry` holds the unfinished
    tails, pass it to the next call (the reference trains on finished episodes only, trainer.rs:206-215).
    A status outside {InProgress, Draw, BlackWin, WhiteWin} -- Option::None of a refused move -- is an error, not an
    end of game."""
    P, G = status.shape
    if status.size and (int(status.min()) < 0 or int(status.max()) > 3):
        raise ValueError("self-play produced a status outside 0..3 (a refused move): the transition stream is corrupt")
    carry = carry if carry is not None else [([], []) for _ in range(G)]
    episodes = []
    for g in range(G):
        bs, ps = carry[g]
        for p in range(P):
            bs.append(boards[p, g])
            ps.append(policy[p, g])
            st = int(status[p, g])
            if st != 0:  # Draw -> 0, BlackWin / WhiteWin -> 1 from the mover's point of view (trainer.rs:157-162)
                episodes.append((np.stack(bs), np.stack(ps), 0.0 if st == 1 else 1.0))
                bs, ps = [], []
        carry[g] = (bs, ps)
    return episodes, carry


# ---------------------------------------------------------------------------------------------- encoders
def encode_nn_input(boards: np.ndarray, turns: np.ndarray, opponent_mode: bool = False) -> np.ndarray:
    """[n,243] memory images of encoder.rs:10-46: floats [0,162) = (cell, {perspective side, other side}) pairs written
    by `encode_board` (environment lib.rs:81-102), floats [162,243) = 1.0 when Black is to move.  (TensorFlow then reads
    the slot as [9,9,3]; the network kernels and `TrainStep` do the same.)"""
    boards = np.asarray(boards).reshape(-1, CELLS)
    turns = np.asarray(turns).reshape(-1)
    n = boards.shape[0]
    img = np.zeros((n, 243), dtype=np.float32)
    persp = turns ^ 1 if opponent_mode else turns          # 0: black's perspective
    black_first = (persp == 0)[:, None]
    is_b, is_w = boards == 1, boards == 2
    pair = img[:, :162].reshape(n, CELLS, 2)
    pair[:, :, 0] = np.where(black_first, is_b, is_w)
    pair[:, :, 1] = np.where(black_first, is_w, is_b)
    img[:, 162:] = (turns == 0)[:, None].astype(np.float32)
    return img


def encode_nn_targets(pi: np.ndarray, z: np.ndarray):
    """encoder.rs:48-68: policy target [n,9,9], value target [n,1]."""
    pi = np.asarray(pi, dtype=np.float32).reshape(-1, BOARD, BOARD)
    return pi, np.asarray(z, dtype=np.float32).reshape(-1, 1)


# ---------------------------------------------------------------------------------------------- gradient step
def forward_logits(params, images: torch.Tensor):
    """The reference network (network.rs:51-262) on torch tensors in the reference's variable layout.
    images [B,243] -> (policy logits [B,81], value [B,1])."""
    (conv_w, conv_b), blocks, (fc0_w, fc0_b, fc1_w, fc1_b, v_w, v_b, p_w, p_b) = params[:2], params[2:23], params[23:]
    B = images.shape[0]
    x = images.reshape(B * CELLS, 3)                       # the 243-float slot read as [81][3]
    x = F.leaky_relu(x @ conv_w.reshape(3, 128) + conv_b, LRELU)
    for r in range(3):
        w0, b0, dw, pw, b1, w2, b2 = blocks[7 * r: 7 * r + 7]
        h = F.leaky_relu(x @ w0.reshape(128, 32) + b0, LRELU)
        h = h.reshape(B, BOARD, BOARD, 32).permute(0, 3, 1, 2)          # depthwise 3x3, SAME, no bias
        h = F.conv2d(h, dw[:, :, :, 0].permute(2, 0, 1).unsqueeze(1), None, padding=1, groups=32)
        h = h.permute(0, 2, 3, 1).reshape(B * CELLS, 32)
        h = F.leaky_relu(h @ pw.reshape(32, 32) + b1, LRELU)
        x = F.leaky_relu(h @ w2.reshape(32, 128) + b2 + x, LRELU)
    flat = x.reshape(B, CELLS * 128)                       # NHWC flatten: (y*9+x)*128 + c
    h = F.leaky_relu(flat @ fc0_w + fc0_b, LRELU)
    h = F.leaky_relu(h @ fc1_w + fc1_b, LRELU)
    return h @ p_w + p_b, torch.tanh(h @ v_w + v_b)


def losses(params, images, pi, z):
    """(p_loss, v_loss, loss) of agent_model.rs:60-73 and network.rs:249-253."""
    logits, v = forward_logits(params, images)
    v_loss = torch.mean((z.reshape(-1, 1) - v) ** 2)
    p_loss = torch.mean(-(pi.reshape(-1, CELLS) * F.log_softmax(logits, dim=1)).sum(dim=1))
    return p_loss, v_loss, p_loss + v_loss


class TrainStep:
    """`AgentModel::train` with the optimizer state of the reference's graph (Adadelta accumulators, never saved)."""

    LEARNING_RATE = 0.01  # agent_model.rs:24

    def __init__(self, params, device="cpu", dtype=torch.float32):
        self.device = torch.device(device)
        self.params = [torch.tensor(np.asarray(p, dtype=np.float32).reshape(s), device=self.device, dtype=dtype, requires_grad=True)
                       for p, s in zip(params, PARAM_SHAPES)]
        # tensorflow::train::AdadeltaOptimizer defaults: rho 0.95, epsilon 1e-8 (== ApplyAdadelta's update rule)
        self.opt = torch.optim.Adadelta(self.params, lr=self.LEARNING_RATE, rho=0.95, eps=1e-8)
        self.steps = 0

    def _t(self, a, dtype=None):
        return torch.as_tensor(np.asarray(a), device=self.device).to(dtype or self.params[0].dtype)

    def train(self, images, pi, z):
        """One optimizer step on the local minibatch (gradients averaged over the process group when one is
        initialised), then the reference's second forward: returns (p_loss, v_loss, loss) AFTER the update."""
        images, pi, z = self._t(images).reshape(-1, 243), self._t(pi), self._t(z)
        self.opt.zero_grad(set_to_none=True)
        _, _, loss = losses(self.params, images, pi, z)
        loss.backward()
        self._average_gradients()
        self.opt.step()
        self.steps += 1
        with torch.no_grad():
            out = torch.stack(losses(self.params, images, pi, z))
            dist = torch.distributed
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                dist.all_reduce(out, op=dist.ReduceOp.SUM)
                out /= dist.get_world_size()
        p_loss, v_loss, total = (float(x) for x in out.tolist())
        return p_loss, v_loss, total

    def _average_gradients(self):
        """Data parallelism of config 5: ONE all-reduce of the 5 643 250 gradients (22.6 MB fp32) per step."""
        dist = torch.distributed
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        flat = torch.cat([p.grad.reshape(-1) for p in self.params])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat /= dist.get_world_size()
        off = 0
        for p in self.params:
            n = p.numel()
            p.grad.copy_(flat[off:off + n].reshape(p.shape))
            off += n

    def numpy_params(self):
        return [p.detach().to(torch.float32).cpu().numpy() for p in self.params]

    def sync_to(self, ctx) -> None:
        """Hand the current weights to the CUDA self-play kernels of `ctx` (omk_net_load_params)."""
        ctx.net_load_params(self.numpy_params())


class AbiTrainStep:
    """`AgentModel::train` through the C ABI (omk_train_step): weights, Adadelta slots and the gradient live in the
    context `ctx`; after every step the self-play kernels of the same context see the new weights (no `sync_to`).
    With `world > 1` a NCCL communicator is attached to the context: `unique_id` comes from rank 0's
    `ctx.train_comm_unique_id()` and reaches the other ranks by any side channel (tools/iteration.py broadcasts it with
    torch.distributed); every step then all-reduces the 22.6 MB gradient once."""

    LEARNING_RATE = 0.01

    def __init__(self, ctx, world: int = 1, rank: int = 0, unique_id: bytes | None = None):
        self.ctx, self.world, self.steps = ctx, world, 0
        if world > 1:
            if unique_id is None:
                raise ValueError("data-parallel training needs rank 0's NCCL unique id")
            ctx.train_comm_init(unique_id, world, rank)

    def train(self, images, pi, z):
        self.steps += 1
        return self.ctx.train_step(images, pi, z)

    def train_replay(self, steps: int, minibatch: int, seed: int):
        """`steps` steps on minibatches sampled from the context's device replay memory (omk_train_replay): losses
        [steps, 3].  The sampler streams continue from this object's step count, so consecutive calls draw fresh ones."""
        losses = self.ctx.train_replay(seed, self.steps, steps, minibatch)
        self.steps += steps
        return losses

    def numpy_params(self):
        return self.ctx.net_get_params()

    def sync_to(self, ctx) -> None:
        if ctx is not self.ctx:
            ctx.net_load_params(self.numpy_params())
