"""ctypes binding of libomok_b200.so -- one method per entry point of include/omok_b200.h.

numpy arrays in, numpy arrays out; every non-zero status raises OmkError with the
library's message.  Nothing here computes: it stages pointers.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np

CELLS = 81
NONE = -1
EVAL_NET, EVAL_HASH = 0, 1
SAMPLE_BEST, SAMPLE_BOLTZMANN = 0, 1

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)

NET_LENS = [384, 128] + [4096, 32, 288, 1024, 32, 4096, 128] * 3 + [10368 * 512, 512, 512 * 512, 512, 512, 1, 512 * 81, 81]
NET_SHAPES = (
    [(1, 1, 3, 128), (128,)]
    + [(1, 1, 128, 32), (32,), (3, 3, 32, 1), (1, 1, 32, 32), (32,), (1, 1, 32, 128), (128,)] * 3
    + [(10368, 512), (512,), (512, 512), (512,), (512, 1), (1,), (512, 81), (81,)]
)


class OmkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"omok_b200 error {code}: {msg}")
        self.code = code


class SelfPlayConfig(C.Structure):
    _fields_ = [
        ("n_games", C.c_int32),
        ("count", C.c_int32),
        ("batch_size", C.c_int32),
        ("epsilon", C.c_float),
        ("alpha", C.c_float),
        ("temperature", C.c_float),
        ("temperature_threshold", C.c_int32),
        ("evaluator", C.c_int32),
    ]


class SelfPlayStats(C.Structure):
    _fields_ = [
        ("simulations", C.c_int64),
        ("positions", C.c_int64),
        ("nn_evals", C.c_int64),
        ("games_finished", C.c_int64),
        ("h2d_bytes", C.c_int64),
        ("d2h_bytes", C.c_int64),
        ("gpu_ms", C.c_float),
        ("kind_ms", C.c_float * 8),
        ("kind_launches", C.c_int64 * 8),
    ]

    KINDS = ("tower", "fc0", "fc1", "heads", "hash", "select_expand", "apply", "move")

    def by_kind(self):
        return {k: (float(self.kind_ms[i]), int(self.kind_launches[i])) for i, k in enumerate(self.KINDS)}


def lib_path() -> str:
    return os.path.join(_HERE, "libomok_b200.so")


def declared_symbols() -> list[str]:
    """Every entry point include/omok_b200.h declares (used by the CPU-side ABI test)."""
    text = open(os.path.join(_ROOT, "include", "omok_b200.h")).read()
    return sorted(set(re.findall(r"OMK_API[^;(]*?\b(omk_\w+)\s*\(", text)))


_lib = None


def load_library():
    """dlopen libomok_b200.so; raises (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise OmkError(-2, f"{path} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    L = C.CDLL(path)
    P = C.POINTER
    i32, i64, u64, f32, vp = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_void_p
    L.omk_last_error.restype = C.c_char_p
    L.omk_version.restype = i32
    L.omk_ctx_create.argtypes = [i32, i32, i32, i32, u64, P(vp)]
    L.omk_ctx_destroy.argtypes = [vp]
    L.omk_ctx_synchronize.argtypes = [vp]
    L.omk_ctx_stream.argtypes = [vp]
    L.omk_ctx_stream.restype = vp
    L.omk_ctx_launch_count.argtypes = [vp]
    L.omk_ctx_launch_count.restype = i64
    L.omk_ctx_transfer_bytes.argtypes = [vp, P(i64), P(i64)]
    L.omk_net_load_params.argtypes = [vp, P(vp), P(i64)]
    L.omk_net_get_params.argtypes = [vp, P(vp), P(i64)]
    L.omk_net_init_random.argtypes = [vp, u64]
    L.omk_net_eval.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    L.omk_net_eval_images.argtypes = [vp, vp, i32, vp, vp]
    L.omk_train_step.argtypes = [vp, vp, vp, vp, i32, vp]
    L.omk_train_backward.argtypes = [vp, vp, vp, vp, i32, P(vp), P(i64)]
    L.omk_train_apply.argtypes = [vp, vp]
    L.omk_train_get_grads.argtypes = [vp, P(vp), P(i64)]
    L.omk_train_reset_optimizer.argtypes = [vp]
    L.omk_train_comm_unique_id.argtypes = [vp, vp]
    L.omk_train_comm_init.argtypes = [vp, vp, i32, i32]
    L.omk_train_comm_destroy.argtypes = [vp]
    L.omk_debug_set_fc0_mode.argtypes = [vp, i32]
    L.omk_debug_set_tower_mode.argtypes = [vp, i32]
    L.omk_debug_set_fc0_chunk.argtypes = [vp, i32]
    L.omk_debug_set_fc0_balance.argtypes = [vp, i32]
    L.omk_debug_set_lane_min_trees.argtypes = [vp, i32]
    L.omk_debug_get_buffer.argtypes = [vp, i32, vp, i64]
    L.omk_debug_tower_timing.argtypes = [vp, vp]
    L.omk_env_reset.argtypes = [vp, vp, i32]
    L.omk_env_step.argtypes = [vp, vp, vp, i32, vp, vp]
    L.omk_env_step_device.argtypes = [vp, vp, i32, vp, vp]
    L.omk_env_get.argtypes = [vp, vp, i32, vp, vp, vp]
    L.omk_env_set.argtypes = [vp, vp, i32, vp, vp]
    L.omk_env_encode.argtypes = [vp, vp, i32, i32, vp]
    L.omk_env_random_playout.argtypes = [vp, i32, i32, vp, vp]
    L.omk_pool_new_games.argtypes = [vp, vp, i32, vp, i32]
    L.omk_pool_search.argtypes = [vp, vp, i32, i32, i32, f32, f32, i32]
    L.omk_search_set_virtual_loss.argtypes = [vp, i32]
    L.omk_pool_sample.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.omk_pool_policy.argtypes = [vp, vp, i32, vp, vp]
    L.omk_pool_ensure_action.argtypes = [vp, vp, vp, i32, i32]
    L.omk_pool_play.argtypes = [vp, vp, vp, i32, vp]
    L.omk_pool_get_env.argtypes = [vp, i32, vp, vp, vp]
    L.omk_pool_get_envs.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.omk_pool_root_stats.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.omk_pool_root_children.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.omk_pool_tree_info.argtypes = [vp, i32, vp, vp]
    L.omk_selfplay_begin.argtypes = [vp, P(SelfPlayConfig)]
    L.omk_selfplay_run.argtypes = [vp, i32, i32, vp, vp, vp, vp, P(SelfPlayStats)]
    L.omk_replay_reset.argtypes = [vp, i64]
    L.omk_replay_info.argtypes = [vp, P(i64), P(i64), P(i64)]
    L.omk_replay_get.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.omk_train_replay.argtypes = [vp, u64, i64, i32, i32, vp, vp]
    L.omk_naive_move.argtypes = [vp, vp, vp, i32, u64, vp, vp, vp]
    L.omk_eval_naive.argtypes = [vp, i32, i32, i32, i32, f32, f32, i32, u64, vp, vp, vp, vp, P(f32)]
    L.omk_opponent_load_params.argtypes = [vp, P(vp), P(i64)]
    L.omk_opponent_from_net.argtypes = [vp]
    L.omk_opponent_eval.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    L.omk_match.argtypes = [vp, i32, i32, i32, i32, f32, f32, i32, vp, vp, vp, vp, P(f32)]
    L.omk_model_load_params.argtypes = [vp, i32, P(vp), P(i64)]
    L.omk_model_from_net.argtypes = [vp, i32]
    L.omk_model_eval.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp]
    L.omk_tournament.argtypes = [vp, i32, vp, i32, i32, i32, i32, f32, f32, i32, vp, vp, vp, vp, P(f32)]
    L.omk_tournament_naive.argtypes = [vp, i32, vp, i32, i32, i32, i32, f32, f32, i32, u64, vp, vp, vp, vp, P(f32)]
    for name in declared_symbols():
        fn = getattr(L, name)  # raises AttributeError if the library lacks a declared symbol
        if name not in ("omk_last_error", "omk_ctx_stream", "omk_ctx_launch_count"):
            fn.restype = i32
    _lib = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _ids(ids):
    return None if ids is None else np.ascontiguousarray(ids, dtype=np.int32)


class Context:
    """One CUDA device, one env pool, one tree pool, one network (omk_ctx)."""

    def __init__(self, device: int = 0, capacity_envs: int = 0, capacity_trees: int = 0, capacity_nodes: int = 4096,
                 seed: int = 0):
        self.L = load_library()
        h = C.c_void_p()
        self.h = None
        self._check(self.L.omk_ctx_create(device, capacity_envs, capacity_trees, capacity_nodes, seed, C.byref(h)))
        self.h = h
        self.capacity_envs, self.capacity_trees, self.capacity_nodes = capacity_envs, capacity_trees, capacity_nodes
        self.seed = seed

    def _check(self, rc: int):
        if rc != 0:
            raise OmkError(rc, self.L.omk_last_error().decode())

    def close(self):
        if self.h is not None:
            self.L.omk_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        self._check(self.L.omk_ctx_synchronize(self.h))

    @property
    def stream(self) -> int:
        return int(self.L.omk_ctx_stream(self.h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.L.omk_ctx_launch_count(self.h))

    @property
    def transfer_bytes(self) -> tuple[int, int]:
        """(host->device, device->host) bytes the API layer has copied for this context since creation."""
        a, b = C.c_int64(), C.c_int64()
        self._check(self.L.omk_ctx_transfer_bytes(self.h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    # ---- network ----
    def net_load_params(self, params):
        arrs = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1) for p in params]
        ptrs = (C.c_void_p * 31)(*[a.ctypes.data for a in arrs])
        lens = (C.c_int64 * 31)(*[a.size for a in arrs])
        self._check(self.L.omk_net_load_params(self.h, ptrs, lens))

    def net_get_params(self):
        arrs = [np.zeros(n, dtype=np.float32) for n in NET_LENS]
        ptrs = (C.c_void_p * 31)(*[a.ctypes.data for a in arrs])
        lens = (C.c_int64 * 31)(*NET_LENS)
        self._check(self.L.omk_net_get_params(self.h, ptrs, lens))
        return [a.reshape(s) for a, s in zip(arrs, NET_SHAPES)]

    def net_init_random(self, seed: int = 0):
        self._check(self.L.omk_net_init_random(self.h, seed))

    def net_eval(self, boards, turns, mode: int = 0, want_v: bool = True):
        boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
        n = boards.shape[0]
        p = np.zeros((n, CELLS), dtype=np.float32)
        v = np.zeros(n, dtype=np.float32) if want_v else None
        self._check(self.L.omk_net_eval(self.h, _ptr(boards), _ptr(turns), n, mode, _ptr(p), _ptr(v)))
        return p, v

    def net_eval_images(self, images, want_v: bool = True):
        images = np.ascontiguousarray(images, dtype=np.float32).reshape(-1, 243)
        n = images.shape[0]
        p = np.zeros((n, CELLS), dtype=np.float32)
        v = np.zeros(n, dtype=np.float32) if want_v else None
        self._check(self.L.omk_net_eval_images(self.h, _ptr(images), n, _ptr(p), _ptr(v)))
        return p, v

    # ---- trainer step (AgentModel::train) ----
    @staticmethod
    def _batch(images, pi, z):
        images = np.ascontiguousarray(images, dtype=np.float32).reshape(-1, 243)
        n = images.shape[0]
        pi = np.ascontiguousarray(pi, dtype=np.float32).reshape(n, CELLS)
        z = np.ascontiguousarray(z, dtype=np.float32).reshape(n)
        return images, pi, z, n

    def train_step(self, images, pi, z):
        """One Adadelta step + the reporting forward: (p_loss, v_loss, loss) after the update."""
        images, pi, z, n = self._batch(images, pi, z)
        out = np.zeros(3, dtype=np.float32)
        self._check(self.L.omk_train_step(self.h, _ptr(images), _ptr(pi), _ptr(z), n, _ptr(out)))
        return float(out[0]), float(out[1]), float(out[2])

    def train_backward(self, images, pi, z):
        """Gradient of the local minibatch's mean loss: (device pointer of the flat buffer, element count)."""
        images, pi, z, n = self._batch(images, pi, z)
        ptr, cnt = C.c_void_p(), C.c_int64()
        self._check(self.L.omk_train_backward(self.h, _ptr(images), _ptr(pi), _ptr(z), n, C.byref(ptr), C.byref(cnt)))
        return int(ptr.value or 0), int(cnt.value)

    def train_apply(self):
        out = np.zeros(3, dtype=np.float32)
        self._check(self.L.omk_train_apply(self.h, _ptr(out)))
        return float(out[0]), float(out[1]), float(out[2])

    def train_get_grads(self):
        arrs = [np.zeros(n, dtype=np.float32) for n in NET_LENS]
        ptrs = (C.c_void_p * 31)(*[a.ctypes.data for a in arrs])
        lens = (C.c_int64 * 31)(*NET_LENS)
        self._check(self.L.omk_train_get_grads(self.h, ptrs, lens))
        return [a.reshape(s) for a, s in zip(arrs, NET_SHAPES)]

    def train_reset_optimizer(self):
        self._check(self.L.omk_train_reset_optimizer(self.h))

    def train_comm_unique_id(self) -> bytes:
        buf = np.zeros(128, dtype=np.uint8)
        self._check(self.L.omk_train_comm_unique_id(self.h, _ptr(buf)))
        return buf.tobytes()

    def train_comm_init(self, unique_id: bytes, nranks: int, rank: int):
        buf = np.frombuffer(unique_id, dtype=np.uint8).copy()
        self._check(self.L.omk_train_comm_init(self.h, _ptr(buf), nranks, rank))

    def train_comm_destroy(self):
        self._check(self.L.omk_train_comm_destroy(self.h))

    def debug_set_fc0_mode(self, mode: int):
        self._check(self.L.omk_debug_set_fc0_mode(self.h, mode))

    def debug_set_tower_mode(self, mode: int):
        self._check(self.L.omk_debug_set_tower_mode(self.h, mode))

    def debug_set_fc0_balance(self, on: bool):
        self._check(self.L.omk_debug_set_fc0_balance(self.h, 1 if on else 0))

    def debug_set_fc0_chunk(self, k_blocks: int):
        self._check(self.L.omk_debug_set_fc0_chunk(self.h, k_blocks))

    def debug_set_lane_min_trees(self, min_trees: int):
        self._check(self.L.omk_debug_set_lane_min_trees(self.h, min_trees))

    def debug_tower_timing(self):
        out = np.zeros(64, dtype=np.int64)
        self._check(self.L.omk_debug_tower_timing(self.h, _ptr(out)))
        return out

    def debug_get_buffer(self, which: int, count: int):
        out = np.zeros(count, dtype=np.float32)
        self._check(self.L.omk_debug_get_buffer(self.h, which, _ptr(out), count))
        return out

    # ---- environment pool ----
    def env_reset(self, ids=None, n=None):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        self._check(self.L.omk_env_reset(self.h, _ptr(ids), n))

    def env_step(self, actions, ids=None, want_legal: bool = True):
        actions = np.ascontiguousarray(actions, dtype=np.uint8)
        ids = _ids(ids)
        n = actions.size
        status = np.zeros(n, dtype=np.int8)
        legal = np.zeros((n, 3), dtype=np.uint32) if want_legal else None
        self._check(self.L.omk_env_step(self.h, _ptr(ids), _ptr(actions), n, _ptr(status), _ptr(legal)))
        return status, legal

    def env_step_device(self, actions_dev: int, n: int, status_dev: int, legal_dev: int):
        self._check(self.L.omk_env_step_device(self.h, actions_dev, n, status_dev, legal_dev))

    def env_get(self, ids=None, n=None):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        boards = np.zeros((n, CELLS), dtype=np.uint8)
        turns = np.zeros(n, dtype=np.uint8)
        legal = np.zeros(n, dtype=np.uint16)
        self._check(self.L.omk_env_get(self.h, _ptr(ids), n, _ptr(boards), _ptr(turns), _ptr(legal)))
        return boards, turns, legal

    def env_set(self, boards, turns, ids=None):
        boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
        ids = _ids(ids)
        self._check(self.L.omk_env_set(self.h, _ptr(ids), boards.shape[0], _ptr(boards), _ptr(turns)))

    def env_encode(self, ids=None, n=None, mode: int = 0):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        out = np.zeros((n, 243), dtype=np.float32)
        self._check(self.L.omk_env_encode(self.h, _ptr(ids), n, mode, _ptr(out)))
        return out

    def env_random_playout(self, n: int, plies: int, trace: bool = True):
        actions = np.zeros((plies, n), dtype=np.uint8) if trace else None
        status = np.zeros((plies, n), dtype=np.int8) if trace else None
        self._check(self.L.omk_env_random_playout(self.h, n, plies, _ptr(actions), _ptr(status)))
        return actions, status

    # ---- tree pool ----
    def pool_new_games(self, ids=None, n=None, streams=None, evaluator: int = EVAL_NET):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        streams = None if streams is None else np.ascontiguousarray(streams, dtype=np.uint32)
        self._check(self.L.omk_pool_new_games(self.h, _ptr(ids), n, _ptr(streams), evaluator))

    def pool_search(self, ids=None, n=None, count=800, batch_size=16, epsilon=0.25, alpha=0.03, evaluator: int = EVAL_NET):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        self._check(self.L.omk_pool_search(self.h, _ptr(ids), n, count, batch_size, epsilon, alpha, evaluator))

    def search_set_virtual_loss(self, enabled: bool):
        """Opt-in, non-reference search mode (see include/omok_b200.h); refused with EVAL_HASH while on."""
        self._check(self.L.omk_search_set_virtual_loss(self.h, 1 if enabled else 0))

    def pool_sample(self, ids=None, n=None, modes=None, temperatures=None):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        modes = None if modes is None else np.ascontiguousarray(modes, dtype=np.uint8)
        temperatures = None if temperatures is None else np.ascontiguousarray(temperatures, dtype=np.float32)
        actions = np.zeros(n, dtype=np.int32)
        policy = np.zeros((n, CELLS), dtype=np.float32)
        self._check(self.L.omk_pool_sample(self.h, _ptr(ids), n, _ptr(modes), _ptr(temperatures), _ptr(actions), _ptr(policy)))
        return actions, policy

    def pool_policy(self, ids=None, n=None):
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        policy = np.zeros((n, CELLS), dtype=np.float32)
        valid = np.zeros(n, dtype=np.uint8)
        self._check(self.L.omk_pool_policy(self.h, _ptr(ids), n, _ptr(policy), _ptr(valid)))
        return policy, valid

    def pool_ensure_action(self, actions, ids=None, evaluator: int = EVAL_NET):
        actions = np.ascontiguousarray(actions, dtype=np.int32)
        ids = _ids(ids)
        self._check(self.L.omk_pool_ensure_action(self.h, _ptr(ids), _ptr(actions), actions.size, evaluator))

    def pool_play(self, actions, ids=None):
        actions = np.ascontiguousarray(actions, dtype=np.int32)
        ids = _ids(ids)
        status = np.zeros(actions.size, dtype=np.int8)
        self._check(self.L.omk_pool_play(self.h, _ptr(ids), _ptr(actions), actions.size, _ptr(status)))
        return status

    def pool_get_env(self, tree: int):
        board = np.zeros(CELLS, dtype=np.uint8)
        turn = C.c_uint8()
        legal = C.c_uint16()
        self._check(self.L.omk_pool_get_env(self.h, tree, _ptr(board), C.byref(turn), C.byref(legal)))
        return board, turn.value, legal.value

    def pool_get_envs(self, ids=None, n=None):
        """Agent.env of many trees in one call: (boards [n,81], turns [n], legal counts [n], root status [n])."""
        ids = _ids(ids)
        n = len(ids) if ids is not None else n
        boards = np.zeros((n, CELLS), dtype=np.uint8)
        turns = np.zeros(n, dtype=np.uint8)
        legal = np.zeros(n, dtype=np.uint16)
        status = np.zeros(n, dtype=np.int8)
        self._check(self.L.omk_pool_get_envs(self.h, _ptr(ids), n, _ptr(boards), _ptr(turns), _ptr(legal), _ptr(status)))
        return boards, turns, legal, status

    def pool_root_stats(self, tree: int):
        n = C.c_uint64()
        w = C.c_float()
        p = C.c_float()
        st = C.c_int32()
        pol = np.zeros(CELLS, dtype=np.float32)
        self._check(self.L.omk_pool_root_stats(self.h, tree, C.byref(n), C.byref(w), C.byref(p), C.byref(st), _ptr(pol)))
        return n.value, w.value, p.value, st.value, pol

    def pool_root_children(self, tree: int):
        a = np.zeros(CELLS, dtype=np.int32)
        n = np.zeros(CELLS, dtype=np.uint64)
        w = np.zeros(CELLS, dtype=np.float32)
        p = np.zeros(CELLS, dtype=np.float32)
        k = C.c_int32()
        self._check(self.L.omk_pool_root_children(self.h, tree, _ptr(a), _ptr(n), _ptr(w), _ptr(p), C.byref(k)))
        return a[: k.value], n[: k.value], w[: k.value], p[: k.value]

    def pool_tree_info(self, tree: int):
        nodes = C.c_int32()
        ctr = C.c_uint32()
        self._check(self.L.omk_pool_tree_info(self.h, tree, C.byref(nodes), C.byref(ctr)))
        return nodes.value, ctr.value

    # ---- self-play driver ----
    def selfplay_begin(self, n_games, count=800, batch_size=16, epsilon=0.25, alpha=0.03, temperature=1.0,
                       temperature_threshold=30, evaluator: int = EVAL_NET):
        cfg = SelfPlayConfig(n_games, count, batch_size, epsilon, alpha, temperature, temperature_threshold, evaluator)
        self._sp_n = n_games
        self._check(self.L.omk_selfplay_begin(self.h, C.byref(cfg)))

    def selfplay_run(self, plies: int, profile: int = 0, want_transitions: bool = True):
        n = self._sp_n
        boards = np.zeros((plies, n, CELLS), dtype=np.uint8) if want_transitions else None
        policy = np.zeros((plies, n, CELLS), dtype=np.float32) if want_transitions else None
        status = np.zeros((plies, n), dtype=np.int8) if want_transitions else None
        actions = np.zeros((plies, n), dtype=np.int32) if want_transitions else None
        stats = SelfPlayStats()
        self._check(self.L.omk_selfplay_run(self.h, plies, int(profile), _ptr(boards), _ptr(policy), _ptr(status),
                                            _ptr(actions), C.byref(stats)))
        return stats, boards, policy, status, actions

    # ---- replay memory on the device ----
    def replay_reset(self, capacity: int):
        """Empty the device replay memory and size it to `capacity` rows (0 frees it).  Create it before
        `selfplay_begin`: the driver feeds the replay memory that exists when it starts."""
        self._check(self.L.omk_replay_reset(self.h, int(capacity)))

    def replay_info(self):
        """(rows held, rows added since the last reset, episodes added since the last reset)."""
        a, b, e = C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self.L.omk_replay_info(self.h, C.byref(a), C.byref(b), C.byref(e)))
        return int(a.value), int(b.value), int(e.value)

    def replay_get(self, rows):
        """Rows by logical index (0 = oldest): (boards [n,81] u8, turns [n] u8, policies [n,81] f32, z [n] f32)."""
        rows = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1)
        n = rows.size
        boards = np.zeros((n, CELLS), dtype=np.uint8)
        turns = np.zeros(n, dtype=np.uint8)
        policy = np.zeros((n, CELLS), dtype=np.float32)
        z = np.zeros(n, dtype=np.float32)
        self._check(self.L.omk_replay_get(self.h, _ptr(rows), n, _ptr(boards), _ptr(turns), _ptr(policy), _ptr(z)))
        return boards, turns, policy, z

    def train_replay(self, seed: int, first_step: int, steps: int, n: int, want_rows: bool = False):
        """`steps` trainer steps on minibatches of min(n, len) rows sampled from the device replay memory (step s on
        sampler stream first_step + s).  Returns losses [steps, 3] ({p_loss, v_loss, loss} after each update) and, with
        `want_rows`, the logical rows of each step [steps, n] (-1 past the minibatch size)."""
        losses = np.zeros((steps, 3), dtype=np.float32)
        rows = np.zeros((steps, n), dtype=np.int64) if want_rows else None
        self._check(self.L.omk_train_replay(self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step), int(steps), int(n),
                                            _ptr(losses), _ptr(rows)))
        return (losses, rows) if want_rows else losses

    # ---- evaluation against the naive player ----
    def naive_move(self, boards, turns, seed: int, streams=None):
        """The naive player's move for every position (DESIGN.md 4): (actions [n] i32, forced [n] u8: 1 if the move wins,
        blocks or fills the last cell, 0 if it was drawn on stream streams[i] (default i) of key mix64(seed ^ K_NAIVE))."""
        boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
        n = boards.shape[0]
        streams = None if streams is None else np.ascontiguousarray(streams, dtype=np.uint32).reshape(n)
        actions = np.zeros(n, dtype=np.int32)
        forced = np.zeros(n, dtype=np.uint8)
        self._check(self.L.omk_naive_move(self.h, _ptr(boards), _ptr(turns), n, int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(streams),
                                          _ptr(actions), _ptr(forced)))
        return actions, forced

    def eval_naive(self, episodes: int, count: int = 800, batch_size: int = 16, epsilon: float = 0.25, alpha: float = 0.03,
                   evaluator: int = EVAL_NET, seed: int = 0, first_tree: int = 0):
        """The trainer's evaluation against the naive player in one call, on trees first_tree .. first_tree + episodes - 1.
        Returns (result (black/naive wins, white/model wins, draws), moves [episodes, 81] i8 (-1 past a game's end),
        final status [episodes] i8, stats dict: simulations, nn_evals, moves, host_syncs, gpu_ms)."""
        result = np.zeros(3, dtype=np.int32)
        moves = np.zeros((episodes, CELLS), dtype=np.int8)
        status = np.zeros(episodes, dtype=np.int8)
        stats = np.zeros(4, dtype=np.int64)
        gpu_ms = C.c_float()
        self._check(self.L.omk_eval_naive(self.h, episodes, first_tree, count, batch_size, epsilon, alpha, evaluator,
                                          int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(result), _ptr(moves), _ptr(status), _ptr(stats),
                                          C.byref(gpu_ms)))
        info = dict(zip(("simulations", "nn_evals", "moves", "host_syncs"), (int(x) for x in stats)))
        info["gpu_ms"] = float(gpu_ms.value)
        return (int(result[0]), int(result[1]), int(result[2])), moves, status, info

    # ---- the opponent network and the arena ----
    def opponent_load_params(self, params):
        """A second set of weights, read only by opponent_eval and match (training, self-play and the searches never see it)."""
        arrs = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1) for p in params]
        ptrs = (C.c_void_p * 31)(*[a.ctypes.data for a in arrs])
        lens = (C.c_int64 * 31)(*[a.size for a in arrs])
        self._check(self.L.omk_opponent_load_params(self.h, ptrs, lens))

    def opponent_from_net(self):
        """The opponent becomes a device-side copy of the network's current weights (e.g. the snapshot before training)."""
        self._check(self.L.omk_opponent_from_net(self.h))

    def opponent_eval(self, boards, turns, mode: int = 0, want_v: bool = True):
        """net_eval with the opponent's weights."""
        boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
        n = boards.shape[0]
        p = np.zeros((n, CELLS), dtype=np.float32)
        v = np.zeros(n, dtype=np.float32) if want_v else None
        self._check(self.L.omk_opponent_eval(self.h, _ptr(boards), _ptr(turns), n, mode, _ptr(p), _ptr(v)))
        return p, v

    def match(self, pairs: int, first_tree: int = 0, count: int = 800, batch_size: int = 8, epsilon: float = 0.0, alpha: float = 1.0,
              evaluator: int = EVAL_NET):
        """The benchmark's arena between the network and the opponent in one call: 2 * pairs games, the network opens games
        0 .. pairs - 1, the opponent the rest; trees first_tree .. first_tree + 4 * pairs - 1.  Returns (result (network wins,
        opponent wins, draws), moves [2 * pairs, 81] i8 (-1 past a game's end), final status [2 * pairs] i8, stats dict:
        simulations, nn_evals, moves, host_syncs, gpu_ms)."""
        games = 2 * pairs
        result = np.zeros(3, dtype=np.int32)
        moves = np.zeros((max(games, 0), CELLS), dtype=np.int8)
        status = np.zeros(max(games, 0), dtype=np.int8)
        stats = np.zeros(4, dtype=np.int64)
        gpu_ms = C.c_float()
        self._check(self.L.omk_match(self.h, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, _ptr(result), _ptr(moves),
                                     _ptr(status), _ptr(stats), C.byref(gpu_ms)))
        info = dict(zip(("simulations", "nn_evals", "moves", "host_syncs"), (int(x) for x in stats)))
        info["gpu_ms"] = float(gpu_ms.value)
        return (int(result[0]), int(result[1]), int(result[2])), moves, status, info

    # ---- model slots and the tournament ----
    def model_load_params(self, slot: int, params):
        """Weights into model slot `slot` (1 .. 15; 1 is the opponent), read only by model_eval, match (slot 1) and tournament."""
        arrs = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1) for p in params]
        ptrs = (C.c_void_p * 31)(*[a.ctypes.data for a in arrs])
        lens = (C.c_int64 * 31)(*[a.size for a in arrs])
        self._check(self.L.omk_model_load_params(self.h, slot, ptrs, lens))

    def model_from_net(self, slot: int):
        """Model slot `slot` becomes a device-side copy of the network's current weights (a snapshot)."""
        self._check(self.L.omk_model_from_net(self.h, slot))

    def model_eval(self, slot: int, boards, turns, mode: int = 0, want_v: bool = True):
        """net_eval with model slot `slot`'s weights (slot 0 is the network)."""
        boards = np.ascontiguousarray(boards, dtype=np.uint8).reshape(-1, CELLS)
        turns = np.ascontiguousarray(turns, dtype=np.uint8).reshape(-1)
        n = boards.shape[0]
        p = np.zeros((n, CELLS), dtype=np.float32)
        v = np.zeros(n, dtype=np.float32) if want_v else None
        self._check(self.L.omk_model_eval(self.h, slot, _ptr(boards), _ptr(turns), n, mode, _ptr(p), _ptr(v)))
        return p, v

    def tournament(self, slots, pairs: int, first_tree: int = 0, count: int = 800, batch_size: int = 8, epsilon: float = 0.0,
                   alpha: float = 1.0, evaluator: int = EVAL_NET):
        """A round-robin of `match` over the model slots `slots` in one call: pairing p = (i, j), i < j in lexicographic order,
        is match(pairs) with slots[i] as the network (left) and slots[j] as the opponent (right), on the trees
        first_tree + 4 * pairs * p ..  Returns (result [P, 3] i32 (left wins, right wins, draws), moves [P, 2 * pairs, 81] i8
        (-1 past a game's end), final status [P, 2 * pairs] i8, stats dict: simulations, nn_evals, moves, host_syncs, gpu_ms)."""
        return self._tournament(slots, 0, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, None)

    def tournament_naive(self, slots, pairs: int, seed: int = 0, first_tree: int = 0, count: int = 800, batch_size: int = 8,
                         epsilon: float = 0.0, alpha: float = 1.0, evaluator: int = EVAL_NET):
        """`tournament` with the naive player (naive_move's rule on seed `seed`) as participant 0 and slots[k] as participant
        k + 1: N = len(slots) + 1 participants, P = N(N-1)/2 pairings over participants, the first len(slots) of them
        (naive, slots[k]) with the naive player left, opening games 0 .. pairs - 1.  Returns `tournament`'s tuple."""
        return self._tournament(slots, 1, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, seed)

    def _tournament(self, slots, extra, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, seed):
        s = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
        n = s.size + extra  # participants
        n_pairings = max(n * (n - 1) // 2, 0)
        games = max(2 * pairs, 0)
        result = np.zeros((n_pairings, 3), dtype=np.int32)
        moves = np.zeros((n_pairings, games, CELLS), dtype=np.int8)
        status = np.zeros((n_pairings, games), dtype=np.int8)
        stats = np.zeros(4, dtype=np.int64)
        gpu_ms = C.c_float()
        outs = (_ptr(result), _ptr(moves), _ptr(status), _ptr(stats), C.byref(gpu_ms))
        args = (self.h, s.size, _ptr(s), pairs, first_tree, count, batch_size, epsilon, alpha, evaluator)
        if seed is None:
            self._check(self.L.omk_tournament(*args, *outs))
        else:
            self._check(self.L.omk_tournament_naive(*args, int(seed) & 0xFFFFFFFFFFFFFFFF, *outs))
        info = dict(zip(("simulations", "nn_evals", "moves", "host_syncs"), (int(x) for x in stats)))
        info["gpu_ms"] = float(gpu_ms.value)
        return result, moves, status, info
