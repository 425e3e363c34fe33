"""tools/iteration.py --score combines the ranks' replay scores weighted by their rows through
sharding.reduce_measurements: float work entries are summed as floats (world_size-2 gloo process group on the CPU)."""
import importlib
import os
import socket
import sys

import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    sh = importlib.import_module("omok-ai_b200.sharding")
    rows, mean = (3, 0.25) if rank == 0 else (1, 1.5)
    q.put((rank, sh.reduce_measurements({"score_s": 0.5 + rank}, {"score_rows": rows, "score_p_loss": mean * rows})))
    dist.destroy_process_group()


def test_row_weighted_means_over_two_ranks():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, (times, work) in res:
        assert times == {"score_s": 1.5}
        assert work == {"score_rows": 4, "score_p_loss": 2.25} and isinstance(work["score_rows"], int)
        assert work["score_p_loss"] / work["score_rows"] == 0.5625  # (3 * 0.25 + 1 * 1.5) / 4
