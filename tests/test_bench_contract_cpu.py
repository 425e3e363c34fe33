"""bench.py's output contract, checked on the CPU through the reference arm (`--impl reference` times the oracle port on the
host cores and needs no GPU): exactly one JSON line on stdout with the keys the driver reads; under torchrun only rank 0
prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = run({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "mcts_simulations_per_sec" and d["unit"] == "simulations/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and abs(cb["value"] - d["value"]) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["steps"] == 1


def test_reference_arm_other_ranks_stay_silent():
    r = run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_steps_below_one_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "--steps" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_writes_float32_rows_within_the_cap(tmp_path):
    """The writer behind `--dump-outputs`: every array as float32 with its values kept, game_index.npy naming the games,
    and above the cap a seeded sample of games that is the same on every call."""
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(3)
    games = 300
    arrays = {"selfplay_boards": rng.integers(0, 3, (games, 81)).astype(np.uint8),
              "selfplay_policy": rng.random((games, 81), dtype=np.float32),
              "selfplay_actions": rng.integers(-1, 81, games).astype(np.int32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays, games)
    assert (np.load(tmp_path / "all" / "game_index.npy") == np.arange(games)).all()
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float32 and (got == a).all(), name
    bench.DUMP_LIMIT_BYTES = 100_000
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), arrays, games)
        assert sum(f.stat().st_size for f in (tmp_path / run).iterdir()) <= bench.DUMP_LIMIT_BYTES
    idx = np.load(tmp_path / "s1" / "game_index.npy")
    assert 0 < len(idx) < games and (idx == np.load(tmp_path / "s2" / "game_index.npy")).all()
    assert (np.load(tmp_path / "s1" / "selfplay_policy.npy") == arrays["selfplay_policy"][idx.astype(int)]).all()
