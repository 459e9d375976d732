"""bench.py's reference arm (the CPU port of the reference algorithm) prints the contract's JSON line."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-games", "300"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "simulated_plays_per_sec" and d["unit"] == "plays/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_rejected_arguments():
    """No timed step, or outputs asked of the CPU arm, is an argument error before anything runs."""
    for extra, msg in ((["--steps", "0"], "--steps must be at least 1"),
                       (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs needs --impl ours")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert r.returncode == 2 and msg in r.stderr and r.stdout == ""


def test_dump_outputs_samples(tmp_path):
    """`--dump-outputs` on outputs larger than its limits (host tensors stand in for the device buffers): a sorted,
    repeatable sample of distinct games / matchups, player boxes cut to their byte budget, 64 MiB at most in all."""
    import numpy as np
    import torch
    import bench
    from fast_monte_carlo_b200 import native
    rng = np.random.default_rng(1)
    g = bench.DUMP_GAMES + 12345
    pts = rng.integers(0, 128, (g, 2))
    words = torch.from_numpy((pts[:, 0] | (pts[:, 1] << 16)).astype(np.int32))
    hist = torch.from_numpy(rng.integers(0, 1 << 20, (70, 2, 128, 128), dtype=np.int32))
    counters = torch.arange(native.N_COUNTERS, dtype=torch.int64)
    ids = bench.sample_ids(g, bench.DUMP_GAMES)
    assert np.array_equal(ids, bench.sample_ids(g, bench.DUMP_GAMES)) and len(np.unique(ids)) == len(ids) == bench.DUMP_GAMES
    assert (np.diff(ids) > 0).all() and np.array_equal(bench.sample_ids(5, 8), np.arange(5))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), words, hist, counters, None)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == ["counters", "hist", "scores"]
    assert all(np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy")) for k, a in got.items())
    assert got["scores"].dtype == np.float32 and np.array_equal(got["scores"], pts[ids])
    assert got["hist"].dtype == np.float64 and np.array_equal(got["hist"], hist.numpy()[bench.sample_ids(70, 64)])
    assert got["counters"].tolist() == list(range(15))
    # a player box of 48 slots: only the first games that fit in DUMP_BOX_BYTES
    n, slots = 40000, 48
    box = torch.from_numpy(rng.integers(0, 1 << 40, (n, 2, slots, 2), dtype=np.int64))
    bench.dump_outputs(str(tmp_path / "p"), words[:n], hist[:1], counters, box)
    players = np.load(tmp_path / "p" / "players.npy")
    keep = bench.DUMP_BOX_BYTES // players[0].nbytes
    assert keep < n and players.shape == (keep, 2, slots, 6) and players.nbytes <= bench.DUMP_BOX_BYTES
    assert np.array_equal(players, native.unpack_player_box(box[:keep].numpy().view(native.PLAYER_REC)[..., 0]),
                          equal_nan=True)
    worst = bench.DUMP_GAMES * 2 * 4 + bench.DUMP_BOX_BYTES + bench.DUMP_MATCHUPS * 2 * 128 * 128 * 8 + 15 * 8
    assert worst <= bench.DUMP_BYTES


def test_reference_arm_player_mode():
    """`--players`: the CPU arm samples names from the synthetic focus sheet too, and says so in `config`."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-games", "200", "--players"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["value"] > 0 and "focus sheet" in d["config"]["players"]
