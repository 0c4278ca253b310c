"""bench.py's orchestration -- K timed steps, collective teardown of the steady-state solver, a second solver for the
end-to-end leg, one JSON line from rank 0 -- executed on the CPU at world_size 1 and 2 (tests/bench_emulated_worker.py:
CUDA emulation + gloo + emulated CUDA IPC).  The numbers are meaningless here; the keys of the contract and the
bookkeeping (edges trained, launches counted, partitions) are checked."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"]


@pytest.mark.parametrize("world", [1, 2])
def test_bench_flow_under_emulation(world, tmp_path):
    subprocess.check_call(["make", "-j8", "-C", os.path.join(ROOT, "tests", "emu")], stdout=subprocess.DEVNULL)
    worker = os.path.join(ROOT, "tests", "bench_emulated_worker.py")
    dump = str(tmp_path / "outputs")
    env = dict(os.environ, GV_EMULATE="1", GV_EMU_IPC="1", GV_EMU_BACKTRACE="1", OMP_NUM_THREADS="1",
               GV_BENCH_DUMP=dump)
    if world == 1:
        command = [sys.executable, worker]
    else:
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        command = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                   "--master-addr", "127.0.0.1", "--master-port", str(port), worker]
    result = subprocess.run(command, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert result.returncode == 0, result.stderr[-4000:]
    lines = [line for line in result.stdout.splitlines() if line.startswith("{")]
    assert len(lines) == 1, result.stdout[-2000:]  # rank 0 alone prints
    line = json.loads(lines[0])
    for key in KEYS:
        assert key in line, key
    assert line["n_gpus"] == world and line["steps"] == 4 and line["warmup"] == 2
    assert line["config"]["num_partition"] == world and line["scaling"] == "weak"
    assert line["value"] > 0 and line["gpu_launches"] > 0
    assert line["roofline"]["bound"] == "hbm" and line["roofline"]["achieved"] > 0
    assert line["e2e"]["value"] > 0 and line["e2e"]["edges"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert "end-to-end train() done" in result.stderr
    assert line["model_quality"]["auc"] > 0 and line["model_quality"]["vertex_norm"] > 0
    if world > 1:  # the multi-rank parity self-check against the oracle's N-worker emulation ran and passed
        assert line["parity_ok"] is True, line.get("parity")
        assert set(line["parity"]) >= {"line_P2", "line_P4", "node2vec_P2", "rotate_adam_P4"} and not line["parity_not_run"]
    # --dump-outputs: rank 0 writes the sample pools of the last step, whole (the toy graph's are small)
    assert sorted(os.listdir(dump)) == ["next_pool.npy", "trained_pool.npy"]
    for name in ("trained_pool", "next_pool"):
        pairs = np.load(os.path.join(dump, name + ".npy"))
        assert pairs.dtype == np.float64 and pairs.ndim == 2 and pairs.shape[1] == 2
        assert len(pairs) > 0 and len(pairs) % (20 * 1000) == 0  # whole blocks of episode_size * batch_size
        assert np.all(pairs == np.floor(pairs)) and pairs.min() >= 0 and pairs.max() < 300


def test_dump_outputs_keeps_a_fixed_sample_of_rows_within_the_budget(tmp_path, monkeypatch):
    import bench
    rows = np.arange(1000, dtype=np.uint32)[:, None] * np.ones((1, 2), dtype=np.uint32)
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 4096 + 2 * 250 * 2 * 8)  # room for a quarter of the rows
    for directory in ("a", "b"):
        bench.dump_outputs(str(tmp_path / directory), {"x": rows, "y": rows + np.uint32(3 << 24)})
    x, y = np.load(str(tmp_path / "a" / "x.npy")), np.load(str(tmp_path / "a" / "y.npy"))
    assert x.dtype == y.dtype == np.float64 and x.shape == y.shape == (250, 2)
    ids = x[:, 0].astype(np.int64)
    assert len(set(ids)) == 250 and np.all(np.diff(ids) > 0)  # distinct rows, in order
    np.testing.assert_array_equal(y[:, 0], ids + (3 << 24))  # the same rows of every array, ids beyond 2^24 exact
    np.testing.assert_array_equal(np.load(str(tmp_path / "b" / "x.npy")), x)  # and the same rows in every run
    total = sum(os.path.getsize(str(tmp_path / "a" / name)) for name in ("x.npy", "y.npy"))
    assert total <= bench.DUMP_BYTES
