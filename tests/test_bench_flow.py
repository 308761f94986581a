"""bench.py's product arm executed end to end WITHOUT a GPU: the CUDA library and torch.cuda are replaced by stand-ins that
follow the real interfaces (tests/fake_gpu.py), so that the control flow the driver launches -- single GPU and the N > 1 path
(shard verification, per-GPU events, leader barriers), alone and under a real torchrun launch with two and three ranks -- cannot
hide a Python error or a dead-lock until it runs on a multi-GPU box.  Nothing here measures anything; the assertions are about
the JSON contract and about every process leaving."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
        "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline")


def _check_line(line, ngpu, strong):
    for key in KEYS:
        assert key in line, key
    assert line["n_gpus"] == ngpu and line["steps"] == 3 and line["unit"] == "images/s"
    assert line["scaling"] == ("strong" if strong else "weak")
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and line["e2e"]["h2d_bytes_per_step"] > 0
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    if ngpu > 1:
        assert "shards checked" in line["config"]["verified"] and str(ngpu) in line["config"]["parallelism"]


@pytest.mark.parametrize("ngpu,extra", [(1, []), (2, []), (4, ["--workload", "yolov3_tiny_uint8", "--global-batch", "16"])])
def test_product_arm_control_flow_and_json_contract(monkeypatch, capsys, ngpu, extra):
    import bench
    import fake_gpu

    undo = fake_gpu.install()
    try:
        monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", str(ngpu), "--steps", "3", "--warmup", "1", "--cpu-window", "0", "--watchdog", "0"] + extra)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
            monkeypatch.delenv(k, raising=False)
        bench.main()
    finally:
        undo()
    _check_line(json.loads(capsys.readouterr().out.strip().splitlines()[-1]), ngpu, bool(extra))


@pytest.mark.parametrize("workload,batch", [("mobilenet_v1_int8", 4), ("yolov5s_int8", 64)])
def test_dump_outputs_writes_every_graph_output_within_the_limit(monkeypatch, capsys, tmp_path, workload, batch):
    """--dump-outputs DIR: one float32 .npy per graph output; whole outputs when they fit in 64 MB, else a seeded sample of each
    (YOLOv5s 640x640 at batch 64 has 4.4 x 10^8 output bytes as float32)."""
    import numpy as np

    import bench
    import fake_gpu

    undo = fake_gpu.install()
    try:
        monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "0", "--cpu-window", "0", "--watchdog", "0", "--workload", workload,
                                          "--batch", str(batch), "--dump-outputs", str(tmp_path / "out")])
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
            monkeypatch.delenv(k, raising=False)
        bench.main()
        g, _ = bench.build_workload(workload, batch)
    finally:
        undo()
    capsys.readouterr()
    files = sorted(os.listdir(tmp_path / "out"))
    assert files == [f"output{i}.npy" for i in range(len(g.outputs))]
    dumps = [np.load(tmp_path / "out" / f) for f in files]
    assert all(a.dtype == np.float32 for a in dumps) and sum(a.nbytes for a in dumps) <= bench.DUMP_LIMIT_BYTES
    whole = sum(g.numel(t) for t in g.outputs) * 4 <= bench.DUMP_LIMIT_BYTES
    assert whole == all(a.shape == g.dims(t) for a, t in zip(dumps, g.outputs))
    if whole:
        assert np.array_equal(dumps[0], (np.arange(dumps[0].size) % 251).astype(g.np_dtype).reshape(dumps[0].shape))


@pytest.mark.parametrize("world", [2, 3])
def test_torchrun_launch_as_the_driver_does_it(world):
    """python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ... with the stand-ins installed in every rank: rank 0
    prints ONE JSON line, the followers follow it through its barriers, every process exits 0 well inside the time limit."""
    import socket

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "bench_fake_gpu_main.py"), "--gpus", str(world), "--steps", "3", "--warmup", "1", "--cpu-window", "0",
           "--workload", "yolov3_tiny_uint8", "--batch", "4"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-600:], r.stderr[-1200:])
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-800:]
    _check_line(json.loads(lines[0]), world, False)


def test_torchrun_launch_leaves_cleanly_when_rank0_fails():
    """An exception in rank 0 in the middle of the run must not leave the followers waiting: the leader tells them to leave on its
    way out, torchrun reports the failure, nobody hangs."""
    import socket
    import time

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "bench_fake_gpu_main.py"), "--gpus", "2", "--steps", "3", "--warmup", "1", "--cpu-window", "0",
           "--workload", "yolov3_tiny_uint8", "--batch", "4"]
    t0 = time.time()
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=dict(os.environ, FAKE_GPU_FAIL="1"))
    assert r.returncode != 0 and "injected failure" in r.stderr
    assert time.time() - t0 < 200
