"""bench.py is what the driver measures with, and its GPU arm cannot run in the build container. This drives
bench.main() end to end on the CPU with the device layer replaced by recorders (fake torch.cuda entry points, fake
JxgContext / Batch), real synthetic frames, the real host front-end and the real oracle: it checks the script's control
flow and the shape of the JSON line, not any number."""
import json
import sys
import types

import pytest


from tests import bench_fakes


@pytest.mark.parametrize("fail_e2e", [False, True])
def test_bench_main_control_flow(monkeypatch, capsys, tmp_path, fail_e2e):
    import numpy as np
    import jxl_rs_b200 as j
    bench = bench_fakes.install(monkeypatch.setattr, fail_e2e)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "3", "--warmup", "3", "--frames", "3",
                                      "--width", "320", "--height", "200", "--cpu-sample-frames", "1", "--lf-tree", "1",
                                      "--dump-outputs", str(tmp_path)])
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    bench.main()
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1
    line = json.loads(out[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["config"]["frames_per_gpu"] == 3
    assert "weighted-predictor" in line["config"]["workload"]
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] > 0
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    if fail_e2e:
        assert line["e2e"]["value"] is None and "injected failure" in line["e2e"]["error"]
        assert line["value"] > 0  # the device-resident measurement survives
    else:
        assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 1000
    # device-resident reruns: 3 warm-up, 1 single-batch stage timing, then exactly --steps timed ones
    assert j.Batch.reruns == 3 + 1 + 3
    # 3 frames of 320x200 fit the dump whole; the device-resident pixels are those of the last timed step
    idx, dev = np.load(tmp_path / "pixel_index.npy"), np.load(tmp_path / "device_rgb.npy")
    assert idx.dtype == np.float64 and np.array_equal(idx, np.arange(320 * 200))
    assert dev.dtype == np.float32 and dev.shape == (3, 320 * 200, 3) and (dev == 100 + j.Batch.reruns).all()
    if fail_e2e:
        assert not (tmp_path / "e2e_rgb.npy").exists()
    else:
        e2e = np.load(tmp_path / "e2e_rgb.npy")
        assert e2e.dtype == np.float32 and e2e.shape == dev.shape and (e2e == j.Batch.runs).all()


def test_dump_sample_is_fixed_and_bounded():
    """--dump-outputs keeps the same pixel positions in every run and stays under 64 MB (both dumped arrays and the
    index) in every BASELINE configuration."""
    import numpy as np
    import bench
    for frames, w, h in ((64, 3840, 2160), (512, 1920, 1080), (1, 16384, 16384), (8, 4096, 4096)):
        idx = bench.sample_index(h, w, frames)
        assert 2 * frames * len(idx) * 3 * 4 + 8 * len(idx) < 64_000_000
        assert len(np.unique(idx)) == len(idx) and 0 <= idx[0] and idx[-1] < w * h
        assert np.array_equal(idx, bench.sample_index(h, w, frames))


def test_bench_two_ranks_over_gloo(tmp_path):
    """The multi-rank control flow (per-rank frame seeds and host-thread share, barriers, max-over-ranks reductions, rank
    0 printing the line) with two CPU processes launched the way the driver launches them."""
    import os
    import socket
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    driver = tmp_path / "drive.py"
    driver.write_text(
        "import sys\n"
        f"sys.path.insert(0, {root!r})\n"
        "from tests import bench_fakes\n"
        "bench = bench_fakes.install(setattr, gloo=True)\n"
        "sys.argv = ['bench.py', '--gpus', '2', '--steps', '2', '--warmup', '3', '--frames', '2', '--width', '200',\n"
        "            '--height', '120', '--cpu-sample-frames', '1']\n"
        "bench.main()\n")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(driver)],
                       capture_output=True, text=True, timeout=300, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    line = json.loads(lines[0])
    assert line["n_gpus"] == 2 and line["e2e"]["value"] > 0 and line["value"] > 0
