"""bench.py's control flow for world_size 1 and 2, on CPU: gloo process group, the renderer replaced by bench.FakeBackend
(`--fake`).  Round 1 shipped a bench that crashed at N>1 because the default command line had never run there (the e2e
check compared against buffers the fused-gather mode never writes); this test runs exactly that command line shape."""
import json
import os
import socket
import subprocess
import sys

import pytest

from conftest import ROOT


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _run(world, extra_env=None, extra_args=()):
    port = _free_port()
    procs = []
    for rank in range(world):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port), OMP_NUM_THREADS="1")
        env.update(extra_env or {})
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "bench.py"), "--fake", "--gpus", str(world), "--steps", "3",
                                       "--warmup", "1", *extra_args], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=300) for p in procs]
    for p, (so, se) in zip(procs, outs):
        assert p.returncode == 0, se[-3000:]
    lines = [l for l in outs[0][0].splitlines() if l.startswith("{")]
    assert len(lines) == 1, outs[0]
    assert outs[0][0].count("\n") == 1 and outs[0][0].startswith("{"), "stdout must hold the JSON line and nothing else"
    assert "library banner" in outs[0][1]                                     # ... the banner went to stderr
    assert all(not [l for l in so.splitlines() if l.startswith("{")] for so, _ in outs[1:])     # only rank 0 prints
    return json.loads(lines[0])


@pytest.mark.parametrize("world,no_symm", [(1, False), (2, False), (2, True)])
def test_default_command_line_runs_every_leg(world, no_symm):
    line = _run(world, {"GMPI_FAKE_NO_SYMM": "1"} if no_symm else None)
    assert line["n_gpus"] == world and line["steps"] == 3 and line["warmup"] == 3 and line["value"] > 0
    assert line["scaling"] == "weak" and line["higher_is_better"] is True and line["gpu_launches"] == 3
    for key in ("metric", "unit", "ms_per_step", "dtype", "data", "config", "roofline", "e2e", "train_step", "configs"):
        assert line.get(key) is not None, key
    assert line["e2e"]["matches_device_resident_run"] and line["e2e"]["h2d_bytes_per_step"] > 0
    assert set(line["configs"]) >= {"C2_ffhq256_fwd", "N1_factored_fwd", "C4_video_512", "C5_train_512"}
    assert line["configs"]["C4_video_512"]["scaling"] == "strong"
    assert f"x{world}" in line["config"]["parallelism"] and "L2" in line["config"]["l2"]
    par = line["collective"]
    if world == 1:
        assert "none" in par
    elif no_symm:
        assert "ncclAllGather" in par
    else:
        assert "fused" in par


@pytest.mark.parametrize("world", [1, 2])
def test_dump_outputs_writes_the_last_timed_step_reproducibly(world, tmp_path):
    """--dump-outputs DIR: the headline's frames (every rank's, after the all-gather) as float32 .npy, the same from run to run;
    --steps sets the number of timed launches."""
    import numpy as np
    runs = []
    for i in range(2 if world == 1 else 1):
        d = tmp_path / f"run{i}"
        line = _run(world, extra_args=("--steps", "5", "--dump-outputs", str(d)))
        assert line["steps"] == 5 and line["gpu_launches"] == 5
        runs.append({k: np.load(d / f"{k}.npy") for k in ("color", "depth", "pixel_index")})
    n_pix = world * 2 * 16 * 16                                       # FakeBackend.sizes: 2 MPIs x 1 view, 16^2, per rank
    got = runs[0]
    assert got["color"].shape == (n_pix, 3) and got["depth"].shape == (n_pix,)
    assert got["color"].dtype == np.float32 and got["depth"].dtype == np.float32
    assert np.array_equal(got["pixel_index"], np.arange(n_pix, dtype=np.float64))
    assert np.all(np.isfinite(got["color"])) and np.all(got["depth"] > 0)
    for other in runs[1:]:
        assert all(np.array_equal(got[k], other[k]) for k in got)


def test_dump_outputs_samples_a_fixed_set_of_pixels_beyond_the_cap(tmp_path):
    import numpy as np
    import torch
    import bench
    gen = torch.Generator().manual_seed(3)
    color, depth = torch.rand(3, 3, 20, 24, generator=gen), torch.rand(3, 1, 20, 24, generator=gen)
    cap = 3 * 1024 + 1000 * 24                                        # headers + 1000 of the 1440 pixels
    shapes = bench.dump_outputs(str(tmp_path / "a"), color, depth, max_bytes=cap)
    assert shapes == {"color": [1000, 3], "depth": [1000], "pixel_index": [1000]}
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= cap
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    p = idx.astype(np.int64)
    assert np.array_equal(p, np.unique(p)) and p.max() < 1440
    v, y, x = p // (20 * 24), p // 24 % 20, p % 24
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "color.npy"), color.numpy()[v, :, y, x])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "depth.npy"), depth.numpy()[v, 0, y, x])
    bench.dump_outputs(str(tmp_path / "b"), color * 2, depth, max_bytes=cap)
    assert np.array_equal(np.load(tmp_path / "b" / "pixel_index.npy"), idx)          # the sample does not depend on the data
    assert bench.DUMP_MAX_BYTES <= 64 * 10**6


def test_reference_arm_only_rank0_prints_and_others_exit_zero():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_usable_cores_respects_affinity():
    import bench
    n = bench.usable_cores()
    assert 1 <= n <= len(os.sched_getaffinity(0))


def test_reference_arm_prints_the_product_arms_config(monkeypatch, capsys):
    """`--impl reference` runs on the product arm's `config` (same object), so the driver can pair the two lines."""
    import argparse
    import bench
    monkeypatch.setattr(bench, "cpu_reference_frames_per_s", lambda steps, warmup, budget_s=0: {
        "value": 0.5, "sample": "stub", "cores": 3, "ms_per_step": 2000.0, "spread": 0.0})
    monkeypatch.setenv("RANK", "0")

    class Out:
        lines = []

        def emit(self, s):
            self.lines.append(s)

    bench.run_reference_arm(argparse.Namespace(steps=2, warmup=1, gpus=4, ref_budget_s=1.0), Out())
    line = json.loads(Out.lines[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 4 and line["cpu_baseline"]["cores"] == 3
    assert line["config"] == bench.headline_config(bench.N_PLANES, bench.RES, bench.BATCH, 4)
    assert line["e2e"] == {"value": 0.5, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["metric"] == bench.METRIC and line["unit"] == "frames/s" and line["higher_is_better"] is True
