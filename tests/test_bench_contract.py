"""bench.py contract on the CPU side: `--impl reference` prints exactly ONE JSON line on stdout with the driver's keys, the same
`config` function serves both arms, and non-zero ranks of a torchrun launch stay silent.  On the GPU: `--dump-outputs` writes
the solution of the last timed step."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    e["OMP_NUM_THREADS"] = "2"
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "lid_driven2D_nx64",
                           "--steps", "1", "--warmup", "0", *extra], capture_output=True, text=True, env=e, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run([])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert KEYS <= set(line)
    assert line["impl"] == "reference" and line["metric"] == "DOF-timesteps/s" and line["higher_is_better"] is True
    assert line["config"]["workload"] == "lid_driven2D_nx64" and line["config"]["dofs"] == 3 * 65 * 65
    assert line["steps"] == 1 and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    r = _run(["--gpus", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_follows_the_weak_scaled_mesh_of_an_n_gpu_run():
    """At N > 1 the GPU arm solves one cavity of nx * sqrt(N) squared: rank 0 of the reference arm marches the same mesh."""
    r = _run(["--gpus", "4"], env={"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "4"})
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert line["n_gpus"] == 4 and line["config"]["global_nx"] == 128 and line["config"]["dofs"] == 3 * 129 * 129
    assert line["config"]["cells_per_gpu"] == 2 * 128 * 128 // 4


def test_steps_below_one_and_dump_outputs_off_the_single_gpu_arm_are_refused(tmp_path):
    """--steps is the number of timed steps, so 0 is an error rather than 1; the CPU arm has no --dump-outputs."""
    for extra in (["--steps", "0"], ["--dump-outputs", str(tmp_path / "out")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *extra],
                           capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and r.stdout == "", r.stderr[-2000:]
    assert not (tmp_path / "out").exists()


def test_dump_outputs_samples_large_arrays_the_same_way_every_time(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    arrays = {"velocity": rng.standard_normal(3000), "pressure": rng.standard_normal(1500).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, a.astype(np.float64))
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 900)
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    total = 0
    for name, a in arrays.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))
        assert got.size == a.size * 900 // 4500 and np.isin(got, a.astype(np.float64)).all()
        total += got.nbytes
    assert total <= 8 * 900


@pytest.mark.gpu
def test_dump_outputs_holds_the_solution_of_the_last_timed_step(tmp_path):
    """K timed steps after W warm-up steps: the dumped velocity and pressure are those of step W + K of the same
    scenario marched directly."""
    import numpy as np
    pytest.importorskip("torch")
    import bench
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "lid_driven2D_nx64", "--steps", "2",
                        "--warmup", "3", "--no-extra", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and line["warmup"] == 3
    u, p = np.load(out / "velocity.npy"), np.load(out / "pressure.npy")
    assert u.dtype == p.dtype == np.float64 and u.shape == (2 * 65 * 65,) and p.shape == (65 * 65,)
    sc = bench.build_scenario(bench.WORKLOADS["lid_driven2D_nx64"], device=0)
    s = sc.solver
    for _ in range(5):
        s.step_device()
    x = s.d_x.cpu().numpy()
    s.hemo.close()
    assert np.linalg.norm(u - x[:2 * s.n]) <= 1e-6 * np.linalg.norm(u)
    pm, qm = p - p.mean(), x[2 * s.n:] - x[2 * s.n:].mean()
    assert np.linalg.norm(pm - qm) <= 1e-6 * np.linalg.norm(qm)
