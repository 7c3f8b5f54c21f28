"""CPU test of bench.py's reference arm (`--impl reference`): the line contract the driver parses, on a small register
(the oracle port of QobjEvo + qutip.sesolve at QuTiP's default options -- the reference's own CPU path for this hot
path, pulser_simulation/simulation.py:729-735).  The GPU arm needs a device and is exercised on the GPU box."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, PB200_BENCH_ATOMS="8", PB200_REF_SAMPLE_STEPS="30", **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                           "--warmup", "0"], env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_line_contract():
    res = _run({})
    assert res.returncode == 0, res.stderr[-400:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "steps/s"
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1e3 * 30 / d["value"]) < 1e-6 * d["ms_per_step"]
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and "30 consecutive" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    res = _run({"RANK": "3", "WORLD_SIZE": "8"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_outputs_format_and_sampling(tmp_path):
    """bench.py --dump-outputs: the final state as float64 (re, im) pairs, the densities, and above the size cap a
    seeded sample of amplitudes that is the same from run to run."""
    code = (
        "import sys, numpy as np; sys.path.insert(0, {root!r}); import bench\n"
        "rng = np.random.default_rng(5); psi = rng.normal(size=64) + 1j * rng.normal(size=64)\n"
        "bench.dump_outputs({full!r}, psi, np.arange(6.0))\n"
        "bench.DUMP_BYTES = 16 * 16\n"
        "bench.dump_outputs({a!r}, psi, np.arange(6.0)); bench.dump_outputs({b!r}, psi, np.arange(6.0))\n"
    ).format(root=ROOT, full=str(tmp_path / "full"), a=str(tmp_path / "a"), b=str(tmp_path / "b"))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-400:]
    import numpy as np

    rng = np.random.default_rng(5)
    psi = rng.normal(size=64) + 1j * rng.normal(size=64)
    full = np.load(tmp_path / "full" / "c2_state.npy")
    assert full.dtype == np.float64 and full.shape == (64, 2)
    np.testing.assert_array_equal(full[:, 0] + 1j * full[:, 1], psi)
    assert sorted(os.listdir(tmp_path / "full")) == ["c2_rydberg_density.npy", "c2_state.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "full" / "c2_rydberg_density.npy"), np.arange(6.0))
    idx = np.load(tmp_path / "a" / "c2_state_index.npy")
    part = np.load(tmp_path / "a" / "c2_state.npy")
    assert idx.dtype == np.float64 and part.shape == (16, 2) and len(np.unique(idx)) == 16
    np.testing.assert_array_equal(part, full[idx.astype(int)])
    np.testing.assert_array_equal(idx, np.load(tmp_path / "b" / "c2_state_index.npy"))


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=300)
    assert res.returncode != 0 and "--steps" in res.stderr
