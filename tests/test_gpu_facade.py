"""The drop-in surface on a real GPU: ``B200Emulator.from_sequence(seq).run()`` (mirror of
``QutipEmulator``, simulation.py:955-1051, 800-883) and ``B200Backend(seq, config).run()`` (mirror of
``QutipBackendV2``, qutip_backend.py:235-325) driven by real ``pulser.Sequence`` objects through the real
``DevicePlan`` (no fake device), checked against the CPU oracle.

pulser-core reaches the GPU as the copy that build() makes under ``oracle/_ref`` (git-ignored, see DESIGN.md
section 5); the tests skip where it is not importable.
"""
from collections import Counter

import numpy as np
import pytest

from pulser_b200 import HAVE_PULSER

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not HAVE_PULSER, reason="pulser-core not importable"),
    pytest.mark.filterwarnings("ignore::DeprecationWarning"),
]

STATE_TOL = 1e-8


@pytest.fixture(scope="module")
def engine(lib):
    from pulser_b200 import engine

    assert engine.device_count() > 0, "GPU tests need a CUDA device"
    return engine


def _oracle_states(spec, psi0, times, order=3):
    from oracle import evolve
    from oracle.ref_hamiltonian import OracleHamiltonian

    return evolve.sesolve(OracleHamiltonian.from_spec(spec), psi0, list(times), order=order, rtol=1e-13, atol=1e-15)


def _c1_sequence():
    import pulser

    reg = pulser.Register.square(2, 6.0, prefix="q")
    seq = pulser.Sequence(reg, pulser.MockDevice)
    seq.declare_channel("ryd", "rydberg_global")
    seq.add(pulser.Pulse.ConstantPulse(1000, 2 * np.pi, np.pi, 0.0), "ryd")
    return seq


def _sweep_sequence(side=2, spacing=6.0, local=False):
    import pulser
    from pulser.waveforms import ConstantWaveform, RampWaveform

    reg = pulser.Register.square(side, spacing, prefix="q")
    seq = pulser.Sequence(reg, pulser.MockDevice)
    seq.declare_channel("ryd", "rydberg_global")
    om = 2 * np.pi * 1.5
    seq.add(pulser.Pulse(RampWaveform(100, 0.0, om), ConstantWaveform(100, -3 * om), 0.0), "ryd")
    seq.add(pulser.Pulse(ConstantWaveform(300, om), RampWaveform(300, -3 * om, om), 0.0), "ryd")
    seq.add(pulser.Pulse(RampWaveform(100, om, 0.0), ConstantWaveform(100, om), 0.0), "ryd")
    if local:
        seq.declare_channel("ram", "raman_local", initial_target="q0")
        seq.add(pulser.Pulse.ConstantPulse(100, 1.0, 0.3, 0.0), "ram")
    return seq


def test_from_sequence_run_c1_against_oracle(engine):
    """BASELINE configs[0] through the facade: every evaluation-time state within 1e-8 of the oracle."""
    from oracle import evolve
    from pulser_b200 import B200Emulator, workloads as W

    emu = B200Emulator.from_sequence(_c1_sequence(), evaluation_times=0.1)
    res = emu.run()
    spec = emu._current_spec
    ref_spec = W.config_c1()
    np.testing.assert_allclose(spec.drives[0].coef, ref_spec.drives[0].coef)
    np.testing.assert_allclose(np.squeeze(spec.interaction_matrix), np.squeeze(ref_spec.interaction_matrix), rtol=1e-12)
    psi0 = evolve.all_ground_state(spec)
    times = emu._eval_times_array
    refs = _oracle_states(spec, psi0, times)
    assert len(res.states) == len(times)
    for got, ref in zip(res.states, refs):
        assert np.max(np.abs(np.asarray(got.full()).reshape(-1) - ref)) < STATE_TOL
    final = np.asarray(res.get_final_state().full()).reshape(-1)
    assert abs(np.linalg.norm(final) - 1.0) < 1e-9
    counts = res.sample_final_state(500)
    assert sum(counts.values()) == 500 and all(len(k) == 4 for k in counts)
    assert emu.last_run_stats["n_launches"] > 0 and emu.last_run_stats["n_applies"] > 0


def test_noisy_run_equals_oracle_backed_run_shot_for_shot(engine, monkeypatch):
    """Doppler + amplitude noise, 30 trajectories: the GPU run and the same facade run on the oracle-backed fake
    device (tests/fake_device.py) with the same seed give the SAME Counter when the trajectories are sampled one
    per device batch (the reference's order of random draws, simulation.py:847-915)."""
    from fake_device import FakeDevicePlan
    from pulser.noise_model import NoiseModel
    from pulser_b200 import B200Emulator
    from pulser_b200 import engine as eng

    noise = NoiseModel(temperature=50.0, amp_sigma=0.05, runs=30, samples_per_run=5)
    seq = _sweep_sequence()
    out = {}
    for kind in ("gpu", "oracle"):
        if kind == "oracle":
            monkeypatch.setattr(eng, "DevicePlan", FakeDevicePlan)
        np.random.seed(1234)
        emu = B200Emulator.from_sequence(seq, noise_model=noise, evaluation_times="Minimal")
        res = emu.run(b200_batch=1)
        assert res.n_measures == 150
        out[kind] = dict(res.results[-1])
    assert abs(sum(out["gpu"].values()) - 1.0) < 1e-12     # relative frequencies of the 150 shots
    assert out["gpu"] == out["oracle"]


def test_spam_state_preparation_errors_through_the_real_plan(engine):
    """ADVICE r01 (high): a bad atom that silences a local channel leaves its trajectory with fewer drive tables than
    its batch mates; DevicePlan pads the missing basis with a zero table instead of refusing the batch."""
    from pulser.noise_model import NoiseModel
    from pulser_b200 import B200Emulator

    import pulser

    reg = pulser.Register.from_coordinates([(0.0, 0.0), (6.0, 0.0)], prefix="q")
    seq = pulser.Sequence(reg, pulser.MockDevice)
    seq.declare_channel("ryd", "rydberg_global")
    seq.declare_channel("ram", "raman_local", initial_target="q0")
    seq.add(pulser.Pulse.ConstantPulse(200, 2 * np.pi, 0.0, 0.0), "ryd")
    seq.add(pulser.Pulse.ConstantPulse(200, 1.0, 0.5, 0.0), "ram")
    noise = NoiseModel(state_prep_error=0.3, runs=12, samples_per_run=10)
    np.random.seed(7)
    emu = B200Emulator.from_sequence(seq, noise_model=noise, evaluation_times="Minimal")
    res = emu.run()  # default batching: all trajectories in one device batch
    assert res.n_measures == 120
    freq = res.results[-1]
    assert abs(sum(freq.values()) - 1.0) < 1e-12 and all(len(k) == 2 for k in freq)


def test_backend_v2_observables_on_the_device(engine):
    """B200Backend(seq, config=B200Config(observables=[Occupation, Energy, BitStrings])).run() against the oracle."""
    import pulser
    from pulser.backend import BitStrings, Energy, Occupation
    from oracle import evolve
    from oracle.ref_hamiltonian import OracleHamiltonian
    from pulser_b200 import B200Backend, B200Config, B200Emulator

    seq = _sweep_sequence()
    ev = [0.5, 1.0]
    cfg = B200Config(observables=[Occupation(evaluation_times=ev), Energy(evaluation_times=ev),
                                  BitStrings(evaluation_times=[1.0], num_shots=200)])
    res = B200Backend(seq, config=cfg).run()
    emu = B200Emulator.from_sequence(seq)
    spec = emu._current_spec
    H = OracleHamiltonian.from_spec(spec)
    psi0 = evolve.all_ground_state(spec)
    tf = spec.total_duration_ns * 1e-3
    refs = evolve.sesolve(H, psi0, [0.0, 0.5 * tf, tf], rtol=1e-13, atol=1e-15)
    n = spec.n_qudits
    idx = np.arange(spec.hilbert_dim)
    r = spec.eigenbasis.index("r")
    for t, ref in zip(ev, refs[1:]):
        p = np.abs(ref) ** 2
        occ = np.array([p[((idx >> (n - 1 - k)) & 1) == r].sum() for k in range(n)])
        got = np.asarray(res.get_result("occupation", t), dtype=float)
        assert np.max(np.abs(got - occ)) < 1e-8
        hm = H.matrix_at(t * tf, 3)
        e_ref = float(np.vdot(ref, hm @ ref).real)
        assert abs(float(res.get_result("energy", t)) - e_ref) < 1e-7 * max(1.0, abs(e_ref))
    bits = res.get_result("bitstrings", 1.0)
    assert sum(bits.values()) == 200 and all(len(k) == n for k in bits)
    assert isinstance(bits, (Counter, dict))


def test_backend_v2_leakage_energy(engine):
    """ADVICE r01 (medium): with a leakage noise model the noiseless Hamiltonian handed to Energy lives in the
    3-level basis (``_get_noiseless_hamiltonian(with_leakage)``, simulation.py:266-297)."""
    import pulser
    from pulser.backend import Energy, Occupation
    from pulser.noise_model import NoiseModel
    from pulser_b200 import B200Backend, B200Config

    reg = pulser.Register.from_coordinates([(0.0, 0.0), (7.0, 0.0)], prefix="q")
    seq = pulser.Sequence(reg, pulser.MockDevice)
    seq.declare_channel("ryd", "rydberg_global")
    seq.add(pulser.Pulse.ConstantPulse(300, 2 * np.pi, 0.5, 0.0), "ryd")
    leak = np.zeros((3, 3)); leak[2, 0] = 1.0  # |x><r|
    noise = NoiseModel(eff_noise_opers=(leak,), eff_noise_rates=(0.2,), with_leakage=True)
    cfg = B200Config(observables=[Energy(evaluation_times=[1.0]), Occupation(evaluation_times=[1.0])], noise_model=noise)
    res = B200Backend(seq, config=cfg).run()
    e = float(res.get_result("energy", 1.0))
    assert np.isfinite(e)
    occ = np.asarray(res.get_result("occupation", 1.0), dtype=float)
    assert occ.shape == (2,) and np.all(occ >= -1e-9) and np.all(occ <= 1 + 1e-9)


def test_simconfig_c4_phrasing_runs_on_the_gpu(engine):
    """BASELINE configs[3] as written: SimConfig(doppler + amplitude noise) -> from_sequence -> run (striping over
    GPUs is exercised by bench.py --gpus N and tests/test_parallel_cpu.py)."""
    from pulser_b200 import B200Emulator, SimConfig

    cfg = SimConfig(noise=("doppler", "amplitude"), runs=16, samples_per_run=4, temperature=50.0, amp_sigma=0.05)
    np.random.seed(5)
    emu = B200Emulator.from_sequence(_sweep_sequence(), config=cfg, evaluation_times="Minimal")
    res = emu.run()
    assert res.n_measures == 64
    freq = res.results[-1]
    assert abs(sum(freq.values()) - 1.0) < 1e-12 and all(len(k) == 4 for k in freq)
