"""Generate the committed golden fixtures from the REAL reference (pulser-core,
imported from the copy that __graft_entry__.build() makes under oracle/_ref)
plus the tight-tolerance oracle.

Run where pulser-core is importable:
    python tests/golden/make_golden.py [--extra | --xy | --slm | --counters | --workloads]

Each ``*.npz`` holds a HamiltonianSpec (what the reference's Hamiltonian
constructor receives, extracted from real pulser objects), an initial state and
the expected output.  Sources of the expected values:
  * ``ref_*``  : numbers hard-coded in the reference's own tests
                 (tests/pulser_simulation/test_simulation.py etc., cited below);
  * ``orc_*``  : oracle (oracle/evolve.py, DOP853 rtol 1e-13) on the same spec;
  * ``pul_*``  : what pulser-core itself computes (drive tables, interaction
                 matrices) for the Sequences that pulser_b200/workloads.py restates.
"""
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import pulser_b200  # noqa: F401,E402  (import hooks)
from pulser import NoiseModel, Pulse, Register, Sequence  # noqa: E402
from pulser._hamiltonian_data import HamiltonianData  # noqa: E402
from pulser.devices import AnalogDevice, DigitalAnalogDevice, MockDevice  # noqa: E402
from pulser.sampler import sampler  # noqa: E402
from pulser.waveforms import BlackmanWaveform, RampWaveform  # noqa: E402

from oracle import evolve  # noqa: E402
from oracle.ref_hamiltonian import OracleHamiltonian  # noqa: E402
from pulser_b200.spec import spec_from_pulser  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def hdata(seq, noise_model=None, n_traj=None, rate=1.0):
    samples = sampler.sample(seq, extended_duration=seq.get_duration())
    T = samples.max_duration
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        hd = HamiltonianData(
            samples.extend_duration(T + 1), seq.register, seq.device,
            noise_model or NoiseModel(), n_traj,
        )
    return hd, T


def specs_of(seq, noise_model=None, n_traj=None, rate=1.0):
    hd, T = hdata(seq, noise_model, n_traj, rate)
    out = []
    for traj, ns, reps in hd.noisy_samples:
        out.append((spec_from_pulser(ns, traj, hd.basis_data, hd.lindblad_data, rate, T), reps))
    return out


def oracle_final(spec, psi0):
    H = OracleHamiltonian.from_spec(spec)
    return evolve.sesolve(H, psi0, [0.0, spec.sampling_times[-1]], rtol=1e-13, atol=1e-15)[-1]


def save(name, spec, **extra):
    spec.save(os.path.join(OUT, name + ".npz"), **extra)
    print("wrote", name)


def main():
    # --- reference golden: test_get_hamiltonian (test_simulation.py:476-588) ---
    reg = Register.from_coordinates([[10, 0], [0, 0]], prefix="atom")
    seq = Sequence(reg, DigitalAnalogDevice)
    seq.declare_channel("ising", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(RampWaveform(1500, 0.0, 2.0), 1.0, 0.0), "ising")
    spec = specs_of(seq, rate=0.01)[0][0]
    save("ref_get_hamiltonian_rate001", spec, t_ns=143.0,
         h00=DigitalAnalogDevice.interaction_coeff / 10**6 - 2 * 1.0)
    np.random.seed(123)
    spec = specs_of(seq, NoiseModel(samples_per_run=1, temperature=20000), 15)[0][0]
    save("ref_get_hamiltonian_doppler", spec, t_ns=144.0, h=np.array(
        [[4.47984523, 0.09606404, 0.09606404, 0.0],
         [0.09606404, 12.03082372, 0.0, 0.09606404],
         [0.09606404, 0.0, -12.97113702, 0.09606404],
         [0.0, 0.09606404, 0.09606404, 0.0]]))
    np.random.seed(456)
    spec = specs_of(seq, NoiseModel(samples_per_run=1, temperature=50.0, trap_depth=150.0,
                                    trap_waist=1.0), 1)[0][0]
    save("ref_get_hamiltonian_register", spec, t_ns=144.0, h=np.array(
        [[4.92294305, 0.09606404, 0.09606404, 0.0],
         [0.09606404, -0.59902269, 0.0, 0.09606404],
         [0.09606404, 0.0, -0.70099956, 0.09606404],
         [0.0, 0.09606404, 0.09606404, 0.0]]))

    # --- reference golden: test_initial_state_sim (test_simulation.py:2156-2190), rtol 1e-2 ---
    seq = Sequence(Register({"q0": (-6, 0), "q1": (0, 0), "q2": (6, 0)}), AnalogDevice)
    seq.declare_channel("ising", "rydberg_global")
    seq.add(Pulse.ConstantPulse(4000, 9.28, 18.7, 0), "ising")
    spec = specs_of(seq)[0][0]
    psi0 = np.ones(8, dtype=complex) / np.sqrt(8)
    gold = np.array([0.28985369 + 0.13530479j, 0.40220557 + 0.0j, 0.27445983 + 0.15541026j,
                     0.29608403 + 0.06155379j, 0.40220557 + 0.0j, 0.36173532 - 0.01617572j,
                     0.29608403 + 0.06155379j, 0.36931122 - 0.15570528j])
    save("ref_initial_state_sim", spec, psi0=psi0, ref_final=gold, orc_final=oracle_final(spec, psi0))

    # --- reference golden: test_qutip_backend (test_qutip_backend.py:43-59), atol 1e-5 ---
    seq = Sequence(Register({"q0": (0, 0)}), MockDevice)
    seq.declare_channel("raman_local", "raman_local", initial_target="q0")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(1000, np.pi), 0, 0), "raman_local")
    spec = specs_of(seq)[0][0]
    psi0 = evolve.all_ground_state(spec)
    save("ref_qutip_backend_pi_pulse", spec, psi0=psi0, ref_final_abs=np.array([0.0, 1.0]),
         orc_final=oracle_final(spec, psi0))

    # --- reference golden: test_add_max_step_and_delays (test_simulation.py:612-633) ---
    seq = Sequence(Register.from_coordinates([(0, 0)], prefix="q"), DigitalAnalogDevice)
    seq.declare_channel("ch", "rydberg_global")
    seq.delay(1500, "ch")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(600, np.pi), 0, 0), "ch")
    seq.delay(2000, "ch")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(600, np.pi / 2), 0, 0), "ch")
    spec = specs_of(seq)[0][0]
    psi0 = evolve.all_ground_state(spec)
    save("ref_delays_occupation", spec, psi0=psi0, ref_r_occupation=0.5,
         orc_final=oracle_final(spec, psi0))

    # --- oracle goldens on real pulser sequences -------------------------------
    # C1 (BASELINE configs[0])
    seq = Sequence(Register.square(2, spacing=6.0, prefix="q"), MockDevice)
    seq.declare_channel("ch", "rydberg_global")
    seq.add(Pulse.ConstantPulse(1000, 2 * np.pi, np.pi, 0), "ch")
    spec = specs_of(seq)[0][0]
    psi0 = evolve.all_ground_state(spec)
    save("orc_c1_square", spec, psi0=psi0, orc_final=oracle_final(spec, psi0))

    # 3-level 'all' basis: raman (digital) + rydberg channels, CCZ-like (test_simulation.py:43-95)
    reg = Register({"control1": np.array([-4.0, 0.0]), "target": np.array([0.0, 4.0]),
                    "control2": np.array([4.0, 0.0])})
    seq = Sequence(reg, DigitalAnalogDevice)
    seq.declare_channel("raman", "raman_local", "control1")
    pi_Y = Pulse.ConstantDetuning(BlackmanWaveform(400, np.pi), 0.0, -np.pi / 2)
    pi_p = Pulse.ConstantDetuning(BlackmanWaveform(400, np.pi), 0.0, 0)
    twopi = Pulse.ConstantDetuning(BlackmanWaveform(400, 2 * np.pi), 0.0, 0)
    seq.add(pi_Y, "raman"); seq.target("target", "raman"); seq.add(pi_Y, "raman")
    seq.declare_channel("ryd", "rydberg_local", "control1")
    seq.add(pi_p, "ryd", protocol="wait-for-all")
    seq.target("control2", "ryd"); seq.add(pi_p, "ryd")
    seq.target("target", "ryd"); seq.add(twopi, "ryd")
    seq.declare_channel("glob", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(600, 0.7 * np.pi), 1.5, 0.3), "glob",
            protocol="wait-for-all")
    spec = specs_of(seq)[0][0]
    psi0 = evolve.all_ground_state(spec)
    save("orc_all_basis_3atoms", spec, psi0=psi0, orc_final=oracle_final(spec, psi0))

    # noisy trajectories (doppler + amplitude, SURVEY 8(d) C4 shape, small)
    np.random.seed(7)
    reg = Register.square(2, spacing=6.5, prefix="q")
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch", "rydberg_global")
    om = 2 * np.pi * 1.5
    seq.add(Pulse.ConstantDetuning(RampWaveform(152, 0, om), -6.0, 0), "ch")
    seq.add(Pulse.ConstantAmplitude(om, RampWaveform(400, -6.0, 8.0), 0), "ch")
    seq.add(Pulse.ConstantDetuning(RampWaveform(200, om, 0), 8.0, 0), "ch")
    nm = NoiseModel(temperature=50.0, amp_sigma=0.05, laser_waist=175.0)
    for i, (spec, reps) in enumerate(specs_of(seq, nm, 3)):
        psi0 = evolve.all_ground_state(spec)
        save(f"orc_noisy_traj{i}", spec, psi0=psi0, orc_final=oracle_final(spec, psi0), reps=reps)


if __name__ == "__main__" and not {"--extra", "--xy", "--slm", "--counters", "--workloads"} & set(sys.argv):
    main()


def extra():
    """Second batch: non-uniform sampling grid (sampling_rate < 1) and leakage + effective noise (Lindblad, d = 3)."""
    reg = Register({"a": (-4.0, 0.0), "b": (0.0, 4.0), "c": (4.0, 0.0)})
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(600, 1.3 * np.pi), -2.0, 0.4), "ch")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(400, 0.6 * np.pi), 3.0, 0.0), "ch")
    spec = specs_of(seq, rate=0.3)[0][0]
    assert len(np.unique(np.round(np.diff(spec.sampling_times), 9))) > 1  # non-uniform grid
    psi0 = evolve.all_ground_state(spec)
    save("orc_sampling_rate_03", spec, psi0=psi0, orc_final=oracle_final(spec, psi0))

    # leakage: eigenbasis (r, g, x) with effective-noise jump operators (reference hamiltonian_data.py:718-738)
    reg = Register({"a": (-3.5, 0.0), "b": (3.5, 0.0)})
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(500, np.pi), 1.0, 0.0), "ch")
    leak = np.zeros((3, 3)); leak[2, 0] = 1.0   # |x><r|
    deph = np.diag([1.0, 0.0, 0.0])
    nm = NoiseModel(with_leakage=True, eff_noise_opers=(leak, deph), eff_noise_rates=(0.3, 0.5))
    spec = specs_of(seq, nm)[0][0]
    assert spec.eigenbasis == ["r", "g", "x"] and spec.collapse_ops.shape == (2, 3, 3)
    from oracle.ref_hamiltonian import OracleHamiltonian as OH
    psi0 = evolve.all_ground_state(spec)
    rho = evolve.mesolve(OH.from_spec(spec), psi0, [0.0, spec.sampling_times[-1]])[-1]
    save("orc_leakage_lindblad", spec, psi0=psi0, orc_rho=rho)


if __name__ == "__main__" and "--extra" in sys.argv:
    extra()


def xy():
    """Third batch: XY mode (microwave channel, eigenbasis u, d)."""
    # reference tests/pulser_simulation/test_simulation.py:1430-1491 (test_get_xy_hamiltonian)
    reg = Register.from_coordinates([[0, 10], [10, 0], [0, 0]], prefix="atom")
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch0", "mw_global")
    seq.set_magnetic_field(0, 1.0, 0.0)
    seq.add(Pulse.ConstantPulse(1500, 3.0, 1.0, 0.0), "ch0")
    spec = specs_of(seq, rate=0.03)[0][0]
    assert spec.eigenbasis == ["u", "d"] and spec.interaction_type == "XY"
    save("ref_get_xy_hamiltonian", spec, t_ns=143.0, c3=MockDevice.interaction_coeff_xy, c6=MockDevice.interaction_coeff)

    # XY evolution of a 4-atom register under a tilted field, full sampling: oracle end state
    reg = Register.from_coordinates([[0, 0], [9, 0], [1, 8], [10, 9]], prefix="a", center=False)
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch0", "mw_global")
    seq.set_magnetic_field(0.4, 1.0, 0.7)
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(400, 1.2 * np.pi), 0.7, 0.3), "ch0")
    seq.add(Pulse.ConstantPulse(200, 2.0, -1.0, 0.0), "ch0")
    spec = specs_of(seq)[0][0]
    psi0 = evolve.all_ground_state(spec)
    save("orc_xy_evolution", spec, psi0=psi0, orc_final=oracle_final(spec, psi0))


if __name__ == "__main__" and "--xy" in sys.argv:
    xy()


def slm():
    """Fourth batch: XY mode with an SLM mask (time-dependent interaction, hamiltonian.py:399-424)."""
    import scipy.sparse as sp

    # reference tests/pulser_simulation/test_simulation.py:1792-1838 (test_mask_two_pulses_xy): the masked
    # Hamiltonian equals (two-qubit H) x 1 while the mask is on and the three-qubit H afterwards.  Checked here
    # on the ORACLE built from the real pulser objects (this pins the oracle's two-term interaction), then the
    # spec and the sample times are stored for the GPU apply_h test.
    reg_three = Register({"q0": (0, 0), "q1": (10, 10), "q2": (-10, -10)})
    reg_two = Register({"q0": (0, 0), "q1": (10, 10)})
    pulse = Pulse.ConstantPulse(100, 10, 0, 0)
    no_pulse = Pulse.ConstantPulse(100, 0, 0, 0)

    def build(reg, pulses, mask=None):
        seq = Sequence(reg, MockDevice)
        seq.declare_channel("ch", "mw_global")
        if mask:
            seq.config_slm_mask(mask)
        for p in pulses:
            seq.add(p, "ch")
        return seq

    seq_masked = build(reg_three, [pulse, pulse, pulse], ["q2"])
    seq_three = build(reg_three, [no_pulse, pulse, pulse])
    seq_two = build(reg_two, [pulse, no_pulse, no_pulse])

    def oracle_of(seq):
        hd, T = hdata(seq)
        traj, ns, _ = next(iter(hd.noisy_samples))
        return OracleHamiltonian.from_pulser(ns, traj, hd.basis_data, hd.lindblad_data, 1.0)

    Hm, H3, H2 = oracle_of(seq_masked), oracle_of(seq_three), oracle_of(seq_two)
    ti, tf = seq_masked._slm_mask_time
    eye2 = sp.identity(2, format="csr")
    for t in Hm.sampling_times:
        hm = Hm.matrix_at(t).toarray()
        if ti <= t * 1000 < tf:  # mask on (sample times strictly inside; the switching sample itself is 1)
            np.testing.assert_allclose(hm, sp.kron(H2.matrix_at(t), eye2).toarray(), atol=1e-12)
        elif t * 1000 > tf:
            np.testing.assert_allclose(hm, H3.matrix_at(t).toarray(), atol=1e-12)
    spec = specs_of(seq_masked)[0][0]
    assert spec.slm_end == tf and spec.slm_targets == [2]
    # spec-built oracle == pulser-built oracle, between samples too (spline of the 0/1 coefficient)
    Hs = OracleHamiltonian.from_spec(spec)
    for t in (0.0, 0.0503, 0.0991, 0.1004, 0.1507, 0.2999):
        np.testing.assert_allclose(Hs.matrix_at(t).toarray(), Hm.matrix_at(t).toarray(), atol=1e-12)
    rng = np.random.default_rng(7)
    psi0 = rng.normal(size=8) + 1j * rng.normal(size=8)
    psi0 /= np.linalg.norm(psi0)
    save("ref_mask_two_pulses_xy", spec, psi0=psi0, orc_final=oracle_final(spec, psi0),
         h_two_kron=np.stack([sp.kron(H2.matrix_at(t), eye2).toarray() for t in (0.01, 0.05, 0.09)]),
         h_three=np.stack([H3.matrix_at(t).toarray() for t in (0.15, 0.2, 0.29)]))

    # a 6-atom register, two masked atoms, tilted field, mask ending inside the first of two pulses' successor
    reg = Register.from_coordinates([[0, 0], [9, 0], [1, 8], [10, 9], [-8, 3], [4, -9]], prefix="a", center=False)
    seq = Sequence(reg, MockDevice)
    seq.declare_channel("ch0", "mw_global")
    seq.set_magnetic_field(0.4, 1.0, 0.7)
    seq.config_slm_mask(["a1", "a4"])
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(300, 1.1 * np.pi), 0.5, 0.2), "ch0")
    seq.add(Pulse.ConstantPulse(300, 2.5, -0.8, 0.0), "ch0")
    spec = specs_of(seq)[0][0]
    assert spec.slm_end == 300 and sorted(spec.slm_targets) == [1, 4]
    psi0 = evolve.all_ground_state(spec)
    save("orc_xy_slm_evolution", spec, psi0=psi0, orc_final=oracle_final(spec, psi0))

    # reference tests/pulser_simulation/test_simulation.py:1960-1998 (test_effective_size_disjoint, mw_global):
    # SPAM leaves atom0 and atom2 unprepared (seed 15092021), the SLM mask covers atom1, so fewer than two good
    # unmasked atoms remain: H(0) = 0.5 * amp * sigma_x on atom3 alone (no interaction, masked atom not driven).
    np.random.seed(15092021)
    seq = Sequence(Register.square(2, prefix="atom"), MockDevice)
    seq.declare_channel("ch0", "mw_global")
    seq.add(Pulse.ConstantPulse(1500, 1, 0, 0), "ch0")
    seq.config_slm_mask(["atom1"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        nm = NoiseModel(samples_per_run=5, state_prep_error=0.4, p_false_pos=0.01, p_false_neg=0.05)
    spec = specs_of(seq, nm, n_traj=15, rate=0.01)[0][0]
    assert list(spec.bad_atoms) == [True, False, True, False], spec.bad_atoms
    assert spec.slm_targets == [1] and spec.slm_end == 1500
    sx3 = np.kron(np.eye(8), np.array([[0.0, 1.0], [1.0, 0.0]]))
    np.testing.assert_allclose(OracleHamiltonian.from_spec(spec).matrix_at(0.0).toarray(), 0.5 * sx3, atol=1e-14)
    save("ref_effective_size_disjoint_xy", spec, h0=0.5 * sx3)


if __name__ == "__main__" and "--slm" in sys.argv:
    slm()


# ---------------------------------------------------------------------------------------------------------------
# Fifth batch: the reference's Counter goldens of its master-equation tests (test_simulation.py:978-1046 test_noises_
# rydberg, :1079-1171 test_noises_digital).  np.random.seed(123); build; run; sample_final_state() -- nothing between
# the seed and the 1000 uniforms of the sampling draws from np.random, so the Counter is a function of the final
# density matrix alone (populations resolved to ~1e-3) and of the sampling recipe.  The oracle reproduces all 14
# EXACTLY (asserted below); the specs + expected counters are the fixtures of the GPU test.
RYDBERG_COUNTERS = [
    (("dephasing",), {"0": 572, "1": 428}, 1),
    (("relaxation",), {"0": 572, "1": 428}, 1),
    (("eff_noise",), {"0": 572, "1": 428}, 1),
    (("depolarizing",), {"0": 561, "1": 439}, 3),
    (("dephasing", "depolarizing", "relaxation"), {"0": 562, "1": 438}, 5),
    (("eff_noise", "dephasing"), {"0": 573, "1": 427}, 2),
    (("eff_noise", "leakage"), {"0": 572, "1": 428}, 1),
]
_DEPH = {"111": 978, "110": 12, "011": 7, "101": 3}
_DEPO = {"111": 827, "101": 63, "011": 59, "110": 40, "010": 5, "001": 4, "000": 1, "100": 1}
_DEPH_DEPO = {"111": 807, "101": 64, "011": 60, "110": 56, "001": 5, "010": 4, "100": 3, "000": 1}
_EFF_DEPH = {"111": 961, "101": 15, "110": 14, "011": 9, "001": 1}
DIGITAL_COUNTERS = [
    (("dephasing",), _DEPH, 1),
    (("eff_noise",), _DEPH, 1),
    (("depolarizing",), _DEPO, 3),
    (("dephasing", "depolarizing"), _DEPH_DEPO, 4),
    (("eff_noise", "dephasing"), _EFF_DEPH, 2),
    (("eff_noise", "leakage"), _DEPH, 1),
    (("eff_noise", "leakage", "dephasing"), _EFF_DEPH, 2),
]


def _legacy_params(noise):
    from pulser.noise_model import _LEGACY_DEFAULTS

    return {
        p: _LEGACY_DEFAULTS[p]
        for p in NoiseModel._find_relevant_params(
            [n for n in noise if n not in ["leakage", "eff_noise"]],
            state_prep_error=_LEGACY_DEFAULTS["state_prep_error"],
            amp_sigma=_LEGACY_DEFAULTS["amp_sigma"],
            laser_waist=_LEGACY_DEFAULTS["laser_waist"],
        )
    }


def counter_case(kind, noise):
    """(sequence, NoiseModel, n_trajectories) of one parametrisation, as the reference test builds it."""
    params = _legacy_params(noise)
    with_leakage = "leakage" in noise
    z = np.diag([1.0, -1.0]).astype(complex)
    if kind == "rydberg":  # test_simulation.py:990-1026
        seq = Sequence(Register.from_coordinates([(0, 0)], prefix="q"), DigitalAnalogDevice)
        seq.declare_channel("ch0", "rydberg_global")
        seq.add(Pulse.ConstantPulse(2500, np.pi, 0, 0), "ch0")
        if with_leakage or "eff_noise" in noise:
            params["eff_noise_opers"] = [np.diag([1.0, 0, 0]).astype(complex) if with_leakage else z]
            params["eff_noise_rates"] = [0.1 if with_leakage else 0.025]
    else:  # test_simulation.py:55-72 (seq_digital), :1115-1146
        reg = Register({"control1": np.array([-4.0, 0.0]), "target": np.array([0.0, 4.0]),
                        "control2": np.array([4.0, 0.0])})
        pi_y = Pulse.ConstantDetuning(BlackmanWaveform(1000, np.pi), 0.0, -np.pi / 2)
        seq = Sequence(reg, DigitalAnalogDevice)
        seq.declare_channel("raman", "raman_local", "control1")
        seq.add(pi_y, "raman")
        seq.target("target", "raman")
        seq.add(pi_y, "raman")
        seq.target("control2", "raman")
        seq.add(pi_y, "raman")
        if "dephasing" in noise:
            params["hyperfine_dephasing_rate"] = 0.05
        if with_leakage or "eff_noise" in noise:
            params["eff_noise_opers"] = [np.diag([0, 1.0, 0]).astype(complex) if with_leakage else z]
            params["eff_noise_rates"] = [0.1 if with_leakage else 0.025]
    n_traj = params.pop("runs", None)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        nm = NoiseModel(with_leakage=with_leakage, **params)
    return seq, nm, n_traj


def counters():
    from collections import Counter

    from oracle import evolve as ev
    from pulser_b200.results import B200Result, CoherentResults, DensityMatrix

    for kind, table in (("rydberg", RYDBERG_COUNTERS), ("digital", DIGITAL_COUNTERS)):
        for noise, expected, n_ops in table:
            from pulser_b200.emulator import B200Emulator

            np.random.seed(123)
            seq, nm, n_traj = counter_case(kind, noise)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                # same constructor path as QutipEmulator.from_sequence (needs no device): what it draws from
                # np.random while building its HamiltonianData is part of the reference's recipe
                sim = B200Emulator.from_sequence(seq, sampling_rate=0.01, noise_model=nm, n_trajectories=n_traj)
            spec = sim._current_spec
            assert len(spec.collapse_ops) == n_ops, (noise, len(spec.collapse_ops))
            psi0 = ev.all_ground_state(spec)
            tf = spec.sampling_times[-1]
            rho = ev.mesolve(OracleHamiltonian.from_spec(spec), psi0, [0.0, tf], rtol=1e-9, atol=1e-11)[-1]
            n, d = spec.n_qudits, spec.dim
            meas = "ground-rydberg" if kind == "rydberg" else "digital"
            res = CoherentResults(
                [B200Result(tuple(spec.qubit_ids), meas, DensityMatrix(rho, [[d] * n, [d] * n]), True, evaluation_time=1.0)],
                n, spec.basis_name, np.array([tf]), meas)
            # the reference seeds ONCE, before building the emulator: the constructor has drawn uniforms from
            # np.random by now (state-preparation draws of HamiltonianData, pulser/_hamiltonian_data/
            # hamiltonian_data.py:795-800) -- count them so that the GPU test, which has no pulser, can put the global
            # stream in the same position
            probe = np.random.get_state()
            nxt = np.random.rand(4)
            np.random.seed(123)
            stream = np.random.rand(64)
            pre_draws = next(k for k in range(60) if np.array_equal(stream[k:k + 4], nxt))
            np.random.set_state(probe)
            got = res.sample_final_state()
            assert got == Counter(expected), (kind, noise, got)
            name = f"ref_counter_{kind}_" + "_".join(noise)
            save(name, spec, psi0=psi0, orc_rho=rho, meas_basis=meas, seed=123, pre_draws=pre_draws,
                 counter_keys=np.array(list(expected)), counter_values=np.array(list(expected.values())))


def eom_counters():
    """reference tests/pulser_simulation/test_simulation.py:2594-2650 (test_eom_limit_det): a NOISELESS three-atom run
    (qutip.sesolve) in EOM mode at the detuning limits; np.random.seed(123); from_sequence; run; sample_final_state()
    == hard-coded Counter.  Pins the Schroedinger path on real QuTiP output the way counters() pins mesolve."""
    import dataclasses
    from collections import Counter

    from pulser.channels import Raman, Rydberg
    from pulser.channels.dmm import DMM
    from pulser.channels.eom import RydbergBeam, RydbergEOM
    from pulser.devices import Device

    from oracle import evolve as ev
    from pulser_b200.emulator import B200Emulator
    from pulser_b200.results import B200Result, CoherentResults, StateVector

    def mod_device():  # tests/conftest.py:29-89 of the reference
        return Device(
            name="ModDevice", dimensions=3, rydberg_level=70, max_atom_num=2000, max_radial_distance=1000,
            min_atom_distance=1, supports_slm_mask=True,
            channel_objects=(
                Rydberg.Global(1000, 200, clock_period=1, min_duration=1, mod_bandwidth=4.0,
                               eom_config=RydbergEOM(mod_bandwidth=30.0, limiting_beam=RydbergBeam.RED,
                                                     max_limiting_amp=50 * 2 * np.pi,
                                                     intermediate_detuning=800 * 2 * np.pi,
                                                     controlled_beams=(RydbergBeam.BLUE,))),
                Rydberg.Local(2 * np.pi * 20, 2 * np.pi * 10, max_targets=2, fixed_retarget_t=0, clock_period=4,
                              min_retarget_interval=220, mod_bandwidth=4.0,
                              eom_config=RydbergEOM(mod_bandwidth=20.0, limiting_beam=RydbergBeam.RED,
                                                    max_limiting_amp=60 * 2 * np.pi,
                                                    intermediate_detuning=700 * 2 * np.pi,
                                                    controlled_beams=tuple(RydbergBeam))),
                Raman.Local(2 * np.pi * 20, 2 * np.pi * 10, max_targets=2, fixed_retarget_t=0,
                            min_retarget_interval=220, clock_period=4, mod_bandwidth=4.0),
            ),
            dmm_objects=(DMM(bottom_detuning=-100, total_bottom_detuning=-10000),
                         DMM(clock_period=4, mod_bandwidth=4.0, bottom_detuning=-50, total_bottom_detuning=-5000)),
        )

    reg = Register({"control1": np.array([-4.0, 0.0]), "target": np.array([0.0, 4.0]),
                    "control2": np.array([4.0, 0.0])})
    for min_detuning_on, expected in (
        (True, {"000": 850, "100": 53, "001": 46, "010": 42, "101": 9}),
        (False, {"000": 879, "010": 49, "100": 40, "001": 32}),
    ):
        dev = mod_device()
        channels = dev.channels
        if not min_detuning_on:
            eom_config = dataclasses.replace(channels["rydberg_global"].eom_config, controlled_beams=(RydbergBeam.RED,))
            channels["rydberg_global"] = dataclasses.replace(channels["rydberg_global"], eom_config=eom_config)
            dev = dataclasses.replace(dev, channel_ids=list(channels), channel_objects=list(channels.values()))
        seq = Sequence(reg, dev)
        seq.declare_channel("ryd_glob", "rydberg_global")
        seq.add(Pulse.ConstantPulse(1000, np.pi / 2, 0, 0), "ryd_glob")
        max_abs_det = seq.declared_channels["ryd_glob"].max_abs_detuning
        detuning_on = -max_abs_det if min_detuning_on else max_abs_det
        seq.enable_eom_mode("ryd_glob", np.pi, detuning_on, correct_phase_drift=True)
        seq.add_eom_pulse("ryd_glob", 1000, 0)
        seq.delay(500, "ryd_glob")
        seq.modify_eom_setpoint("ryd_glob", np.pi / 2, 0, 0, correct_phase_drift=True)
        seq.add_eom_pulse("ryd_glob", 1000, 0)
        np.random.seed(123)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sim = B200Emulator.from_sequence(seq)
        spec = sim._current_spec
        psi0 = ev.all_ground_state(spec)
        final = oracle_final(spec, psi0)
        n, d = spec.n_qudits, spec.dim
        res = CoherentResults(
            [B200Result(tuple(spec.qubit_ids), "ground-rydberg", StateVector(final, [[d] * n, [1] * n]), True,
                        evaluation_time=1.0)],
            n, spec.basis_name, np.array([spec.sampling_times[-1]]), "ground-rydberg")
        probe = np.random.get_state()
        nxt = np.random.rand(4)
        np.random.seed(123)
        stream = np.random.rand(64)
        pre_draws = next(k for k in range(60) if np.array_equal(stream[k:k + 4], nxt))
        np.random.set_state(probe)
        got = res.sample_final_state()
        assert got == Counter(expected), (min_detuning_on, got)
        save("ref_counter_eom_" + ("min_detuning" if min_detuning_on else "max_detuning"), spec, psi0=psi0,
             orc_final=final, meas_basis="ground-rydberg", seed=123, pre_draws=pre_draws,
             counter_keys=np.array(list(expected)), counter_values=np.array(list(expected.values())))


def expect_leakage():
    """reference tests/pulser_simulation/test_simresults.py:339-361 (test_expect, "With leakage"): single atom, Blackman
    pi pulse, collapse operator |x><g| at rate 0.5, sampling_rate 0.1; the reference hard-codes
    <|r><r|>(T) = 0.7804005 (atol 1e-6), a QuTiP mesolve output.  With the 10 ns sampling grid the number depends on
    the QobjEvo coefficient interpolation at the 1e-6 level: cubic spline (QuTiP 5 default) gives 0.780400534, linear
    0.780401390, step 0.778431246 -- the seven printed digits select the cubic spline."""
    from oracle import evolve as ev
    from pulser_b200.emulator import B200Emulator

    seq = Sequence(Register.from_coordinates([(0, 0)], prefix="q"), DigitalAnalogDevice)
    seq.declare_channel("ryd", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(1000, np.pi), 0.0, 0), "ryd")
    eff = np.zeros((3, 3), dtype=complex)
    eff[2, 1] = 1.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sim = B200Emulator.from_sequence(
            seq, noise_model=NoiseModel(eff_noise_rates=[0.5], eff_noise_opers=[eff], with_leakage=True),
            sampling_rate=0.1)
    spec = sim._current_spec
    psi0 = ev.all_ground_state(spec)
    tf = spec.sampling_times[-1]
    vals = {}
    for order in (3, 1):
        rho = ev.mesolve(OracleHamiltonian.from_spec(spec), psi0, [0.0, tf], order=order, rtol=1e-11, atol=1e-13)[-1]
        vals[order] = rho[0, 0].real
    assert abs(vals[3] - 0.7804005) < 5e-8 and abs(vals[1] - 0.7804005) > 5e-7, vals
    rho = ev.mesolve(OracleHamiltonian.from_spec(spec), psi0, [0.0, tf], rtol=1e-11, atol=1e-13)[-1]
    save("ref_expect_leakage", spec, psi0=psi0, orc_rho=rho, ref_value=0.7804005, linear_value=vals[1])


if __name__ == "__main__" and "--counters" in sys.argv:
    if "--eom-only" not in sys.argv and "--expect-only" not in sys.argv:
        counters()
    if "--expect-only" not in sys.argv:
        eom_counters()
    expect_leakage()


def workloads():
    """pul_workloads.npz: what pulser-core computes for the Sequences that pulser_b200/workloads.py restates as plain
    arrays (tests/test_oracle_cpu.py compares the restatements with it).  Drive tables are stored as a seeded sample
    of their columns plus a digest of all of them (tests/helpers.py::table_sample), the rest in full."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import table_sample
    from pulser.devices import AnalogDevice
    from pulser_b200 import workloads as W

    out = {}

    def put(case, spec, tables=True):
        out[f"{case}_eigenbasis"] = np.array(spec.eigenbasis)
        out[f"{case}_basis_name"] = np.array(spec.basis_name)
        out[f"{case}_interaction_type"] = np.array(spec.interaction_type)
        out[f"{case}_interaction_matrix"] = spec.interaction_matrix
        out[f"{case}_sampling_times"] = spec.sampling_times
        out[f"{case}_drive_bases"] = np.array([d.basis for d in spec.drives])
        for i, d in enumerate(spec.drives):
            if tables:
                out[f"{case}_d{i}_coef_cols"], out[f"{case}_d{i}_coef_digest"] = table_sample(d.coef)
                out[f"{case}_d{i}_det_cols"], out[f"{case}_d{i}_det_digest"] = table_sample(d.det)
            else:
                out[f"{case}_d{i}_coef"], out[f"{case}_d{i}_det"] = d.coef, d.det

    om = 2 * np.pi * 1.5
    U = om / 2

    def sweep(seq):
        seq.declare_channel("ch", "rydberg_global")
        seq.add(Pulse.ConstantDetuning(RampWaveform(500, 0, om), -6 * U, 0), "ch")
        seq.add(Pulse.ConstantAmplitude(om, RampWaveform(2500, -6 * U, 2 * U), 0), "ch")
        seq.add(Pulse.ConstantDetuning(RampWaveform(1000, om, 0), 2 * U, 0), "ch")
        return seq

    # C1: 2 x 2 square, one constant pi pulse
    seq = Sequence(Register.square(2, spacing=6.0, prefix="q"), MockDevice)
    seq.declare_channel("ch", "rydberg_global")
    seq.add(Pulse.ConstantPulse(1000, 2 * np.pi, np.pi, 0), "ch")
    put("c1", specs_of(seq)[0][0])
    # C2 at 9 atoms: the blockade sweep on the random disc register
    n = 9
    coords = W.disc_register(n, 38.0, 5.0, n)
    put("c2", specs_of(sweep(Sequence(Register.from_coordinates(coords, center=False, prefix="q"), AnalogDevice)))[0][0])
    # C3 at 5 atoms: raman pi/2 - rydberg pi - raman pi/2 in the 'all' basis
    n = 5
    coords = W.disc_register(n, 22.0, 6.0, 100 + n)
    seq = Sequence(Register.from_coordinates(coords, center=False, prefix="q"), MockDevice)
    seq.declare_channel("ram", "raman_global")
    seq.declare_channel("ryd", "rydberg_global")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(500, np.pi / 2), 0, 0), "ram")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(1000, np.pi), 0, 0), "ryd", protocol="wait-for-all")
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(500, np.pi / 2), 0, 0), "ram", protocol="wait-for-all")
    put("c3", specs_of(seq)[0][0])
    # C4: two doppler + amplitude noise trajectories of the 4 x 4 sweep, with the noise they drew
    seq = sweep(Sequence(Register.square(4, spacing=6.0, prefix="q"), MockDevice))
    np.random.seed(3)
    hd, T = hdata(seq, NoiseModel(temperature=50.0, amp_sigma=0.05, laser_waist=175.0), 2)
    for i, (tr, ns, _) in enumerate(hd.noisy_samples):
        put(f"c4_{i}", spec_from_pulser(ns, tr, hd.basis_data, hd.lindblad_data, 1.0, T))
        out[f"c4_{i}_doppler"] = np.array([tr.doppler_detune[q] for q in seq.register.qubit_ids])
        out[f"c4_{i}_amp"] = np.array(tr.amp_fluctuations["ch"])
    # XY: a global microwave pulse under a tilted field, 5 atoms, 120 ns (small: tables in full)
    n, T, field = 5, 120, (0.3, 1.0, 0.5)
    coords = W.disc_register(n, 30.0, 8.0, 9)
    seq = Sequence(Register.from_coordinates(coords, center=False, prefix="q"), MockDevice)
    seq.declare_channel("mw", "mw_global")
    seq.set_magnetic_field(*field)
    seq.add(Pulse.ConstantDetuning(BlackmanWaveform(T, 1.5 * np.pi), 0.8, 0), "mw")
    put("xy", specs_of(seq)[0][0], tables=False)
    np.savez_compressed(os.path.join(OUT, "pul_workloads.npz"), **out)
    print("wrote pul_workloads")


if __name__ == "__main__" and "--workloads" in sys.argv:
    workloads()
