"""CPU tests: the oracle against the reference's own golden numbers, the
matrix-free oracle against the literal restatement, workloads against what
pulser-core computes (tests/golden/pul_workloads.npz)."""
import glob
import os

import numpy as np
import pytest

from helpers import assert_table_equal, random_local_spec, random_state
from oracle import evolve
from oracle.matfree import MatFreeHamiltonian
from oracle.ref_hamiltonian import OracleHamiltonian
from pulser_b200 import HAVE_PULSER, workloads as W
from pulser_b200.spec import HamiltonianSpec

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    path = os.path.join(GOLD, name + ".npz")
    with np.load(path, allow_pickle=False) as data:
        return HamiltonianSpec.from_npz(data), {k: data[k] for k in data.files}


def test_golden_get_hamiltonian_h00():
    """reference tests/pulser_simulation/test_simulation.py:489-494"""
    spec, extra = load("ref_get_hamiltonian_rate001")
    H = OracleHamiltonian.from_spec(spec)
    h = H.matrix_at(float(extra["t_ns"]) / 1000).toarray()
    assert np.isclose(h[0, 0], float(extra["h00"]))
    assert np.allclose(h, h.conj().T)


@pytest.mark.parametrize("name", ["ref_get_hamiltonian_doppler", "ref_get_hamiltonian_register"])
def test_golden_get_hamiltonian_noisy(name):
    """reference test_simulation.py:496-588 (assert_allclose default rtol 1e-7)"""
    spec, extra = load(name)
    H = OracleHamiltonian.from_spec(spec)
    h = H.matrix_at(float(extra["t_ns"]) / 1000).toarray()
    np.testing.assert_allclose(h, extra["h"], rtol=1e-7, atol=1e-8)


def test_golden_get_xy_hamiltonian():
    """reference tests/pulser_simulation/test_simulation.py:1430-1491 (test_get_xy_hamiltonian)"""
    spec, extra = load("ref_get_xy_hamiltonian")
    c3, c6 = float(extra["c3"]), float(extra["c6"])
    h = OracleHamiltonian.from_spec(spec).matrix_at(float(extra["t_ns"]) / 1000).toarray()
    assert h[1, 2] == c3 / 10**3
    assert abs(h[1, 4] - (-2 * c3 / 10**3)) < 1e-10
    assert h[0, 1] == 0.5 * 3.0
    n_d = np.array([0, 1, 1, 2, 1, 2, 2, 3])
    vdw = np.array([2 + 1 / 8, 1 / 8, 1, 0, 1, 0, 0, 0]) * c6 / 1e6
    np.testing.assert_array_almost_equal(np.diag(h).real, -1.0 * n_d + vdw)
    # matrix-free oracle == literal restatement in XY mode
    v = random_state(8, 3)
    assert np.max(np.abs(MatFreeHamiltonian(spec).apply(0.143, v) - h @ v)) < 1e-12


def test_xy_workload_matrix_free_equals_literal():
    spec = W.config_xy(n=5, seed=2, t_total=60, local_rows=True, magnetic_field=(0.3, 1.0, 0.5))
    H = OracleHamiltonian.from_spec(spec)
    v = random_state(32, 1)
    for t in (0.004, 0.0313):
        assert np.max(np.abs(MatFreeHamiltonian(spec).apply(t, v) - H.matrix_at(t) @ v)) < 1e-11


def test_golden_initial_state_sim():
    """reference test_simulation.py:2156-2190 pins the 3-atom final state to
    rtol 1e-2 (generated with an older pulser/QuTiP).  The restatement agrees
    to 5.8e-3 max-abs; the residual is the zero-padded last nanosecond
    (SURVEY.md Appendix C.3), so the check here is max-abs < 1e-2."""
    spec, extra = load("ref_initial_state_sim")
    H = OracleHamiltonian.from_spec(spec)
    out = evolve.sesolve(H, extra["psi0"], [0, spec.sampling_times[-1]], rtol=1e-10, atol=1e-12)[-1]
    out = out * np.exp(-1j * np.angle(out[np.argmax(np.abs(out))]))
    assert np.max(np.abs(out - extra["ref_final"])) < 1e-2
    f = extra["orc_final"]
    f = f * np.exp(-1j * np.angle(f[np.argmax(np.abs(f))]))
    assert np.max(np.abs(out - f)) < 1e-8


def test_golden_pi_pulse_digital():
    """reference tests/pulser_simulation/test_qutip_backend.py:43-59 (atol 1e-5)"""
    spec, extra = load("ref_qutip_backend_pi_pulse")
    assert spec.eigenbasis == ["g", "h"] and not spec.has_interaction()
    H = OracleHamiltonian.from_spec(spec)
    out = evolve.sesolve(H, extra["psi0"], [0, spec.sampling_times[-1]], rtol=1e-10, atol=1e-12)[-1]
    np.testing.assert_allclose(np.abs(out), extra["ref_final_abs"], atol=1e-5)
    assert np.max(np.abs(out - extra["orc_final"])) < 1e-8


def test_golden_delays_occupation():
    """reference test_simulation.py:612-633: final |r> occupation 0.5 (1e-4)"""
    spec, extra = load("ref_delays_occupation")
    f = extra["orc_final"]
    assert np.all(np.isfinite(f))
    assert abs(abs(f[0]) ** 2 - float(extra["ref_r_occupation"])) < 1e-4


def test_zvode_adams_default_options_match_tight_oracle():
    """QuTiP-default stand-in (adams, atol 1e-8, rtol 1e-6, max_step 1 ns)
    agrees with the tight oracle at the reference's own accuracy (~1e-5)."""
    spec = W.config_c1()
    H = OracleHamiltonian.from_spec(spec)
    psi0 = evolve.all_ground_state(spec)
    tf = spec.sampling_times[-1]
    tight = evolve.sesolve(H, psi0, [0, tf])[-1]
    loose, stats = evolve.sesolve(H, psi0, [0, tf], method="zvode-adams", rtol=1e-6, atol=1e-8,
                                  max_step=1e-3, nsteps=100000, return_stats=True)
    assert np.max(np.abs(loose[-1] - tight)) < 1e-4
    assert stats["rhs_calls"] >= spec.total_duration_ns  # >= 1 RHS per ns (SURVEY 0.6)


@pytest.mark.parametrize("builder", [
    lambda: W.config_c1(),
    lambda: W.config_c2(n=6, seed=3),
    lambda: random_local_spec(5, T=64, seed=2),
])
def test_matfree_equals_literal_restatement(builder):
    spec = builder()
    mf = MatFreeHamiltonian(spec)
    H = OracleHamiltonian.from_spec(spec)
    v = random_state(spec.hilbert_dim, 1)
    for t in (0.0, 0.0123, spec.sampling_times[-1] * 0.77):
        ref = H.matrix_at(t) @ v
        assert np.max(np.abs(mf.apply(t, v) - ref)) < 1e-12 * max(1.0, np.max(np.abs(ref)))


def test_matfree_all_basis():
    spec, _ = load("orc_all_basis_3atoms")
    assert spec.dim == 3 and spec.basis_name == "all" and len(spec.drives) == 2
    mf = MatFreeHamiltonian(spec)
    H = OracleHamiltonian.from_spec(spec)
    v = random_state(27, 5)
    for t in (0.2, 1.0, 1.9):
        assert np.max(np.abs(mf.apply(t, v) - H.matrix_at(t) @ v)) < 1e-12


def test_spec_roundtrip(tmp_path):
    spec = random_local_spec(4, T=32, seed=8)
    p = str(tmp_path / "s.npz")
    spec.save(p)
    back = HamiltonianSpec.load(p)
    assert back.eigenbasis == spec.eigenbasis
    np.testing.assert_array_equal(back.drives[0].coef, spec.drives[0].coef)
    np.testing.assert_array_equal(back.interaction_matrix, spec.interaction_matrix)


def test_fixtures_present():
    assert len(glob.glob(os.path.join(GOLD, "*.npz"))) >= 11


def load_pulser_case(case):
    """What pulser-core computed for one of the Sequences that workloads.py restates (make_golden.py --workloads)."""
    with np.load(os.path.join(GOLD, "pul_workloads.npz"), allow_pickle=False) as data:
        return {k[len(case) + 1:]: data[k] for k in data.files if k.startswith(case + "_")}


def assert_drive_equals_pulser(ref, i, drive):
    assert_table_equal(drive.coef, ref[f"d{i}_coef_cols"], ref[f"d{i}_coef_digest"])
    assert_table_equal(drive.det, ref[f"d{i}_det_cols"], ref[f"d{i}_det_digest"])


class TestAgainstPulser:
    def _spec(self, seq, rate=1.0):
        from pulser import NoiseModel
        from pulser._hamiltonian_data import HamiltonianData
        from pulser.sampler import sampler
        from pulser_b200.spec import spec_from_pulser

        samples = sampler.sample(seq, extended_duration=seq.get_duration())
        T = samples.max_duration
        hd = HamiltonianData(samples.extend_duration(T + 1), seq.register, seq.device, NoiseModel(), None)
        traj, ns, _ = next(iter(hd.noisy_samples))
        return spec_from_pulser(ns, traj, hd.basis_data, hd.lindblad_data, rate, T), (ns, traj, hd)

    def test_workload_c1_c2_equal_pulser(self):
        """C1 (2 x 2 square, constant pi pulse, MockDevice) and C2 at 9 atoms (blockade sweep on the disc register,
        AnalogDevice) as pulser-core builds them."""
        ref = load_pulser_case("c1")
        b = W.config_c1()
        assert_drive_equals_pulser(ref, 0, b.drives[0])
        np.testing.assert_allclose(ref["interaction_matrix"], b.interaction_matrix, rtol=1e-15)

        n = 9
        ref = load_pulser_case("c2")
        b = W.config_c2(n=n)
        assert_drive_equals_pulser(ref, 0, b.drives[0])
        np.testing.assert_allclose(ref["interaction_matrix"], b.interaction_matrix, rtol=1e-14)
        np.testing.assert_array_equal(ref["sampling_times"], b.sampling_times)

    @pytest.mark.skipif(not HAVE_PULSER, reason="pulser-core not importable here")
    def test_spec_extraction_equals_direct_restatement(self):
        """OracleHamiltonian.from_pulser walks the nested dict itself
        (hamiltonian.py:426-431); from_spec goes through the product's spec."""
        from pulser import Pulse, Register, Sequence
        from pulser.devices import DigitalAnalogDevice
        from pulser.waveforms import BlackmanWaveform

        reg = Register({"a": (-4.0, 0.0), "b": (0.0, 4.0), "c": (4.0, 0.0)})
        seq = Sequence(reg, DigitalAnalogDevice)
        seq.declare_channel("raman", "raman_local", "a")
        seq.add(Pulse.ConstantDetuning(BlackmanWaveform(200, np.pi), 0.0, -np.pi / 2), "raman")
        seq.declare_channel("ryd", "rydberg_local", "b")
        seq.add(Pulse.ConstantDetuning(BlackmanWaveform(200, np.pi), 1.0, 0.4), "ryd")
        seq.declare_channel("glob", "rydberg_global")
        seq.add(Pulse.ConstantDetuning(BlackmanWaveform(300, 1.0), -2.0, 0.0), "glob")
        for rate in (1.0, 0.3):
            spec, (ns, traj, hd) = self._spec(seq, rate)
            A = OracleHamiltonian.from_spec(spec)
            B = OracleHamiltonian.from_pulser(ns, traj, hd.basis_data, hd.lindblad_data, rate)
            np.testing.assert_array_equal(A.sampling_times, B.sampling_times)
            for t in (0.01, 0.25, 0.41):
                assert abs(A.matrix_at(t) - B.matrix_at(t)).max() < 1e-12


def test_fast_terms_equal_kron_terms():
    from oracle.fast_terms import global_ising_hamiltonian

    spec = W.config_c2(n=7, seed=4)
    A = global_ising_hamiltonian(spec)
    B = OracleHamiltonian.from_spec(spec)
    assert len(A.terms) == len(B.terms) == 6  # interaction(+dag), amp(+dag), det(+dag)
    for t in (0.3, 2.2, 3.7):
        assert abs(A.matrix_at(t) - B.matrix_at(t)).max() < 1e-13


def test_workloads_c3_c4_equal_pulser():
    """The numpy restatements of BASELINE configs C3 / C4 equal what pulser-core produces: C3 at 5 atoms (raman pi/2 -
    rydberg pi - raman pi/2, MockDevice), and two doppler + amplitude noise trajectories of C4 rebuilt from the noise
    pulser-core drew for them (np.random.seed(3))."""
    ref = load_pulser_case("c3")
    mine = W.config_c3(5)
    assert list(ref["eigenbasis"]) == mine.eigenbasis == ["r", "g", "h"] and str(ref["basis_name"]) == "all"
    for a in mine.drives:
        i = list(ref["drive_bases"]).index(a.basis)
        assert_drive_equals_pulser(ref, i, a)
    np.testing.assert_allclose(mine.interaction_matrix, ref["interaction_matrix"], rtol=1e-14)

    coords = W.square_register(4, 6.0)
    base = W.ising_global_spec(coords, W.C6_LEVEL_70, *W.blockade_sweep_waveforms())
    for i in range(2):
        ref = load_pulser_case(f"c4_{i}")
        mine = W.noisy_trajectory_spec(base, coords, ref["doppler"], float(ref["amp"]), 175.0)
        assert_drive_equals_pulser(ref, 0, mine.drives[0])
    assert abs(W.doppler_sigma(50.0) - 0.600149981254686) < 1e-15


def test_xy_workload_equals_pulser():
    """workloads.config_xy restates what pulser-core produces for a global microwave pulse under a tilted field."""
    n, T, field = 5, 120, (0.3, 1.0, 0.5)
    mine = W.config_xy(n=n, seed=9, t_total=T, magnetic_field=field)
    ref = load_pulser_case("xy")
    assert list(ref["eigenbasis"]) == mine.eigenbasis and str(ref["interaction_type"]) == "XY"
    assert np.allclose(ref["interaction_matrix"], mine.interaction_matrix, rtol=1e-12, atol=0)
    assert np.allclose(ref["d0_coef"], mine.drives[0].coef, rtol=1e-12, atol=1e-15)
    assert np.allclose(ref["d0_det"], mine.drives[0].det, rtol=1e-12, atol=1e-15)


def test_golden_xy_slm_mask_two_pulses():
    """reference tests/pulser_simulation/test_simulation.py:1792-1838 (test_mask_two_pulses_xy): the oracle built
    from the plain spec reproduces the (two-qubit H) x 1 / three-qubit H matrices that make_golden.py --slm derived
    from the real pulser objects, and the reference's coefficient arrays (hamiltonian.py:405-421)."""
    from oracle.ref_hamiltonian import OracleHamiltonian

    spec, extra = load("ref_mask_two_pulses_xy")
    c = spec.slm_coefficient()
    assert c is not None and len(c) == len(spec.sampling_times)
    assert set(np.unique(c)) == {0.0, 1.0} and c[0] == 0.0 and c[-1] == 1.0
    # _adapt_to_sampling_rate indexes a (T)-long array with T + 1 indices: the switch lands one sample late
    assert c[spec.slm_end] == 0.0 and c[spec.slm_end + 1] == 1.0
    orc = OracleHamiltonian.from_spec(spec)
    for t, ref in zip((0.01, 0.05, 0.09), extra["h_two_kron"]):
        np.testing.assert_allclose(orc.matrix_at(t).toarray(), ref, atol=1e-12)
    for t, ref in zip((0.15, 0.2, 0.29), extra["h_three"]):
        np.testing.assert_allclose(orc.matrix_at(t).toarray(), ref, atol=1e-12)


def test_xy_slm_matrix_free_equals_literal():
    """oracle/matfree.py (the GPU tests' apply_h reference) handles the masked interaction like the literal oracle."""
    from oracle.matfree import MatFreeHamiltonian
    from oracle.ref_hamiltonian import OracleHamiltonian

    spec, _ = load("orc_xy_slm_evolution")
    mf = MatFreeHamiltonian(spec)
    orc = OracleHamiltonian.from_spec(spec)
    rng = np.random.default_rng(3)
    v = rng.normal(size=spec.hilbert_dim) + 1j * rng.normal(size=spec.hilbert_dim)
    for t in (0.05, 0.2995, 0.3004, 0.45):
        np.testing.assert_allclose(mf.apply(t, v), orc.matrix_at(t) @ v, atol=1e-11)


def test_doubled_xy_spec_is_the_commutator_generator():
    """pulser_b200/lindblad.py::doubled_spec in XY mode with an SLM mask: the 2N-qudit Hamiltonian is
    H (x) 1 - 1 (x) H^T, between samples too (host logic of the XY master equation)."""
    from oracle.ref_hamiltonian import OracleHamiltonian
    from pulser_b200.lindblad import doubled_spec

    spec = W.config_xy(n=3, seed=4, t_total=300, magnetic_field=(0.3, 1.0, 0.5))
    spec.slm_end, spec.slm_targets = 120, [1]
    d = doubled_spec(spec)
    assert d.slm_targets == [1, 4] and np.array_equal(d.slm_coefficient(), spec.slm_coefficient())
    H, Hd = OracleHamiltonian.from_spec(spec), OracleHamiltonian.from_spec(d)
    eye = np.eye(8)
    for t in (0.05, 0.1207, 0.25):
        h = H.matrix_at(t).toarray()
        np.testing.assert_allclose(Hd.matrix_at(t).toarray(), np.kron(h, eye) - np.kron(eye, h.T), atol=1e-12)


def test_golden_effective_size_disjoint_xy():
    """reference tests/pulser_simulation/test_simulation.py:1960-1998 (test_effective_size_disjoint, mw_global):
    two unprepared atoms + one SLM-masked atom leave H(0) = 0.5 amp sigma_x on the last atom."""
    from oracle.ref_hamiltonian import OracleHamiltonian

    spec, extra = load("ref_effective_size_disjoint_xy")
    assert list(spec.bad_atoms) == [True, False, True, False] and spec.slm_targets == [1]
    np.testing.assert_allclose(OracleHamiltonian.from_spec(spec).matrix_at(0.0).toarray(), extra["h0"], atol=1e-14)


# ---------------------------------------------------------------------------
# The reference's Counter goldens of its master-equation tests: real QuTiP mesolve outputs, sampled with seed 123.
def _counter_fixture_names():
    import glob

    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLD, "ref_counter_*.npz")))


def _sample_like_the_reference(spec, state, extra):
    from pulser_b200.results import B200Result, CoherentResults, DensityMatrix, StateVector

    n, d = spec.n_qudits, spec.dim
    meas = str(extra["meas_basis"])
    wrapped = DensityMatrix(state, [[d] * n, [d] * n]) if np.ndim(state) == 2 else StateVector(state, [[d] * n, [1] * n])
    res = CoherentResults(
        [B200Result(tuple(spec.qubit_ids), meas, wrapped, True, evaluation_time=1.0)],
        n, spec.basis_name, np.array([spec.sampling_times[-1]]), meas)
    np.random.seed(int(extra["seed"]))
    np.random.rand(int(extra["pre_draws"]))  # what the reference's constructor drew before the run
    return res.sample_final_state()


@pytest.mark.parametrize("name", _counter_fixture_names())
def test_oracle_mesolve_reproduces_reference_counters(name):
    """reference tests/pulser_simulation/test_simulation.py:978-1046 (test_noises_rydberg) and :1079-1171
    (test_noises_digital): the hard-coded Counters come out EXACTLY -- every one of the 1000 shots lands in the same
    bin, which pins the oracle's Lindblad evolution (collapse operators, rates, QobjEvo interpolation) on real QuTiP
    output to the resolution of the sampling, and the sampling recipe itself.  Every master-equation case is
    re-integrated here; tests/golden/make_golden.py --counters asserted the same equalities when it wrote the
    fixtures."""
    from collections import Counter

    from oracle import evolve
    from oracle.ref_hamiltonian import OracleHamiltonian

    spec, extra = load(name)
    expected = Counter(dict(zip((str(k) for k in extra["counter_keys"]), (int(v) for v in extra["counter_values"]))))
    if "_eom_" in name:  # test_simulation.py:2594-2650 (test_eom_limit_det): noiseless sesolve run
        psi = extra["orc_final"]
        if os.environ.get("PB200_SLOW_TESTS") == "1":  # re-integration: 20 s each (detunings of 1000 rad/us)
            psi = evolve.sesolve(OracleHamiltonian.from_spec(spec), extra["psi0"], [0.0, spec.sampling_times[-1]],
                                 rtol=1e-12, atol=1e-14)[-1]
            assert np.max(np.abs(psi - extra["orc_final"])) < 1e-8
        assert _sample_like_the_reference(spec, psi, extra) == expected
        return
    # integrator steps bounded by one sampling interval (the coefficients are smooth splines in between)
    rho = evolve.mesolve(OracleHamiltonian.from_spec(spec), extra["psi0"], [0.0, spec.sampling_times[-1]],
                         rtol=1e-9, atol=1e-11, max_step=float(np.min(np.diff(spec.sampling_times))))[-1]
    assert np.max(np.abs(rho - extra["orc_rho"])) < 1e-6  # (steps may straddle spline knots at this max_step)
    assert _sample_like_the_reference(spec, rho, extra) == expected


def test_golden_expect_leakage_pins_the_interpolation_order():
    """reference tests/pulser_simulation/test_simresults.py:339-361 (test_expect, leakage case): QuTiP's mesolve gave
    <|r><r|>(T) = 0.7804005 on a 10 ns sampling grid.  The oracle reproduces all seven digits with the cubic-spline
    coefficients (QuTiP 5's default ``order=3``, until now an assumption taken from its documentation); with linear
    interpolation the seventh digit is off by nine -- the reference number discriminates between the two."""
    from oracle import evolve
    from oracle.ref_hamiltonian import OracleHamiltonian

    spec, extra = load("ref_expect_leakage")
    tf = spec.sampling_times[-1]
    H = OracleHamiltonian.from_spec(spec)
    cubic = evolve.mesolve(H, extra["psi0"], [0.0, tf], order=3, rtol=1e-10, atol=1e-12)[-1][0, 0].real
    linear = evolve.mesolve(H, extra["psi0"], [0.0, tf], order=1, rtol=1e-10, atol=1e-12)[-1][0, 0].real
    ref = float(extra["ref_value"])
    assert ref == 0.7804005
    assert abs(cubic - ref) < 5e-8          # every printed digit
    assert abs(linear - ref) > 5e-7         # 0.7804014 would have been printed
    assert abs(cubic - extra["orc_rho"][0, 0].real) < 1e-9


def test_oracle_role_table_matches_product_table():
    """oracle/matfree.py keeps its own (to, from) table (restated from hamiltonian.py:340-352); it must agree with
    the one the product uses."""
    from oracle.matfree import BASIS_ROLES as oracle_roles
    from pulser_b200.spec import BASIS_ROLES as product_roles

    assert oracle_roles == product_roles
