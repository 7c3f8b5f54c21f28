"""Shared builders of seeded test inputs (no pulser needed)."""
from __future__ import annotations

import hashlib

import numpy as np

from pulser_b200 import workloads as W
from pulser_b200.spec import DriveTable, HamiltonianSpec


def chain_coords(n: int, spacing: float = 7.0, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    pts = np.array([[i * spacing, 0.0] for i in range(n)], dtype=float)
    return pts + rng.uniform(-0.8, 0.8, size=pts.shape)


def random_local_spec(
    n: int, T: int = 200, seed: int = 1, phase: bool = True, c6: float = W.C6_LEVEL_60
) -> HamiltonianSpec:
    """Per-qubit smooth random amp/det/phase tables (a noisy-trajectory look-alike)."""
    rng = np.random.default_rng(seed)
    t = np.arange(T + 1) / T
    base_amp = 8.0 * np.sin(np.pi * t) ** 2
    base_det = -10.0 + 25.0 * t
    coef = np.zeros((n, T + 1), dtype=complex)
    det = np.zeros((n, T + 1))
    for k in range(n):
        a = base_amp * rng.uniform(0.7, 1.1)
        ph = (rng.uniform(-1, 1) + rng.uniform(-2, 2) * t) if phase else 0.0
        coef[k] = 0.5 * a * np.exp(-1j * ph)
        det[k] = base_det + rng.normal(0, 2.0)
        det[k, -1] = 0.0
        coef[k, -1] = 0.0
    coords = chain_coords(n, 7.0, seed)
    return HamiltonianSpec(
        n_qudits=n, dim=2, eigenbasis=["r", "g"], basis_name="ground-rydberg",
        interaction_type="ising",
        sampling_times=np.arange(T + 1, dtype=float) / 1000,
        total_duration_ns=T,
        interaction_matrix=W.interaction_matrix(coords, c6),
        bad_atoms=np.zeros(n, dtype=bool),
        drives=[DriveTable("ground-rydberg", coef, det, False)],
        collapse_ops=np.zeros((0, 2, 2), dtype=complex),
        qubit_ids=[f"q{i}" for i in range(n)],
    )


def random_state(D: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    v = rng.normal(size=D) + 1j * rng.normal(size=D)
    return v / np.linalg.norm(v)


def digest(a: np.ndarray) -> str:
    """sha256 of an array's shape, dtype and values (-0.0 read as 0.0): equal digests mean equal arrays."""
    a = np.ascontiguousarray(a) + np.zeros((), dtype=np.asarray(a).dtype)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def table_sample(a: np.ndarray, n: int = 64) -> tuple[np.ndarray, str]:
    """A fixed, seeded sample of the columns (time samples) of a drive table, and the digest of the whole table."""
    cols = np.sort(np.random.default_rng(0).choice(a.shape[-1], size=min(n, a.shape[-1]), replace=False))
    return a[..., cols], digest(a)


def assert_table_equal(a: np.ndarray, cols_ref: np.ndarray, digest_ref) -> None:
    """``a`` equals the table that ``table_sample`` summarised: the sampled columns first (a readable failure), then
    every element through the digest."""
    cols, d = table_sample(a, cols_ref.shape[-1])
    np.testing.assert_array_equal(cols, cols_ref)
    assert d == str(digest_ref)
