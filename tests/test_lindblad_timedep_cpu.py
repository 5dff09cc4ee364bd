"""Host side of time-dependent Lindblad problems (no GPU): the piecewise Chebyshev structure that the Lindblad kernels
evaluate at their adaptive stage times must reproduce the callables to 1e-13 at off-node times, also beyond the
evolution time, and every time dependence it cannot represent must be refused."""
import numpy as np
import pytest

from qoc_b200.core.plan import (LindbladTimeStructure, NonlinearHamiltonian, extract_lindblad_time_structure,
                                _lindblad_is_time_dependent)
from tests.problems import Problem, rand_herm

SX = np.array([[0, 1], [1, 0]], dtype=complex)
SY = np.array([[0, -1j], [1j, 0]])
SZ = np.diag([1.0, -1.0]).astype(complex)
SM = np.array([[0, 1], [0, 0]], dtype=complex)


def _max_h_error(st, h, K, cc, seed=0, count=300):
    """largest |H_fit(x, t) - h(u, t)| / scale over random controls and random times in [0, t_max]."""
    rng = np.random.default_rng(seed)
    worst = 0.0
    for t in rng.uniform(0.0, st.t_max, count):
        u = None
        x = np.zeros(0)
        if K:
            u = rng.standard_normal(K) + (1j * rng.standard_normal(K) if cc else 0.0)
            x = np.concatenate([u.real, u.imag]) if cc else u
        got = np.asarray(h(u, t), dtype=complex)
        worst = max(worst, np.abs(got - st.hamiltonian(x, t)).max() / max(1.0, np.abs(got).max()))
    return worst


@pytest.mark.parametrize("cc", [False, True])
@pytest.mark.parametrize("n", [2, 5])
def test_problem_td_hamiltonian(n, cc):
    p = Problem(n, 4, 2, 1, 2, complex_controls=cc, seed=11)
    h = p.hamiltonian_td_numpy()
    t_max = p.T + 1.5
    st = extract_lindblad_time_structure(h, p.K, cc, p.T, p.N, t_max)
    assert isinstance(st, LindbladTimeStructure)
    assert st.t_max >= t_max and st.degree <= 24 and 1 <= st.KC <= 16 and st.L == 0
    assert st.series.shape == (st.segments, st.degree + 1, st.KC * (1 + st.KR))
    assert st.KR == p.K * (2 if cc else 1)
    assert _max_h_error(st, h, p.K, cc) < 1e-13
    # beyond the evolution time in particular
    rng = np.random.default_rng(3)
    for t in rng.uniform(p.T, st.t_max, 20):
        x = rng.standard_normal(st.KR)
        u = x[:p.K] + 1j * x[p.K:] if cc else x
        assert np.abs(h(u, t) - st.hamiltonian(x, t)).max() < 1e-13 * max(1.0, np.abs(h(u, t)).max())


def test_gaussian_envelope_drive():
    T, N = 6.0, 7
    h0 = 0.5 * SZ

    def h(u, t):
        env = np.exp(-(t - T / 2) ** 2 / (2 * 1.2 ** 2))
        return h0 + env * (u[0].real * (np.cos(2.0 * t) * SX + np.sin(2.0 * t) * SY) + u[0].imag * SY)
    st = extract_lindblad_time_structure(h, 1, True, T, N, T + 2.0)
    assert _max_h_error(st, h, 1, True) < 1e-13


def test_time_dependent_drift_without_controls():
    rng = np.random.default_rng(2)
    h0, d = rand_herm(rng, 3), rand_herm(rng, 3)
    h = lambda u, t: h0 + np.cos(1.3 * t) * d + 0.2 * t * t * np.eye(3)
    st = extract_lindblad_time_structure(h, 0, False, 2.0, 3, 3.0)
    assert st.KR == 0 and st.KC >= 1
    assert _max_h_error(st, h, 0, False) < 1e-13


@pytest.mark.parametrize("kind", ["rate", "phase", "both"])
def test_time_dependent_dissipation(kind):
    T, N = 3.0, 4
    ops = np.stack([SM, SZ])

    def ld(t):
        g = np.array([0.1, 0.05])
        o = ops.copy()
        if kind in ("rate", "both"):
            g = g * np.array([1.0 + 0.5 * np.sin(0.7 * t), np.exp(-0.2 * t)])
        if kind in ("phase", "both"):
            o[0] = np.exp(1j * 2.5 * t) * (1.0 + 0.1 * t) * o[0]
        return g, o
    assert _lindblad_is_time_dependent(ld, T)
    st = extract_lindblad_time_structure(None, 0, False, T, N, T + 2.0, lindblad_data=ld)
    assert st.KC == 0 and st.L == 2 and st.series.shape[2] == 2
    rng = np.random.default_rng(4)
    for t in rng.uniform(0.0, st.t_max, 200):
        g, o = ld(t)
        want = g * np.array([np.abs(o[l]).max() / np.abs(st.rate_ops[l]).max() for l in range(2)]) ** 2
        assert np.abs(st.rates(t) - want).max() < 1e-13 * max(1.0, want.max())
        for l in range(2):                       # the fixed direction reproduces the operator up to its scalar
            b = st.rate_ops[l]
            f = np.vdot(b, o[l]) / np.vdot(b, b)
            assert np.abs(o[l] - f * b).max() < 1e-13


def test_hamiltonian_and_dissipation_together():
    p = Problem(2, 3, 1, 1, 2, complex_controls=True, seed=5)
    h = p.hamiltonian_td_numpy()
    ld = lambda t: (np.array([0.02 * (1 + 0.3 * np.cos(t))]), np.stack([SM]))
    st = extract_lindblad_time_structure(h, 1, True, p.T, p.N, p.T + 1.0, lindblad_data=ld)
    assert st.series.shape[2] == st.KC * 3 + 1
    assert _max_h_error(st, h, 1, True) < 1e-13
    for t in np.linspace(0.0, st.t_max, 57):
        assert abs(st.rates(t)[0] - 0.02 * (1 + 0.3 * np.cos(t))) < 1e-15


def test_time_independent_dissipation_is_recognised():
    assert not _lindblad_is_time_dependent(lambda t: (np.array([0.1]), np.stack([SM])), 2.0)


# --- refused ------------------------------------------------------------------------------------------------------
def test_square_pulse_raises():
    T, N = 4.0, 5
    h = lambda u, t: 0.5 * SZ + u[0] * SX + (1.0 if 0.3 * T < t < 0.6 * T else 0.0) * SY
    with pytest.raises(NotImplementedError):
        extract_lindblad_time_structure(h, 1, False, T, N, T + 1.0)


def test_dissipator_changing_direction_raises():
    ld = lambda t: (np.array([0.1]), np.stack([np.cos(t) * SM + np.sin(t) * SM.T]))
    with pytest.raises(NotImplementedError):
        extract_lindblad_time_structure(None, 0, False, 2.0, 3, 3.0, lindblad_data=ld)


def test_changing_operator_count_raises():
    ld = lambda t: ((np.array([0.1]), np.stack([SM])) if t < 1.0 else (np.array([0.1, 0.2]), np.stack([SM, SZ])))
    with pytest.raises(NotImplementedError):
        extract_lindblad_time_structure(None, 0, False, 2.0, 3, 3.0, lindblad_data=ld)


def test_non_affine_raises():
    h = lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX + u[0] ** 2 * SY
    with pytest.raises(NonlinearHamiltonian):
        extract_lindblad_time_structure(h, 1, False, 2.0, 3, 3.0)


def test_more_than_16_channels_raises():
    rng = np.random.default_rng(9)
    mats = [rand_herm(rng, 5) for _ in range(17)]
    h = lambda u, t: sum(np.cos((k + 1) * 0.37 * t + k) * m for k, m in enumerate(mats))
    with pytest.raises(NotImplementedError):
        extract_lindblad_time_structure(h, 0, False, 2.0, 3, 3.0)
