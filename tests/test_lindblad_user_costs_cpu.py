"""CPU: the host half of user-defined costs - the 4-point central differences that turn a user `cost(...)` into cotangents of
states, densities and controls (`central_differences`, `explicit_control_grad`), checked against analytic cotangents, and the
rule that decides which costs are user-defined (`is_user_cost`)."""
import numpy as np
import pytest

from qoc_b200.core.plan import central_differences, explicit_control_grad, is_user_cost


def rel(a, b):
    return np.linalg.norm((np.asarray(a) - np.asarray(b)).ravel()) / max(np.linalg.norm(np.asarray(b).ravel()), 1e-300)


def _cot(f, z):
    dre, dim = central_differences(f, z)
    return dre - 1j * dim


def _rand_c(rng, shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def test_overlap_modulus_cotangent():
    """|tr(M^dag rho)|: cotangent conj(z) conj(M) / |z| with z = tr(M^dag rho)."""
    rng = np.random.default_rng(0)
    M, rho = _rand_c(rng, (4, 4)), _rand_c(rng, (4, 4))
    z = np.trace(M.conj().T @ rho)
    assert rel(_cot(lambda r: abs(np.trace(M.conj().T @ r)), rho), np.conj(z) * M.conj() / abs(z)) < 1e-9


def test_purity_cotangent_on_a_density_set():
    """sum_d Re tr(rho_d^2) on a D x n x n set: cotangent 2 rho_d^T (every entry on its own, not the Hermitian restriction)."""
    rng = np.random.default_rng(1)
    rho = _rand_c(rng, (2, 3, 3))
    f = lambda r: float(np.real(np.trace(r @ r, axis1=-2, axis2=-1).sum()))
    assert rel(_cot(f, rho), 2 * np.swapaxes(rho, -1, -2)) < 1e-9


def test_quartic_population_cotangent_on_states():
    """sum_s |psi_s,last|^4 on S x n x 1 states: cotangent 4 |psi|^2 conj(psi) at the last level."""
    rng = np.random.default_rng(2)
    psi = _rand_c(rng, (3, 5, 1))
    want = np.zeros_like(psi)
    want[:, -1, 0] = 4 * np.abs(psi[:, -1, 0]) ** 2 * np.conj(psi[:, -1, 0])
    assert rel(_cot(lambda q: float(np.sum(np.abs(q[:, -1, 0]) ** 4)), psi), want) < 1e-9


@pytest.mark.parametrize("complex_controls", [False, True])
def test_explicit_control_grad(complex_controls):
    """0.01 sum |u|^2 -> 0.02 u (d/dRe u + i d/dIm u); a function that ignores the controls -> None."""
    rng = np.random.default_rng(3)
    u = _rand_c(rng, (5, 2)) if complex_controls else rng.standard_normal((5, 2))
    g = explicit_control_grad(lambda c: 0.01 * float(np.sum(np.abs(c) ** 2)), u)
    assert g.dtype == u.dtype and rel(g, 0.02 * u) < 1e-9
    assert explicit_control_grad(lambda c: 1.5, u) is None


def test_real_arrays_have_no_imaginary_part():
    dre, dim = central_differences(lambda x: float(np.sum(x ** 3)), np.array([0.5, -2.0]))
    assert dim is None and rel(dre, 3 * np.array([0.5, -2.0]) ** 2) < 1e-9


def test_user_cost_classification():
    import qoc_b200.standard.costs as sc
    from qoc_b200.models.cost import Cost
    builtins = [sc.TargetStateInfidelity, sc.TargetStateInfidelityTime, sc.ForbidStates, sc.TargetDensityInfidelity,
                sc.TargetDensityInfidelityTime, sc.ForbidDensities, sc.ControlNorm, sc.ControlVariation, sc.ControlArea,
                sc.ControlBandwidthMax]
    for cls in builtins:
        assert not is_user_cost(object.__new__(cls)), cls

    class Purity(Cost):
        requires_step_evaluation = True

        def cost(self, controls, densities, step):
            return 0.0

    class Leakage(Cost):
        def cost(self, controls, densities, step):
            return 0.0

    class ScaledTarget(sc.TargetDensityInfidelity):            # keeps the built-in's device hook
        def cost(self, controls, densities, step):
            return 2 * super().cost(controls, densities, step)
    assert is_user_cost(Purity()) and is_user_cost(Leakage())
    assert not is_user_cost(object.__new__(ScaledTarget))
