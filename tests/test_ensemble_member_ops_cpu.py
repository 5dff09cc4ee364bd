"""CPU: `ensemble_hamiltonians` (members that differ in drift and control operators) on `SchroedingerPlan`, `LindbladPlan` and
`EnsembleShardedPlan` validates every member before any device call, takes the drift-only route exactly when every member's
operators equal member 0's, and the two new C-ABI calls are bound with their header signatures."""
import ctypes

import numpy as np
import pytest

import qoc_b200.standard as std
from qoc_b200 import _lib
from qoc_b200.core.plan import LindbladPlan, NonlinearHamiltonian, SchroedingerPlan, ensemble_member_structures
from qoc_b200.core.sharded import EnsembleShardedPlan
from qoc_b200.models import MagnusPolicy
from qoc_b200.models.cost import Cost

N_, M_, T_ = 5, 5, 1.0
SX = np.array([[0, 1], [1, 0]], dtype=complex)
SY = np.array([[0, -1j], [1j, 0]])
SZ = np.diag([1.0, -1.0]).astype(complex)


def _cuda():
    import torch
    return torch.cuda.is_available()


def _member(eps=0.0, det=0.0, xt=0.0):
    """H = (1 + det) SZ / 2 + (1 + eps) u0 SX + u1 (SY + xt SX): amplitude error eps, detuning det, crosstalk xt."""
    return lambda u, t: 0.5 * (1.0 + det) * SZ + (1.0 + eps) * u[0] * SX + u[1] * (SY + xt * SX)


NOMINAL = _member()
AMPLITUDE = [_member(eps=e) for e in (-0.1, 0.0, 0.1)]
DRIFT_ONLY = [_member(det=d) for d in (-0.2, 0.0, 0.2)]


def _states():
    return np.array([[[1.0], [0.0]]], dtype=complex)


def _schroedinger(members=AMPLITUDE, costs=None, hamiltonian=NOMINAL, n=2, **kw):
    init = np.zeros((1, n, 1), dtype=complex)
    init[0, 0, 0] = 1.0
    costs = [std.TargetStateInfidelity(init)] if costs is None else costs
    return SchroedingerPlan(hamiltonian, init, costs, T_, N_, control_eval_count=M_, control_count=2,
                            ensemble_hamiltonians=members, **kw)


def _lindblad(members=AMPLITUDE, costs=None, hamiltonian=NOMINAL, lindblad_data=None, **kw):
    rho0 = np.zeros((1, 2, 2), dtype=complex)
    rho0[0, 0, 0] = 1.0
    targ = np.zeros((1, 2, 2), dtype=complex)
    targ[0, 1, 1] = 1.0
    a = np.array([[0, 1], [0, 0]], dtype=complex)
    lind = (lambda t: (np.array([0.05]), a[None])) if lindblad_data is None else lindblad_data
    costs = [std.TargetDensityInfidelity(targ)] if costs is None else costs
    return LindbladPlan(rho0, costs, T_, N_, hamiltonian=hamiltonian, lindblad_data=lind, control_eval_count=M_,
                        control_count=2, ensemble_hamiltonians=members, **kw)


class PurityPenalty(Cost):
    requires_step_evaluation = False

    def cost(self, controls, states, step):
        return float(np.abs(states[0, 0, 0]) ** 2)


# --- the fast-path decision -------------------------------------------------------------------------------------------
def test_drift_only_members_share_operators():
    h0s, a_ops = ensemble_member_structures(DRIFT_ONLY, 2, 2, False, T_)
    assert h0s.shape == (3, 2, 2) and a_ops.shape == (2, 2, 2)
    assert np.array_equal(a_ops, ensemble_member_structures([NOMINAL], 2, 2, False, T_)[1])
    assert np.array_equal(h0s[2], 0.6 * SZ)


@pytest.mark.parametrize("members", [AMPLITUDE, [_member(), _member(xt=0.05)], [_member(), _member(eps=1e-15)]],
                         ids=["amplitude", "crosstalk", "last-bit"])
def test_differing_operators_are_per_member(members):
    h0s, a_ops = ensemble_member_structures(members, 2, 2, False, T_)
    assert a_ops.shape == (len(members), 2, 2, 2) and a_ops.flags["C_CONTIGUOUS"]
    assert h0s.shape == (len(members), 2, 2)


def test_member_operators_of_complex_controls():
    members = [lambda u, t, s=s: 0.5 * SZ + s * (u[0] * SX + np.conj(u[0]) * SX.conj().T) for s in (0.9, 1.1)]
    _, a_ops = ensemble_member_structures(members, 2, 1, True, T_)
    assert a_ops.shape == (2, 2, 2, 2)                   # [E][Re u, Im u][n][n]
    assert np.allclose(a_ops[1], a_ops[0] * 1.1 / 0.9, rtol=0, atol=1e-15)


# --- refusals before any device call ----------------------------------------------------------------------------------
@pytest.mark.parametrize("members", [
    [],                                                    # no members
    [NOMINAL, "not callable"],
    [NOMINAL, lambda u, t: np.eye(3) + u[0] * np.eye(3)],   # another n
    [NOMINAL, lambda u, t: SZ + u[0] * SX + u[2] * SY],     # more controls than the plan's
], ids=["empty", "not-callable", "other-n", "other-control-count"])
@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_bad_members_raise_value_error(make, members):
    with pytest.raises(ValueError):
        make(members)


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_drifts_and_hamiltonians_together_raise_value_error(make):
    with pytest.raises(ValueError, match="not both"):
        make(AMPLITUDE, ensemble_drifts=np.array([0.5 * SZ] * 3))


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_time_dependent_member_not_implemented(make):
    members = [NOMINAL, lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX + u[1] * SY]
    with pytest.raises(NotImplementedError, match="read `time`"):
        make(members)


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_time_dependent_nominal_hamiltonian_not_implemented(make):
    with pytest.raises(NotImplementedError, match="time-dependent hamiltonian"):
        make(AMPLITUDE, hamiltonian=lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX + u[1] * SY)


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_nonlinear_member_raises(make):
    members = [NOMINAL, lambda u, t: 0.5 * SZ + u[0] * SX + u[1] ** 2 * SY]
    with pytest.raises(NonlinearHamiltonian):
        make(members)


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_user_costs_on_member_ensembles_not_implemented(make):
    with pytest.raises(NotImplementedError, match="user-defined"):
        make(AMPLITUDE, costs=[PurityPenalty()])


def test_lindblad_members_without_hamiltonian_raise_value_error():
    with pytest.raises(ValueError, match="None"):
        _lindblad(AMPLITUDE, hamiltonian=None)


def test_lindblad_member_counts_must_agree():
    with pytest.raises(ValueError, match="members"):
        _lindblad(AMPLITUDE, ensemble_rates=np.full((2, 1), 0.04))


def test_state_sharding_of_member_ensembles_not_implemented():
    with pytest.raises(NotImplementedError, match="state sharding"):
        _schroedinger(AMPLITUDE, state_slice=(0, 1))


def test_large_dimension_keeps_its_refusal():
    """n > 64 is refused by the plan creation itself, with or without a device."""
    n = 72
    h0 = np.diag(np.linspace(-1, 1, n)).astype(complex)
    x = np.eye(n, k=1, dtype=complex) + np.eye(n, k=-1, dtype=complex)
    members = [lambda u, t, s=s: h0 + s * u[0] * x + u[1] * 1j * (np.eye(n, k=1) - np.eye(n, k=-1)) for s in (0.9, 1.1)]
    with pytest.raises(RuntimeError, match="ensembles are not implemented for hilbert_size > 64"):
        _schroedinger(members, hamiltonian=members[0], n=n)


@pytest.mark.parametrize("kw", [dict(), dict(ensemble_drifts=np.array([0.5 * SZ] * 3), ensemble_hamiltonians=AMPLITUDE)],
                         ids=["neither", "both"])
def test_sharded_plan_needs_one_kind_of_members(kw):
    with pytest.raises(ValueError, match="exactly one"):
        EnsembleShardedPlan(NOMINAL, _states(), [], T_, N_, **kw)


@pytest.mark.skipif(_cuda(), reason="checks that valid members reach the device")
@pytest.mark.parametrize("make, members, kw", [
    (_schroedinger, AMPLITUDE, dict()),
    (_schroedinger, DRIFT_ONLY, dict()),
    (_schroedinger, AMPLITUDE, dict(magnus_policy=MagnusPolicy.M4)),
    (_lindblad, AMPLITUDE, dict()),
    (_lindblad, AMPLITUDE, dict(ensemble_rates=np.full((3, 1), 0.02))),
    (_lindblad, AMPLITUDE, dict(lindblad_data=lambda t: (np.array([0.05 * (1 + 0.5 * np.sin(t))]),
                                                         np.array([[[0, 1], [0, 0]]], dtype=complex)))),
])
def test_valid_members_pass_validation(make, members, kw):
    with pytest.raises(RuntimeError, match="no CUDA device"):
        make(members, **kw)


# --- the C ABI --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["qocb_set_member_operators", "qocb_lindblad_set_member_operators"])
def test_member_operator_calls_are_bound(name):
    lib = _lib.load()
    assert name in _lib.EXPORTS
    fn = getattr(lib, name)
    assert fn.argtypes == [ctypes.c_void_p, ctypes.c_void_p]
    assert fn(None, None) == -1                            # a null plan is refused without touching a device
