"""CPU: `LindbladPlan(ensemble_drifts=..., ensemble_rates=...)` validates its members before any device call, and the ctypes
mirror of `qocb_lindblad_problem` carries the new `ensemble_count` field in the header's order."""
import os
import re

import numpy as np
import pytest

import qoc_b200.standard as std
from qoc_b200 import _lib
from qoc_b200.core.plan import LindbladPlan
from qoc_b200.models.cost import Cost

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_, M_, T_ = 5, 5, 1.0


def _cuda():
    import torch
    return torch.cuda.is_available()


def _problem(n=2, td_h=False, td_l=False, with_h=True):
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    h0 = np.diag(np.arange(n)).astype(complex)
    if td_h:
        ham = lambda u, t: h0 + np.cos(3.0 * t) * (u[0] * a + np.conj(u[0]) * a.conj().T)
    else:
        ham = lambda u, t: h0 + u[0] * a + np.conj(u[0]) * a.conj().T
    gam = np.array([0.05])
    lind = (lambda t: (gam * (1.0 + 0.5 * np.sin(t)), a[None])) if td_l else (lambda t: (gam, a[None]))
    rho0 = np.zeros((1, n, n), dtype=complex)
    rho0[0, 0, 0] = 1.0
    targ = np.zeros((1, n, n), dtype=complex)
    targ[0, -1, -1] = 1.0
    kw = dict(hamiltonian=ham if with_h else None, lindblad_data=lind, control_eval_count=M_ if with_h else 0,
              control_count=1 if with_h else 0, complex_controls=with_h)
    return rho0, [std.TargetDensityInfidelity(targ)], kw


def _drifts(E, n=2):
    return np.array([np.diag(np.arange(n)) * (1.0 + 0.1 * e) for e in range(E)], dtype=complex)


def _plan(drifts=None, rates=None, costs=None, **pk):
    rho0, c, kw = _problem(**pk)
    return LindbladPlan(rho0, c if costs is None else costs, T_, N_, ensemble_drifts=drifts, ensemble_rates=rates, **kw)


class PurityPenalty(Cost):
    requires_step_evaluation = False

    def cost(self, controls, densities, step):
        return float(np.real(np.trace(densities[0] @ densities[0])))


@pytest.mark.parametrize("drifts, rates", [
    (np.zeros((3, 3, 3)), None),                   # wrong n
    (np.zeros((3, 2)), None),                      # not [E][n][n]
    (np.zeros((0, 2, 2)), None),                   # no members
    (None, np.zeros((3, 2))),                      # wrong L
    (None, np.zeros(3)),                           # not [E][L]
    (None, np.ones((2, 1)) * (1 + 1j)),            # complex rates
    ("E3", np.ones((2, 1))),                       # members disagree
])
def test_bad_shapes_raise_value_error(drifts, rates):
    if isinstance(drifts, str):
        drifts = _drifts(3)
    with pytest.raises(ValueError):
        _plan(drifts, rates)


def test_drifts_without_hamiltonian_raise_value_error():
    with pytest.raises(ValueError, match="None"):
        _plan(_drifts(2), None, with_h=False)


def test_rates_without_operators_raise_value_error():
    rho0, c, kw = _problem()
    kw["lindblad_data"] = None
    with pytest.raises(ValueError, match="no operators"):
        LindbladPlan(rho0, c, T_, N_, ensemble_rates=np.ones((2, 1)), **kw)


def test_drifts_with_time_dependent_hamiltonian_not_implemented():
    with pytest.raises(NotImplementedError, match="time-dependent hamiltonian"):
        _plan(_drifts(2), None, td_h=True)


def test_rates_with_time_dependent_lindblad_data_not_implemented():
    with pytest.raises(NotImplementedError, match="time-dependent lindblad_data"):
        _plan(None, np.full((2, 1), 0.04), td_l=True)


@pytest.mark.parametrize("which", ["drifts", "rates"])
def test_user_costs_on_ensembles_not_implemented(which):
    rho0, c, kw = _problem()
    members = dict(ensemble_drifts=_drifts(2)) if which == "drifts" else dict(ensemble_rates=np.full((2, 1), 0.04))
    with pytest.raises(NotImplementedError, match="user-defined"):
        LindbladPlan(rho0, c + [PurityPenalty()], T_, N_, **members, **kw)


@pytest.mark.skipif(_cuda(), reason="checks that valid members reach the device")
@pytest.mark.parametrize("pk, drifts, rates", [
    (dict(), _drifts(3), None),
    (dict(), None, np.full((4, 1), 0.02)),
    (dict(), _drifts(2), np.full((2, 1), 0.02)),
    (dict(td_h=True), None, np.full((2, 1), 0.02)),         # one component varies, the other is time-dependent
    (dict(td_l=True), _drifts(2), None),
    (dict(with_h=False), None, np.full((2, 1), 0.02)),
])
def test_valid_members_pass_validation(pk, drifts, rates):
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _plan(drifts, rates, **pk)


def test_lindblad_problem_struct_matches_header():
    header = open(os.path.join(ROOT, "include", "qocb200.h")).read()
    body = header[:header.index("} qocb_lindblad_problem;")]
    body = body[body.rindex("typedef struct {"):]
    fields = re.findall(r"(?:int32_t|double)\s+([a-z_0-9]+);", body)
    assert fields == [f[0] for f in _lib.LindbladProblem._fields_]
    assert fields.index("ensemble_count") == fields.index("time_dependent_rates") + 1
