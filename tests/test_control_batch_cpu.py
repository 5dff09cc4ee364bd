"""CPU: control batches (`SchroedingerPlan(control_batch=B)`) and `grape_schroedinger_discrete_batch` refuse what they do not
serve before any device call, valid arguments reach the device, malformed initial controls raise ValueError, and the three
new C-ABI calls are bound with their header signatures."""
import ctypes

import numpy as np
import pytest

import qoc_b200 as qoc
import qoc_b200.standard as std
from qoc_b200 import _lib
from qoc_b200.core.plan import SchroedingerPlan, make_schroedinger_plan
from qoc_b200.core.schroedingerdiscrete import _adam_rows
from qoc_b200.models import MagnusPolicy
from qoc_b200.models.cost import Cost

N_, M_, T_ = 5, 4, 1.0
SX = np.array([[0, 1], [1, 0]], dtype=complex)
SY = np.array([[0, -1j], [1j, 0]])
SZ = np.diag([1.0, -1.0]).astype(complex)
NOMINAL = lambda u, t: 0.5 * SZ + u[0] * SX + u[1] * SY


def _cuda():
    import torch
    return torch.cuda.is_available()


def _init(n=2):
    init = np.zeros((1, n, 1), dtype=complex)
    init[0, 0, 0] = 1.0
    return init


def _plan(B=3, hamiltonian=NOMINAL, costs=None, n=2, **kw):
    init = _init(n)
    costs = [std.TargetStateInfidelity(init)] if costs is None else costs
    return SchroedingerPlan(hamiltonian, init, costs, T_, N_, control_eval_count=M_, control_count=2, control_batch=B, **kw)


def _grape(initial_controls, **kw):
    init = _init()
    kw.setdefault("iteration_count", 2)
    return qoc.grape_schroedinger_discrete_batch(2, M_, [std.TargetStateInfidelity(init)], T_, NOMINAL, init, N_,
                                                 initial_controls, **kw)


class PurityPenalty(Cost):
    requires_step_evaluation = False

    def cost(self, controls, states, step):
        return float(np.abs(states[0, 0, 0]) ** 2)


# --- refusals before any device call ----------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(ensemble_drifts=np.array([0.5 * SZ] * 3)),
                                dict(ensemble_hamiltonians=[NOMINAL] * 3),
                                dict(slice_range=(0, 2)), dict(state_slice=(0, 1))],
                         ids=["ensemble-drifts", "ensemble-hamiltonians", "slice-range", "state-slice"])
def test_batch_combinations_not_implemented(kw):
    with pytest.raises(NotImplementedError, match="control batches"):
        _plan(**kw)


def test_user_costs_not_implemented():
    with pytest.raises(NotImplementedError, match="user-defined costs"):
        _plan(costs=[PurityPenalty()])


def test_time_dependent_hamiltonian_not_implemented():
    with pytest.raises(NotImplementedError, match="time-dependent"):
        _plan(hamiltonian=lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX + u[1] * SY)


@pytest.mark.parametrize("make", [_plan, lambda **kw: make_schroedinger_plan(
    kw["hamiltonian"], _init(), [std.TargetStateInfidelity(_init())], T_, N_, control_eval_count=M_, control_count=2,
    control_batch=3)], ids=["plan", "make_schroedinger_plan"])
def test_nonlinear_hamiltonian_not_implemented(make):
    """a plain NotImplementedError, so that make_schroedinger_plan does not route a batch to NonlinearSchroedingerPlan."""
    from qoc_b200.core.plan import NonlinearHamiltonian
    with pytest.raises(NotImplementedError, match="affine") as info:
        make(hamiltonian=lambda u, t: 0.5 * SZ + u[0] * SX + u[1] ** 2 * SY)
    assert not isinstance(info.value, NonlinearHamiltonian)


def test_large_dimension_not_implemented():
    n = 72
    h0 = np.diag(np.linspace(-1, 1, n)).astype(complex)
    x = np.eye(n, k=1, dtype=complex) + np.eye(n, k=-1, dtype=complex)
    with pytest.raises(NotImplementedError, match="hilbert_size > 64"):
        _plan(hamiltonian=lambda u, t: h0 + u[0] * x + u[1] * 1j * (np.eye(n, k=1) - np.eye(n, k=-1)), n=n)


@pytest.mark.parametrize("B", [0, -2, 2.5, True, "4"])
def test_bad_batch_size_raises_value_error(B):
    with pytest.raises(ValueError, match="control_batch"):
        _plan(B=B)


@pytest.mark.skipif(_cuda(), reason="checks that valid batches reach the device")
@pytest.mark.parametrize("kw", [dict(), dict(B=1), dict(magnus_policy=MagnusPolicy.M4, store_tape=False),
                                dict(costs=[std.TargetStateInfidelity(_init()), std.ControlNorm(2, M_)])])
def test_valid_batches_reach_the_device(kw):
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _plan(**kw)


# --- the driver -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("controls", [np.zeros((M_, 2)), np.zeros((3, M_, 3)), np.zeros((3, M_ + 1, 2)),
                                      np.zeros((0, M_, 2)), np.zeros((2, M_, 2), dtype=complex),
                                      np.full((2, M_, 2), "x"), np.full((2, M_, 2), 3.0)],
                         ids=["2d", "controls", "steps", "empty", "complex", "strings", "over-max-norm"])
def test_bad_initial_controls_raise_value_error(controls):
    with pytest.raises(ValueError):
        _grape(controls)


def test_real_initial_controls_for_complex_program_raise_value_error():
    with pytest.raises(ValueError):
        _grape(np.zeros((2, M_, 2)), complex_controls=True)


@pytest.mark.parametrize("kw, match", [(dict(optimizer=std.LBFGSB()), "L-BFGS-B"),
                                       (dict(save_file_path="run.h5"), "save"),
                                       (dict(optimizer=object()), "Adam or SGD")])
def test_driver_refusals(kw, match):
    with pytest.raises(NotImplementedError, match=match):
        _grape(np.zeros((2, M_, 2)), **kw)


@pytest.mark.skipif(_cuda(), reason="checks that a valid run reaches the device")
def test_valid_driver_run_reaches_the_device():
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _grape(np.full((3, M_, 2), 0.1))


def test_driver_is_exported():
    assert "grape_schroedinger_discrete_batch" in qoc.__all__


@pytest.mark.parametrize("kw", [dict(), dict(scale_grads=0.7, clip_grads=0.05), dict(learning_rate_decay=3.0)])
def test_adam_rows_are_independent_adam_updates(kw):
    """each row of the vectorised update is exactly `Adam.update` on that row alone (own moments, step count and norm)."""
    rng = np.random.default_rng(0)
    B, P = 3, 8
    params, moment, square, steps = rng.standard_normal((B, P)), np.zeros((B, P)), np.zeros((B, P)), np.zeros((B, 1))
    singles = [std.Adam(learning_rate=0.1, **kw) for _ in range(B)]
    for s in singles:
        s.gradient_moment, s.gradient_square_moment = np.zeros(P), np.zeros(P)
    rows = [params[b].copy() for b in range(B)]
    for it in range(4):
        grads = rng.standard_normal((B, P)) * (1 + np.arange(B))[:, None]
        idx = np.arange(B) if it < 2 else np.array([0, 2])          # row 1 stops after two updates
        params[idx], moment[idx], square[idx], steps[idx] = _adam_rows(singles[0], params[idx], grads[idx], moment[idx],
                                                                       square[idx], steps[idx])
        for b in idx:
            rows[b] = singles[b].update(grads[b], rows[b])
    for b in range(B):
        assert np.array_equal(params[b], rows[b]), b


# --- the C ABI --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name, nargs", [("qocb_set_control_batch", 1), ("qocb_batch_cost", 4),
                                         ("qocb_batch_cost_and_grad", 5)])
def test_batch_calls_are_bound(name, nargs):
    lib = _lib.load()
    assert name in _lib.EXPORTS
    fn = getattr(lib, name)
    assert fn.argtypes == [ctypes.c_void_p] * nargs
    assert fn(*([None] * nargs)) == -1                      # a null plan is refused without touching a device
