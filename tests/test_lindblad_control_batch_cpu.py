"""CPU: Lindblad control batches (`LindbladPlan(control_batch=B)`) and `grape_lindblad_discrete_batch` refuse what they do not
serve before any device call, valid arguments reach the device, malformed initial controls raise ValueError, the lockstep
helper shared with the Schroedinger driver updates every start as `Adam.update` would, and the three new C-ABI calls are
bound with their header signatures."""
import ctypes

import numpy as np
import pytest

import qoc_b200 as qoc
import qoc_b200.standard as std
from qoc_b200 import _lib
from qoc_b200.core.common import grape_lockstep
from qoc_b200.core.plan import LindbladPlan
from qoc_b200.models import GrapeLindbladResult
from qoc_b200.models.cost import Cost

N_, M_, T_ = 4, 5, 1.0
SX = np.array([[0, 1], [1, 0]], dtype=complex)
SY = np.array([[0, -1j], [1j, 0]])
SZ = np.diag([1.0, -1.0]).astype(complex)
SM = np.array([[0, 1], [0, 0]], dtype=complex)
NOMINAL = lambda u, t: 0.5 * SZ + u[0] * SX + u[1] * SY
DECAY = lambda t: (np.array([0.05]), SM[None])
RHO0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
TARG = np.array([[[0, 0], [0, 1]]], dtype=complex)


def _cuda():
    import torch
    return torch.cuda.is_available()


def _plan(B=3, hamiltonian=NOMINAL, costs=None, **kw):
    costs = [std.TargetDensityInfidelity(TARG)] if costs is None else costs
    kw.setdefault("control_count", 2)
    return LindbladPlan(RHO0, costs, T_, N_, hamiltonian=hamiltonian, lindblad_data=DECAY, control_eval_count=M_,
                        control_batch=B, **kw)


def _grape(initial_controls, **kw):
    kw.setdefault("iteration_count", 2)
    return qoc.grape_lindblad_discrete_batch(2, M_, [std.TargetDensityInfidelity(TARG)], T_, RHO0, N_, initial_controls,
                                             hamiltonian=NOMINAL, lindblad_data=DECAY, **kw)


class PurityPenalty(Cost):
    requires_step_evaluation = False

    def cost(self, controls, densities, step):
        return float(np.real(np.trace(densities[0] @ densities[0])))


# --- refusals before any device call ----------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(ensemble_drifts=np.array([0.5 * SZ] * 3)),
                                dict(ensemble_rates=np.array([[0.05]] * 3)),
                                dict(ensemble_hamiltonians=[NOMINAL] * 3)],
                         ids=["ensemble-drifts", "ensemble-rates", "ensemble-hamiltonians"])
def test_batch_with_ensembles_not_implemented(kw):
    with pytest.raises(NotImplementedError, match="control batches"):
        _plan(**kw)


@pytest.mark.parametrize("B", [1, 3])
def test_user_costs_not_implemented(B):
    with pytest.raises(NotImplementedError, match="user-defined costs"):
        _plan(B=B, costs=[std.TargetDensityInfidelity(TARG), PurityPenalty()])


@pytest.mark.parametrize("kw", [dict(hamiltonian=None, control_count=0), dict(hamiltonian=None), dict(control_count=0)],
                         ids=["no-hamiltonian", "no-hamiltonian-with-count", "no-controls"])
def test_nothing_to_batch_raises_value_error(kw):
    with pytest.raises(ValueError, match="no controls to batch"):
        _plan(**kw)


@pytest.mark.parametrize("B", [0, -2, 2.5, True, "4"])
def test_bad_batch_size_raises_value_error(B):
    with pytest.raises(ValueError, match="control_batch"):
        _plan(B=B)


@pytest.mark.skipif(_cuda(), reason="checks that valid batches reach the device")
@pytest.mark.parametrize("kw", [dict(), dict(B=1), dict(B=np.int64(4), complex_controls=True),
                                dict(costs=[std.TargetDensityInfidelity(TARG), std.ControlNorm(2, M_)]),
                                dict(hamiltonian=lambda u, t: 0.5 * np.cos(t) * SZ + u[0] * SX + u[1] * SY)],
                         ids=["plain", "one-start", "complex", "control-norm", "time-dependent"])
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
                                       (dict(save_file_path="run.h5"), "grape_lindblad_discrete to save"),
                                       (dict(optimizer=object()), "Adam or SGD")])
def test_driver_refusals(kw, match):
    with pytest.raises(NotImplementedError, match=match):
        _grape(np.zeros((2, M_, 2)), **kw)


@pytest.mark.skipif(_cuda(), reason="checks that a valid run reaches the device")
def test_valid_driver_run_reaches_the_device():
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _grape(np.full((3, M_, 2), 0.1))


def test_driver_is_exported():
    import qoc_b200.core as core
    assert "grape_lindblad_discrete_batch" in qoc.__all__ and "grape_lindblad_discrete_batch" in core.__all__


# --- the lockstep helper against per-start Adam.update ----------------------------------------------------------------
def _quadratic(targets, calls):
    """a batched evaluate on the host: error_b = |u_b - t_b|^2, with complex grads dE/dRe u + i dE/dIm u."""
    def evaluate(controls):
        calls.append(controls.copy())
        d = controls - targets
        return np.sum(np.abs(d) ** 2, axis=(1, 2)), 2 * d, np.abs(d)
    return evaluate


@pytest.mark.parametrize("cc", [False, True], ids=["real", "complex"])
@pytest.mark.parametrize("adam_kw", [dict(), dict(scale_grads=0.7, clip_grads=0.05), dict(learning_rate_decay=3.0)],
                         ids=["plain", "scale-clip", "decay"])
def test_lockstep_follows_per_start_adam(cc, adam_kw):
    """each start of the shared lockstep helper takes the steps of its own `Adam.update`, with clipping to the max norms
    and `impose_control_conditions` applied before each evaluation; a start at `min_error` stops updating.  (The row norm of
    `scale_grads` may differ from the 1-D norm of `Adam.update` in the last bit, hence 1e-13 and not equality.)"""
    close = lambda a, b: np.allclose(a, b, rtol=1e-13, atol=1e-15)
    rng = np.random.default_rng(3)
    B, M, K, its = 3, 4, 2, 5
    dtype = complex if cc else float
    u0 = 0.3 * rng.standard_normal((B, M, K)).astype(dtype)
    targets = 0.6 * rng.standard_normal((B, M, K)).astype(dtype)
    if cc:
        u0 = u0 + 0.3j * rng.standard_normal((B, M, K))
        targets = targets + 0.6j * rng.standard_normal((B, M, K))
    norms = np.full(K, 0.5)
    impose = lambda c: c * 0.99
    from qoc_b200.core.common import clip_control_norms, slap_controls, strip_controls
    first = u0[1].copy()
    clip_control_norms(first, norms)
    targets[1] = impose(first)                            # start 1 sits at its minimum: it stops after one iteration
    calls = []
    got = grape_lockstep(_quadratic(targets, calls), u0.copy(), cc, norms, impose, its, 0, 1e-30,
                         std.Adam(learning_rate=0.1, **adam_kw), GrapeLindbladResult, "best_final_densities")
    for b in range(B):
        opt = std.Adam(learning_rate=0.1, **adam_kw)
        P = 2 * M * K if cc else M * K
        opt.gradient_moment, opt.gradient_square_moment = np.zeros(P), np.zeros(P)
        params = strip_controls(cc, u0[b]).astype(np.float64)
        best = (np.inf, None, None)
        for it in range(its):
            c = slap_controls(cc, params, (M, K))
            clip_control_norms(c, norms)
            c = impose(c)
            assert close(calls[it][b], c), (b, it)
            err = float(np.sum(np.abs(c - targets[b]) ** 2))
            if err < best[0]:
                best = (err, c.copy(), it)
            if err <= 1e-30:
                break
            params = opt.update(strip_controls(cc, 2 * (c - targets[b])), params)
        assert close(got[b].best_error, best[0]) and close(got[b].best_controls, best[1]), b
        assert got[b].best_iteration == best[2], b
        assert close(got[b].best_final_densities, np.abs(best[1] - targets[b])), b
    assert got[1].best_iteration == 0 and got[1].best_error == 0.0


def test_lockstep_sgd():
    rng = np.random.default_rng(4)
    u0, targets = rng.standard_normal((2, 3, 1)), rng.standard_normal((2, 3, 1))
    calls = []
    grape_lockstep(_quadratic(targets, calls), u0.copy(), False, np.full(1, 10.0), None, 3, 0, 0,
                   std.SGD(learning_rate=0.25), GrapeLindbladResult, "best_final_densities")
    u = u0.copy()
    for it in range(3):
        assert np.array_equal(calls[it], u)
        u = u - 0.25 * 2 * (u - targets)


def test_lockstep_stops_when_every_start_stopped(capsys):
    u0 = np.zeros((2, 3, 1))
    calls = []
    got = grape_lockstep(_quadratic(np.zeros((2, 3, 1)), calls), u0, False, np.ones(1), None, 10, 1, 0.0,
                         std.Adam(), GrapeLindbladResult, "best_final_densities")
    assert len(calls) == 1 and all(r.best_error == 0.0 for r in got)
    assert "stopped 2/2" in capsys.readouterr().out


# --- the C ABI --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name, nargs", [("qocb_lindblad_set_control_batch", 1), ("qocb_lindblad_batch_cost", 4),
                                         ("qocb_lindblad_batch_cost_and_grad", 5)])
def test_batch_calls_are_bound(name, nargs):
    lib = _lib.load()
    assert name in _lib.EXPORTS
    fn = getattr(lib, name)
    assert fn.argtypes == [ctypes.c_void_p] * nargs
    assert fn(*([None] * nargs)) == -1                      # a null plan is refused without touching a device
