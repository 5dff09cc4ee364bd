"""GPU: user-defined `Cost` subclasses on the Lindblad path (qoc/models/cost.py:5-51) - costs that only provide
`cost(controls, densities, step)`, evaluated where the reference evaluates them (qoc/core/lindbladdiscrete.py:384-441): at
every cost step when `requires_step_evaluation`, else once on the final densities.  The device runs the forward pass with its
tape (qocb_lindblad_forward), the host evaluates the user costs on the stored densities and differentiates them by central
differences, and the reverse pass is seeded with those cotangents at their steps (qocb_lindblad_backward).

Pins: the built-in density costs rewritten as plain NumPy subclasses (same forward, so final densities are bit-identical, and
the same gradient up to the differences' error), and the torch oracle with the step grid frozen under the contract of
include/qocb200.h (cost and densities within 1e-9, gradient within 1e-7)."""
import numpy as np
import pytest

from qoc_b200.models.cost import Cost
from tests.problems import Problem, haar_columns, rand_herm

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _dens(rng, n, count):
    v = haar_columns(rng, n, count).T
    return np.einsum("di,dj->dij", v, v.conj())


def _dissipator(n, L, seed):
    rng = np.random.default_rng(seed)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    ops = np.array([a, rand_herm(rng, n) * 0.5, a.T.copy()][:L]).reshape(L, n, n)
    return np.linspace(0.08, 0.03, L), ops


# --- the built-in density costs as plain NumPy user costs (qoc_b200/standard/costs.py, same normalisations and flags) -------
class TwinTarget(Cost):
    """TargetDensityInfidelity (norm 1) and TargetDensityInfidelityTime (norm (N-1)//cost_eval_step): final step only."""
    requires_step_evaluation = False

    def __init__(self, targets, cost_multiplier=1.0, norm=1.0):
        super().__init__(cost_multiplier)
        self.targets, self.norm = np.asarray(targets), norm

    def cost(self, controls, densities, step):
        D, n = self.targets.shape[0], self.targets.shape[1]
        fid = sum(abs(np.trace(t.conj().T @ r)) for t, r in zip(self.targets, densities)) / (D * n)
        return (1 - fid) / self.norm * self.cost_multiplier


class TwinForbid(Cost):
    """ForbidDensities: every cost step."""
    requires_step_evaluation = True

    def __init__(self, forbidden, N, cost_eval_step=1, cost_multiplier=1.0):
        super().__init__(cost_multiplier)
        self.forbidden = [np.asarray(f) for f in forbidden]
        self.norm = ((N - 1) // cost_eval_step) * len(self.forbidden)

    def cost(self, controls, densities, step):
        tot = 0.0
        for f, r in zip(self.forbidden, densities):
            n = r.shape[-1]
            tot += sum(abs(np.trace(m.conj().T @ r) / n) ** 2 for m in f) / len(f)
        return tot / self.norm * self.cost_multiplier


def _builtin_costs(std, targ, forb, N, ces, K, M):
    return [std.TargetDensityInfidelity(targ, cost_multiplier=0.8),
            std.ForbidDensities(forb, N, cost_eval_step=ces, cost_multiplier=0.4),
            std.TargetDensityInfidelityTime(N, targ, cost_eval_step=ces, cost_multiplier=0.3),
            std.ControlNorm(K, M, cost_multiplier=0.05)]


def _twin_costs(std, targ, forb, N, ces, K, M):
    return [TwinTarget(targ, 0.8), TwinForbid(forb, N, ces, 0.4), TwinTarget(targ, 0.3, (N - 1) // ces),
            std.ControlNorm(K, M, cost_multiplier=0.05)]


TWIN_CASES = [  # n, D, L, complex controls, cost_eval_step, slices
    (2, 1, 1, True, 1, 3),
    (3, 2, 0, False, 2, 4),
    (5, 1, 2, True, 3, 4),       # N-1 = 4 is not a cost step: the forbid twin is never evaluated at the final step
    (8, 2, 1, False, 1, 3),
    (16, 1, 2, True, 2, 4),
    (3, 1, 2, False, 3, 6),
]


@pytest.mark.parametrize("n,D,L,cc,ces,slices", TWIN_CASES)
def test_builtin_twins_match_builtins(n, D, L, cc, ces, slices):
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    K = 2
    p = Problem(n, slices, K, 1, 2, complex_controls=cc, seed=60 + n, M=6, h0_norm=0.8, drive_norm=0.3)
    rng = np.random.default_rng(n + 10 * D)
    rho0, targ = _dens(rng, n, D), _dens(rng, n, D)
    forb = np.array([_dens(rng, n, 2) for _ in range(D)])
    gam, ops = _dissipator(n, L, n)
    ld = (lambda t: (gam, ops)) if L else None
    plans = {}
    for key, make in (("builtin", _builtin_costs), ("twin", _twin_costs)):
        plans[key] = LindbladPlan(rho0, make(std, targ, forb, p.N, ces, K, p.M), p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                                  lindblad_data=ld, control_eval_count=p.M, control_count=K, complex_controls=cc,
                                  cost_eval_step=ces)
    assert len(plans["twin"].user_costs) == 3 and not plans["builtin"].user_costs
    e_b, g_b, f_b = plans["builtin"].cost_and_grad(p.controls)
    e_u, g_u, f_u = plans["twin"].cost_and_grad(p.controls)
    e_c, f_c = plans["twin"].cost(p.controls)
    assert np.array_equal(f_u, f_b) and np.array_equal(f_c, f_b)
    assert abs(e_u - e_b) <= 1e-12 * abs(e_b) and abs(e_c - e_b) <= 1e-12 * abs(e_b), (e_u, e_c, e_b)
    assert g_u.shape == p.controls.shape and g_u.dtype == p.controls.dtype
    assert rel(g_u, g_b) < 1e-8, rel(g_u, g_b)
    for plan in plans.values():
        plan.close()


# --- non-linear user costs against the torch oracle ---------------------------------------------------------------------
def _nonlinear_costs():
    import torch

    class Purity(Cost):
        """sum_d (1 - tr rho_d^2) at every cost step"""
        requires_step_evaluation = True

        def cost(self, controls, densities, step):
            return self.cost_multiplier * np.sum(1 - np.trace(densities @ densities, axis1=-2, axis2=-1))

    class Leakage(Cost):
        """squared population of the top level on the final densities, with an explicit control-energy term"""
        requires_step_evaluation = False

        def cost(self, controls, densities, step):
            pop = np.real(densities[:, -1, -1])
            return self.cost_multiplier * (np.sum(pop ** 2) + 0.01 * np.sum(np.abs(controls) ** 2))

    class PurityT(object):
        requires_step_evaluation = True

        def __init__(self, cost_multiplier=1.0):
            self.cost_multiplier = cost_multiplier

        def cost(self, controls, densities, step):
            return self.cost_multiplier * torch.sum(1 - torch.real(torch.einsum("dij,dji->d", densities, densities)))

    class LeakageT(object):
        requires_step_evaluation = False

        def __init__(self, cost_multiplier=1.0):
            self.cost_multiplier = cost_multiplier

        def cost(self, controls, densities, step):
            pop = torch.real(densities[:, -1, -1])
            return self.cost_multiplier * (torch.sum(pop ** 2) + 0.01 * torch.sum(torch.abs(controls) ** 2))
    return Purity, Leakage, PurityT, LeakageT


def _mixed_costs(mod, user, targ, forb, N, ces, K, M):
    Purity, Leakage = user
    return [Purity(0.3), mod.TargetDensityInfidelity(targ, cost_multiplier=0.8),
            mod.ForbidDensities(forb, N, cost_eval_step=ces, cost_multiplier=0.4), Leakage(0.7),
            mod.ControlNorm(K, M, cost_multiplier=0.05)]


@pytest.mark.parametrize("n,D,L,cc,ces,slices", [(3, 2, 1, True, 1, 3), (5, 1, 2, False, 2, 4), (8, 1, 1, True, 3, 4)])
def test_nonlinear_user_costs_vs_oracle(n, D, L, cc, ces, slices):
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    Purity, Leakage, PurityT, LeakageT = _nonlinear_costs()
    K = 2
    p = Problem(n, slices, K, 1, 2, complex_controls=cc, seed=80 + n, M=5, h0_norm=0.8, drive_norm=0.3)
    rng = np.random.default_rng(3 * n + D)
    rho0, targ = _dens(rng, n, D), _dens(rng, n, D)
    forb = np.array([_dens(rng, n, 1) for _ in range(D)])
    gam, ops = _dissipator(n, L, n + 1)
    plan = LindbladPlan(rho0, _mixed_costs(std, (Purity, Leakage), targ, forb, p.N, ces, K, p.M), p.T, p.N,
                        hamiltonian=p.hamiltonian_numpy(), lindblad_data=lambda t: (gam, ops), control_eval_count=p.M,
                        control_count=K, complex_controls=cc, cost_eval_step=ces)
    err, grads, finals = plan.cost_and_grad(p.controls)
    err_f, finals_f = plan.cost(p.controls)
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(p.controls, orc.make_hamiltonian(p.h0, p.drives, cc),
                                                      orc.make_lindblad_data(gam, ops), rho0,
                                                      _mixed_costs(orc, (PurityT, LeakageT), targ, forb, p.N, ces, K, p.M),
                                                      p.T, p.N, cost_eval_step=ces, freeze_steps=True)
    assert abs(err - o_err) < 1e-9 and abs(err_f - o_err) < 1e-9, (err, err_f, o_err)
    assert rel(finals, o_fin) < 1e-9 and rel(finals_f, o_fin) < 1e-9
    assert grads.shape == p.controls.shape and grads.dtype == p.controls.dtype
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    plan.close()


# --- time-dependent problems ---------------------------------------------------------------------------------------------
def test_timedep_problem_with_user_step_cost_vs_oracle():
    """the rotating-frame drive and modulated decay rate of tests/test_gpu_lindblad_timedep.py with a purity step cost."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    from tests.test_gpu_lindblad_timedep import _rotating_problem
    Purity, _, PurityT, _ = _nonlinear_costs()
    n, T, M, N, h, oh, ld, old, rho0, targ = _rotating_problem()
    u = 0.2 * (1 - 1j) / np.sqrt(2) * np.ones((M, 1), dtype=complex)     # the initial controls of that file's GRAPE test
    plan = LindbladPlan(rho0, [Purity(0.5), std.TargetDensityInfidelity(targ)], T, N, hamiltonian=h, lindblad_data=ld,
                        control_eval_count=M, control_count=1, complex_controls=True)
    assert plan.series is not None
    err, grads, finals = plan.cost_and_grad(u)
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(u, oh, old, rho0, [PurityT(0.5), orc.TargetDensityInfidelity(targ)], T, N,
                                                      freeze_steps=True)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    plan.close()


def test_user_step_cost_with_series_extension():
    """weak dynamics put the initial-step probe far beyond T + dt (tests/test_gpu_lindblad_timedep.py): the forward pass of
    the split evaluation returns -5, the plan extends its table and runs the forward pass again before seeding the reverse."""
    import torch
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan

    class UpperPop(Cost):
        """squared population of the upper level at every cost step"""
        requires_step_evaluation = True

        def cost(self, controls, densities, step):
            return np.sum(np.real(densities[:, 1, 1]) ** 2)

    class UpperPopT(object):
        requires_step_evaluation = True

        def cost(self, controls, densities, step):
            return torch.sum(torch.real(densities[:, 1, 1]) ** 2)
    sx = np.array([[0, 1], [1, 0]], dtype=complex)
    sz = np.diag([1.0, -1.0]).astype(complex)
    eps, w, T, N, M = 2e-3, 0.8, 2.0, 3, 4
    h = lambda u, t: eps * (np.cos(w * t) * sz + u[0] * sx)
    oh = lambda u, t: eps * (np.cos(w * float(t)) * torch.as_tensor(sz) + u[0] * torch.as_tensor(sx))
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    u = np.array([[0.3], [-0.2], [0.5], [0.1]])
    plan = LindbladPlan(rho0, [UpperPop()], T, N, hamiltonian=h, control_eval_count=M, control_count=1)
    err, grads, finals = plan.cost_and_grad(u)
    assert plan.range_extensions > 0
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(u, oh, None, rho0, [UpperPopT()], T, N, freeze_steps=True)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    plan.close()


def test_no_hamiltonian_user_cost_with_explicit_controls():
    """hamiltonian = None: the densities do not see the controls, so the gradient is the user cost's explicit control term."""
    from qoc_b200.core.plan import LindbladPlan
    Purity, Leakage, _, _ = _nonlinear_costs()
    n, D, N, M = 3, 2, 4, 5
    rng = np.random.default_rng(9)
    rho0 = _dens(rng, n, D)
    gam, ops = _dissipator(n, 2, 2)
    u = rng.standard_normal((M, 1)) + 1j * rng.standard_normal((M, 1))
    plan = LindbladPlan(rho0, [Purity(0.5), Leakage(2.0)], 3.0, N, lindblad_data=lambda t: (gam, ops), control_eval_count=M,
                        control_count=1, complex_controls=True)
    err, grads, finals = plan.cost_and_grad(u)
    dens = plan.intermediate_densities()
    want = sum(0.5 * np.sum(1 - np.trace(dens[k] @ dens[k], axis1=-2, axis2=-1)).real for k in range(1, N))
    want += 2.0 * (np.sum(dens[-1][:, -1, -1].real ** 2) + 0.01 * np.sum(np.abs(u) ** 2))
    assert abs(err - want) < 1e-12
    assert grads.dtype == u.dtype and rel(grads, 2.0 * 0.02 * u) < 1e-8, rel(grads, 0.04 * u)
    plan.close()


# --- the split C ABI -----------------------------------------------------------------------------------------------------
def test_split_abi_is_bit_identical_and_keeps_the_tape_rule():
    import qoc_b200.standard as std
    from qoc_b200 import _lib
    from qoc_b200.core.plan import LindbladPlan
    n, D, K = 4, 2, 2
    p = Problem(n, 3, K, 1, 2, complex_controls=True, seed=5, M=5, h0_norm=0.8, drive_norm=0.3)
    rng = np.random.default_rng(1)
    rho0, targ = _dens(rng, n, D), _dens(rng, n, D)
    forb = np.array([_dens(rng, n, 2) for _ in range(D)])
    gam, ops = _dissipator(n, 2, 4)
    plan = LindbladPlan(rho0, _builtin_costs(std, targ, forb, p.N, 1, K, p.M), p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                        lindblad_data=lambda t: (gam, ops), control_eval_count=p.M, control_count=K, complex_controls=True)
    lib, x = plan.lib, plan._real_channels(p.controls)
    c1, c2 = np.zeros(1), np.zeros(1)
    g1, g2 = np.zeros((p.M, 2 * K)), np.zeros((p.M, 2 * K))
    f1, f2 = (np.empty((D, n, n), dtype=np.complex128) for _ in range(2))
    plan._check(lib.qocb_lindblad_cost_and_grad(plan.handle, _lib.ptr(x), _lib.ptr(c1), _lib.ptr(g1), _lib.ptr(f1)))
    plan._check(lib.qocb_lindblad_forward(plan.handle, _lib.ptr(x), _lib.ptr(c2), _lib.ptr(f2)))
    plan._check(lib.qocb_lindblad_backward(plan.handle, None, _lib.ptr(g2)))
    assert np.array_equal(c1, c2) and np.array_equal(g1, g2) and np.array_equal(f1, f2)
    g3 = np.zeros_like(g2)                                  # a zero seed table changes nothing either
    zero = np.zeros((p.N, D, n, n), dtype=np.complex128)
    plan._check(lib.qocb_lindblad_backward(plan.handle, _lib.ptr(zero), _lib.ptr(g3)))
    assert np.array_equal(g3, g1)
    plan.cost(p.controls)                                   # overwrites the densities without a tape
    with pytest.raises(RuntimeError):
        plan._check(lib.qocb_lindblad_backward(plan.handle, None, _lib.ptr(g2)))
    plan.close()
    fresh = LindbladPlan(rho0, _builtin_costs(std, targ, forb, p.N, 1, K, p.M), p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                         lindblad_data=lambda t: (gam, ops), control_eval_count=p.M, control_count=K, complex_controls=True)
    with pytest.raises(RuntimeError):
        fresh._check(fresh.lib.qocb_lindblad_backward(fresh.handle, None, _lib.ptr(g2)))
    fresh.close()


# --- public programs -----------------------------------------------------------------------------------------------------
def test_grape_lindblad_with_user_step_cost_matches_oracle_driven_optimisation():
    """cfg2-like problem with a purity step cost next to the target: `grape_lindblad_discrete` with Adam against the same host
    optimiser fed by the oracle's cost and frozen-grid gradient; the error descends."""
    import qoc_b200 as qoc
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    from tests.problems import numpy_hamiltonian
    Purity, _, PurityT, _ = _nonlinear_costs()
    n, T, M, N, k = 2, 10.0, 11, 3, 6
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    h0 = np.diag(np.arange(n) - 0.5).astype(complex)
    rho0 = np.zeros((1, n, n), dtype=complex); rho0[0, 0, 0] = 1
    targ = np.zeros((1, n, n), dtype=complex); targ[0, 1, 1] = 1
    gam = np.array([2e-2])
    u0 = 0.1 * (1 - 1j) / np.sqrt(2) * np.ones((M, 1), dtype=complex)
    errors = []

    class Rec(std.Adam):
        def run(self, function, iteration_count, initial_params, jacobian, args=()):
            def jac(params, *a_):
                g, term = jacobian(params, *a_)
                errors.append(a_[1].error)
                return g, term
            return super().run(function, iteration_count, initial_params, jac, args=args)
    res = qoc.grape_lindblad_discrete(1, M, [std.TargetDensityInfidelity(targ), Purity(0.2)], T, rho0, N,
                                      complex_controls=True, hamiltonian=numpy_hamiltonian(h0, a[None], True),
                                      lindblad_data=lambda t: (gam, a[None]), initial_controls=u0.copy(), iteration_count=k,
                                      log_iteration_step=0, optimizer=Rec())
    o_err = []
    oh, old = orc.make_hamiltonian(h0, a[None], True), orc.make_lindblad_data(gam, a[None])

    def o_fun(params, *a_):
        return 0.0, False

    def o_jac(params, *a_):
        u = slap_controls(True, params, (M, 1))
        e, g, _ = orc.lindblad_cost_and_grad(u, oh, old, rho0, [orc.TargetDensityInfidelity(targ), PurityT(0.2)], T, N,
                                             freeze_steps=True)
        o_err.append(e)
        return strip_controls(True, g), False
    std.Adam().run(o_fun, k, strip_controls(True, u0.copy()), o_jac)
    assert len(errors) == k and len(o_err) == k
    assert np.abs(np.array(errors) - np.array(o_err)).max() < 1e-8, (errors, o_err)
    assert errors[-1] < errors[0] and res.best_error == min(errors)


def test_evolve_lindblad_with_user_costs_and_saved_densities(monkeypatch):
    """`evolve_lindblad_discrete` returns the oracle's error with user costs, and `save_intermediate_densities` writes the
    same rows as the same evolution without them."""
    import torch
    import qoc_b200 as qoc
    from oracle import qoc_oracle as orc
    from tests import fake_h5py
    from tests.problems import numpy_hamiltonian
    files = fake_h5py.install(monkeypatch)
    Purity, Leakage, PurityT, LeakageT = _nonlinear_costs()
    n, D, N, T, ces = 3, 2, 5, 3.0, 2
    p = Problem(n, 4, 1, 1, 2, complex_controls=True, seed=21, M=4, h0_norm=0.8, drive_norm=0.3)
    rng = np.random.default_rng(21)
    rho0 = _dens(rng, n, D)
    gam, ops = _dissipator(n, 1, 6)
    ham, ld = numpy_hamiltonian(p.h0, p.drives, True), (lambda t: (gam, ops))
    kw = dict(controls=p.controls, cost_eval_step=ces, hamiltonian=ham, lindblad_data=ld, save_intermediate_densities=True)
    res = qoc.evolve_lindblad_discrete(T, rho0, N, costs=[Purity(0.5), Leakage(1.5)], save_file_path="/u/a.h5", **kw)
    plain = qoc.evolve_lindblad_discrete(T, rho0, N, costs=[], save_file_path="/u/b.h5", **kw)
    o_err, o_fin = orc.evaluate_lindblad(torch.as_tensor(p.controls), orc.make_hamiltonian(p.h0, p.drives, True), orc.make_lindblad_data(gam, ops),
                                         rho0, [PurityT(0.5), LeakageT(1.5)], T, N, cost_eval_step=ces)
    assert abs(res.error - float(o_err)) < 1e-9 and rel(res.final_densities, o_fin.numpy()) < 1e-9
    a, b = np.asarray(files["/u/a.h5"]["intermediate_densities"]), np.asarray(files["/u/b.h5"]["intermediate_densities"])
    assert a.size == N * D * n * n and np.array_equal(a, b)
    assert np.array_equal(a.reshape(N, D, n, n)[-1], res.final_densities)


def test_state_costs_are_still_refused():
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    rho0 = _dens(np.random.default_rng(0), 2, 1)
    psi = np.array([[[1.0], [0.0]]], dtype=complex)
    with pytest.raises(NotImplementedError):
        LindbladPlan(rho0, [std.TargetStateInfidelity(psi)], 1.0, 3, lindblad_data=lambda t: (np.array([0.1]),
                                                                                                np.eye(2, dtype=complex)[None]))
