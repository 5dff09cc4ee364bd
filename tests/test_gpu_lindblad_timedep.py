"""GPU tests of time-dependent Lindblad problems: `hamiltonian(controls, time)` that reads `time` and `lindblad_data(time)`
that varies with time, evaluated by the kernels at the adaptive Runge-Kutta stage times from piecewise Chebyshev series.

The pin is the torch oracle, which calls the callables at the true stage times (oracle/qoc_oracle.py:469-486), under the
contract of include/qocb200.h: cost and final densities within 1e-9, gradient within 1e-7 of the oracle with the step grid
frozen (`freeze_steps=True`)."""
import numpy as np
import pytest

from tests.problems import Problem, haar_columns, rand_herm

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _dens(rng, n, count):
    v = haar_columns(rng, n, count).T
    return np.einsum("di,dj->dij", v, v.conj())


def _lindblad_pair(kind, n, L, seed):
    """(numpy callable, torch callable) of a dissipator family:
    static: constant; rate: modulated rates; phase: operators rotating in phase (with a growing modulus); both."""
    import torch
    rng = np.random.default_rng(seed)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    ops = [a, rand_herm(rng, n) * 0.5, a.T.copy()][:L]
    ops = np.array(ops).reshape(L, n, n)
    g0 = np.linspace(0.08, 0.03, L) if L else np.zeros(0)

    def ld(t):
        t = float(t)
        g, o = g0.copy(), ops.copy()
        if kind in ("rate", "both"):
            g = g * (1.0 + 0.5 * np.sin(0.9 * t + np.arange(L)))
        if kind in ("phase", "both") and L:
            o[0] = np.exp(1j * 1.7 * t) * (1.0 + 0.05 * t) * o[0]
        return g, o
    return ld, (lambda t: tuple(torch.as_tensor(x) for x in ld(t)))


def _costs(mod, targ, forb, N, ces, K, M, with_control):
    out = [mod.TargetDensityInfidelity(targ, cost_multiplier=0.8),
           mod.ForbidDensities(forb, N, cost_eval_step=ces, cost_multiplier=0.4),
           mod.TargetDensityInfidelityTime(N, targ, cost_eval_step=ces, cost_multiplier=0.3)]
    if with_control:
        out.append(mod.ControlNorm(K, M, cost_multiplier=0.05))
    return out


CASES = [  # n, D, L, complex controls, cost_eval_step, dissipator
    (2, 1, 1, True, 1, "phase"),
    (3, 2, 0, False, 2, None),
    (3, 1, 2, False, 1, "static"),
    (5, 1, 2, True, 2, "rate"),
    (8, 2, 1, False, 1, "both"),
    (16, 1, 1, True, 2, "rate"),
]


@pytest.mark.parametrize("n,D,L,cc,ces,kind", CASES)
def test_timedep_lindblad_vs_oracle(n, D, L, cc, ces, kind):
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    K, slices = 2, 4
    p = Problem(n, slices, K, 1, 2, complex_controls=cc, seed=40 + n, M=6, h0_norm=0.8, drive_norm=0.3)
    N, M, T = p.N, p.M, p.T
    rng = np.random.default_rng(n + 10 * D)
    rho0, targ = _dens(rng, n, D), _dens(rng, n, D)
    forb = np.array([_dens(rng, n, 2) for _ in range(D)])
    ld, old = _lindblad_pair(kind, n, L, n) if L else (None, None)
    plan = LindbladPlan(rho0, _costs(std, targ, forb, N, ces, K, M, True), T, N, hamiltonian=p.hamiltonian_td_numpy(),
                        lindblad_data=ld, control_eval_count=M, control_count=K, complex_controls=cc, cost_eval_step=ces)
    assert plan.series is not None and plan.series.KC >= 1
    assert plan.series.L == (L if kind not in (None, "static") else 0)
    err, grads, finals = plan.cost_and_grad(p.controls)
    err_f, finals_f = plan.cost(p.controls)
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(p.controls, p.hamiltonian_td_torch(), old, rho0,
                                                      _costs(orc, targ, forb, N, ces, K, M, True), T, N,
                                                      cost_eval_step=ces, freeze_steps=True)
    assert abs(err - o_err) < 1e-9 and abs(err_f - o_err) < 1e-9, (err, err_f, o_err)
    assert rel(finals, o_fin) < 1e-9 and rel(finals_f, o_fin) < 1e-9
    assert grads.shape == p.controls.shape and grads.dtype == p.controls.dtype
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    assert rel(plan.intermediate_densities()[-1], o_fin) < 1e-9
    plan.close()


def test_timedep_dissipation_without_hamiltonian():
    from oracle import qoc_oracle as orc
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    n, D, L, N, T = 3, 2, 2, 4, 3.0
    rng = np.random.default_rng(7)
    rho0, targ = _dens(rng, n, D), _dens(rng, n, D)
    forb = np.array([_dens(rng, n, 1) for _ in range(D)])
    ld, old = _lindblad_pair("both", n, L, 3)
    costs = lambda mod: _costs(mod, targ, forb, N, 1, 0, 0, False)
    plan = LindbladPlan(rho0, costs(std), T, N, lindblad_data=ld)
    assert plan.series is not None and plan.series.KC == 0 and plan.series.L == L
    err, finals = plan.cost(None)
    o_err, o_fin = orc.evaluate_lindblad(None, None, old, rho0, costs(orc), T, N)
    assert abs(err - float(o_err)) < 1e-9 and rel(finals, o_fin.numpy()) < 1e-9
    plan.close()


def test_stage_times_beyond_the_table_extend_it():
    """weak dynamics make the initial-step probe t0 + h0 (h0 = 0.01 d0/d1) land far beyond T + dt; the oracle's right-hand
    side is called there, and the plan must extend its series to reproduce it."""
    import torch
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    sx = np.array([[0, 1], [1, 0]], dtype=complex)
    sz = np.diag([1.0, -1.0]).astype(complex)
    eps, w, T, N, M = 2e-3, 0.8, 2.0, 3, 4
    h = lambda u, t: eps * (np.cos(w * t) * sz + u[0] * sx)
    seen = []

    def oh(u, t):
        seen.append(float(t))
        return eps * (np.cos(w * float(t)) * torch.as_tensor(sz) + u[0] * torch.as_tensor(sx))
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    targ = np.array([[[0.5, 0.5], [0.5, 0.5]]], dtype=complex)
    u = np.array([[0.3], [-0.2], [0.5], [0.1]])
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=h, control_eval_count=M,
                        control_count=1)
    t_max0 = plan.series.t_max
    err, grads, finals = plan.cost_and_grad(u)
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(u, oh, None, rho0, [orc.TargetDensityInfidelity(targ)], T, N,
                                                      freeze_steps=True)
    dt = T / (N - 1)
    assert max(seen) > T + dt and t_max0 < max(seen)
    assert plan.range_extensions >= 1 and plan.series.t_max >= max(seen)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7
    ext = plan.range_extensions                                   # the extended table now covers every evaluation
    plan.cost_and_grad(u)
    assert plan.range_extensions == ext
    plan.close()


def test_time_independent_callables_build_no_series():
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    p = Problem(3, 3, 1, 1, 2, complex_controls=True, seed=1)
    rho0 = _dens(np.random.default_rng(0), 3, 1)
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(rho0)], p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                        lindblad_data=lambda t: (np.array([0.1]), np.diag([1.0, 2.0, 3.0]).astype(complex)[None]),
                        control_eval_count=p.M, control_count=1, complex_controls=True)
    assert plan.series is None
    plan.cost_and_grad(p.controls)
    plan.close()


def _rotating_problem():
    import torch
    n, T, M, N = 2, 6.0, 7, 4
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    h0 = np.diag(np.arange(n) - 0.5).astype(complex) * 0.2
    w = 0.6

    def h(u, t):
        ph = np.exp(1j * w * t)
        return h0 + u[0] * ph * a + np.conjugate(u[0] * ph) * a.conj().T

    def oh(u, t):
        t = float(t)
        ph = complex(np.cos(w * t), np.sin(w * t))
        return torch.as_tensor(h0) + u[0] * ph * torch.as_tensor(a) + torch.conj(u[0] * ph) * torch.as_tensor(a.conj().T)
    ld, old = _lindblad_pair("rate", n, 1, 2)
    rho0 = np.zeros((1, n, n), dtype=complex); rho0[0, 0, 0] = 1
    targ = np.zeros((1, n, n), dtype=complex); targ[0, 1, 1] = 1
    return n, T, M, N, h, oh, ld, old, rho0, targ


def test_grape_timedep_lindblad_matches_oracle_driven_optimisation():
    """a rotating-frame drive with a modulated decay rate: `grape_lindblad_discrete` with Adam against the same host optimiser
    fed by the oracle's cost and frozen-grid gradient."""
    import qoc_b200 as qoc
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    n, T, M, N, h, oh, ld, old, rho0, targ = _rotating_problem()
    k = 5
    u0 = 0.2 * (1 - 1j) / np.sqrt(2) * np.ones((M, 1), dtype=complex)
    errors = []

    class Rec(std.Adam):
        def run(self, function, iteration_count, initial_params, jacobian, args=()):
            def jac(params, *a_):
                g, term = jacobian(params, *a_)
                errors.append(a_[1].error)
                return g, term
            return super().run(function, iteration_count, initial_params, jac, args=args)
    res = qoc.grape_lindblad_discrete(1, M, [std.TargetDensityInfidelity(targ)], T, rho0, N, complex_controls=True,
                                      hamiltonian=h, lindblad_data=ld, initial_controls=u0.copy(), iteration_count=k,
                                      log_iteration_step=0, optimizer=Rec())
    o_err = []

    def o_fun(params, *a_):
        return 0.0, False

    def o_jac(params, *a_):
        u = slap_controls(True, params, (M, 1))
        e, g, _ = orc.lindblad_cost_and_grad(u, oh, old, rho0, [orc.TargetDensityInfidelity(targ)], T, N, freeze_steps=True)
        o_err.append(e)
        return strip_controls(True, g), False
    std.Adam().run(o_fun, k, strip_controls(True, u0.copy()), o_jac)
    assert len(errors) == k and len(o_err) == k
    assert np.abs(np.array(errors) - np.array(o_err)).max() < 1e-8, (errors, o_err)
    assert errors[-1] < errors[0] and res.best_error == min(errors)


def test_evolve_timedep_lindblad_saves_intermediate_densities(monkeypatch):
    """`evolve_lindblad_discrete` with a time-dependent drift and dissipator: every saved intermediate density equals the
    oracle's final density over the same number of intervals (intervals are integrated independently)."""
    import torch
    import qoc_b200 as qoc
    from oracle import qoc_oracle as orc
    from tests import fake_h5py
    files = fake_h5py.install(monkeypatch)
    n, N, dt = 3, 5, 0.75
    rng = np.random.default_rng(12)
    h0, d = rand_herm(rng, n) * 0.5, rand_herm(rng, n) * 0.3
    h = lambda u, t: h0 + np.cos(1.1 * t) * d
    oh = lambda u, t: torch.as_tensor(h0 + np.cos(1.1 * float(t)) * d)
    ld, old = _lindblad_pair("both", n, 2, 5)
    rho0 = _dens(rng, n, 2)
    res = qoc.evolve_lindblad_discrete((N - 1) * dt, rho0, N, hamiltonian=h, lindblad_data=ld, save_file_path="/e/l.h5",
                                       save_intermediate_densities=True)
    dens = np.asarray(files["/e/l.h5"]["intermediate_densities"]).reshape(N, 2, n, n)
    assert np.allclose(dens[0], rho0) and rel(dens[-1], res.final_densities) < 1e-14
    for k in (2, N - 1):
        _, o_fin = orc.evaluate_lindblad(None, oh, old, rho0, [], k * dt, k + 1)
        assert rel(dens[k], o_fin.numpy()) < 1e-9
