"""GPU: Lindblad ensembles (`LindbladPlan(ensemble_drifts=..., ensemble_rates=...)`): robust control over a spread of drifts
(detunings) and decay rates, one CTA per member in one launch, with the member mean as cost and gradient.

Pins: every member is bit-identical to a one-member plan built with its drift and rates and the same control operators
(cost, densities at every step, gradient, stats), and the mean is the member-order sum divided by E, bit for bit; the mean
matches the mean of the torch oracle with the step grid frozen under the contract of include/qocb200.h (cost and densities
1e-9, gradient 1e-7)."""
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


def _dissipator(n, L, seed):
    rng = np.random.default_rng(seed)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    ops = np.array([a, rand_herm(rng, n) * 0.5, a.T.copy()][:L]).reshape(L, n, n)
    return np.linspace(0.08, 0.03, L), ops


def _costs(mod, kind, targ, forb, N, ces, K, M):
    out = []
    if kind in ("target", "all"):
        out.append(mod.TargetDensityInfidelity(targ, cost_multiplier=0.8))
    if kind in ("forbid", "all"):
        out += [mod.ForbidDensities(forb, N, cost_eval_step=ces, cost_multiplier=0.4),
                mod.TargetDensityInfidelityTime(N, targ, cost_eval_step=ces, cost_multiplier=0.3)]
    if kind == "all":
        out.append(mod.ControlNorm(K, M, cost_multiplier=0.05))
    return out


class Case(object):
    """a seeded problem with E members: detunings spread the drift, rates spread around gamma."""

    def __init__(self, n, D, L, cc, ces, E, kind, slices=3, seed=0, vary=("drift", "rate")):
        from qoc_b200.core.plan import extract_hamiltonian_structure
        self.K, self.cc, self.ces, self.E, self.kind = 2, cc, ces, E, kind
        self.p = p = Problem(n, slices, self.K, 1, 2, complex_controls=cc, seed=70 + n + seed, M=5, h0_norm=0.8,
                             drive_norm=0.3)
        rng = np.random.default_rng(100 * n + 10 * D + L + seed)
        self.rho0, self.targ = _dens(rng, n, D), _dens(rng, n, D)
        self.forb = np.array([_dens(rng, n, 2) for _ in range(D)])
        self.gam, self.ops = _dissipator(n, L, n + seed)
        self.h0, self.a_ops = extract_hamiltonian_structure(p.hamiltonian_numpy(), self.K, cc, p.T)
        det = np.diag(np.linspace(-0.5, 0.5, n)).astype(complex)
        self.drifts = None
        if "drift" in vary:
            self.drifts = np.array([self.h0 + 0.3 * rng.uniform(-1, 1) * det for _ in range(E)])
        self.rates = None
        if "rate" in vary and L:
            self.rates = np.array([self.gam * rng.uniform(0.5, 1.5, L) for _ in range(E)])

    def member(self, e):
        h0 = self.h0 if self.drifts is None else self.drifts[e]
        gam = self.gam if self.rates is None else self.rates[e]
        return h0, gam

    def plan(self, e=None, **kw):
        """the ensemble (e None) or the one-member plan of member e."""
        import qoc_b200.standard as std
        from qoc_b200.core.plan import LindbladPlan
        p, L = self.p, self.ops.shape[0]
        if e is None:
            h0, gam, ens = self.h0, self.gam, dict(ensemble_drifts=self.drifts, ensemble_rates=self.rates)
        else:
            (h0, gam), ens = self.member(e), {}
        return LindbladPlan(self.rho0, _costs(std, self.kind, self.targ, self.forb, p.N, self.ces, self.K, p.M), p.T, p.N,
                            hamiltonian=p.hamiltonian_numpy(), lindblad_data=(lambda t: (gam, self.ops)) if L else None,
                            control_eval_count=p.M, control_count=self.K, complex_controls=self.cc,
                            cost_eval_step=self.ces, structure=(h0, self.a_ops), **ens, **kw)


def _check_members(case, members):
    u = case.p.controls
    ens = case.plan()
    err, grads, finals = ens.cost_and_grad(u)
    costs, mgrads, mstats = ens.member_results()
    dens = ens.intermediate_densities()
    E, N, D, n = case.E, case.p.N, case.rho0.shape[0], case.rho0.shape[1]
    assert finals.shape == (E, D, n, n) and dens.shape == (E, N, D, n, n)
    assert mgrads.shape == (E,) + u.shape and mgrads.dtype == u.dtype and grads.dtype == u.dtype
    assert ens.stats() == {"attempts": sum(s["attempts"] for s in mstats), "accepted": sum(s["accepted"] for s in mstats)}
    for e in members:
        one = case.plan(e)
        e1, g1, f1 = one.cost_and_grad(u)
        assert e1 == costs[e], (e, e1, costs[e])
        assert np.array_equal(g1, mgrads[e]), e
        assert np.array_equal(f1, finals[e]) and np.array_equal(one.intermediate_densities(), dens[e]), e
        assert one.stats() == mstats[e], e
        one.close()
    s, g = 0.0, 0.0
    for e in range(E):
        s, g = s + costs[e], g + mgrads[e]
    g = g.real / E + 1j * (g.imag / E) if np.iscomplexobj(g) else g / E   # NumPy's complex / real is not (re / E, im / E)
    if case.kind == "all":             # the control cost is added once to the mean, once to every member
        assert abs(err - s / E) <= 1e-14 * (1 + abs(err)) and rel(grads, g) < 1e-14
    else:
        assert err == s / E and np.array_equal(grads, g)
    err_c, finals_c = ens.cost(u)                               # the forward pass without its tape
    assert err_c == err and np.array_equal(finals_c, finals)
    ens.close()


@pytest.mark.parametrize("n,D,L,cc,ces,E,kind", [
    (2, 1, 1, True, 1, 5, "all"),
    (2, 2, 2, False, 2, 2, "forbid"),
    (3, 2, 0, False, 2, 5, "target"),
    (3, 1, 1, True, 1, 37, "all"),
    (8, 2, 2, True, 1, 37, "all"),
    (8, 1, 1, False, 2, 2, "target"),
    (16, 1, 2, True, 1, 5, "forbid"),
    (16, 2, 1, False, 2, 2, "all"),
])
def test_members_match_single_plans(n, D, L, cc, ces, E, kind):
    _check_members(Case(n, D, L, cc, ces, E, kind), range(E))


@pytest.mark.parametrize("vary", [("drift",), ("rate",)])
def test_one_varied_component(vary):
    _check_members(Case(3, 1, 2, True, 1, 5, "all", vary=vary), range(5))


def test_global_memory_working_set():
    """n = 32, D = 1: the working sets of both kernels exceed shared memory and live in each member's global slice."""
    _check_members(Case(32, 1, 1, True, 1, 3, "target", slices=2), range(3))


def test_more_members_than_sms():
    """E = 300 at n = 2 (32-thread CTAs): a seeded sample of members against single plans."""
    rng = np.random.default_rng(5)
    _check_members(Case(2, 1, 1, True, 1, 300, "all"), sorted(rng.choice(300, 6, replace=False)))


def test_one_member_ensemble_is_the_plain_plan():
    case = Case(3, 2, 1, True, 1, 1, "all")
    u = case.p.controls
    a = case.plan().cost_and_grad(u)
    b = case.plan(0).cost_and_grad(u)
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert a[2].shape == b[2].shape


@pytest.mark.parametrize("n,D,L,cc,ces,E", [(2, 1, 1, True, 1, 4), (3, 2, 2, False, 2, 3)])
def test_mean_matches_oracle(n, D, L, cc, ces, E):
    from oracle import qoc_oracle as orc
    case = Case(n, D, L, cc, ces, E, "all")
    p, u = case.p, case.p.controls
    ens = case.plan()
    err, grads, finals = ens.cost_and_grad(u)
    o_err, o_grad, o_fin = 0.0, 0.0, []
    for e in range(E):
        h0, gam = case.member(e)
        oe, og, of = orc.lindblad_cost_and_grad(u, orc.make_hamiltonian(h0, p.drives, cc), orc.make_lindblad_data(gam, case.ops),
                                                case.rho0, _costs(orc, "all", case.targ, case.forb, p.N, ces, case.K, p.M),
                                                p.T, p.N, cost_eval_step=ces, freeze_steps=True)
        o_err, o_grad = o_err + oe / E, o_grad + og / E
        o_fin.append(of)
    assert abs(err - o_err) < 1e-9, (err, o_err)
    assert rel(finals, np.array(o_fin)) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    ens.close()


# --- time dependence ----------------------------------------------------------------------------------------------------
def _oracle_mean(u, members, rho0, costs, T, N):
    from oracle import qoc_oracle as orc
    out = [orc.lindblad_cost_and_grad(u, oh, old, rho0, costs, T, N, freeze_steps=True) for oh, old in members]
    E = len(out)
    return sum(o[0] for o in out) / E, sum(o[1] for o in out) / E, np.array([o[2] for o in out])


def test_timedep_hamiltonian_with_member_rates():
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    from tests.test_gpu_lindblad_timedep import _rotating_problem
    n, T, M, N, h, oh, ld, old, rho0, targ = _rotating_problem()
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    rates = np.array([[0.02], [0.05], [0.11]])
    u = 0.2 * (1 - 1j) / np.sqrt(2) * np.ones((M, 1), dtype=complex)
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=h, lindblad_data=lambda t: (rates[0], a[None]),
                        control_eval_count=M, control_count=1, complex_controls=True, ensemble_rates=rates)
    assert plan.series is not None and plan.series.KC > 0
    err, grads, finals = plan.cost_and_grad(u)
    o_err, o_grad, o_fin = _oracle_mean(u, [(oh, orc.make_lindblad_data(r, a[None])) for r in rates], rho0,
                                        [orc.TargetDensityInfidelity(targ)], T, N)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    plan.close()


def test_timedep_rates_with_member_drifts():
    import torch
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    from tests.test_gpu_lindblad_timedep import _lindblad_pair
    n, T, M, N = 3, 3.0, 5, 4
    ld, old = _lindblad_pair("rate", n, 2, 7)
    rng = np.random.default_rng(11)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    h0 = np.diag(np.arange(n) - 1.0).astype(complex) * 0.4
    drifts = np.array([h0 + d * np.diag([1.0, 0.0, -1.0]) for d in (-0.1, 0.0, 0.07, 0.15)])
    rho0, targ = _dens(rng, n, 1), _dens(rng, n, 1)
    u = 0.3 * (rng.standard_normal((M, 1)) + 1j * rng.standard_normal((M, 1)))
    ham = lambda c, t: h0 + c[0] * a + np.conjugate(c[0]) * a.conj().T
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=ham, lindblad_data=ld,
                        control_eval_count=M, control_count=1, complex_controls=True, ensemble_drifts=drifts)
    assert plan.series is not None and plan.series.KC == 0
    err, grads, finals = plan.cost_and_grad(u)
    members = [(orc.make_hamiltonian(d, a[None], True), old) for d in drifts]
    o_err, o_grad, o_fin = _oracle_mean(u, members, rho0, [orc.TargetDensityInfidelity(targ)], T, N)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)
    plan.close()


def test_timedep_series_extension_over_members():
    """weak dynamics take steps far beyond T + dt; the table is extended to the largest stage time over the members."""
    import torch
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    sx = np.array([[0, 1], [1, 0]], dtype=complex)
    sz = np.diag([1.0, -1.0]).astype(complex)
    sm = np.array([[0, 1], [0, 0]], dtype=complex)
    eps, w, T, N, M = 2e-3, 0.8, 2.0, 3, 4
    h = lambda u, t: eps * (np.cos(w * t) * sz + u[0] * sx)
    oh = lambda u, t: eps * (np.cos(w * float(t)) * torch.as_tensor(sz) + u[0] * torch.as_tensor(sx))
    rates = np.array([[1e-4], [3e-4], [1e-3]])
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    targ = np.array([[[0.5, 0.5], [0.5, 0.5]]], dtype=complex)
    u = np.array([[0.3], [-0.2], [0.5], [0.1]])
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=h, lindblad_data=lambda t: (rates[0], sm[None]),
                        control_eval_count=M, control_count=1, ensemble_rates=rates)
    err, grads, finals = plan.cost_and_grad(u)
    assert plan.range_extensions >= 1
    o_err, o_grad, o_fin = _oracle_mean(u, [(oh, orc.make_lindblad_data(r, sm[None])) for r in rates], rho0,
                                        [orc.TargetDensityInfidelity(targ)], T, N)
    assert abs(err - o_err) < 1e-9 and rel(finals, o_fin) < 1e-9
    assert rel(grads, o_grad) < 1e-7
    plan.close()


# --- tape overflow and the C ABI's refusals -------------------------------------------------------------------------------
def test_one_member_overflows_its_tape():
    """a stiffer member needs more accepted steps than the others: with a per-member capacity between the two, that member
    overflows, the evaluation raises the -4 error, and a plan with enough capacity evaluates the same ensemble."""
    case = Case(3, 1, 1, True, 1, 4, "target", vary=("drift",))
    case.drifts[2] = case.drifts[2] * 6.0
    u = case.p.controls
    ref = case.plan()
    err, grads, finals = ref.cost_and_grad(u)
    acc = sorted(s["accepted"] for s in ref.member_results()[2])
    assert acc[-1] > acc[-2] + 1, acc
    small = case.plan(max_rk_steps=(acc[-1] + acc[-2]) // 2)
    with pytest.raises(RuntimeError, match="rc=-4.*tape is full"):
        small.cost_and_grad(u)
    small.close()
    again = case.plan()
    e2, g2, f2 = again.cost_and_grad(u)
    assert e2 == err and np.array_equal(g2, grads) and np.array_equal(f2, finals)
    ref.close()
    again.close()


def test_c_abi_refusals():
    from qoc_b200 import _lib
    case = Case(2, 1, 1, True, 1, 3, "target")
    ens, one = case.plan(), case.plan(0)
    lib = ens.lib
    assert lib.qocb_lindblad_set_ensemble(one.handle, None, None) == -1
    x = case.p.controls
    x = np.ascontiguousarray(np.concatenate([x.real, x.imag], axis=1))
    out = np.zeros(1)
    fd = np.zeros((3, 1, 2, 2), dtype=complex)
    assert lib.qocb_lindblad_forward(ens.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)) == -1
    assert lib.qocb_lindblad_backward(ens.handle, None, None) == -1
    rates_td = np.ones((3, 1))
    su = ens._setup
    h0 = np.ascontiguousarray(su["h0"])
    a_ops = np.ascontiguousarray(su["a_ops"])
    # set_operators resets the members: an evaluation then needs set_ensemble again
    assert lib.qocb_lindblad_set_operators(ens.handle, _lib.ptr(h0), _lib.ptr(a_ops), _lib.ptr(su["gammas"]),
                                           _lib.ptr(su["lops"])) == 0
    assert lib.qocb_lindblad_cost(ens.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)) == -1
    assert lib.qocb_lindblad_set_ensemble(ens.handle, _lib.ptr(case.drifts), _lib.ptr(rates_td * 0.05)) == 0
    assert lib.qocb_lindblad_cost(ens.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)) == 0
    ens.close()
    one.close()


# --- GRAPE ----------------------------------------------------------------------------------------------------------------
def test_grape_on_ensemble_mean_matches_oracle_driven_adam():
    """robust control of a decaying qubit: Adam on the E = 8 member mean against the same optimiser fed by the oracle."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    n, T, N, M, E, k = 2, 2.0, 5, 6, 8, 4
    rng = np.random.default_rng(21)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    h0 = np.diag([-0.5, 0.5]).astype(complex)
    drifts = np.array([h0 * (1 + d) for d in rng.uniform(-0.1, 0.1, E)])
    rates = rng.uniform(0.01, 0.05, (E, 1))
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    targ = np.array([[[0, 0], [0, 1]]], dtype=complex)
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=numpy_hamiltonian(h0, a[None], True),
                        lindblad_data=lambda t: (rates[0], a[None]), control_eval_count=M, control_count=1,
                        complex_controls=True, ensemble_drifts=drifts, ensemble_rates=rates)
    u0 = 0.3 * (1 - 1j) / np.sqrt(2) * np.ones((M, 1), dtype=complex)
    members = [(orc.make_hamiltonian(d, a[None], True), orc.make_lindblad_data(r, a[None])) for d, r in zip(drifts, rates)]
    errors, o_errors = [], []

    def jac(params):
        e, g, _ = plan.cost_and_grad(slap_controls(True, params, (M, 1)))
        errors.append(e)
        return strip_controls(True, g), False

    def o_jac(params):
        e, g, _ = _oracle_mean(slap_controls(True, params, (M, 1)), members, rho0, [orc.TargetDensityInfidelity(targ)], T, N)
        o_errors.append(e)
        return strip_controls(True, g), False
    std.Adam().run(lambda p: (0.0, False), k, strip_controls(True, u0.copy()), jac)
    std.Adam().run(lambda p: (0.0, False), k, strip_controls(True, u0.copy()), o_jac)
    assert len(errors) == k and len(o_errors) == k
    assert np.abs(np.array(errors) - np.array(o_errors)).max() < 1e-8, (errors, o_errors)
    assert errors[-1] < errors[0]
    plan.close()
