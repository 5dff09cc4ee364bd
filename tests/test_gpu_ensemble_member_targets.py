"""GPU: ensembles whose members differ in their initial states / densities and cost targets (`ensemble_initial_states`,
`ensemble_initial_densities`, `ensemble_costs`: band-selective and multi-target pulses), Schroedinger and Lindblad paths.

Pins: identical member data forced through the new calls is bit-identical to shared data (cost, gradient, final and
intermediate states, launch count); the member mean matches the mean of the torch oracle over members, each with its own
initial states and costs (Schroedinger 1e-10, Lindblad on the frozen step grid 1e-9 / 1e-7); every member equals a one-member
plan built from its data (Schroedinger 1e-12, Lindblad bit for bit); a one-rank member-sharded plan equals the unsharded one;
band-selective inversion under Adam follows the oracle-driven Adam."""
import copy
import socket

import numpy as np
import pytest

from tests.problems import Problem, haar_columns, numpy_hamiltonian

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _policy(order):
    from qoc_b200.models import MagnusPolicy
    return {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}[order]


def _member_problems(p, E, seed):
    """E copies of `p`, each with its own Haar initial, target and forbidden states (same S, F, cost kinds and weights)."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(E):
        q = copy.copy(p)
        n, S = p.n, p.S
        q.initial_states = np.ascontiguousarray(haar_columns(rng, n, S).T)[:, :, None]
        q.target_states = np.ascontiguousarray(haar_columns(rng, n, S).T)[:, :, None]
        if p.F > 0:
            q.forbidden_states = np.array([np.ascontiguousarray(haar_columns(rng, n, p.forbidden_states.shape[1]).T)[:, :, None]
                                           for _ in range(S)])
        out.append(q)
    return out


def _schroedinger(p, std, **kw):
    from qoc_b200.core.plan import SchroedingerPlan
    return SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                            control_count=p.K, complex_controls=p.complex_controls, magnus_policy=_policy(p.order),
                            cost_eval_step=p.cost_eval_step, **kw)


def _results(plan, u):
    err, grads, finals = plan.cost_and_grad(u)
    err_f, finals_f = plan.cost(u)
    return err, grads, finals, plan.intermediate_states(), err_f, finals_f


# --- pointer plumbing: identical member data through the new calls ---------------------------------------------------
@pytest.mark.parametrize("n,K,cc,order,ces,step,F,tape", [
    (2, 2, False, 2, 1, False, 0, True),
    (8, 2, True, 4, 1, True, 2, True),        # M4, KR = 4: product-free
    (8, 4, True, 4, 2, True, 2, False),       # M4, KR = 8: explicit commutators, recompute tape
    (32, 2, False, 4, 1, False, 3, True),
    (32, 1, True, 6, 2, True, 0, True),
    (64, 2, False, 2, 1, True, 2, False),
    (64, 1, True, 6, 1, False, 1, True),
])
def test_identical_member_data_is_bit_identical(n, K, cc, order, ces, step, F, tape):
    import qoc_b200.standard as std
    p = Problem(n, 6, K, 2, order, complex_controls=cc, F=F, seed=n + K, cost_eval_step=ces, step_target=step)
    E = 3
    z = np.diag(np.linspace(-1, 1, n)).astype(complex) * 0.2
    drifts = np.array([p.h0 + d * z for d in (-1.0, 0.3, 1.0)])
    shared = _schroedinger(p, std, ensemble_drifts=drifts, store_tape=tape)
    forced = _schroedinger(p, std, ensemble_drifts=drifts, store_tape=tape,
                           ensemble_initial_states=np.array([p.initial_states] * E),
                           ensemble_costs=[p.costs(std) for _ in range(E)])
    ra, rb = _results(shared, p.controls), _results(forced, p.controls)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert shared.launch_count() == forced.launch_count() and shared.launch_count(False) == forced.launch_count(False)
    shared.close(); forced.close()


# --- physics against the oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,E,S,order,cc,route,ces,tape", [
    (2, 64, 1, 2, True, "alone", 1, True),
    (2, 7, 4, 6, False, "drifts", 2, True),
    (5, 7, 4, 4, True, "hamiltonians", 1, False),
    (5, 2, 5, 4, False, "alone", 2, True),            # S = 5: dense reverse pass
    (16, 2, 1, 6, True, "drifts", 1, True),
    (32, 7, 4, 2, False, "alone", 2, False),
    (32, 2, 5, 4, True, "hamiltonians", 1, True),
    (60, 2, 4, 4, False, "hamiltonians", 1, True),
    (64, 2, 1, 4, True, "alone", 1, True),
    (64, 7, 1, 6, False, "drifts", 2, True),
])
def test_member_mean_matches_oracle(n, E, S, order, cc, route, ces, tape):
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import SchroedingerPlan
    F = 2 if S < n else 0
    p = Problem(n, 4, 2, S, order, complex_controls=cc, F=F, seed=3 * n + E, cost_eval_step=ces, step_target=ces > 1)
    members = _member_problems(p, E, seed=n + S)
    rng = np.random.default_rng(E)
    drives = np.array([p.drives * (1.0 + rng.uniform(-0.1, 0.1)) for _ in range(E)]) if route == "hamiltonians" else \
        np.array([p.drives] * E)
    drifts = np.array([p.h0 + rng.uniform(-0.2, 0.2) * np.diag(np.linspace(-1, 1, n)) for _ in range(E)]) \
        if route == "drifts" else np.array([p.h0] * E)
    kw = dict(ensemble_initial_states=np.array([q.initial_states for q in members]),
              ensemble_costs=[q.costs(std) for q in members],
              store_tape=tape)
    if route == "drifts":
        kw["ensemble_drifts"] = drifts
    hams = [numpy_hamiltonian(drifts[e], drives[e], cc) for e in range(E)]
    if route == "hamiltonians":
        kw["ensemble_hamiltonians"] = hams
    costs = p.costs(std) + [std.ControlNorm(2, p.M, cost_multiplier=0.01)]
    plan = SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, costs, p.T, p.N, control_eval_count=p.M, control_count=2,
                            complex_controls=cc, magnus_policy=_policy(order), cost_eval_step=ces, **kw)
    err, grads, finals = plan.cost_and_grad(p.controls)
    inter = plan.intermediate_states()
    assert finals.shape == (E, S, n, 1) and inter.shape == (E, p.N, S, n, 1)
    plan.close()
    o_err, o_grad = 0.0, 0.0
    cn = orc.ControlNorm(2, p.M, cost_multiplier=0.01)
    for e in range(E):
        v, g, f = orc.schroedinger_cost_and_grad(p.controls, orc.make_hamiltonian(drifts[e], drives[e], cc),
                                                 members[e].initial_states, members[e].costs(orc) + [cn], p.T, p.N,
                                                 order=order, cost_eval_step=ces)
        o_err, o_grad = o_err + v / E, o_grad + g / E
        assert rel(finals[e], f) < 1e-10, e
    assert abs(err - o_err) <= 1e-10 * abs(o_err) and rel(grads, o_grad) < 1e-10
    for e in sorted({0, E // 2, E - 1}):                          # each member against a plan built from its data
        q = members[e]
        one = SchroedingerPlan(hams[e], q.initial_states, q.costs(std) + [std.ControlNorm(2, p.M, cost_multiplier=0.01)],
                               p.T, p.N, control_eval_count=p.M, control_count=2, complex_controls=cc,
                               magnus_policy=_policy(order), cost_eval_step=ces, store_tape=tape)
        e1, _, f1 = one.cost_and_grad(p.controls)
        assert rel(f1, finals[e]) < 1e-12 and rel(one.intermediate_states(), inter[e]) < 1e-12, e
        one.close()


def test_member_data_with_incoherent_targets():
    """neglect_relative_pahse=True (the incoherent kind) with member targets and step costs, M4 complex controls."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    p = Problem(8, 4, 2, 3, 4, complex_controls=True, F=2, seed=17, cost_eval_step=2, step_target=True, neglect_phase=True)
    E = 4
    members = _member_problems(p, E, seed=2)
    plan = _schroedinger(p, std, ensemble_initial_states=np.array([q.initial_states for q in members]),
                         ensemble_costs=[q.costs(std) for q in members])
    err, grads, finals = plan.cost_and_grad(p.controls)
    plan.close()
    outs = [orc.schroedinger_cost_and_grad(p.controls, orc.make_hamiltonian(p.h0, p.drives, True), q.initial_states,
                                           q.costs(orc), p.T, p.N, order=4, cost_eval_step=2) for q in members]
    assert abs(err - np.mean([o[0] for o in outs])) <= 1e-10 * abs(err)
    assert rel(grads, np.mean([o[1] for o in outs], axis=0)) < 1e-10
    assert rel(finals, np.array([o[2] for o in outs])) < 1e-10


def test_member_sharded_plan_single_rank_group():
    import torch
    import torch.distributed as dist
    import qoc_b200.standard as std
    from qoc_b200.core.sharded import EnsembleShardedPlan
    own_group = not dist.is_initialized()
    if own_group:
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1,
                                device_id=torch.device("cuda", 0))
    try:
        p = Problem(16, 8, 2, 3, 4, complex_controls=True, F=1, seed=9)
        E = 5
        members = _member_problems(p, E, seed=1)
        kw = dict(control_eval_count=p.M, control_count=2, complex_controls=True, magnus_policy=_policy(4),
                  ensemble_drifts=[p.h0] * E, ensemble_initial_states=np.array([q.initial_states for q in members]),
                  ensemble_costs=[q.costs(std) for q in members])
        plan = EnsembleShardedPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, **kw)
        err, grads, finals = plan.cost_and_grad(p.controls)
        plan.close()
        ref = _schroedinger(p, std, **{k: v for k, v in kw.items() if k.startswith("ensemble")})
        r_err, r_grads, r_fin = ref.cost_and_grad(p.controls)
        ref.close()
        assert abs(err - r_err) < 1e-13 and rel(grads, r_grads) < 1e-12 and np.array_equal(finals, r_fin)
    finally:
        if own_group:
            dist.destroy_process_group()


def _band(E):
    """E detunings in [-1, 1]; the members with |delta| <= 0.5 are in the band."""
    det = np.linspace(-1.0, 1.0, E)
    return det, np.abs(det) <= 0.5


def test_grape_band_selective_inversion_matches_oracle_driven_adam():
    """Adam on the E = 8 member mean of a band-selective inversion: in-band detunings target |1>, the others |0>."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    from qoc_b200.core.plan import SchroedingerPlan
    T, N, M, E, k = 6.0, 31, 31, 8, 6
    sx, sz = np.array([[0, 1], [1, 0]], dtype=complex), np.diag([0.5, -0.5]).astype(complex)
    det, band = _band(E)
    drifts = np.array([d * sz for d in det])
    init = np.array([[[1], [0]]], dtype=complex)
    targ = [np.array([[[0], [1]]] if b else [[[1], [0]]], dtype=complex) for b in band]
    plan = SchroedingerPlan(numpy_hamiltonian(0 * sz, sx[None], False), init, [std.TargetStateInfidelity(targ[0])], T, N,
                            control_eval_count=M, control_count=1, ensemble_drifts=drifts,
                            ensemble_costs=[[std.TargetStateInfidelity(t)] for t in targ])
    u0 = 0.25 * np.sin(np.linspace(0, np.pi, M))[:, None]
    o_members = [orc.make_hamiltonian(h, sx[None], False) for h in drifts]
    errors, o_errors = [], []

    def jac(params):
        e, g, _ = plan.cost_and_grad(slap_controls(False, params, (M, 1)))
        errors.append(e)
        return strip_controls(False, g), False

    def o_jac(params):
        u = slap_controls(False, params, (M, 1))
        out = [orc.schroedinger_cost_and_grad(u, h, init, [orc.TargetStateInfidelity(t)], T, N) for h, t in zip(o_members, targ)]
        o_errors.append(sum(o[0] for o in out) / E)
        return strip_controls(False, sum(o[1] for o in out) / E), False
    std.Adam().run(lambda q: (0.0, False), k, strip_controls(False, u0.copy()), jac)
    std.Adam().run(lambda q: (0.0, False), k, strip_controls(False, u0.copy()), o_jac)
    assert len(errors) == k and len(o_errors) == k
    assert np.abs(np.array(errors) - np.array(o_errors)).max() < 1e-10, (errors, o_errors)
    assert errors[-1] < errors[0]
    plan.close()


# --- Lindblad ---------------------------------------------------------------------------------------------------------
class LCase(object):
    """E members with their own initial densities and target / forbidden densities, optionally also their own drifts,
    rates or control operators."""

    def __init__(self, n, D, L, cc, E, also=None, ces=1, seed=0):
        from tests.test_gpu_lindblad_ensemble import _dens, _dissipator
        self.n, self.D, self.cc, self.E, self.K, self.ces, self.also = n, D, cc, E, 2, ces, also
        self.p = p = Problem(n, 3, 2, 1, 2, complex_controls=cc, seed=40 + n + seed, M=5, h0_norm=0.8, drive_norm=0.3)
        rng = np.random.default_rng(7 * n + D + L + seed)
        self.rho0 = np.array([_dens(rng, n, D) for _ in range(E)])
        self.targ = np.array([_dens(rng, n, D) for _ in range(E)])
        self.forb = np.array([[_dens(rng, n, 2) for _ in range(D)] for _ in range(E)])
        self.gam, self.ops = _dissipator(n, L, n + seed)
        det = np.diag(np.linspace(-0.5, 0.5, n)).astype(complex)
        self.drifts = np.array([p.h0 + 0.3 * rng.uniform(-1, 1) * det for _ in range(E)]) if also == "drifts" else \
            np.array([p.h0] * E)
        self.drives = np.array([p.drives * (1 + rng.uniform(-0.1, 0.1)) for _ in range(E)]) if also == "hamiltonians" else \
            np.array([p.drives] * E)
        self.rates = np.array([self.gam * rng.uniform(0.5, 1.5, L) for _ in range(E)]) if also == "rates" and L else None

    def costs(self, mod, e):
        from tests.test_gpu_lindblad_ensemble import _costs
        return _costs(mod, "all", self.targ[e], self.forb[e], self.p.N, self.ces, self.K, self.p.M)

    def lind(self, gam):
        return (lambda t: (gam, self.ops)) if self.ops.shape[0] else None

    def member_costs(self, mod, e):
        return [c for c in self.costs(mod, e) if not isinstance(c, mod.ControlNorm)]

    def plan(self, e=None):
        import qoc_b200.standard as std
        from qoc_b200.core.plan import LindbladPlan
        p = self.p
        kw = dict(control_eval_count=p.M, control_count=self.K, complex_controls=self.cc, cost_eval_step=self.ces)
        if e is None:
            if self.also == "drifts":
                kw["ensemble_drifts"] = self.drifts
            if self.also == "hamiltonians":
                kw["ensemble_hamiltonians"] = [numpy_hamiltonian(self.drifts[m], self.drives[m], self.cc) for m in range(self.E)]
            return LindbladPlan(self.rho0[0], self.costs(std, 0), p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                                lindblad_data=self.lind(self.gam), ensemble_rates=self.rates,
                                ensemble_initial_densities=self.rho0,
                                ensemble_costs=[self.member_costs(std, m) for m in range(self.E)], **kw)
        gam = self.gam if self.rates is None else self.rates[e]
        if self.also == "drifts":                # the ensemble's control operators: those probed from the nominal hamiltonian
            from qoc_b200.core.plan import extract_hamiltonian_structure
            kw["structure"] = (self.drifts[e], extract_hamiltonian_structure(p.hamiltonian_numpy(), self.K, self.cc, p.T)[1])
        return LindbladPlan(self.rho0[e], self.costs(std, e), p.T, p.N,
                            hamiltonian=numpy_hamiltonian(self.drifts[e], self.drives[e], self.cc),
                            lindblad_data=self.lind(gam), **kw)


def _check_members(case, members):
    u = case.p.controls
    ens = case.plan()
    err, grads, finals = ens.cost_and_grad(u)
    costs, mgrads, mstats = ens.member_results()
    dens = ens.intermediate_densities()
    assert abs(err - (np.sum(costs) / case.E)) < 1e-12 * max(1.0, abs(err))
    for e in members:
        one = case.plan(e)
        e1, g1, f1 = one.cost_and_grad(u)
        assert e1 == costs[e] and np.array_equal(g1, mgrads[e]), e
        assert np.array_equal(f1, finals[e]) and np.array_equal(one.intermediate_densities(), dens[e]), e
        assert one.stats() == mstats[e], e
        one.close()
    ens.close()


@pytest.mark.parametrize("n,D,L,cc,E,also,ces", [
    (2, 1, 1, True, 5, None, 1),             # 32 threads
    (2, 2, 0, False, 300, None, 2),          # E = 300
    (3, 2, 2, False, 4, "drifts", 1),
    (3, 1, 2, True, 3, "rates", 2),
    (8, 1, 1, False, 3, "hamiltonians", 1),  # 32 threads
    (8, 2, 2, True, 5, "rates", 1),          # 128 threads
    (16, 1, 1, True, 3, "drifts", 2),        # 256 threads
    (16, 2, 2, False, 2, "hamiltonians", 1),
    (32, 1, 1, False, 2, None, 1),           # global-memory working set
])
def test_lindblad_members_match_single_plans(n, D, L, cc, E, also, ces):
    case = LCase(n, D, L, cc, E, also, ces)
    _check_members(case, sorted({0, 1, E // 2, E - 1}))


@pytest.mark.parametrize("n,D,L,cc,E,also", [
    (2, 1, 1, True, 4, "rates"),
    (3, 2, 2, False, 3, None),
    (8, 1, 1, True, 2, "hamiltonians"),
])
def test_lindblad_mean_matches_oracle(n, D, L, cc, E, also):
    from oracle import qoc_oracle as orc
    case = LCase(n, D, L, cc, E, also)
    p, u = case.p, case.p.controls
    ens = case.plan()
    err, grads, finals = ens.cost_and_grad(u)
    ens.close()
    o_err, o_grad, o_fin = 0.0, 0.0, []
    for e in range(E):
        gam = case.gam if case.rates is None else case.rates[e]
        old = orc.make_lindblad_data(gam, case.ops) if L else None
        oe, og, of = orc.lindblad_cost_and_grad(u, orc.make_hamiltonian(case.drifts[e], case.drives[e], cc), old, case.rho0[e],
                                                case.costs(orc, e), p.T, p.N, freeze_steps=True)
        o_err, o_grad = o_err + oe / E, o_grad + og / E
        o_fin.append(of)
    assert abs(err - o_err) < 1e-9, (err, o_err)
    assert rel(finals, np.array(o_fin)) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)


def test_lindblad_identical_member_data_is_bit_identical():
    import qoc_b200.standard as std
    from tests.test_gpu_lindblad_ensemble import Case, _costs
    case = Case(8, 2, 2, True, 1, 4, "all")
    u = case.p.controls
    shared = case.plan()
    forced = case.plan(ensemble_initial_densities=np.array([case.rho0] * 4),
                       ensemble_costs=[[c for c in _costs(std, "all", case.targ, case.forb, case.p.N, 1, case.K, case.p.M)
                                        if not isinstance(c, std.ControlNorm)] for _ in range(4)])
    ra, rb = shared.cost_and_grad(u), forced.cost_and_grad(u)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert np.array_equal(shared.intermediate_densities(), forced.intermediate_densities())
    for x, y in zip(shared.member_results(), forced.member_results()):
        assert np.array_equal(np.asarray(x), np.asarray(y)) if not isinstance(x, list) else x == y
    shared.close(); forced.close()


def test_lindblad_member_data_with_time_dependent_hamiltonian():
    """member densities and targets on a hamiltonian that reads `time` (Chebyshev series): each member bit-identical to its
    one-member plan."""
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    from tests.test_gpu_lindblad_ensemble import _dens
    rng = np.random.default_rng(8)
    n, E, N, T = 3, 3, 4, 1.0
    h0 = np.diag([0.0, 0.4, 0.9]).astype(complex)
    x = np.eye(n, k=1, dtype=complex) + np.eye(n, k=-1, dtype=complex)
    ham = lambda u, t: h0 + np.cos(1.3 * t) * u[0] * x
    rho0, targ = np.array([_dens(rng, n, 1) for _ in range(E)]), np.array([_dens(rng, n, 1) for _ in range(E)])
    u = rng.standard_normal((5, 1)) * 0.5
    kw = dict(hamiltonian=ham, control_eval_count=5, control_count=1)
    ens = LindbladPlan(rho0[0], [std.TargetDensityInfidelity(targ[0])], T, N, ensemble_initial_densities=rho0,
                       ensemble_costs=[[std.TargetDensityInfidelity(t)] for t in targ], **kw)
    err, grads, finals = ens.cost_and_grad(u)
    costs, mgrads, _ = ens.member_results()
    ens.close()
    for e in range(E):
        one = LindbladPlan(rho0[e], [std.TargetDensityInfidelity(targ[e])], T, N, **kw)
        e1, g1, f1 = one.cost_and_grad(u)
        assert e1 == costs[e] and np.array_equal(g1, mgrads[e]) and np.array_equal(f1, finals[e]), e
        one.close()


def test_lindblad_band_selective_inversion_with_t1_matches_oracle_driven_adam():
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    from qoc_b200.core.plan import LindbladPlan
    T, N, M, E, k = 4.0, 9, 9, 8, 6
    sx, sz = np.array([[0, 1], [1, 0]], dtype=complex), np.diag([0.5, -0.5]).astype(complex)
    det, band = _band(E)
    drifts = np.array([d * sz for d in det])
    lower = np.array([[0, 1], [0, 0]], dtype=complex)
    gam = np.array([0.02])
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    targ = [np.array([[[0, 0], [0, 1]]] if b else [[[1, 0], [0, 0]]], dtype=complex) for b in band]
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ[0])], T, N, hamiltonian=numpy_hamiltonian(0 * sz, sx[None], False),
                        lindblad_data=lambda t: (gam, lower[None]), control_eval_count=M, control_count=1,
                        ensemble_drifts=drifts, ensemble_costs=[[std.TargetDensityInfidelity(t)] for t in targ])
    u0 = 0.3 * np.sin(np.linspace(0, np.pi, M))[:, None]
    old = orc.make_lindblad_data(gam, lower[None])
    o_members = [orc.make_hamiltonian(h, sx[None], False) for h in drifts]
    errors, o_errors = [], []

    def jac(params):
        e, g, _ = plan.cost_and_grad(slap_controls(False, params, (M, 1)))
        errors.append(e)
        return strip_controls(False, g), False

    def o_jac(params):
        u = slap_controls(False, params, (M, 1))
        out = [orc.lindblad_cost_and_grad(u, h, old, rho0, [orc.TargetDensityInfidelity(t)], T, N, freeze_steps=True)
               for h, t in zip(o_members, targ)]
        o_errors.append(sum(o[0] for o in out) / E)
        return strip_controls(False, sum(o[1] for o in out) / E), False
    std.Adam().run(lambda q: (0.0, False), k, strip_controls(False, u0.copy()), jac)
    std.Adam().run(lambda q: (0.0, False), k, strip_controls(False, u0.copy()), o_jac)
    assert len(errors) == k and len(o_errors) == k
    assert np.abs(np.array(errors) - np.array(o_errors)).max() < 1e-9, (errors, o_errors)
    assert errors[-1] < errors[0]
    plan.close()
