"""GPU: robust-control ensembles whose members differ in their control operators (`ensemble_hamiltonians`: drive-amplitude
and crosstalk errors), Schroedinger and Lindblad paths.

Pins: per-member operators only move pointers (identical copies in every member are bit-identical to shared operators);
the member mean matches the mean of the torch oracle over members, each with its own hamiltonian (Schroedinger 1e-10,
Lindblad on the frozen step grid 1e-9 / 1e-7); every member equals a one-member plan built from its hamiltonian (Schroedinger
1e-12, Lindblad bit for bit); a non-Hermitian member sends the whole plan to the general LU; drift-only members take the
`ensemble_drifts` route bit for bit; member sharding and an Adam trajectory follow the unsharded plan and the oracle."""
import socket

import numpy as np
import pytest

from tests.problems import Problem, numpy_hamiltonian

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _policy(order):
    from qoc_b200.models import MagnusPolicy
    return {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}[order]


def _member_drives(p, E, kind, seed=0):
    """[E][K][n][n]: amplitude (1 + eps_e) D_k with eps in [-0.1, 0.1], or crosstalk: channel 0 of member e also drives
    delta_e D_1."""
    rng = np.random.default_rng(seed)
    out = []
    for e in range(E):
        d = p.drives.copy()
        if kind == "amplitude":
            d = d * (1.0 + rng.uniform(-0.1, 0.1))
        else:
            d[0] = d[0] + rng.uniform(-0.1, 0.1) * d[1]
        out.append(d)
    return np.array(out)


def _schroedinger(p, std, members=None, **kw):
    from qoc_b200.core.plan import SchroedingerPlan
    return SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                            control_count=p.K, complex_controls=p.complex_controls, magnus_policy=_policy(p.order),
                            cost_eval_step=p.cost_eval_step, ensemble_hamiltonians=members, **kw)


def _results(plan, u):
    err, grads, finals = plan.cost_and_grad(u)
    err_f, finals_f = plan.cost(u)
    return err, grads, finals, plan.intermediate_states(), err_f, finals_f


# --- pointer plumbing: identical operators through qocb_set_member_operators -----------------------------------------
@pytest.mark.parametrize("n,K,cc,order,ces,step", [
    (2, 2, False, 2, 1, False),
    (8, 2, True, 4, 1, True),               # M4, KR = 4: product-free with per-member Cs
    (8, 4, True, 4, 2, True),               # M4, KR = 8: explicit commutators
    (32, 2, False, 4, 1, False),
    (32, 1, True, 6, 2, True),
    (64, 2, False, 2, 1, True),
    (64, 3, False, 4, 1, False),
    (64, 1, True, 6, 1, False),
])
def test_identical_member_operators_are_bit_identical(n, K, cc, order, ces, step):
    import qoc_b200.standard as std
    from qoc_b200 import _lib
    p = Problem(n, 6, K, 2, order, complex_controls=cc, F=1, seed=n + K, cost_eval_step=ces, step_target=step)
    E = 3
    z = np.diag(np.linspace(-1, 1, n)).astype(complex) * 0.2
    drifts = np.array([p.h0 + d * z for d in (-1.0, 0.3, 1.0)])
    shared = _schroedinger(p, std, ensemble_drifts=drifts)
    forced = _schroedinger(p, std, ensemble_drifts=drifts)
    a_ops = np.ascontiguousarray(np.broadcast_to(forced.structure[1], (E,) + forced.structure[1].shape))
    _lib.check(forced.lib.qocb_set_member_operators(forced.handle, _lib.ptr(a_ops)), forced.handle)
    ra, rb = _results(shared, p.controls), _results(forced, p.controls)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert shared.launch_count() == forced.launch_count()
    shared.close(); forced.close()


# --- physics against the oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,E,S,order,cc,kind", [
    (2, 64, 1, 2, True, "amplitude"),
    (2, 7, 4, 6, False, "crosstalk"),
    (5, 7, 4, 4, True, "crosstalk"),
    (16, 2, 1, 6, True, "amplitude"),
    (32, 7, 4, 2, False, "amplitude"),
    (60, 2, 4, 4, False, "crosstalk"),
    (64, 2, 1, 4, True, "amplitude"),
    (64, 7, 1, 6, False, "crosstalk"),
])
def test_member_mean_matches_oracle(n, E, S, order, cc, kind):
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import SchroedingerPlan
    p = Problem(n, 4, 2, S, order, complex_controls=cc, F=1 if S < n else 0, seed=3 * n + E)
    drives = _member_drives(p, E, kind, seed=n)
    members = [numpy_hamiltonian(p.h0, d, cc) for d in drives]
    plan = _schroedinger(p, std, members)
    err, grads, finals = plan.cost_and_grad(p.controls)
    assert finals.shape == (E, S, n, 1)
    plan.close()
    o_err, o_grad = 0.0, 0.0
    for e in range(E):
        v, g, f = orc.schroedinger_cost_and_grad(p.controls, orc.make_hamiltonian(p.h0, drives[e], cc), p.initial_states,
                                                 p.costs(orc), p.T, p.N, order=order)
        o_err, o_grad = o_err + v / E, o_grad + g / E
        assert rel(finals[e], f) < 1e-10, e
    assert abs(err - o_err) <= 1e-10 * abs(o_err) and rel(grads, o_grad) < 1e-10
    for e in sorted({0, E // 2, E - 1}):                          # each member against a plan built from its hamiltonian
        one = SchroedingerPlan(members[e], p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M, control_count=2,
                               complex_controls=cc, magnus_policy=_policy(order))
        assert rel(one.cost(p.controls)[1], finals[e]) < 1e-12, e
        one.close()


def test_non_hermitian_member_takes_the_general_path(monkeypatch):
    """member 1's drive carries a loss term: the pivot-free LU must be off for the whole plan, so QOCB_NO_NOPIV=1 changes
    nothing."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    p = Problem(16, 5, 2, 2, 4, seed=11)
    drives = _member_drives(p, 3, "amplitude", seed=2)
    drives[1, 0] = drives[1, 0] - 0.05j * np.diag(np.linspace(0, 1, 16))
    members = [numpy_hamiltonian(p.h0, d, False) for d in drives]
    runs = []
    for env in (None, "1"):
        with monkeypatch.context() as m:
            if env:
                m.setenv("QOCB_NO_NOPIV", env)
            plan = _schroedinger(p, std, members)
        runs.append(plan.cost_and_grad(p.controls))
        plan.close()
    assert runs[0][0] == runs[1][0] and np.array_equal(runs[0][1], runs[1][1]) and np.array_equal(runs[0][2], runs[1][2])
    o_err, o_grad = 0.0, 0.0
    for e in range(3):
        v, g, f = orc.schroedinger_cost_and_grad(p.controls, orc.make_hamiltonian(p.h0, drives[e], False), p.initial_states,
                                                 p.costs(orc), p.T, p.N, order=4)
        o_err, o_grad = o_err + v / 3, o_grad + g / 3
        assert rel(runs[0][2][e], f) < 1e-10
    assert abs(runs[0][0] - o_err) <= 1e-10 * abs(o_err) and rel(runs[0][1], o_grad) < 1e-10


@pytest.mark.parametrize("order,cc", [(2, False), (4, True), (6, False)])
def test_drift_only_members_take_the_drift_route(order, cc):
    """a diagonal drift and drives without a diagonal make the probed operators exact (H(e_k) - H(0) rounds otherwise), so
    every member's operators equal member 0's bit for bit and the plan takes the `ensemble_drifts` route."""
    import qoc_b200.standard as std
    from qoc_b200.core.plan import ensemble_member_structures
    p = Problem(8, 6, 2, 2, order, complex_controls=cc, seed=5)
    p.h0 = np.diag(np.diag(p.h0))
    p.drives = p.drives - np.array([np.diag(np.diag(d)) for d in p.drives])
    z = np.diag(np.linspace(-1, 1, 8)).astype(complex) * 0.2
    drifts = np.array([p.h0 + d * z for d in (-1.0, -0.2, 0.5, 1.0)])
    members = [numpy_hamiltonian(h, p.drives, cc) for h in drifts]
    assert ensemble_member_structures(members, 8, 2, cc, p.T)[1].ndim == 3
    a = _schroedinger(p, std, members)
    b = _schroedinger(p, std, ensemble_drifts=drifts)
    for x, y in zip(_results(a, p.controls), _results(b, p.controls)):
        assert np.array_equal(x, y)
    assert a.launch_count() == b.launch_count() and a.launch_count(False) == b.launch_count(False)
    a.close(); b.close()


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
        members = [numpy_hamiltonian(p.h0, d, True) for d in _member_drives(p, 5, "amplitude", seed=4)]
        kw = dict(control_eval_count=p.M, control_count=2, complex_controls=True, magnus_policy=_policy(4))
        plan = EnsembleShardedPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N,
                                   ensemble_hamiltonians=members, **kw)
        err, grads, finals = plan.cost_and_grad(p.controls)
        plan.close()
        ref = _schroedinger(p, std, members)
        r_err, r_grads, r_fin = ref.cost_and_grad(p.controls)
        ref.close()
        assert abs(err - r_err) < 1e-13 and rel(grads, r_grads) < 1e-12 and np.array_equal(finals, r_fin)
    finally:
        if own_group:
            dist.destroy_process_group()


def test_grape_amplitude_robust_pi_pulse_matches_oracle_driven_adam():
    """Adam on the E = 8 member mean of a pi pulse whose drive amplitude is off by up to +-10 %, against the same optimiser
    fed by the oracle."""
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.common import slap_controls, strip_controls
    from qoc_b200.core.plan import SchroedingerPlan
    n, T, N, M, E, k = 2, 4.0, 21, 21, 8, 5
    sx = np.array([[0, 1], [1, 0]], dtype=complex)
    h0 = np.diag([0.0, 0.05]).astype(complex)
    scale = np.linspace(0.9, 1.1, E)
    members = [numpy_hamiltonian(h0, s * sx[None], False) for s in scale]
    init = np.array([[[1], [0]]], dtype=complex)
    targ = np.array([[[0], [1]]], dtype=complex)
    plan = SchroedingerPlan(members[E // 2], init, [std.TargetStateInfidelity(targ)], T, N, control_eval_count=M,
                            control_count=1, ensemble_hamiltonians=members)
    u0 = 0.3 * np.ones((M, 1))
    o_members = [orc.make_hamiltonian(h0, s * sx[None], False) for s in scale]
    errors, o_errors = [], []

    def jac(params):
        e, g, _ = plan.cost_and_grad(slap_controls(False, params, (M, 1)))
        errors.append(e)
        return strip_controls(False, g), False

    def o_jac(params):
        u = slap_controls(False, params, (M, 1))
        out = [orc.schroedinger_cost_and_grad(u, h, init, [orc.TargetStateInfidelity(targ)], T, N) for h in o_members]
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
    """E members with amplitude or crosstalk spreads of the control operators, optionally with their own rates."""

    def __init__(self, n, D, L, cc, E, kind, rates, seed=0):
        from tests.test_gpu_lindblad_ensemble import _dens, _dissipator
        self.n, self.cc, self.E, self.K = n, cc, E, 2
        self.p = p = Problem(n, 3, 2, 1, 2, complex_controls=cc, seed=90 + n + seed, M=5, h0_norm=0.8, drive_norm=0.3)
        rng = np.random.default_rng(10 * n + D + L + seed)
        self.rho0, self.targ = _dens(rng, n, D), _dens(rng, n, D)
        self.forb = np.array([_dens(rng, n, 2) for _ in range(D)])
        self.gam, self.ops = _dissipator(n, L, n + seed)
        self.drives = _member_drives(p, E, kind, seed=n + seed)
        self.members = [numpy_hamiltonian(p.h0, d, cc) for d in self.drives]
        self.rates = np.array([self.gam * rng.uniform(0.5, 1.5, L) for _ in range(E)]) if rates and L else None

    def costs(self, mod):
        from tests.test_gpu_lindblad_ensemble import _costs
        return _costs(mod, "all", self.targ, self.forb, self.p.N, 1, self.K, self.p.M)

    def lind(self, gam):
        return (lambda t: (gam, self.ops)) if self.ops.shape[0] else None

    def plan(self, e=None):
        import qoc_b200.standard as std
        from qoc_b200.core.plan import LindbladPlan
        p = self.p
        kw = dict(control_eval_count=p.M, control_count=self.K, complex_controls=self.cc)
        if e is None:
            return LindbladPlan(self.rho0, self.costs(std), p.T, p.N, hamiltonian=p.hamiltonian_numpy(),
                                lindblad_data=self.lind(self.gam), ensemble_hamiltonians=self.members,
                                ensemble_rates=self.rates, **kw)
        gam = self.gam if self.rates is None else self.rates[e]
        return LindbladPlan(self.rho0, self.costs(std), p.T, p.N, hamiltonian=self.members[e], lindblad_data=self.lind(gam), **kw)


@pytest.mark.parametrize("n,D,L,cc,E,kind,rates", [
    (2, 1, 1, True, 5, "amplitude", True),
    (2, 2, 0, False, 3, "crosstalk", False),
    (3, 2, 2, False, 4, "amplitude", False),
    (3, 1, 2, True, 3, "crosstalk", True),
    (8, 2, 2, True, 5, "crosstalk", True),
    (8, 1, 0, False, 2, "amplitude", False),
    (16, 1, 1, True, 3, "amplitude", True),
    (16, 2, 2, False, 2, "crosstalk", False),
])
def test_lindblad_members_match_single_plans(n, D, L, cc, E, kind, rates):
    case = LCase(n, D, L, cc, E, kind, rates)
    u = case.p.controls
    ens = case.plan()
    assert ens._members[2].shape == (E, case.K * (2 if cc else 1), n, n)        # per-member operators
    err, grads, finals = ens.cost_and_grad(u)
    costs, mgrads, mstats = ens.member_results()
    dens = ens.intermediate_densities()
    for e in range(E):
        one = case.plan(e)
        e1, g1, f1 = one.cost_and_grad(u)
        assert e1 == costs[e] and np.array_equal(g1, mgrads[e]), e
        assert np.array_equal(f1, finals[e]) and np.array_equal(one.intermediate_densities(), dens[e]), e
        assert one.stats() == mstats[e], e
        one.close()
    ens.close()


@pytest.mark.parametrize("n,D,L,cc,E,kind,rates", [
    (2, 1, 1, True, 4, "amplitude", True),
    (3, 2, 2, False, 3, "crosstalk", False),
    (8, 1, 1, True, 2, "crosstalk", True),
])
def test_lindblad_mean_matches_oracle(n, D, L, cc, E, kind, rates):
    from oracle import qoc_oracle as orc
    case = LCase(n, D, L, cc, E, kind, rates)
    p, u = case.p, case.p.controls
    ens = case.plan()
    err, grads, finals = ens.cost_and_grad(u)
    ens.close()
    o_err, o_grad, o_fin = 0.0, 0.0, []
    for e in range(E):
        gam = case.gam if case.rates is None else case.rates[e]
        old = orc.make_lindblad_data(gam, case.ops) if L else None
        oe, og, of = orc.lindblad_cost_and_grad(u, orc.make_hamiltonian(p.h0, case.drives[e], cc), old, case.rho0,
                                                case.costs(orc), p.T, p.N, freeze_steps=True)
        o_err, o_grad = o_err + oe / E, o_grad + og / E
        o_fin.append(of)
    assert abs(err - o_err) < 1e-9, (err, o_err)
    assert rel(finals, np.array(o_fin)) < 1e-9
    assert rel(grads, o_grad) < 1e-7, rel(grads, o_grad)


def test_lindblad_identical_member_operators_are_bit_identical():
    from qoc_b200 import _lib
    from tests.test_gpu_lindblad_ensemble import Case
    case = Case(8, 2, 2, True, 1, 4, "all")
    u = case.p.controls
    shared, forced = case.plan(), case.plan()
    a_ops = np.ascontiguousarray(np.broadcast_to(case.a_ops, (4,) + case.a_ops.shape))
    forced._check(forced.lib.qocb_lindblad_set_member_operators(forced.handle, _lib.ptr(a_ops)))
    ra, rb = shared.cost_and_grad(u), forced.cost_and_grad(u)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert np.array_equal(shared.intermediate_densities(), forced.intermediate_densities())
    shared.close(); forced.close()
