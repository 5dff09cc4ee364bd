"""CPU: members with their own initial states / densities and cost targets (`ensemble_initial_states`,
`ensemble_initial_densities`, `ensemble_costs`) on `SchroedingerPlan`, `LindbladPlan` and `EnsembleShardedPlan`: every refusal
is raised before any device call, member cost lists must repeat the term structure of `costs`, the member vector and matrix
tables hold the oracle's targets, the four C-ABI calls are bound, and a world-size-2 gloo run of the units protocol slices
the member data as `EnsembleShardedPlan` does."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import qoc_b200.standard as std
from qoc_b200 import _lib
from qoc_b200.core.plan import LindbladPlan, SchroedingerPlan, member_cost_terms, is_user_cost
from qoc_b200.core.sharded import EnsembleShardedPlan, TorchDistComm, member_share, units_evaluate
from qoc_b200.models.cost import Cost

N_, M_, T_ = 5, 5, 1.0
SX = np.array([[0, 1], [1, 0]], dtype=complex)
SZ = np.diag([1.0, -1.0]).astype(complex)
KET = [np.array([[1.0], [0.0]], dtype=complex), np.array([[0.0], [1.0]], dtype=complex)]
H = lambda u, t: 0.5 * SZ + u[0] * SX


def _cuda():
    return torch.cuda.is_available()


class PurityPenalty(Cost):
    requires_step_evaluation = False

    def cost(self, controls, states, step):
        return float(np.abs(states[0, 0, 0]) ** 2)


def _targets(E):
    """member e targets |1> for even e, |0> otherwise (one state)"""
    return [[std.TargetStateInfidelity(KET[1 - e % 2][None])] for e in range(E)]


def _schroedinger(E=3, hamiltonian=H, costs=None, n=2, **kw):
    init = np.zeros((1, n, 1), dtype=complex)
    init[0, 0, 0] = 1.0
    kw.setdefault("ensemble_costs", _targets(E) if n == 2 else None)
    costs = [std.TargetStateInfidelity(init)] if costs is None else costs
    return SchroedingerPlan(hamiltonian, init, costs, T_, N_, control_eval_count=M_, control_count=1, **kw)


def _dens(k):
    return (KET[k] @ KET[k].conj().T)[None]


def _lindblad(E=3, hamiltonian=H, costs=None, lindblad_data=None, **kw):
    kw.setdefault("ensemble_costs", [[std.TargetDensityInfidelity(_dens(e % 2))] for e in range(E)])
    a = np.array([[0, 1], [0, 0]], dtype=complex)
    lind = (lambda t: (np.array([0.05]), a[None])) if lindblad_data is None else lindblad_data
    costs = [std.TargetDensityInfidelity(_dens(1))] if costs is None else costs
    return LindbladPlan(_dens(0), costs, T_, N_, hamiltonian=hamiltonian, lindblad_data=lind, control_eval_count=M_,
                        control_count=1, **kw)


# --- refusals before any device call ----------------------------------------------------------------------------------
@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_control_batch_refused(make):
    with pytest.raises(NotImplementedError, match="control batches cannot be combined with ensemble_initial"):
        make(control_batch=2)


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_user_cost_in_member_list_refused(make):
    base = _targets(3) if make is _schroedinger else [[std.TargetDensityInfidelity(_dens(1))]] * 3
    with pytest.raises(NotImplementedError, match="user-defined"):
        make(ensemble_costs=[base[0], base[1] + [PurityPenalty()], base[2]])


@pytest.mark.parametrize("make", [_schroedinger, _lindblad], ids=["schroedinger", "lindblad"])
def test_user_cost_in_costs_refused(make):
    costs = ([std.TargetStateInfidelity(KET[1][None]), PurityPenalty()] if make is _schroedinger else
             [std.TargetDensityInfidelity(_dens(1)), PurityPenalty()])
    with pytest.raises(NotImplementedError, match="user-defined"):
        make(costs=costs)


def test_time_dependent_schroedinger_refused():
    with pytest.raises(NotImplementedError, match="time-dependent"):
        _schroedinger(hamiltonian=lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX)


def test_nonlinear_schroedinger_refused_without_rerouting():
    with pytest.raises(NotImplementedError, match="affine") as err:
        _schroedinger(hamiltonian=lambda u, t: 0.5 * SZ + u[0] ** 2 * SX)
    assert type(err.value) is NotImplementedError          # not NonlinearHamiltonian: no silent fall-back to another plan


def test_lindblad_time_dependence_follows_the_ensemble_rules():
    td = lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX
    with pytest.raises(NotImplementedError, match="time-dependent"):
        _lindblad(hamiltonian=td, ensemble_drifts=np.array([0.5 * SZ] * 3))
    with pytest.raises(NotImplementedError, match="time-dependent"):
        _lindblad(ensemble_rates=np.full((3, 1), 0.02),
                  lindblad_data=lambda t: (np.array([0.05 * (1 + 0.5 * np.sin(t))]), np.array([[[0, 1], [0, 0]]], dtype=complex)))


@pytest.mark.parametrize("make, kw", [
    (_schroedinger, dict(ensemble_initial_states=np.array([[KET[0]]] * 2))),
    (_schroedinger, dict(ensemble_drifts=np.array([0.5 * SZ] * 4))),
    (_schroedinger, dict(ensemble_hamiltonians=[H] * 2)),
    (_lindblad, dict(ensemble_initial_densities=np.array([_dens(0)] * 4))),
    (_lindblad, dict(ensemble_rates=np.full((2, 1), 0.02))),
    (_lindblad, dict(ensemble_drifts=np.array([0.5 * SZ] * 2))),
], ids=["s-states", "s-drifts", "s-hamiltonians", "l-densities", "l-rates", "l-drifts"])
def test_member_counts_must_agree(make, kw):
    with pytest.raises(ValueError, match="member count"):
        make(**kw)


@pytest.mark.parametrize("make, kw", [
    (_schroedinger, dict(ensemble_initial_states=np.zeros((3, 2, 2, 1)))),       # another S
    (_schroedinger, dict(ensemble_initial_states=np.zeros((3, 1, 2)))),          # no trailing axis
    (_lindblad, dict(ensemble_initial_densities=np.zeros((3, 2, 2, 2)))),        # another D
], ids=["s-S", "s-ndim", "l-D"])
def test_member_state_shapes(make, kw):
    with pytest.raises(ValueError, match="shape"):
        make(**kw)


def test_large_dimension_refused():
    n = 72
    h = lambda u, t: np.diag(np.linspace(-1, 1, n)).astype(complex) + u[0] * (np.eye(n, k=1) + np.eye(n, k=-1))
    init = np.zeros((3, 1, n, 1), dtype=complex)
    with pytest.raises(NotImplementedError, match="hilbert_size > 64"):
        _schroedinger(hamiltonian=h, n=n, ensemble_initial_states=init)


def test_sharding_refused():
    with pytest.raises(NotImplementedError, match="state sharding"):
        _schroedinger(state_slice=(0, 1))
    with pytest.raises(NotImplementedError, match="time-slice"):
        _schroedinger(slice_range=(0, 2))


# --- term-structure matching ------------------------------------------------------------------------------------------
def _forbid(F, mult=1.0):
    return std.ForbidStates([np.array([KET[k % 2] for k in range(F)])], N_, cost_multiplier=mult)


@pytest.mark.parametrize("member_costs", [
    [std.TargetStateInfidelity(KET[1][None], cost_multiplier=2.0), _forbid(2)],       # multiplier
    [std.TargetStateInfidelity(KET[1][None]), _forbid(3)],                            # forbidden count
    [std.TargetStateInfidelity(KET[1][None], neglect_relative_pahse=True), _forbid(2)],  # kind
    [std.TargetStateInfidelityTime(N_, KET[1][None]), _forbid(2)],                    # step flag and weight
    [std.TargetStateInfidelity(KET[1][None])],                                        # a missing term
    [_forbid(2), std.TargetStateInfidelity(KET[1][None])],                            # another order
    [std.TargetStateInfidelity(KET[1][None]), _forbid(2), std.ControlNorm(1, M_)],    # a control cost
], ids=["multiplier", "forbid-count", "kind", "step", "missing", "order", "control-cost"])
def test_member_lists_must_repeat_the_term_structure(member_costs):
    costs = [std.TargetStateInfidelity(KET[0][None]), _forbid(2), std.ControlNorm(1, M_)]
    good = [std.TargetStateInfidelity(KET[1][None]), _forbid(2)]
    with pytest.raises(ValueError):
        _schroedinger(costs=costs, ensemble_costs=[good, member_costs, good])


def test_density_member_lists_must_repeat_the_term_structure():
    forb = lambda F, m=1.0: std.ForbidDensities([np.array([_dens(0)[0]] * F)], N_, cost_multiplier=m)
    costs = [std.TargetDensityInfidelity(_dens(1)), forb(2)]
    with pytest.raises(ValueError):
        _lindblad(costs=costs, ensemble_costs=[costs, [std.TargetDensityInfidelity(_dens(0)), forb(3)]])
    with pytest.raises(ValueError):
        _lindblad(costs=costs, ensemble_costs=[costs, [std.TargetDensityInfidelity(_dens(0)), forb(2, 0.5)]])


def test_ensemble_costs_must_be_lists():
    with pytest.raises(ValueError):
        _schroedinger(ensemble_costs=[std.TargetStateInfidelity(KET[1][None])] * 3)
    with pytest.raises(ValueError):
        _schroedinger(ensemble_costs=[])


# --- packing of the member tables -------------------------------------------------------------------------------------
def test_member_vectors_hold_the_oracle_targets():
    from oracle import qoc_oracle as orc
    rng = np.random.default_rng(3)
    n, S, E, F = 4, 2, 3, 3

    def ket():
        v = rng.standard_normal((n, 1)) + 1j * rng.standard_normal((n, 1))
        return v / np.linalg.norm(v)
    targ = [np.array([ket() for _ in range(S)]) for _ in range(E)]
    forb = [[np.array([ket() for _ in range(F if s == 0 else 1)]) for s in range(S)] for e in range(E)]   # counts [3, 1]
    lists = [[std.TargetStateInfidelityTime(N_, targ[e], cost_multiplier=0.5), std.ForbidStates(forb[e], N_)]
             for e in range(E)]
    terms = member_cost_terms(lists[0], lists, lambda c: c.device_terms(S, n), is_user_cost)
    assert [t[:3] for t in terms] == [(0, 1, 0.5 / (N_ - 1)), (2, 1, 1.0 / ((N_ - 1) * S))]
    assert terms[0][3].shape == (E, S, 1, n) and terms[1][3].shape == (E, S, F, n)
    assert np.array_equal(terms[1][4], [F, 1])
    for e in range(E):
        o_t = orc.TargetStateInfidelityTime(N_, targ[e])
        assert np.array_equal(terms[0][3][e, :, 0], o_t.target_states_dagger.conj().resolve_conj().numpy()[:, 0, :])
        o_f = orc.ForbidStates(forb[e], N_)
        for s in range(S):
            k = o_f.fdag[s].shape[0]
            assert np.array_equal(terms[1][3][e, s, :k], o_f.fdag[s].conj().resolve_conj().numpy()[:, 0, :])
            assert not terms[1][3][e, s, k:].any()


def test_member_matrices_hold_the_oracle_targets():
    from oracle import qoc_oracle as orc
    rng = np.random.default_rng(4)
    n, D, E = 3, 2, 4
    targ = [rng.standard_normal((D, n, n)) + 1j * rng.standard_normal((D, n, n)) for _ in range(E)]
    lists = [[std.TargetDensityInfidelity(t)] for t in targ]
    terms = member_cost_terms(lists[0], lists, lambda c: c.device_terms_density(D, n), is_user_cost)
    assert len(terms) == 1 and terms[0][3].shape == (E, D, 1, n, n)
    for e in range(E):
        tdag = orc.TargetDensityInfidelity(targ[e]).tdag.resolve_conj().numpy()
        assert np.array_equal(terms[0][3][e, :, 0], np.conj(np.swapaxes(tdag, -1, -2)))


@pytest.mark.skipif(_cuda(), reason="checks that valid member data reaches the device")
@pytest.mark.parametrize("make, kw", [
    (_schroedinger, dict()),
    (_schroedinger, dict(ensemble_initial_states=np.array([[KET[e % 2]] for e in range(3)]))),
    (_schroedinger, dict(ensemble_drifts=np.array([0.5 * SZ] * 3))),
    (_schroedinger, dict(ensemble_hamiltonians=[lambda u, t, s=s: 0.5 * SZ + s * u[0] * SX for s in (0.9, 1.0, 1.1)])),
    (_lindblad, dict()),
    (_lindblad, dict(ensemble_initial_densities=np.array([_dens(e % 2) for e in range(3)]), ensemble_rates=np.full((3, 1), 0.02))),
    (_lindblad, dict(hamiltonian=lambda u, t: 0.5 * SZ + np.cos(t) * u[0] * SX)),
])
def test_valid_member_data_passes_validation(make, kw):
    with pytest.raises(RuntimeError, match="no CUDA device"):
        make(**kw)


# --- the C ABI --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name, args", [
    ("qocb_set_member_states", [ctypes.c_void_p, ctypes.c_void_p]),
    ("qocb_add_member_cost", [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.c_void_p,
                              ctypes.c_void_p, ctypes.c_int32]),
    ("qocb_lindblad_set_member_densities", [ctypes.c_void_p, ctypes.c_void_p]),
    ("qocb_lindblad_add_member_cost", [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_int32]),
])
def test_member_data_calls_are_bound(name, args):
    lib = _lib.load()
    assert name in _lib.EXPORTS
    fn = getattr(lib, name)
    assert fn.argtypes == args
    null = [0 if a in (ctypes.c_int32, ctypes.c_double) else None for a in args]
    assert fn(*null) == -1                               # a null plan is refused without touching a device


@pytest.mark.gpu
def test_c_abi_refuses_member_data_on_control_batches():
    lib = _lib.load()
    s = _schroedinger(ensemble_costs=None, control_batch=2)
    psi = np.zeros((2, 1, 2), dtype=complex)
    assert lib.qocb_set_member_states(s.handle, _lib.ptr(psi)) == -1
    assert lib.qocb_add_member_cost(s.handle, 0, 0, 1.0, _lib.ptr(psi), None, 1) == -1
    s.close()
    lp = _lindblad(ensemble_costs=None, control_batch=2)
    rho = np.zeros((2, 1, 2, 2), dtype=complex)
    mats = np.zeros((2, 1, 1, 2, 2), dtype=complex)
    assert lib.qocb_lindblad_set_member_densities(lp.handle, _lib.ptr(rho)) == -1
    assert lib.qocb_lindblad_add_member_cost(lp.handle, 0, 0, 1.0, _lib.ptr(mats), None, 1) == -1
    lp.close()
    n = 72                                                   # the large path refuses member data
    h = lambda u, t: np.diag(np.linspace(-1, 1, n)).astype(complex) + u[0] * (np.eye(n, k=1) + np.eye(n, k=-1))
    big = _schroedinger(hamiltonian=h, n=n, ensemble_costs=None)
    assert lib.qocb_set_member_states(big.handle, _lib.ptr(np.zeros((1, 1, n), dtype=complex))) == -1
    big.close()


# --- member slicing of EnsembleShardedPlan, world size 2 over gloo ----------------------------------------------------
def test_sharded_plan_needs_one_kind_of_members():
    with pytest.raises(ValueError, match="exactly one"):
        EnsembleShardedPlan(H, np.array([KET[0]]), [], T_, N_, ensemble_costs=_targets(3))


def test_member_share_partitions_every_argument():
    drifts, states, costs = np.arange(5), np.arange(10, 15), list("abcde")
    got = [member_share(r, 2, ensemble_drifts=drifts, ensemble_initial_states=states, ensemble_costs=costs,
                        ensemble_hamiltonians=None) for r in range(2)]
    assert [g[1] for g in got] == [(0, 2), (2, 5)] and all(g[2] == 5 for g in got)
    assert list(got[1][0]["ensemble_initial_states"]) == [12, 13, 14] and got[1][0]["ensemble_costs"] == ["c", "d", "e"]
    assert "ensemble_hamiltonians" not in got[0][0]
    with pytest.raises(ValueError, match="member count"):
        member_share(0, 2, ensemble_drifts=drifts, ensemble_costs=costs[:4])


def _units_problem():
    """E = 5 members: detuned drifts, member initial states and member targets / forbidden states (oracle terms)."""
    from oracle import adjoint_model as am
    from tests.problems import Problem
    p = Problem(4, 7, 2, 2, 4, complex_controls=False, F=2, seed=31, cost_eval_step=1, step_target=True)
    rng = np.random.default_rng(5)
    E, n, S = 5, 4, 2

    def kets(k):
        v = rng.standard_normal((k, n)) + 1j * rng.standard_normal((k, n))
        return v / np.linalg.norm(v, axis=1, keepdims=True)
    drifts = np.array([p.h0 + 0.1 * e * np.diag(np.linspace(-1, 1, n)) for e in range(E)])
    psi0 = np.array([kets(S) for _ in range(E)])
    cnt = p.N - 1
    terms = [[am.CostTerm(0, [kets(1) for _ in range(S)], 1.0, cnt, True),
              am.CostTerm(2, [kets(2), kets(1)], 0.7, cnt * S, True)] for _ in range(E)]
    return p, drifts, p.drives, psi0, terms


class MemberTargetEngine(object):
    """members of this rank (`member_share`) on the NumPy adjoint model, each with its own drift, initial states and cost
    terms; packs [mean gradient | mean cost] weighted by local / total members, as CudaUnitEngine does."""

    def __init__(self, rank, world, x, drifts, a_ops, psi0, terms, T, N, order):
        local, self.span, E = member_share(rank, world, drifts=drifts, psi0=psi0, terms=terms)
        self.weight = (self.span[1] - self.span[0]) / float(E)
        self.local, self.rest = local, (x, a_ops, T, N, order)

    def forward(self, with_grad):
        from oracle import adjoint_model as am
        x, a_ops, T, N, order = self.rest
        outs = [am.cost_and_grad(x, h, a_ops, p0, t, T, N, order)
                for h, p0, t in zip(self.local["drifts"], self.local["psi0"], self.local["terms"])]
        self.cost = np.mean([o[0] for o in outs])
        self.grad = np.mean([o[1] for o in outs], axis=0)
        return None

    def backward(self, coh):
        pass

    def pack(self, with_grad):
        g = self.grad if with_grad else np.zeros_like(self.grad)
        return torch.from_numpy(np.concatenate([g.ravel(), [self.cost]]) * self.weight)


def _units_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        p, drifts, a_ops, psi0, terms = _units_problem()
        eng = MemberTargetEngine(rank, world, p.controls, drifts, a_ops, psi0, terms, p.T, p.N, 4)
        res = units_evaluate(eng, TorchDistComm(), True)
        q.put((rank, eng.span, res.numpy().copy()))
    finally:
        dist.destroy_process_group()


def test_member_targets_units_protocol_gloo():
    from oracle import adjoint_model as am
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_units_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    outs = sorted(q.get(timeout=120) for _ in range(2))
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    p, drifts, a_ops, psi0, terms = _units_problem()
    ref = [am.cost_and_grad(p.controls, drifts[e], a_ops, psi0[e], terms[e], p.T, p.N, 4) for e in range(5)]
    cost, grad = np.mean([r[0] for r in ref]), np.mean([r[1] for r in ref], axis=0)
    assert [o[1] for o in outs] == [(0, 2), (2, 5)]
    for _, _, res in outs:
        assert abs(res[-1] - cost) < 1e-13 * max(1.0, abs(cost))
        assert np.abs(res[:-1].reshape(grad.shape) - grad).max() < 1e-13 * max(1.0, np.abs(grad).max())
    # the members differ: a protocol that dropped the member data would not match
    assert abs(ref[0][0] - ref[1][0]) > 1e-3
