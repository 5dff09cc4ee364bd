"""GPU parity on Pade denominators that need row interchanges and on non-Hermitian Hamiltonians (tests/pivot_problems.py).

The random problems of the other modules never make partial pivoting swap a row, and every one of them is Hermitian, so
the row bookkeeping of the pivoted LU, the permutations on the tapes, the transposed solves of the reverse passes and
the general (non-Hermitian) kernel path were never compared with a reference.  Oracle: oracle/qoc_oracle.py at 1e-10
relative (cost, final states, gradient); per-slice propagators at 1e-12."""
import numpy as np
import pytest

from tests import pivot_problems as pp
from tests.test_gpu_parity import VARIANTS
from tests.test_gpu_sharded import emulate

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _mods():
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import SchroedingerPlan
    from qoc_b200.models import MagnusPolicy
    return std, orc, SchroedingerPlan, {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}


def _kw(p, pol, **extra):
    kw = dict(control_eval_count=p.M, control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order],
              cost_eval_step=p.cost_eval_step)
    kw.update(extra)
    return kw


_ORACLE = {}


def _oracle(p, key=None):
    """(cost, grad, final states) of the oracle; cached per case (the GPU modes share it)."""
    if key is not None and key in _ORACLE:
        return _ORACLE[key]
    _, orc, _, _ = _mods()
    out = orc.schroedinger_cost_and_grad(p.controls, p.hamiltonian_torch(), p.initial_states, p.costs(orc), p.T, p.N,
                                         order=p.order, cost_eval_step=p.cost_eval_step)
    if key is not None:
        _ORACLE[key] = out
    return out


def _plan(p, env=None, monkeypatch=None, **extra):
    std, _, Plan, pol = _mods()
    if env:
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            return Plan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, **_kw(p, pol, **extra))
    return Plan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, **_kw(p, pol, **extra))


def _run(p, env=None, monkeypatch=None, **extra):
    plan = _plan(p, env, monkeypatch, **extra)
    err, grads, finals = plan.cost_and_grad(p.controls)
    err_f, finals_f = plan.cost(p.controls)
    plan.close()
    return err, grads, finals, err_f, finals_f


def _assert_oracle(got, want, label=""):
    err, grads, finals, err_f, finals_f = got
    o_err, o_grad, o_fin = want
    assert abs(err - o_err) <= RTOL * max(abs(o_err), 1e-3), (label, err, o_err)
    assert abs(err_f - o_err) <= RTOL * max(abs(o_err), 1e-3), (label, err_f, o_err)
    assert rel(finals, o_fin) < RTOL and rel(finals_f, o_fin) < RTOL, (label, rel(finals, o_fin), rel(finals_f, o_fin))
    assert grads.shape == np.shape(o_grad) and rel(grads, o_grad) < RTOL, (label, rel(grads, o_grad))


# --- 1. per-slice forward: localises a forward fault to a slice and an LU bracket ---------------------------------------
@pytest.mark.parametrize("case", pp.PER_SLICE, ids=lambda c: "%s_n%d" % (c[0], c[1]))
def test_propagators_per_slice(case):
    import torch
    _, orc, _, _ = _mods()
    family, n, slices, K, S, order = case
    p = pp.make(family, n, slices, K=K, S=S, order=order, seed=n)
    plan = _plan(p)
    plan.cost_and_grad(p.controls)
    U = plan.propagators()
    plan.close()
    bad = []
    for j, a in enumerate(p.magnus_matrices()):
        want = orc.expm_pade(torch.as_tensor(a)).numpy()
        e = rel(U[j], want)
        if not e < 1e-12:
            norm, s, q = pp.scaled_denominator(a)
            bad.append((j, pp.bracket(norm), s, pp.row_swaps(q), e))
    assert not bad, bad


# --- 2. evaluation matrix: H, N, L x Magnus order x state count x cost kind x tape mode ------------------------------------
@pytest.mark.parametrize("mode", ["tape", "recompute", "onechunk"])
@pytest.mark.parametrize("case", pp.EVAL_CASES, ids=pp.case_id)
def test_eval_vs_oracle(case, mode):
    p = pp.from_case(case)
    extra = dict(store_tape=mode != "recompute")
    if mode == "onechunk":
        extra["chunks_per_member"] = 1
    _assert_oracle(_run(p, **extra), _oracle(p, case), pp.case_id(case))


# --- 3. three levels, chunk boundaries and every A/B switch on swap data ---------------------------------------------------
@pytest.mark.parametrize("case", pp.THREE_LEVEL, ids=["final_cost", "step_costs"])
def test_three_level_and_switches(case, monkeypatch):
    """310 slices at n = 64 take the three-level boundary scheme; every A/B switch must reproduce the default, the
    default the oracle"""
    p = pp.from_case(case)
    base = _run(p)
    _assert_oracle(base, _oracle(p))
    e0, g0, f0 = base[:3]
    for env in VARIANTS + [{"QOCB_NO_COMM": "1"}]:
        e1, g1, f1 = _run(p, env, monkeypatch)[:3]
        assert abs(e1 - e0) <= 1e-10 * max(abs(e0), 1e-3), env
        assert rel(f1, f0) < 1e-10 and rel(g1, g0) < 1e-10, (env, rel(f1, f0), rel(g1, g0))
        if env == {"QOCB_NO_NOPIV": "1"}:        # the default ran the Hermitian fast path (pivot-free LU, half products)
            assert not np.array_equal(g1, g0)


def test_full_length_swap_pulse():
    """n = 64, 2000 slices: swap slices in every chunk, tape formats (Krylov / full) mixed inside chunks"""
    p = pp.from_case(pp.FULL_LENGTH)
    _assert_oracle(_run(p), _oracle(p))


# --- 4. path proof on non-Hermitian data ------------------------------------------------------------------------------
NONHERM = [c for c in pp.EVAL_CASES if c[0] in ("N", "L") and c[1] in (16, 64)]


@pytest.mark.parametrize("case", NONHERM, ids=pp.case_id)
def test_nonhermitian_ignores_nopiv_switch(case, monkeypatch):
    """QOCB_NO_NOPIV=1 only clears the Hermitian flag: on non-Hermitian operators the results are bit-identical"""
    p = pp.from_case(case)
    a = _run(p)
    b = _run(p, {"QOCB_NO_NOPIV": "1"}, monkeypatch)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("n", pp.EDGE_NS)
@pytest.mark.parametrize("edge", pp.EDGES, ids=["below_rule", "above_rule"])
def test_hermitian_classification_edge(n, edge, monkeypatch):
    p = pp.edge_problem(n, edge)
    a = _run(p)
    _assert_oracle(a, _oracle(p))               # below the rule: the Hermitian fast path on a nearly Hermitian drift
    b = _run(p, {"QOCB_NO_NOPIV": "1"}, monkeypatch)
    if edge > 1e-13:                            # above the rule: the general path already
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    else:                                       # below it: the fast path ran (results differ in rounding only)
        assert abs(a[0] - b[0]) <= 1e-12 * max(abs(a[0]), 1e-3) and rel(a[1], b[1]) < 1e-10
        assert not np.array_equal(a[1], b[1])


def test_ensemble_with_one_nonhermitian_member(monkeypatch):
    std, orc, Plan, pol = _mods()
    p = pp.from_case(pp.ENSEMBLE)
    E = 4
    z = np.diag(np.linspace(-1, 1, 16)).astype(complex) * 0.05
    drifts = np.stack([p.h0 + d * z for d in np.random.default_rng(2).normal(0, 1.0, E)])
    drifts[2] = drifts[2] - 0.5j * np.diag(np.linspace(0.0, 0.05, 16))
    assert [pp.is_hermitian(d) for d in drifts] == [True, True, False, True]
    runs = []
    for env in (None, {"QOCB_NO_NOPIV": "1"}):
        plan = _plan(p, env, monkeypatch, ensemble_drifts=drifts)
        runs.append(plan.cost_and_grad(p.controls))
        plan.close()
    err, grads, finals = runs[0]
    assert err == runs[1][0] and np.array_equal(grads, runs[1][1]) and np.array_equal(finals, runs[1][2])
    o_err, o_grad = 0.0, 0.0
    for e in range(E):
        v, g, f = orc.schroedinger_cost_and_grad(p.controls, p.hamiltonian_torch(drifts[e]), p.initial_states, p.costs(orc),
                                                 p.T, p.N, order=4)
        o_err, o_grad = o_err + v / E, o_grad + g / E
        assert rel(finals[e], f) < RTOL
    assert abs(err - o_err) <= RTOL * abs(o_err) and rel(grads, o_grad) < RTOL


# --- 5. large-dimension path ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", pp.LARGE_CASES + pp.LARGE_OWN_LU, ids=pp.case_id)
def test_large_dim_vs_oracle(case, monkeypatch):
    """N: cuBLAS getrf / getrs with row swaps of Q^T.  H: a slice at or above 2.5 moves the whole plan to getrf / getrs,
    so the result is bit-identical to QOCB_LARGE_CUBLAS_LU=1.  HS: every slice below 2.5, the own block LU stays in use
    (pivots inside its diagonal blocks) and must agree with getrf / getrs without being bit-identical to it."""
    p = pp.from_case(case)
    plan = _plan(p)
    err, grads, finals = plan.cost_and_grad(p.controls)
    err_f, finals_f = plan.cost(p.controls)
    U = plan.propagators()
    plan.close()
    _assert_oracle((err, grads, finals, err_f, finals_f), _oracle(p), pp.case_id(case))
    if p.family in ("H", "HS"):
        assert np.abs(U @ U.conj().transpose(0, 2, 1) - np.eye(p.n)).max() < 1e-11
        e1, g1, f1 = _run(p, {"QOCB_LARGE_CUBLAS_LU": "1"}, monkeypatch)[:3]
        assert abs(e1 - err) <= 1e-12 * max(abs(err), 1e-3) and rel(f1, finals) < 1e-11 and rel(g1, grads) < 1e-10
        if p.family == "H":
            assert e1 == err and np.array_equal(g1, grads) and np.array_equal(f1, finals)
        else:
            assert not np.array_equal(g1, grads)


# --- 6. sharded engines on swap data ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,world", pp.TIME_SHARDED, ids=lambda c: pp.case_id(c) if isinstance(c, tuple) else "w%d" % c)
def test_time_sharded(case, world):
    std, orc, _, pol = _mods()
    from qoc_b200.core.sharded import CudaShardEngine
    p = pp.from_case(case)
    engines = [CudaShardEngine(r, world, p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, **_kw(p, pol))
               for r in range(world)]
    cost, g, finals = emulate(engines, p.controls, True)
    cost0, _, finals0 = emulate(engines, p.controls, False)
    for e in engines:
        e.close()
    o_err, o_grad, o_fin = _oracle(p)
    assert abs(cost - o_err) <= RTOL * abs(o_err) and abs(cost0 - o_err) <= RTOL * abs(o_err)
    assert rel(g, o_grad) < RTOL and rel(finals, o_fin) < RTOL and rel(finals0, o_fin) < RTOL


@pytest.mark.parametrize("case", pp.STATE_SHARDED, ids=pp.case_id)
def test_state_sharded_coherent(case):
    std, orc, Plan, pol = _mods()
    from qoc_b200.core.sharded import CudaStateEngine, slice_bounds
    from tests.test_gpu_units import _emulate_state_shards
    p = pp.from_case(case)
    costs = p.costs(std) + [std.TargetStateInfidelity(p.target_states, cost_multiplier=0.3)]
    ocosts = p.costs(orc) + [orc.TargetStateInfidelity(p.target_states, cost_multiplier=0.3)]
    world = 3
    b = slice_bounds(p.S, world)
    plans = [Plan(p.hamiltonian_numpy(), p.initial_states, costs, p.T, p.N, state_slice=(b[g], b[g + 1]), **_kw(p, pol))
             for g in range(world)]
    engines = [CudaStateEngine(pl, 0) for pl in plans]
    res = _emulate_state_shards(engines, p.controls, True)
    res0 = _emulate_state_shards(engines, p.controls, False)
    finals = np.concatenate([pl.final_states() for pl in plans])
    for e, pl in zip(engines, plans):
        e.close()
        pl.close()
    g = res[:-1].reshape(p.M, -1)
    grads = g[:, :p.K] + 1j * g[:, p.K:] if p.complex_controls else g
    o_err, o_grad, o_fin = orc.schroedinger_cost_and_grad(p.controls, p.hamiltonian_torch(), p.initial_states, ocosts, p.T, p.N,
                                                          order=4, cost_eval_step=p.cost_eval_step)
    assert abs(res[-1] - o_err) <= RTOL * abs(o_err) and abs(res0[-1] - o_err) <= RTOL * abs(o_err)
    assert rel(grads, o_grad) < RTOL and rel(finals, o_fin) < RTOL


# --- 7. time-dependent and non-linear callables -----------------------------------------------------------------------
def _loss_callables(p, nonlinear):
    """family L operators in a rotating frame: H(u, t) = H0 - i Gamma/2 + u e^{i w t} C + conj(u e^{i w t}) C'
    (time-dependent, affine); nonlinear: H0 - i Gamma/2 + x0^2 C_h + sin(x1 + w t) E with C_h = C + C', E = C - C'."""
    import math
    import torch
    w = 0.23
    h0, c, cp = p.h0, p.ops[0], p.partners[0]
    ch, en = c + cp, c - cp
    cdt = torch.complex128
    th0, tc, tcp, tch, ten = (torch.as_tensor(m, dtype=cdt) for m in (h0, c, cp, ch, en))
    if nonlinear:
        def h_np(u, t):
            return h0 + u[0] ** 2 * ch + np.sin(u[1] + w * t) * en

        def h_t(u, t):
            return th0 + u[0] ** 2 * tch + torch.sin(u[1] + w * float(t)) * ten
    else:
        def h_np(u, t):
            ph = np.exp(1j * w * t)
            return h0 + u[0] * ph * c + np.conjugate(u[0] * ph) * cp

        def h_t(u, t):
            ph = complex(math.cos(w * float(t)), math.sin(w * float(t)))
            return th0 + u[0] * ph * tc + torch.conj(u[0] * ph) * tcp
    return h_np, h_t


def test_time_dependent_loss_callable():
    std, orc, Plan, pol = _mods()
    p = pp.make("L", 12, 30, K=1, S=3, order=4, F=2, cost_eval_step=4, step_target=True, seed=31)
    h_np, h_t = _loss_callables(p, False)
    plan = Plan(h_np, p.initial_states, p.costs(std), p.T, p.N, **_kw(p, pol))
    assert len(plan.structure) == 4
    err, grads, finals = plan.cost_and_grad(p.controls)
    err_f, finals_f = plan.cost(p.controls)
    plan.close()
    want = orc.schroedinger_cost_and_grad(p.controls, h_t, p.initial_states, p.costs(orc), p.T, p.N, order=4, cost_eval_step=4)
    _assert_oracle((err, grads, finals, err_f, finals_f), want)


def test_nonlinear_loss_callable():
    std, orc, _, pol = _mods()
    from qoc_b200.core.plan import NonlinearSchroedingerPlan, make_schroedinger_plan
    q = pp.make("L", 8, 20, K=1, S=2, order=4, F=2, cost_eval_step=3, step_target=True, seed=41)
    h_np, h_t = _loss_callables(q, True)
    rng = np.random.default_rng(5)
    controls = 0.6 * rng.standard_normal((q.M, 2))
    kw = dict(control_eval_count=q.M, control_count=2, complex_controls=False, magnus_policy=pol[4], cost_eval_step=3)
    plan = make_schroedinger_plan(h_np, q.initial_states, q.costs(std), q.T, q.N, **kw)
    assert isinstance(plan, NonlinearSchroedingerPlan)
    err, grads, finals = plan.cost_and_grad(controls)
    plan.close()
    o_err, o_grad, o_fin = orc.schroedinger_cost_and_grad(controls, h_t, q.initial_states, q.costs(orc), q.T, q.N, order=4,
                                                          cost_eval_step=3)
    assert abs(err - o_err) <= RTOL * abs(o_err) and rel(finals, o_fin) < RTOL
    assert rel(grads, o_grad) < 1e-8, rel(grads, o_grad)


# --- 8. standalone hooks on slice matrices with real permutations -------------------------------------------------------
@pytest.mark.parametrize("n", pp.EXPM_NS)
def test_standalone_expm_and_vjp(n):
    import torch
    _, orc, _, _ = _mods()
    from qoc_b200.standard.functions import expm, expm_vjp
    a = pp.expm_stack(n)
    rng = np.random.default_rng(n)
    ubar = rng.standard_normal(a.shape) + 1j * rng.standard_normal(a.shape)
    got = expm(a)
    out, abar = expm_vjp(a, ubar)
    for b in range(a.shape[0]):
        at = torch.tensor(a[b], requires_grad=True)
        u = orc.expm_pade(at)
        torch.sum(torch.as_tensor(ubar[b]) * u).real.backward()
        want = u.detach().numpy()
        assert rel(got[b], want) < 1e-12 and rel(out[b], want) < 1e-12, (b, rel(got[b], want), rel(out[b], want))
        assert rel(abar[b], np.conj(at.grad.numpy())) < 1e-11, (b, rel(abar[b], np.conj(at.grad.numpy())))


# --- 9. properties independent of the oracle ------------------------------------------------------------------------
def test_loss_norms_non_increasing():
    p = pp.make("L", 16, 400, K=2, S=3, order=2, seed=5)
    plan = _plan(p)
    plan.cost_and_grad(p.controls)
    nr = np.linalg.norm(plan.intermediate_states()[..., 0], axis=-1)
    plan.close()
    assert np.all(np.diff(nr, axis=0) < 0) and nr[-1].min() > np.exp(-1.6)


@pytest.mark.parametrize("case", pp.FD_CASES, ids=pp.case_id)
def test_gradient_vs_central_difference(case):
    p = pp.from_case(case)
    plan = _plan(p)
    err, grads, _ = plan.cost_and_grad(p.controls)
    rng = np.random.default_rng(1)
    v = rng.standard_normal(p.controls.shape) * np.abs(p.controls).max()
    if p.complex_controls:
        v = v + 1j * rng.standard_normal(p.controls.shape) * np.abs(p.controls).max()
    eps = 1e-6
    ep, _ = plan.cost(p.controls + eps * v)
    em, _ = plan.cost(p.controls - eps * v)
    plan.close()
    fd = (ep - em) / (2 * eps)
    dd = np.sum(grads.real * v.real + grads.imag * v.imag)
    assert abs(fd - dd) < 1e-6 * max(1.0, abs(fd)), (fd, dd)
