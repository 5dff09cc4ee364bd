"""GPU: control batches (`SchroedingerPlan(control_batch=B)`, qocb_set_control_batch) and the multi-start driver
`grape_schroedinger_discrete_batch`.

Pins: every start equals a one-member plan given that start's controls (cost and final states 1e-12 relative, gradient
1e-12), over n, B, S (Krylov and dense reverse passes), every Magnus form, real and complex controls, coherent / incoherent /
forbid costs with step costs, ControlNorm and the recompute tape; each start matches the oracle within 1e-10; B = 1 is
bit-identical to an ordinary plan; identical controls give bit-identical starts; a lossy hamiltonian takes the pivoted LU;
the driver follows B separate `grape_schroedinger_discrete` runs."""
import numpy as np
import pytest

from tests.problems import Problem

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300)


def _policy(order):
    from qoc_b200.models import MagnusPolicy
    return {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}[order]


def _costs(p, mod, control_norm):
    costs = p.costs(mod)
    if control_norm:
        costs.append(mod.ControlNorm(p.K, p.M, cost_multiplier=0.13, max_control_norms=np.full(p.K, 2.0)))
    return costs


def _plan(p, control_norm=False, **kw):
    import qoc_b200.standard as std
    from qoc_b200.core.plan import SchroedingerPlan
    return SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, _costs(p, std, control_norm), p.T, p.N,
                            control_eval_count=p.M, control_count=p.K, complex_controls=p.complex_controls,
                            magnus_policy=_policy(p.order), cost_eval_step=p.cost_eval_step, **kw)


def _batch_controls(p, B, seed):
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((B, p.M, p.K)) * 0.5
    if p.complex_controls:
        u = (u + 1j * rng.standard_normal((B, p.M, p.K)) * 0.5) / np.sqrt(2)
    return u


# n, B, S, K, order, complex, step costs (cost_eval_step 2), forbidden states, incoherent target, ControlNorm, store_tape
GRID = [
    (2, 150, 1, 2, 2, False, False, 0, False, False, True),
    (2, 7, 4, 1, 6, True, True, 0, True, True, True),
    (5, 7, 5, 2, 4, True, True, 0, False, True, True),            # M4 product-free, KR = 4
    (5, 2, 1, 1, 2, False, True, 1, True, False, False),
    (16, 2, 4, 4, 4, True, True, 1, False, False, True),          # M4 with explicit commutators, KR = 8
    (16, 150, 1, 2, 4, False, False, 1, True, True, True),
    (32, 7, 4, 2, 6, False, True, 1, False, True, False),
    (32, 2, 5, 3, 2, True, False, 1, True, False, True),
    (60, 2, 5, 2, 4, False, True, 1, False, True, True),          # S = 5: dense reverse pass
    (64, 2, 4, 1, 4, True, False, 1, True, False, True),          # Krylov reverse pass
    (64, 7, 1, 3, 6, False, True, 1, False, True, False),
    (64, 2, 5, 4, 4, True, False, 1, False, True, True),          # KR = 8 at n = 64
]
IDS = ["n{}-B{}-S{}-K{}-M{}{}{}".format(g[0], g[1], g[2], g[3], g[4], "c" if g[5] else "r", "-step" if g[6] else "")
       for g in GRID]


@pytest.mark.parametrize("n,B,S,K,order,cc,step,F,incoherent,cnorm,tape", GRID, ids=IDS)
def test_every_start_matches_a_one_member_plan(n, B, S, K, order, cc, step, F, incoherent, cnorm, tape):
    p = Problem(n, 9, K, S, order, complex_controls=cc, F=F if S < n else 0, seed=7 * n + B, M=6,
                cost_eval_step=2 if step else 1, step_target=step, neglect_phase=incoherent)
    u = _batch_controls(p, B, seed=n + S)
    batch = _plan(p, cnorm, store_tape=tape, control_batch=B)
    errs, grads, finals = batch.cost_and_grad(u)
    states = batch.intermediate_states()
    errs_f, finals_f = batch.cost(u)
    assert errs.shape == (B,) and grads.shape == (B, p.M, K) and finals.shape == (B, S, n, 1)
    assert states.shape == (B, p.N, S, n, 1)
    assert grads.dtype == (np.complex128 if cc else np.float64)
    assert np.array_equal(errs, errs_f) and np.array_equal(finals, finals_f)
    one = _plan(p, cnorm, store_tape=tape)
    for b in range(B):
        e1, g1, f1 = one.cost_and_grad(u[b])
        assert abs(errs[b] - e1) <= 1e-12 * abs(e1), (b, errs[b], e1)
        assert rel(grads[b], g1) < 1e-12, b
        assert rel(finals[b], f1) < 1e-12, b
        if b in (0, B - 1):
            assert rel(states[b], one.intermediate_states()) < 1e-12, b
    one.close(); batch.close()


@pytest.mark.parametrize("n,B,S,K,order,cc,step,cnorm", [
    (2, 7, 1, 2, 2, True, True, True),
    (5, 7, 4, 2, 4, False, True, False),
    (16, 2, 4, 4, 4, True, False, True),
    (32, 2, 1, 1, 6, False, True, True),
])
def test_starts_match_the_oracle(n, B, S, K, order, cc, step, cnorm):
    from oracle import qoc_oracle as orc
    p = Problem(n, 6, K, S, order, complex_controls=cc, F=1 if S < n else 0, seed=n + 100, M=5,
                cost_eval_step=2 if step else 1, step_target=step)
    u = _batch_controls(p, B, seed=n)
    plan = _plan(p, cnorm, control_batch=B)
    errs, grads, finals = plan.cost_and_grad(u)
    plan.close()
    o_errs, o_grads = [], []
    for b in range(B):
        v, g, f = orc.schroedinger_cost_and_grad(u[b], orc.make_hamiltonian(p.h0, p.drives, cc), p.initial_states,
                                                 _costs(p, orc, cnorm), p.T, p.N, order=order,
                                                 cost_eval_step=p.cost_eval_step)
        o_errs.append(v); o_grads.append(g)
        assert abs(errs[b] - v) <= 1e-10 * abs(v) and rel(grads[b], g) < 1e-10 and rel(finals[b], f) < 1e-10, b
    assert abs(errs.mean() - np.mean(o_errs)) <= 1e-10 * abs(np.mean(o_errs))
    assert rel(grads.mean(axis=0), np.mean(o_grads, axis=0)) < 1e-10


@pytest.mark.parametrize("n,S,K,order,cc,step,tape", [
    (2, 1, 2, 2, False, False, True),
    (16, 4, 2, 4, True, True, True),
    (16, 2, 4, 4, True, False, False),
    (64, 2, 2, 4, False, False, True),          # streaming Magnus adjoint and Krylov reverse pass
    (64, 5, 1, 6, True, True, True),
])
def test_batch_of_one_is_bit_identical(n, S, K, order, cc, step, tape):
    p = Problem(n, 12, K, S, order, complex_controls=cc, F=1 if S < n else 0, seed=n + K, M=7,
                cost_eval_step=2 if step else 1, step_target=step)
    ordinary, batch = _plan(p, True, store_tape=tape), _plan(p, True, store_tape=tape, control_batch=1)
    assert ordinary.launch_count() == batch.launch_count()
    for trial in range(3):                                        # plain launches, then the captured graph
        u = _batch_controls(p, 1, seed=trial)
        e0, g0, f0 = ordinary.cost_and_grad(u[0])
        s0 = ordinary.intermediate_states()
        e1, g1, f1 = batch.cost_and_grad(u)
        s1 = batch.intermediate_states()
        assert e1[0] == e0 and np.array_equal(g1[0], g0) and np.array_equal(f1[0], f0) and np.array_equal(s1[0], s0)
        c0, fc0 = ordinary.cost(u[0])
        c1, fc1 = batch.cost(u)
        assert c1[0] == c0 and np.array_equal(fc1[0], fc0)
    ordinary.close(); batch.close()


@pytest.mark.parametrize("n,B,order,cc", [(16, 7, 4, True), (64, 3, 6, False), (5, 150, 2, False)])
def test_identical_controls_give_identical_starts(n, B, order, cc):
    p = Problem(n, 10, 2, 2, order, complex_controls=cc, F=1, seed=n, M=6, cost_eval_step=2, step_target=True)
    u = np.repeat(_batch_controls(p, 1, seed=3), B, axis=0)
    plan = _plan(p, control_batch=B)
    errs, grads, finals = plan.cost_and_grad(u)
    states = plan.intermediate_states()
    plan.close()
    for b in range(1, B):
        assert errs[b] == errs[0] and np.array_equal(grads[b], grads[0]) and np.array_equal(finals[b], finals[0])
        assert np.array_equal(states[b], states[0])


def test_lossy_hamiltonian_takes_the_pivoted_lu(monkeypatch):
    """a non-Hermitian drive: the pivot-free LU is off, so QOCB_NO_NOPIV=1 changes no bit; every start still matches its
    one-member plan."""
    p = Problem(16, 8, 2, 2, 4, F=1, seed=5, M=5)
    p.drives = p.drives.copy()
    p.drives[0] = p.drives[0] - 0.05j * np.diag(np.linspace(0, 1, 16))
    u = _batch_controls(p, 7, seed=1)
    runs = []
    for env in (None, "1"):
        with monkeypatch.context() as m:
            if env:
                m.setenv("QOCB_NO_NOPIV", env)
            plan = _plan(p, control_batch=7)
        runs.append(plan.cost_and_grad(u))
        plan.close()
    for x, y in zip(runs[0], runs[1]):
        assert np.array_equal(x, y)
    one = _plan(p)
    for b in range(7):
        e1, g1, f1 = one.cost_and_grad(u[b])
        assert abs(runs[0][0][b] - e1) <= 1e-12 * abs(e1) and rel(runs[0][1][b], g1) < 1e-12 and rel(runs[0][2][b], f1) < 1e-12
    one.close()


@pytest.mark.parametrize("cc,adam_kw,norms,stop", [
    (False, dict(), None, False),
    (True, dict(scale_grads=0.5, clip_grads=0.02), None, False),
    (False, dict(clip_grads=0.05), 0.45, False),
    (True, dict(), 0.4, False),
    (False, dict(), None, True),
], ids=["plain", "scale-clip", "norm-clip", "complex-norm-clip", "min-error"])
def test_multistart_adam_follows_separate_runs(cc, adam_kw, norms, stop):
    import qoc_b200 as qoc
    import qoc_b200.standard as std
    p = Problem(4, 8, 2, 2, 4, complex_controls=cc, F=1, seed=21, M=5, h0_norm=0.5, drive_norm=0.6)
    B, its = 4, 6
    u = _batch_controls(p, B, seed=9) * 0.6
    mx = None if norms is None else np.full(p.K, norms)
    if mx is not None:                                           # feasible start, clipped on the way
        u = u / np.maximum(1.0, np.abs(u).max(axis=(1, 2), keepdims=True) / norms)
    costs = _costs(p, std, True)
    common = dict(complex_controls=cc, cost_eval_step=1, magnus_policy=_policy(p.order), max_control_norms=mx,
                  log_iteration_step=1000)

    def batch_run(iterations, min_error):
        return qoc.grape_schroedinger_discrete_batch(p.K, p.M, costs, p.T, p.hamiltonian_numpy(), p.initial_states, p.N,
                                                     u, iteration_count=iterations, min_error=min_error,
                                                     optimizer=std.Adam(learning_rate=0.08, **adam_kw), **common)
    # min-error: the lowest error any start reaches within its first 3 updates, so that start stops early
    min_error = min(r.best_error for r in batch_run(4, 0)) if stop else 0
    got = batch_run(its, min_error)
    assert len(got) == B
    for b in range(B):
        ref = qoc.grape_schroedinger_discrete(p.K, p.M, costs, p.T, p.hamiltonian_numpy(), p.initial_states, p.N,
                                              initial_controls=u[b].copy(), iteration_count=its, min_error=min_error,
                                              optimizer=std.Adam(learning_rate=0.08, **adam_kw), **common)
        assert got[b].best_iteration == ref.best_iteration, b
        assert abs(got[b].best_error - ref.best_error) <= 1e-10 * abs(ref.best_error), b
        assert rel(got[b].best_controls, ref.best_controls) < 1e-10, b
        assert rel(got[b].best_final_states, ref.best_final_states) < 1e-10, b
    if stop:
        assert min(r.best_iteration for r in got) < its - 1


def test_single_start_calls_refuse_a_batch():
    """buffer sizes of the [M][KR] calls would be wrong on a batch; the batch calls need a batch; operators and batches are
    set in one order only."""
    from qoc_b200 import _lib
    p = Problem(8, 5, 2, 2, 4, F=1, seed=2, M=4)
    batch, ordinary = _plan(p, control_batch=3), _plan(p)
    lib, x, out = batch.lib, np.zeros((p.M, p.K)), np.zeros(3)
    g, fs = np.zeros((3, p.M, p.K)), np.zeros((3, p.S, p.n), dtype=complex)
    for rc in (lib.qocb_cost(batch.handle, _lib.ptr(x), _lib.ptr(out), None),
               lib.qocb_cost_and_grad(batch.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(x), None),
               lib.qocb_forward(batch.handle, _lib.ptr(x), _lib.ptr(out), None),
               lib.qocb_backward(batch.handle, None, _lib.ptr(x))):
        assert rc == -1 and b"qocb_batch_cost" in lib.qocb_last_error(batch.handle)
    a_ops = np.ascontiguousarray(np.broadcast_to(batch.structure[1], (3,) + batch.structure[1].shape))
    assert lib.qocb_set_member_operators(batch.handle, _lib.ptr(a_ops)) == -1
    assert lib.qocb_set_control_batch(ordinary.handle) == -1 and b"before" in lib.qocb_last_error(ordinary.handle)
    u = np.ascontiguousarray(_batch_controls(p, 3, seed=0))
    assert lib.qocb_batch_cost(ordinary.handle, _lib.ptr(u), _lib.ptr(out), None) == -1
    assert lib.qocb_batch_cost_and_grad(ordinary.handle, _lib.ptr(u), _lib.ptr(out), _lib.ptr(g), _lib.ptr(fs)) == -1
    errs, _, _ = batch.cost_and_grad(u)                          # the refusals left the batch plan usable
    assert np.isfinite(errs).all()
    batch.close(); ordinary.close()
