"""GPU: Lindblad control batches (`LindbladPlan(control_batch=B)`): B independent control sets of one problem, one CTA per
start in one launch of each kernel, for multi-start GRAPE (`grape_lindblad_discrete_batch`).

Pins: every start is bit-identical to a one-member plan given that start's controls (cost, final densities, densities at
every step, gradient, stats), on every launch layout (32, 128 and 256 threads, shared and global working sets), for
time-independent and time-dependent problems; B = 1 is the ordinary plan; starts against the torch oracle with the step
grid frozen under the contract of include/qocb200.h (cost and densities 1e-9, gradient 1e-7); the multi-start driver
follows separate `grape_lindblad_discrete` runs."""
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


def _lindblad_pair(kind, n, L, seed):
    """(numpy callable, torch callable) of a dissipator family: rate: modulated rates; phase: operators rotating in phase
    (with a growing modulus); both."""
    import torch
    rng = np.random.default_rng(seed)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(complex)
    ops = np.array([a, rand_herm(rng, n) * 0.5, a.T.copy()][:L]).reshape(L, n, n)
    g0 = np.linspace(0.08, 0.03, L)

    def ld(t):
        t = float(t)
        g, o = g0.copy(), ops.copy()
        if kind in ("rate", "both"):
            g = g * (1.0 + 0.5 * np.sin(0.9 * t + np.arange(L)))
        if kind in ("phase", "both"):
            o[0] = np.exp(1j * 1.7 * t) * (1.0 + 0.05 * t) * o[0]
        return g, o
    return ld, (lambda t: tuple(torch.as_tensor(x) for x in ld(t)))


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


def _starts(u, B, seed):
    """B seeded starts around the pulse u: a +-30 % scale and an added 10 % of noise per entry, so step counts differ."""
    rng = np.random.default_rng(seed)
    scale = np.abs(u).max()
    noise = rng.uniform(-1, 1, (B,) + u.shape)
    if np.iscomplexobj(u):
        noise = noise + 1j * rng.uniform(-1, 1, (B,) + u.shape)
    return u[None] * rng.uniform(0.7, 1.3, (B, 1, 1)) + 0.1 * scale * noise


class Case(object):
    """a seeded time-independent problem (or, td=True, its time-dependent twin) with B starts."""

    def __init__(self, n, D, L, cc, ces, kind, slices=3, seed=0, td=False):
        from qoc_b200.core.plan import extract_hamiltonian_structure
        self.K, self.cc, self.ces, self.kind, self.td = 2, cc, ces, kind, td
        self.p = p = Problem(n, slices, self.K, 1, 2, complex_controls=cc, seed=70 + n + seed, M=5, h0_norm=0.8,
                             drive_norm=0.3)
        rng = np.random.default_rng(100 * n + 10 * D + L + seed)
        self.rho0, self.targ = _dens(rng, n, D), _dens(rng, n, D)
        self.forb = np.array([_dens(rng, n, 2) for _ in range(D)])
        self.gam, self.ops = _dissipator(n, L, n + seed)
        self.structure = None if td else extract_hamiltonian_structure(p.hamiltonian_numpy(), self.K, cc, p.T)
        self.ld = self.old = None
        if td and L:
            self.ld, self.old = _lindblad_pair("both", n, L, n + seed)
        elif L:
            self.ld = lambda t: (self.gam, self.ops)

    def plan(self, B=None, **kw):
        import qoc_b200.standard as std
        from qoc_b200.core.plan import LindbladPlan
        p = self.p
        return LindbladPlan(self.rho0, _costs(std, self.kind, self.targ, self.forb, p.N, self.ces, self.K, p.M), p.T, p.N,
                            hamiltonian=p.hamiltonian_td_numpy() if self.td else p.hamiltonian_numpy(),
                            lindblad_data=self.ld, control_eval_count=p.M, control_count=self.K, complex_controls=self.cc,
                            cost_eval_step=self.ces, structure=self.structure, control_batch=B, **kw)


def _check_starts(case, B, starts, seed=1):
    u = _starts(case.p.controls, B, seed)
    bp = case.plan(B)
    errs, grads, finals = bp.cost_and_grad(u)
    costs, mgrads, mstats = bp.member_results()
    dens = bp.intermediate_densities()
    N, D, n = case.p.N, case.rho0.shape[0], case.rho0.shape[1]
    assert errs.shape == (B,) and finals.shape == (B, D, n, n) and dens.shape == (B, N, D, n, n)
    assert grads.shape == u.shape and grads.dtype == u.dtype and mgrads.dtype == u.dtype
    assert np.array_equal(costs, errs) and np.array_equal(mgrads, grads)
    assert bp.stats() == {"attempts": sum(s["attempts"] for s in mstats), "accepted": sum(s["accepted"] for s in mstats)}
    if B > 2:                                                    # the starts' step sequences really differ
        assert len({(s["attempts"], s["accepted"]) for s in mstats}) > 1, mstats
    exact = case.kind != "all"                  # ControlNorm is added on the host: 1e-14 relative
    for b in starts:
        one = case.plan()
        e1, g1, f1 = one.cost_and_grad(u[b])
        if exact:
            assert e1 == errs[b] and np.array_equal(g1, grads[b]), b
        else:
            assert abs(e1 - errs[b]) <= 1e-14 * abs(e1) and rel(grads[b], g1) <= 1e-14, b
        assert np.array_equal(f1, finals[b]) and np.array_equal(one.intermediate_densities(), dens[b]), b
        assert one.stats() == mstats[b], b
        assert one.range_extensions == bp.range_extensions == 0
        one.close()
    errs_c, finals_c = bp.cost(u)                                # the forward pass without its tape
    assert np.array_equal(errs_c, errs) and np.array_equal(finals_c, finals)
    bp.close()


def _sample(B, k=6, seed=0):
    return range(B) if B <= 7 else sorted({0, B - 1} | set(np.random.default_rng(seed).choice(B, k, replace=False).tolist()))


@pytest.mark.parametrize("n,D,L,cc,ces,B,kind", [
    (2, 1, 1, True, 1, 7, "all"),            # 32 threads
    (2, 2, 2, False, 2, 150, "forbid"),
    (3, 2, 0, False, 2, 7, "target"),
    (3, 1, 1, True, 1, 2, "all"),
    (8, 2, 2, True, 1, 7, "all"),            # 128 threads
    (8, 1, 1, False, 2, 150, "target"),      # 32 threads
    (16, 1, 2, True, 1, 7, "forbid"),        # 128 threads
    (16, 2, 1, False, 2, 2, "all"),          # 256 threads
])
def test_starts_match_single_plans(n, D, L, cc, ces, B, kind):
    _check_starts(Case(n, D, L, cc, ces, kind), B, _sample(B))


def test_global_memory_working_set():
    """n = 32, D = 1: the working sets of both kernels exceed shared memory and live in each start's global slice."""
    _check_starts(Case(32, 1, 1, True, 1, "target", slices=2), 3, range(3))


def test_more_starts_than_sms():
    """B = 640 at n = 2: more than four starts per SM, a seeded sample against single plans."""
    _check_starts(Case(2, 1, 1, True, 1, "all"), 640, _sample(640, k=5, seed=3))


def test_one_start_is_the_ordinary_plan():
    case = Case(3, 2, 1, True, 1, "all")
    u = case.p.controls
    bp, one = case.plan(1), case.plan()
    e, g, f = bp.cost_and_grad(u[None])
    e1, g1, f1 = one.cost_and_grad(u)
    assert e.shape == (1,) and e[0] == e1 and np.array_equal(g[0], g1) and np.array_equal(f[0], f1)
    assert np.array_equal(bp.intermediate_densities()[0], one.intermediate_densities())
    assert bp.stats() == one.stats()
    bp.close(); one.close()


def test_identical_controls_give_identical_starts():
    case = Case(8, 2, 2, True, 1, "all")
    B = 5
    u = np.ascontiguousarray(np.broadcast_to(case.p.controls, (B,) + case.p.controls.shape))
    bp = case.plan(B)
    errs, grads, finals = bp.cost_and_grad(u)
    dens = bp.intermediate_densities()
    _, _, stats = bp.member_results()
    for b in range(1, B):
        assert errs[b] == errs[0] and np.array_equal(grads[b], grads[0]) and np.array_equal(finals[b], finals[0])
        assert np.array_equal(dens[b], dens[0]) and stats[b] == stats[0]
    bp.close()


@pytest.mark.parametrize("n,D,L,cc,ces,B", [(2, 1, 1, True, 1, 4), (3, 2, 2, False, 2, 3)])
def test_starts_match_oracle(n, D, L, cc, ces, B):
    from oracle import qoc_oracle as orc
    case = Case(n, D, L, cc, ces, "all")
    p = case.p
    u = _starts(p.controls, B, 5)
    bp = case.plan(B)
    errs, grads, finals = bp.cost_and_grad(u)
    for b in range(B):
        oe, og, of = orc.lindblad_cost_and_grad(u[b], orc.make_hamiltonian(case.structure[0], p.drives, cc),
                                                orc.make_lindblad_data(case.gam, case.ops), case.rho0,
                                                _costs(orc, "all", case.targ, case.forb, p.N, ces, case.K, p.M), p.T, p.N,
                                                cost_eval_step=ces, freeze_steps=True)
        assert abs(errs[b] - oe) < 1e-9, (b, errs[b], oe)
        assert rel(finals[b], of) < 1e-9, b
        assert rel(grads[b], og) < 1e-7, (b, rel(grads[b], og))
    bp.close()


# --- time dependence ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,D,L,cc,ces,B", [(2, 1, 1, True, 1, 5), (3, 2, 2, False, 2, 4), (8, 1, 1, True, 1, 3)])
def test_timedep_starts_match_single_plans(n, D, L, cc, ces, B):
    """a hamiltonian reading `time` and a lindblad_data varying with time: the Chebyshev table is shared and every start
    forms its channel coefficients from its own controls, so every start is still bit-identical to a one-member plan."""
    case = Case(n, D, L, cc, ces, "forbid", td=True)
    bp = case.plan(B)
    assert bp.series is not None and bp.series.KC >= 1 and bp.series.L == L
    bp.close()
    _check_starts(case, B, range(B))


def test_timedep_batch_extends_the_table_and_matches_oracle():
    """weak dynamics take stage times far beyond T + dt: the table is extended to the largest stage time over the starts,
    and every start keeps the Lindblad bars against the oracle."""
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
    rho0 = np.array([[[1, 0], [0, 0]]], dtype=complex)
    targ = np.array([[[0.5, 0.5], [0.5, 0.5]]], dtype=complex)
    u = np.array([[[0.3], [-0.2], [0.5], [0.1]], [[0.1], [0.4], [-0.3], [0.2]], [[-0.5], [0.2], [0.1], [0.6]]])
    plan = LindbladPlan(rho0, [std.TargetDensityInfidelity(targ)], T, N, hamiltonian=h,
                        lindblad_data=lambda t: (np.array([3e-4]), sm[None]), control_eval_count=M, control_count=1,
                        control_batch=3)
    errs, grads, finals = plan.cost_and_grad(u)
    assert plan.range_extensions >= 1
    for b in range(3):
        oe, og, of = orc.lindblad_cost_and_grad(u[b], oh, orc.make_lindblad_data(np.array([3e-4]), sm[None]), rho0,
                                                [orc.TargetDensityInfidelity(targ)], T, N, freeze_steps=True)
        assert abs(errs[b] - oe) < 1e-9 and rel(finals[b], of) < 1e-9, b
        assert rel(grads[b], og) < 1e-7, (b, rel(grads[b], og))
    plan.close()


# --- the C ABI's refusals -----------------------------------------------------------------------------------------------
def test_c_abi_refusals():
    from qoc_b200 import _lib
    case = Case(2, 1, 1, True, 1, "target")
    batch, ordinary = case.plan(3), case.plan()
    lib, M, K = batch.lib, case.p.M, case.K
    x, out = np.zeros((M, 2 * K)), np.zeros(3)
    g, fd = np.zeros((3, M, 2 * K)), np.zeros((3, 1, 2, 2), dtype=complex)
    for rc in (lib.qocb_lindblad_cost(batch.handle, _lib.ptr(x), _lib.ptr(out), None),
               lib.qocb_lindblad_cost_and_grad(batch.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(x), None),
               lib.qocb_lindblad_forward(batch.handle, _lib.ptr(x), _lib.ptr(out), None),
               lib.qocb_lindblad_backward(batch.handle, None, _lib.ptr(x))):
        assert rc == -1 and b"qocb_lindblad_batch_cost" in lib.qocb_lindblad_last_error(batch.handle)
    assert lib.qocb_lindblad_set_ensemble(batch.handle, None, None) == -1
    a_ops = np.ascontiguousarray(np.broadcast_to(batch._setup["a_ops"], (3,) + batch._setup["a_ops"].shape))
    assert lib.qocb_lindblad_set_member_operators(batch.handle, _lib.ptr(a_ops)) == -1
    assert lib.qocb_lindblad_set_control_batch(ordinary.handle) == -1
    assert b"before" in lib.qocb_lindblad_last_error(ordinary.handle)
    u = np.ascontiguousarray(batch._batch_channels(_starts(case.p.controls, 3, 0)))
    assert lib.qocb_lindblad_batch_cost(ordinary.handle, _lib.ptr(u), _lib.ptr(out), None) == -1
    assert lib.qocb_lindblad_batch_cost_and_grad(ordinary.handle, _lib.ptr(u), _lib.ptr(out), _lib.ptr(g), _lib.ptr(fd)) == -1
    # plans without controls have nothing to batch
    import ctypes
    for have_h, KR, M_ in ((0, 0, 0), (1, 0, 0)):
        pb = _lib.LindbladProblem(hilbert_size=2, density_count=1, control_count=KR, control_eval_count=M_,
                                  system_eval_count=3, cost_eval_step=1, lindblad_count=1, have_hamiltonian=have_h,
                                  device=0, max_rk_steps=0, channel_count=0, time_dependent_rates=0, ensemble_count=3,
                                  evolution_time=1.0)
        h = ctypes.c_void_p()
        assert lib.qocb_lindblad_create(ctypes.byref(pb), ctypes.byref(h)) == 0
        assert lib.qocb_lindblad_set_control_batch(h) == -1 and b"needs controls" in lib.qocb_lindblad_last_error(h)
        lib.qocb_lindblad_destroy(h)
    errs, _, _ = batch.cost_and_grad(_starts(case.p.controls, 3, 0))   # the refusals left the batch plan usable
    assert np.isfinite(errs).all()
    batch.close(); ordinary.close()


# --- GRAPE ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cc,opt,norms,stop", [
    (True, dict(), None, False),
    (False, dict(scale_grads=0.5, clip_grads=0.02), None, False),
    (True, dict(clip_grads=0.05), 0.3, False),
    (False, "sgd", 0.3, False),
    (True, dict(), None, True),
], ids=["adam", "scale-clip", "norm-clip", "sgd-norm-clip", "min-error"])
def test_multistart_follows_separate_runs(cc, opt, norms, stop):
    import qoc_b200 as qoc
    import qoc_b200.standard as std
    case = Case(2, 1, 1, cc, 1, "target")
    p = case.p
    B, its = 4, 6
    u = _starts(p.controls, B, 9) * 0.6
    mx = None if norms is None else np.full(p.K, norms)
    if mx is not None:                                           # feasible start, clipped on the way
        u = u / np.maximum(1.0, np.abs(u).max(axis=(1, 2), keepdims=True) / norms)
    costs = _costs(std, "target", case.targ, case.forb, p.N, 1, p.K, p.M)
    make_opt = (lambda: std.SGD(learning_rate=0.5)) if opt == "sgd" else (lambda: std.Adam(learning_rate=0.08, **opt))
    common = dict(complex_controls=cc, hamiltonian=p.hamiltonian_numpy(), lindblad_data=case.ld, max_control_norms=mx,
                  log_iteration_step=1000)

    def batch_run(iterations, min_error):
        return qoc.grape_lindblad_discrete_batch(p.K, p.M, costs, p.T, case.rho0, p.N, u, iteration_count=iterations,
                                                 min_error=min_error, optimizer=make_opt(), **common)
    # min-error: the lowest error any start reaches within its first 3 updates, so that start stops early
    min_error = min(r.best_error for r in batch_run(4, 0)) if stop else 0
    got = batch_run(its, min_error)
    assert len(got) == B
    for b in range(B):
        ref = qoc.grape_lindblad_discrete(p.K, p.M, costs, p.T, case.rho0, p.N, initial_controls=u[b].copy(),
                                          iteration_count=its, min_error=min_error, optimizer=make_opt(), **common)
        assert got[b].best_iteration == ref.best_iteration, b
        assert abs(got[b].best_error - ref.best_error) <= 1e-9, b
        assert rel(got[b].best_controls, ref.best_controls) < 1e-9, b
        assert rel(got[b].best_final_densities, ref.best_final_densities) < 1e-9, b
    if stop:
        assert min(r.best_iteration for r in got) < its - 1
